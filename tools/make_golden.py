#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on CPU.

Run in the build container only (the GPU box has no /root/reference):

    python tools/make_golden.py

The reference modules are imported as they are; three `sys.modules` shims stand in for packages that
are missing / removed in this image and that the hot path never calls (SURVEY §8c):
`torchvision.models.utils` (backbone/origin/vgg.py:8), `openpyxl`, `thop` (utils/misc.py:11-12); and
`torch.utils.model_zoo.load_url` returns {} (no network: backbone/origin/resnet.py:208-215 then keeps
the seeded random init).

apex (DDP / SyncBN / amp) is not part of /root/reference, so the W=2 vectors are produced from the
reference's own model / loss / optimizer with apex's published semantics restated as the equivalent
single-process computation: SyncBN over W ranks == BatchNorm over the rank-concatenated batch, and
the DDP gradient mean == gradient of mean_r(loss_r).  (Parity unpinned for apex itself.)
"""
from __future__ import annotations

import hashlib
import os
import sys
import types

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from distributed_sod_project_b200.synthetic import synth_batch  # noqa: E402

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def install_reference():
    if not os.path.isdir(REF):
        raise SystemExit("reference not present; golden vectors can only be regenerated in the build container")
    sys.path.insert(0, REF)
    m = types.ModuleType("torchvision.models.utils")
    m.load_state_dict_from_url = lambda *a, **k: {}
    sys.modules["torchvision.models.utils"] = m
    for name in ("openpyxl", "thop"):
        mm = types.ModuleType(name)
        mm.load_workbook = mm.Workbook = mm.profile = None
        sys.modules[name] = mm
    import torch.utils.model_zoo as mz
    mz.load_url = lambda *a, **k: {}


def loss_kats():
    from loss.CEL import CEL
    cases = {}
    g = torch.Generator().manual_seed(7)
    specs = {
        "n1": (1,), "n7": (7,), "n1000": (1000,), "n4097": (4097,), "img": (2, 1, 24, 24),
    }
    for name, shape in specs.items():
        x = torch.randn(*shape, generator=g, dtype=torch.float64) * 3
        t = (torch.rand(*shape, generator=g, dtype=torch.float64) * 255).round() / 255
        cases[name] = (x, t)
    x = torch.randn(513, generator=g, dtype=torch.float64) * 2
    cases["mask_zero"] = (x, torch.zeros(513, dtype=torch.float64))
    cases["mask_one"] = (x.clone(), torch.ones(513, dtype=torch.float64))
    cases["binary"] = (x.clone(), (torch.rand(513, generator=g) > 0.5).double())
    big = torch.tensor([-88.0, -30.0, -10.0, 0.0, 10.0, 30.0, 88.0, 5.0, -5.0] * 3, dtype=torch.float64)
    cases["extreme"] = (big, (torch.rand(27, generator=g) > 0.5).double())
    out = {}
    for name, (x, t) in cases.items():
        for red in ("mean", "sum"):
            xr = x.clone().requires_grad_(True)
            bce = torch.nn.BCEWithLogitsLoss(reduction=red)(xr, t)
            celv = CEL()(xr, t)
            (bce + celv).backward()
            out[f"{name}/{red}/x"] = x.numpy(); out[f"{name}/{red}/t"] = t.numpy()
            out[f"{name}/{red}/bce"] = bce.item(); out[f"{name}/{red}/cel"] = celv.item()
            out[f"{name}/{red}/grad"] = xr.grad.numpy()
    # get_total_loss string contract (fp32, as the training loop sees it)
    from utils.pipeline_ops import get_total_loss
    x, t = cases["img"]
    tot, strs = get_total_loss(x.float(), t.float(), [torch.nn.BCEWithLogitsLoss(), CEL()])
    out["total_loss/value"] = tot.item(); out["total_loss/strings"] = np.array(strs)
    np.savez_compressed(os.path.join(OUT, "loss_kat.npz"), **out)
    print("loss_kat:", len(out), "arrays")


class _Tiny(torch.nn.Module):
    """names exercise the three f3_trick classes: div_2* (no group), div* (backbone), other (head)"""

    def __init__(self):
        super().__init__()
        self.div_2 = torch.nn.Linear(5, 7)
        self.div_4 = torch.nn.Linear(7, 6)
        self.div_16 = torch.nn.Linear(6, 3, bias=False)
        self.head = torch.nn.Linear(3, 2)
        self.classifier = torch.nn.Linear(2, 1)


def sgd_kats():
    from utils.pipeline_ops import CustomScheduler, make_optimizer
    torch.manual_seed(3)
    out = {}
    for kind in ("f3_trick", "sgd_trick", "sgd_all"):
        torch.manual_seed(3)
        net = _Tiny()
        opt = make_optimizer(net, kind, dict(lr=0.05, momentum=0.9, weight_decay=5e-4, nesterov=False))
        names = [n for n, _ in net.named_parameters()]
        out[f"{kind}/names"] = np.array(names)
        out[f"{kind}/group_of"] = np.array([next((gi for gi, g in enumerate(opt.param_groups)
                                                   if any(p is q for q in g["params"])), -1)
                                            for _, p in net.named_parameters()])
        out[f"{kind}/group_lr"] = np.array([g["lr"] for g in opt.param_groups])
        out[f"{kind}/group_wd"] = np.array([g["weight_decay"] for g in opt.param_groups])
        out[f"{kind}/p0"] = np.concatenate([p.detach().numpy().ravel() for p in net.parameters()])
        sched = CustomScheduler(opt, total_num=4, scheduler_type="poly", scheduler_info=dict(lr_decay=0.9, warmup_epoch=1))
        g = torch.Generator().manual_seed(11)
        for it in range(4):
            sched.step(opt, curr_epoch=it)
            out[f"{kind}/lr{it}"] = np.array([gr["lr"] for gr in opt.param_groups])
            grads = []
            for p in net.parameters():
                p.grad = torch.randn(p.shape, generator=g)
                grads.append(p.grad.numpy().ravel().copy())
            out[f"{kind}/g{it}"] = np.concatenate(grads)
            opt.step()
            out[f"{kind}/p{it + 1}"] = np.concatenate([p.detach().numpy().ravel() for p in net.parameters()])
    # scheduler table
    for kind in ("poly", "poly_warmup", "cosine_warmup", "f3_sche"):
        net = _Tiny()
        opt = make_optimizer(net, "f3_trick", dict(lr=0.05, momentum=0.9, weight_decay=5e-4, nesterov=False))
        sched = CustomScheduler(opt, total_num=30, scheduler_type=kind, scheduler_info=dict(lr_decay=0.9, warmup_epoch=3))
        rows = []
        for e in range(30):
            try:
                sched.step(opt, curr_epoch=e)
            except ZeroDivisionError:
                # the warmup branches shrink self.total_num on EVERY call (utils/pipeline_ops.py:206,217),
                # so the reference itself divides by zero late in the schedule; record up to there
                break
            rows.append([float(np.real(g["lr"])) if not isinstance(g["lr"], complex) else np.nan
                         for g in opt.param_groups])
        out[f"sched/{kind}"] = np.array(rows)
    np.savez_compressed(os.path.join(OUT, "sgd_kat.npz"), **out)
    print("sgd_kat:", len(out), "arrays")


def _probe_params(model):
    """small fixed probes of the post-step parameters (full state is 100 MB)"""
    sd = dict(model.named_parameters())
    keys = ["div_2.0.weight", "div_4.1.0.conv1.weight", "div_32.2.bn3.weight", "div_32.2.conv3.weight",
            "trans32.weight", "sim2.bnh_2.bias", "upconv1.basicconv.0.weight", "classifier.weight", "classifier.bias"]
    return {k: sd[k].detach().reshape(-1)[:64].numpy().copy() for k in keys}


def step_vectors(model_name: str, world: int, bs: int, size: int, iters: int, tag: str, keep_logits=(0,), logits_stride: int = 1):
    """reference model + reference loss/optimizer, apex semantics restated (see module docstring)."""
    import network
    from loss.CEL import CEL
    from utils.misc import init_seed
    from utils.pipeline_ops import get_total_loss, make_optimizer
    init_seed(0)
    model = getattr(network, model_name)()
    opt = make_optimizer(model, "f3_trick", dict(lr=0.05, momentum=0.9, weight_decay=5e-4, nesterov=False))
    loss_funcs = [torch.nn.BCEWithLogitsLoss(reduction="mean"), CEL()]
    model.train()
    out = {"meta": np.array([world, bs, size, iters]), "logits_stride": np.array(logits_stride)}
    for it in range(iters):
        batches = [synth_batch(1234 + r + 1000 * it, bs, size) for r in range(world)]
        x = torch.cat([b[0] for b in batches]); m = torch.cat([b[1] for b in batches])
        preds = model(x)                                   # BN over the concatenated batch == SyncBN
        per_rank, strs = [], []
        for r in range(world):
            l, s = get_total_loss(preds[r * bs:(r + 1) * bs], m[r * bs:(r + 1) * bs], loss_funcs)
            per_rank.append(l); strs.append(s)
        loss = sum(per_rank) / world                       # grad == DDP mean of per-rank grads
        opt.zero_grad()
        loss.backward()
        opt.step()
        out[f"loss{it}"] = np.array([l.item() for l in per_rank])
        out[f"items{it}"] = np.array(strs)
        if it in keep_logits:
            # per-pixel logits, spatially subsampled for the large configurations (file size); the test compares the
            # same pixels of the GPU result
            out[f"logits{it}"] = preds.detach().numpy()[:, :, ::logits_stride, ::logits_stride].copy()
        for k, v in _probe_params(model).items():
            out[f"param{it}/{k}"] = v
        print(tag, it, [round(l.item(), 5) for l in per_rank], flush=True)
    np.savez_compressed(os.path.join(OUT, f"step_{tag}.npz"), **out)


def tensor_digest(t: torch.Tensor) -> str:
    """sha256 over dtype, shape and the raw bytes of a tensor: equal digests == bit-identical tensors"""
    t = t.detach().contiguous()
    return hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode() + t.numpy().tobytes()).hexdigest()


def model_vectors():
    """the reference res50 right after `init_seed(0)`: a digest of every state_dict entry (the full state is 100 MB) and
    its output on one seeded input, in eval mode and then in train mode"""
    import network
    from utils.misc import init_seed
    init_seed(0)
    model = network.res50()
    sd = model.state_dict()
    names, digests = list(sd), [tensor_digest(v) for v in sd.values()]      # before a train-mode forward moves the BN buffers
    x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        out_eval = model.eval()(x)
        out_train = model.train()(x)
    np.savez_compressed(os.path.join(OUT, "model_res50_init.npz"), names=np.array(names), digests=np.array(digests),
                        x=x.numpy(), out_eval=out_eval.numpy(), out_train=out_train.numpy())
    print("model_res50_init:", len(names), "state_dict entries")


def main():
    os.makedirs(OUT, exist_ok=True)
    install_reference()
    torch.set_num_threads(8)
    if "--only-320" in sys.argv:      # round 2: the benched configuration pinned with logits (bs 4 and bs 16 at 320x320)
        step_vectors("res50", 1, 4, 320, 3, "res50_w1_s320", keep_logits=(0, 1), logits_stride=2)
        step_vectors("res50", 1, 16, 320, 2, "res50_w1_s320_bs16", keep_logits=(0, 1), logits_stride=4)
        return
    if "--only-model" in sys.argv:
        model_vectors()
        return
    model_vectors()
    loss_kats()
    sgd_kats()
    # 64x64 / bs 2 leaves 8 samples under the deepest BN: a deliberately ill-conditioned edge case (kept for the
    # first-iteration checks); 128x128 / bs 4 is the well-conditioned small configuration
    step_vectors("res50", 1, 2, 64, 6, "res50_w1_s64", keep_logits=(0, 5))
    step_vectors("cp_res50", 1, 2, 64, 3, "cp_res50_w1_s64", keep_logits=(0,))
    step_vectors("res50", 2, 2, 64, 4, "res50_w2_s64", keep_logits=(0, 3))
    step_vectors("res50", 1, 4, 128, 4, "res50_w1_s128", keep_logits=(0,))
    step_vectors("res50", 2, 4, 128, 4, "res50_w2_s128", keep_logits=(0,))
    step_vectors("res50", 1, 4, 320, 3, "res50_w1_s320", keep_logits=(0, 1), logits_stride=2)   # BASELINE config 1 shape
    step_vectors("res50", 1, 16, 320, 2, "res50_w1_s320_bs16", keep_logits=(0, 1), logits_stride=4)   # the benched batch size


if __name__ == "__main__":
    main()
