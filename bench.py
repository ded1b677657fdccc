#!/usr/bin/env python
"""bench.py — images/sec of one training iteration of TestModel (ResNet-50 encoder, 320×320, bs 16/GPU, bf16)
through the B200 hot path, with the CPU reference timed beside it.

    python bench.py [--gpus N --steps K --warmup W]                      # this repo's arm
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference [--steps K --warmup W]              # the reference's algorithm on host cores
    python bench.py --sweep                                              # BASELINE config 5 (needs ≥2 ranks)
    python bench.py --dump-outputs DIR ...                               # also save the last timed step's outputs

One JSON line on stdout (rank 0).  `value` = whole-job images/s with the batch already resident in HBM;
`e2e` = the same through `Trainer.step_from_host` (pinned host batch → H2D → iteration → loss D2H);
`roofline` = the dominant hand-written kernel (SyncBN backward) replayed on the model's 84 layer shapes and
timed with CUDA events on the launching stream; `cpu_baseline` = the oracle restatement of the reference loop
on the host cores (bounded sample).  Nothing here reads the reference project.

`--dump-outputs DIR` writes what the last of the `--steps` timed iterations returned to rank 0 as float32 arrays:
DIR/loss.npy (the rank-mean loss), DIR/loss_items.npy (the fused loss kernel's 8 report scalars: bce, cel, total,
Σp, Σt, Σp·t, unreduced bce sum, n; absent for `--impl torch`) and DIR/logits.npy (N×1×H×W, at most 16×1×384×384 =
9.4 MB).  The inputs and the initial weights are seeded, so two builds run with the same arguments can be compared
output for output.  Two runs of one build with the same arguments compute the same arrays: cuDNN picks its algorithms
by heuristics here rather than by timing them, since algorithms that round differently make two runs of the training
loop drift apart step by step.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

SIZE, BS = 320, 16
METRIC, UNIT = "images_per_sec", "img/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch"])
    ap.add_argument("--model", default="res50", choices=["res50", "cp_res50"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-batch", type=int, default=4)
    ap.add_argument("--sweep", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay of the iteration")
    ap.add_argument("--multiscale", action="store_true",
                    help="BASELINE config 4: one size of {256,320,384} per batch (rank-shared RNG), as the reference's multi-scale collate")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the untimed world>1 parity leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the ride-along measurements (multi-scale, sweep, stock-torch arm)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (float32)")
    return ap.parse_args()


def dump_outputs(out_dir: str, outputs) -> None:
    """`--dump-outputs`: the (loss, loss items, logits) that `forward_backward_update` returned, as float32 .npy files"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in zip(("loss", "loss_items", "logits"), outputs):
        if isinstance(t, torch.Tensor):
            np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms; started before warm-up so that it is already
    streaming when the (possibly sub-second) timed region runs; `mark()` brackets the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index, self.t0, self.t1 = [], None, index, None, None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark(self):
        if self.t0 is None:
            self.t0 = time.time()
        else:
            self.t1 = time.time()

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)            # let the last in-window sample arrive
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        t0, t1 = self.t0 or 0.0, self.t1 or float("inf")
        inside = [r for t, r in self.rows if t0 <= t <= t1 + 0.15]
        if not inside and self.rows:     # region shorter than the sampling period: the samples that bracket it
            inside = [r for t, r in self.rows if t0 - 0.3 <= t <= t1 + 0.3] or [self.rows[-1][1]]
        sm, mx, reasons = [], [], set()
        for r in inside:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port of the reference loop; test infrastructure used as the reported baseline)
# ----------------------------------------------------------------------------------------------------
def cpu_reference(model_name: str, batch: int, steps: int, warmup: int):
    from oracle.step import OracleTrainer
    from distributed_sod_project_b200 import network
    from distributed_sod_project_b200.synthetic import synth_batch
    cores = pick_threads(getattr(network, model_name))
    torch.set_num_threads(cores)
    tr = OracleTrainer(getattr(network, model_name), world_size=1, seed=0)
    batches = [synth_batch(1234 + i, batch, SIZE) for i in range(2)]
    for i in range(warmup):
        tr.step(*batches[i % 2])
    t0 = time.perf_counter()
    for i in range(steps):
        tr.step(*batches[i % 2])
    dt = (time.perf_counter() - t0) / steps
    return {"value": batch / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} steps of bs={batch} at {SIZE}x{SIZE} fp32 ({model_name}, oracle/step.py restatement of "
                      f"reference train.py:284-310 on my network plugin, {cores} torch threads, world 1)",
            "ms_per_step": dt * 1e3}


def pick_threads(factory) -> int:
    """torch intra-op thread count that is actually fastest on this host: the box may expose far more logical CPUs
    than the container is allowed to use (128 visible on the GPU pool; over-subscription made a step >100 s)."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    try:   # cgroup v2 quota
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            avail = max(1, min(avail, int(int(q) / int(per) + 0.5)))
    except (OSError, ValueError):
        pass
    cands = sorted({c for c in (4, 8, 16, 32, 64) if c <= avail} | {min(avail, 64)})
    model = factory().train()
    x = torch.randn(2, 3, 160, 160)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        model(x).sum().backward()
        t0 = time.perf_counter()
        model(x).sum().backward()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        if dt > 4 * best_t:
            break
    return best


def _cpu_world_worker(rank, world, port, model_name, batch, steps, warmup, threads, out_path):
    """one CPU rank of the reference's DDP + SyncBN loop over gloo (oracle/step.py restatement)"""
    # under torchrun the parent's environment says "use the elastic agent's store" (TORCHELASTIC_USE_AGENT_STORE) and carries
    # the NCCL job's rank variables: this CPU job is a separate group with a TCP store of its own
    for k in [k for k in os.environ if k.startswith(("TORCHELASTIC_", "GROUP_", "ROLE_", "LOCAL_WORLD", "TORCH_NCCL"))]:
        os.environ.pop(k, None)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.set_num_threads(threads)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    from oracle.step import OracleTrainer
    from distributed_sod_project_b200 import network
    from distributed_sod_project_b200.synthetic import synth_batch
    tr = OracleTrainer(getattr(network, model_name), world_size=world, seed=0)
    batches = [synth_batch(1234 + rank + 100 * i, batch, SIZE) for i in range(2)]
    for i in range(warmup):
        tr.step(*batches[i % 2])
    dist.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        tr.step(*batches[i % 2])
    dist.barrier()
    dt = (time.perf_counter() - t0) / steps
    if rank == 0:
        json.dump({"dt": dt}, open(out_path, "w"))
    dist.destroy_process_group()


def cpu_reference_world(model_name: str, world: int, batch: int, steps: int, warmup: int):
    """BASELINE.md §3 rows 3-4: the reference's distributed loop (apex DDP + SyncBN semantics restated over gloo) with
    `world` CPU ranks on this host, the available cores split between them"""
    import socket
    import tempfile
    import torch.multiprocessing as mp
    from distributed_sod_project_b200 import network
    cores = pick_threads(getattr(network, model_name))
    threads = max(1, cores // world)
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = os.path.join(tempfile.mkdtemp(), "cpu_world.json")
    mp.spawn(_cpu_world_worker, args=(world, port, model_name, batch, steps, warmup, threads, out), nprocs=world, join=True)
    dt = json.load(open(out))["dt"]
    return {"value": world * batch / dt, "unit": UNIT, "cores": threads * world, "kind": "port",
            "sample": f"{steps} steps of bs={batch}/rank x {world} gloo ranks at {SIZE}x{SIZE} fp32 ({model_name}, oracle/step.py: "
                      f"reference train.py:284-310 with apex DDP + SyncBN semantics over gloo, {threads} torch threads per rank)",
            "ms_per_step": dt * 1e3}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, args.steps)
    warm = max(1, min(args.warmup, 3))
    world = max(1, args.gpus)
    if world > 1:
        # the reference's distributed configuration on the host CPU: one gloo rank per GPU of the arm it is compared with;
        # per-rank batch shrinks with the world so that a step stays a bounded sample (bs 4, 2, 1, 1 at 1, 2, 4, 8 ranks)
        batch = max(1, args.cpu_batch // world)
        steps = min(steps, 10)
        res = cpu_reference_world(args.model, world, batch, steps, min(warm, 2))
    else:
        batch = args.cpu_batch
        res = cpu_reference(args.model, batch, steps, warm)
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": f"TestModel {args.model} {SIZE}x{SIZE}, one training iteration (fwd+BCE/CEL+bwd+SGD"
                                   + (f", DDP + SyncBN over gloo, {world} CPU ranks" if world > 1 else "") + "), "
                                   f"CPU sample bs={batch}" + ("/rank" if world > 1 else "")},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# roofline of the dominant hand-written kernel
# ----------------------------------------------------------------------------------------------------
def bn_roofline(trace, dtype, iters=5):
    """replay every SyncBN backward launch of one iteration (same shapes, same fusion flags), each from a cold L2, timed
    with CUDA events on the launching stream (see `span` below)."""
    from distributed_sod_project_b200 import syncbn as _sbn
    from distributed_sod_project_b200.syncbn import raw_backward
    _sbn.FORCE_LOCAL = True
    esz = 2 if dtype != torch.float32 else 4
    layers = []
    for (n, c, h, w, has_pre, has_res, relu) in trace:
        mk = lambda: torch.randn((n, c, h, w), device="cuda", dtype=dtype).contiguous(memory_format=torch.channels_last)  # noqa: E731
        x, dy = mk(), mk()
        pre = mk() if has_pre else None
        y = mk() if relu else None
        weight = torch.ones(c, device="cuda")
        mean = torch.zeros(c, device="cuda"); invstd = torch.ones(c, device="cuda")
        elems = n * c * h * w
        # algorithmic bytes = compulsory traffic: every input operand read ONCE, every output written once
        # (SURVEY §8d's 10 B/elem assumed two passes over dy,x; the kernel keeps its strip in shared memory between
        # the reduction and the elementwise phase, so the honest denominator is the single-pass figure: 6 B/elem
        # for plain bf16 backward, +2 B/elem per fused operand)
        from_x = _sbn.MASK_FROM_X and relu and not has_res        # experimental variant: y is not read at all
        reads = 2 + (1 if has_pre else 0) + (1 if relu and not from_x else 0)
        byts = (reads + 1 + (1 if has_res else 0)) * esz * elems
        layers.append(((dy, x, pre, y, weight, mean, invstd, relu, has_res), dict(bias=torch.zeros(c, device="cuda")), byts))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    reps = 4

    def span(fn):
        """milliseconds (CUDA events on the launching stream) of `reps` x [flush L2, fn]"""
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            flush.zero_()
            fn()
        e.record()
        e.synchronize()
        return s.elapsed_time(e)

    # Every launch starts cold: a 256 MB write flushes the 126 MB L2 before it, INSIDE the event pair, and the flush's own
    # time (measured the same way, median) is subtracted.  A pair of events around one 15 µs kernel would mostly measure the
    # events themselves (≈4 µs); here the kernel's launch overlaps the preceding flush, as it overlaps the preceding
    # convolution in the real iteration.
    for _ in range(3):
        span(lambda: None)
    flush_ms = sorted(span(lambda: None) for _ in range(9))[4]
    total_ms, total_bytes = 0.0, 0
    for (a, kw, byts) in layers:
        raw_backward(*a, **kw)                     # warm-up (kernel attributes, allocator)
        ms = sorted(span(lambda: raw_backward(*a, **kw)) for _ in range(iters))[iters // 2]      # exactly reps launches per span
        total_ms += max(ms - flush_ms, 0.0) / reps
        total_bytes += byts
    _sbn.FORCE_LOCAL = False
    n = len(layers)
    return total_bytes / (total_ms * 1e-3) / 1e9, total_ms / n, total_bytes / n


class TorchEagerTrainer:
    """Same iteration with stock PyTorch on the GPU (nn.BatchNorm2d, torch losses, torch.optim.SGD(fused=True),
    bf16 autocast, channels-last): NOT the reference arm — the "what you get without this repo's kernels" line."""

    def __init__(self, model_name, dtype):
        from distributed_sod_project_b200 import network
        from distributed_sod_project_b200.utils import init_seed

        class StockCEL(torch.nn.Module):          # loss/CEL.py:15-20 in plain torch ops (this arm must not use oracle/)
            def forward(self, pred, target):
                p = pred.sigmoid()
                inter = p * target
                return ((p - inter).sum() + (target - inter).sum()) / (p.sum() + target.sum() + 1e-6)

        init_seed(0)
        self.model = getattr(network, model_name)().cuda().to(memory_format=torch.channels_last)
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        if self.world > 1:      # the stock multi-GPU recipe: nn.SyncBatchNorm + DistributedDataParallel over NCCL
            self.model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(self.model)
        named = list(self.model.named_parameters())
        groups = [{"params": [p for n, p in named if n.startswith("div") and not n.startswith("div_2")], "lr": 0.005},
                  {"params": [p for n, p in named if not n.startswith("div")], "lr": 0.05}]
        self.opt = torch.optim.SGD(groups, momentum=0.9, weight_decay=5e-4, fused=True)
        self.loss_funcs = [torch.nn.BCEWithLogitsLoss(), StockCEL()]
        self.dtype = dtype
        self.model.train()
        self.net = self.model
        if self.world > 1:
            self.net = torch.nn.parallel.DistributedDataParallel(self.model, device_ids=[torch.cuda.current_device()],
                                                                 gradient_as_bucket_view=True)
        self._pinned = torch.zeros(1).pin_memory()

    def forward_backward_update(self, x, m):
        x = x.contiguous(memory_format=torch.channels_last)
        with torch.autocast("cuda", dtype=self.dtype, enabled=self.dtype != torch.float32):
            preds = self.net(x)
        loss = sum(f(preds.float(), m) for f in self.loss_funcs)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self.opt.step()
        return loss.detach(), None, preds

    def step_from_host(self, xh, mh):
        loss, _, _ = self.forward_backward_update(xh.cuda(non_blocking=True), mh.cuda(non_blocking=True))
        self._pinned.copy_(loss.reshape(1), non_blocking=True)

    def last_loss(self):
        torch.cuda.synchronize()
        return float(self._pinned[0])

    @property
    def module(self):
        return self.model


# ----------------------------------------------------------------------------------------------------
# untimed parity leg for world > 1 (runs on the timed processes, after the timed region)
# ----------------------------------------------------------------------------------------------------
def parity_check(tr, rank: int, world: int) -> dict:
    """Cross-rank correctness of the kernels that only exist at world > 1, against torch's NCCL equivalents on the
    same inputs (reference semantics: apex DDP + SyncBN, train.py:180-185; apex is absent, torch's SyncBatchNorm /
    all_reduce / SGD are the in-image stand-ins SURVEY §8c names):
      1. parameters (and the bf16 shadow) bit-identical on all ranks after the timed steps;
      2. sod_syncbn_fwd/bwd on three layer shapes vs torch.nn.SyncBatchNorm;
      3. sod_allreduce_sgd on the real gradient bucket vs dist.all_reduce + the SGD-momentum formula;
      4. at world 2: the fp32 training trajectory vs the reference's golden vectors (tests/golden/step_res50_w2_s128.npz).
    Every verdict is all-reduced (MIN) so that all ranks agree; the caller exits non-zero on a mismatch."""
    import numpy as np
    from distributed_sod_project_b200 import comm
    from distributed_sod_project_b200.syncbn import SyncBatchNorm
    dev = torch.device("cuda", torch.cuda.current_device())
    out: dict = {}

    def agree(flag: bool) -> bool:
        t = torch.tensor([1 if flag else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(int(t.item()))

    def relerr(a, b) -> float:
        a, b = a.detach().double(), b.detach().double()
        return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))

    flat = tr.optimizer.flat
    # 1 ---------------------------------------------------------------------------------------------------------
    ref = flat.param.clone(); dist.broadcast(ref, 0)
    same = torch.equal(ref, flat.param)
    if flat.shadow16 is not None:
        ref16 = flat.shadow16.clone(); dist.broadcast(ref16, 0)
        same = same and torch.equal(ref16, flat.shadow16)
    out["params_identical"] = agree(same)
    # 2 ---------------------------------------------------------------------------------------------------------
    bn_rows = []
    ok_bn = True
    for (shape, dt, tol) in (((16, 64, 80, 80), torch.float32, 2e-4), ((16, 256, 20, 20), torch.float32, 2e-4),
                             ((16, 2048, 10, 10), torch.float32, 2e-4), ((16, 64, 80, 80), torch.bfloat16, 3e-2)):
        g = torch.Generator(device="cpu").manual_seed(4242 + rank)
        c = shape[1]
        x0 = (torch.randn(shape, generator=g) * (1.0 + 0.5 * rank) + 0.3 * rank).to(dt).to(dev).contiguous(memory_format=torch.channels_last)
        dy = torch.randn(shape, generator=g).to(dt).to(dev).contiguous(memory_format=torch.channels_last)
        mine, theirs = SyncBatchNorm(c).to(dev), torch.nn.SyncBatchNorm(c).to(dev)
        with torch.no_grad():
            for bn in (mine, theirs):
                bn.weight.copy_(torch.linspace(0.5, 1.5, c)); bn.bias.copy_(torch.linspace(-0.3, 0.3, c))
        res = []
        for bn in (mine, theirs):
            x = x0.clone().requires_grad_(True)
            y = bn(x) if bn is theirs else bn.fused_forward(x)
            y.backward(dy)
            res.append((y.detach(), x.grad, bn.weight.grad, bn.bias.grad, bn.running_mean.clone(), bn.running_var.clone()))
        errs = {k: relerr(a, b) for k, a, b in zip(("y", "dx", "dgamma", "dbeta", "running_mean", "running_var"), res[0], res[1])}
        good = all(v < tol for v in errs.values())
        ok_bn = ok_bn and good
        bn_rows.append({"shape": list(shape), "dtype": str(dt).replace("torch.", ""), "tol": tol, **{k: float(f"{v:.3g}") for k, v in errs.items()}})
    out["syncbn_vs_torch_nccl"] = {"ok": agree(ok_bn), "cases": bn_rows}
    # 3 ---------------------------------------------------------------------------------------------------------
    opt = tr.optimizer
    snap_p, snap_v = flat.param.clone(), flat.mom.clone()
    snap_s = flat.shadow16.clone() if flat.shadow16 is not None else None
    opt.gather_momentum()                                   # the reference SGD below needs the full momentum on every rank
    v_full = flat.mom.clone()

    def one_exchange(bf16_wire: bool):
        """random per-rank gradients → fused kernel vs dist.all_reduce + the SGD formula.  bf16_wire: the convolution
        parameters' gradients are placed in the bf16 buffer (as backward leaves them) and cross NVLink in bf16."""
        with torch.no_grad():
            flat.param.copy_(snap_p); flat.mom.copy_(v_full)
        opt.zero_grad()                                     # also drops the weight gradients autograd left from the last step
        g = torch.Generator(device="cpu").manual_seed(777 + rank + (1000 if bf16_wire else 0))
        grad = (torch.randn(flat.numel, generator=g) * 1e-2).to(dev)
        if bf16_wire:
            plan = opt._segment_plan()
            eff = torch.zeros_like(grad)
            for b, e, _, bf16_part in plan:
                if bf16_part:
                    flat.grad16[b:e].copy_(grad[b:e])                  # rounds to bf16
                    eff[b:e] = flat.grad16[b:e].float()
                else:
                    flat.grad.data[b:e].copy_(grad[b:e])               # behind autograd's back, like the SyncBN kernels do
                    eff[b:e] = grad[b:e]
            assert opt._bf16_exclusive()
        else:
            flat.grad.copy_(grad)                                      # fp32 everywhere ...
            flat.master_grads_seen = True                              # ... which is what a run outside autocast leaves: fp32 wire format
            if flat.grad16 is not None:
                flat.grad16.zero_()
            eff = grad
        parts = [torch.empty_like(eff) for _ in range(world)]
        dist.all_gather(parts, eff)
        gsum = parts[0].clone()
        for t in parts[1:]:
            gsum += t                                                  # rank order, fp32: what the peer-load path computes
        gavg = gsum / world
        exp_p, exp_v = snap_p.clone(), v_full.clone()
        for grp, (b, e) in zip(opt.param_groups, flat.ranges):
            if e > b:
                gg = gavg[b:e] + grp["weight_decay"] * exp_p[b:e]
                exp_v[b:e] = grp["momentum"] * exp_v[b:e] + gg
                exp_p[b:e] = exp_p[b:e] - grp["lr"] * exp_v[b:e]
        torch.cuda.synchronize(); dist.barrier()
        opt.step()
        torch.cuda.synchronize()
        lo, hi = opt.shard_bounds(rank, world)
        e_p = relerr(flat.param, exp_p)
        e_v = relerr(flat.mom[lo:hi], exp_v[lo:hi]) if hi > lo else 0.0
        cleared = float(flat.grad.abs().max()) == 0.0 and (flat.grad16 is None or float(flat.grad16.float().abs().max()) == 0.0)
        ref = flat.param.clone(); dist.broadcast(ref, 0)
        good = e_p < 1e-5 and e_v < 1e-5 and cleared and torch.equal(ref, flat.param)
        return {"ok": agree(good), "elems": flat.numel, "param_relerr": float(f"{e_p:.3g}"),
                "momentum_shard_relerr": float(f"{e_v:.3g}"), "grads_cleared": cleared}

    out["allreduce_sgd_vs_nccl_plus_sgd"] = one_exchange(bf16_wire=False)
    if flat.grad16 is not None and flat.grad16_off:
        out["allreduce_sgd_bf16_wire_vs_nccl_plus_sgd"] = one_exchange(bf16_wire=True)
    with torch.no_grad():                                    # put the training state back
        flat.param.copy_(snap_p); flat.mom.copy_(snap_v)
        if snap_s is not None:
            flat.shadow16.copy_(snap_s)
    torch.cuda.synchronize(); dist.barrier()
    # 4 ---------------------------------------------------------------------------------------------------------
    gpath = os.path.join(ROOT, "tests", "golden", "step_res50_w2_s128.npz")
    if world == 2 and os.path.exists(gpath):
        from distributed_sod_project_b200.engine import Trainer
        from distributed_sod_project_b200.synthetic import synth_batch
        gold = np.load(gpath)
        _, bs, size, _ = (int(v) for v in gold["meta"])
        tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
        torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.benchmark = False
        try:
            t2 = Trainer(model_name="res50", dtype=torch.float32, channels_last=True)
            errs, ok_g = [], True
            for it in range(2):
                xb, mb = synth_batch(1234 + rank + 1000 * it, bs, size)
                o = t2.step(xb.cuda(), mb.cuda())
                # the reference value is this rank's LOCAL loss; step() returns the rank mean (train.py:306)
                want = float(np.mean(gold[f"loss{it}"]))
                e = abs(o["loss"] - want) / abs(want)
                errs.append(float(f"{e:.3g}"))
                ok_g = ok_g and e < 1e-3
                if it == 0:
                    ref_l = gold["logits0"][rank * bs:(rank + 1) * bs]
                    le = float(np.abs(o["preds"].float().cpu().numpy() - ref_l).max() / np.abs(ref_l).max())
                    errs.append(float(f"{le:.3g}"))
                    ok_g = ok_g and le < 1e-3
            t2.check_errors()
        finally:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = tf32
        out["golden_w2_fp32"] = {"ok": agree(ok_g), "loss0_logits0_loss1_relerr": errs, "tol": 1e-3}
    for a in (getattr(tr.model, "arena", None), comm.small_arena()):
        if a is not None:
            a.check_error()
    out["ok"] = all(v.get("ok", True) if isinstance(v, dict) else bool(v) for v in out.values())
    return out


# ----------------------------------------------------------------------------------------------------
# ride-along measurements (BASELINE configs 4 and 5, SyncBN exchange cost, same-box stock-torch comparator)
# ----------------------------------------------------------------------------------------------------
def extra_pipeline(tr, rank, world, timed, steps=12):
    """SURVEY §8f.2 measured: the batch leaves the host as uint8 (what the loader's workers produce before ToTensor), is
    uploaded and pre-processed by `sod_preprocess_batch` one batch ahead on a side stream (`DevicePrefetcher`), and the
    iteration consumes it — end to end per step: pinned uint8 H2D + pre-processing kernel + iteration + loss D2H."""
    from distributed_sod_project_b200.pipeline import DevicePrefetcher, preprocess_batch
    g = torch.Generator().manual_seed(99 + rank)
    host = [(torch.randint(0, 256, (BS, SIZE, SIZE, 3), generator=g, dtype=torch.uint8).pin_memory(),
             torch.randint(0, 256, (BS, SIZE, SIZE), generator=g, dtype=torch.uint8).pin_memory(), None) for _ in range(4)]
    pinned = torch.zeros(1).pin_memory()

    def epoch(n):
        pre = DevicePrefetcher([host[i % 4] for i in range(n)], size_list=None)
        for x, m, _ in pre:
            red, _, _ = tr.forward_backward_update(x, m, report=False)
            pinned.copy_(red.reshape(1), non_blocking=True)

    epoch(3)
    ms = timed(lambda i: epoch(steps) if i == 0 else None, 1)
    img_d, msk_d = host[0][0].cuda(), host[0][1].cuda()
    for _ in range(3):
        preprocess_batch(img_d, msk_d)
    us = timed(lambda i: preprocess_batch(img_d, msk_d), 20) / 20 * 1e3
    px = BS * SIZE * SIZE
    return {"value": world * BS * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
            "h2d_bytes_per_step": 4 * px, "h2d_bytes_per_step_fp32_loader": 16 * px,
            "preprocess_kernel_us": us, "preprocess_kernel_gbs": 20 * px / (us * 1e-6) / 1e9,
            "note": "uint8 HWC image + uint8 mask in, normalised channels-last fp32 image + fp32 mask out (20 B/pixel of traffic)"}


def extra_multiscale(tr, rank, world, timed, steps=12):
    """BASELINE config 4: multi-scale {256,320,384}, one size per batch (rank-shared RNG), on the trainer that was just
    timed — two more graphs are captured (the 320 one exists), then `steps` iterations are timed like the headline."""
    import random as _random
    from distributed_sod_project_b200.synthetic import synth_batch
    sizes = (256, 320, 384)
    dev = {}
    for k, sz in enumerate(sizes):
        dev[sz] = [tuple(t.cuda() for t in synth_batch(4321 + rank + 100 * i + k, BS, sz)) for i in range(2)]
    for sz in sizes:                                    # warm-up: capture the missing graphs, run each size twice
        for i in range(2):
            tr.forward_backward_update(*dev[sz][i])
    rng = _random.Random(7)
    order = [sizes[rng.randrange(3)] for _ in range(steps)]
    ms = timed(lambda i: tr.forward_backward_update(*dev[order[i]][i % 2]), steps)
    tr.check_errors()
    return {"value": world * BS * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "sizes": list(sizes),
            "order": order, "graphs": len(getattr(tr, "_graphs", {})),
            "note": "one captured graph per size, learning rates from the device table; same timing discipline as the headline"}


def extra_sweep(world, timed):
    """BASELINE config 5 (short form; `--sweep` is the long one): peer-memory all-reduce vs torch NCCL, fp32, in place"""
    if world < 2:
        return None
    from distributed_sod_project_b200 import comm
    sizes = [64 << 10, 1 << 20, 16 << 20, 99_625_220 // 16 * 16]
    arena = comm.Arena(payload_bytes=sizes[-1] + 4096)
    off = arena.alloc(sizes[-1])
    rows = []
    for nbytes in sizes:
        n = nbytes // 4
        ref = torch.zeros(n, device="cuda")
        arena.view(off, n, torch.float32).zero_()
        row = {"bytes": nbytes}
        for name, fn in (("nccl", lambda: dist.all_reduce(ref)), ("sod", lambda: arena.allreduce_(off, n, algo=0))):
            for _ in range(3):
                fn()
            iters = 20 if nbytes <= (16 << 20) else 8
            us = timed(lambda i: fn(), iters) / iters * 1e3
            row[name] = {"us": us, "bus_gbs": 2 * (world - 1) / world * nbytes / (us * 1e-6) / 1e9}
        row["frac_of_nvlink_900"] = row["sod"]["bus_gbs"] / 900.0
        rows.append(row)
    arena.check_error()
    return {"world": world, "multicast": arena.has_multicast, "rows": rows}


def extra_syncbn_exchange(world, timed, dtype):
    """what one SyncBN statistics exchange costs across ranks: the same layer through the same kernel with and without
    the cross-rank hop (FORCE_LOCAL), next to an NCCL all-reduce of the 2C-float payload the reference's SyncBN sends"""
    if world < 2:
        return None
    from distributed_sod_project_b200 import syncbn as _sbn
    from distributed_sod_project_b200.syncbn import SyncBatchNorm
    out = {}
    for (n, c, h, w) in ((16, 256, 20, 20), (16, 64, 80, 80)):
        x = torch.randn((n, c, h, w), device="cuda", dtype=dtype).contiguous(memory_format=torch.channels_last)
        bn = SyncBatchNorm(c).cuda()
        res = {}
        with torch.no_grad():
            for tag, local_only in (("world", False), ("local", True)):
                _sbn.FORCE_LOCAL = local_only
                try:
                    for _ in range(5):
                        bn.fused_forward(x, relu=True)
                    res[tag] = timed(lambda i: bn.fused_forward(x, relu=True), 50) / 50 * 1e3
                finally:
                    _sbn.FORCE_LOCAL = False
        payload = torch.zeros(2 * c, device="cuda")
        for _ in range(5):
            dist.all_reduce(payload)
        nccl = timed(lambda i: dist.all_reduce(payload), 50) / 50 * 1e3
        extra_us = max(res["world"] - res["local"], 1e-3)
        out[f"{n}x{c}x{h}x{w}"] = {"fwd_us_world": res["world"], "fwd_us_local": res["local"], "exchange_us": extra_us,
                                   "nccl_allreduce_2C_us": nccl, "payload_bytes": 8 * c,
                                   "bus_gbs": 2 * (world - 1) / world * 8 * c / (extra_us * 1e-6) / 1e9}
    return out


def extra_torch_arm(args, dtype, rank, world, timed, steps=8):
    """the same iteration with stock PyTorch on the same GPUs (world > 1: nn.SyncBatchNorm + DistributedDataParallel over
    NCCL) — the comparator SURVEY §2 names, measured in the same process right after the headline"""
    from distributed_sod_project_b200.synthetic import synth_batch
    tt = TorchEagerTrainer(args.model, dtype)
    batches = [tuple(t.cuda() for t in synth_batch(1234 + rank + 100 * i, BS, SIZE)) for i in range(2)]
    for i in range(3):
        tt.forward_backward_update(*batches[i % 2])
    ms = timed(lambda i: tt.forward_backward_update(*batches[i % 2]), steps)
    del tt
    torch.cuda.empty_cache()
    return {"value": world * BS * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
            "what": "nn.BatchNorm2d" if world == 1 else "nn.SyncBatchNorm + DistributedDataParallel (NCCL)"}


def run_b200_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from distributed_sod_project_b200 import _lib, syncbn
    from distributed_sod_project_b200.engine import Trainer
    from distributed_sod_project_b200.synthetic import synth_batch

    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    args.warmup = max(3, args.warmup)          # timing rule: at least 3 warm-up iterations
    # cuDNN's heuristics, not its autotuner: the autotuner times candidate algorithms afresh in every process and may
    # pick different ones, so two runs on the same inputs would round differently and drift apart as training proceeds
    torch.backends.cudnn.benchmark = False
    log('building trainer')
    if args.impl == "torch":
        tr = TorchEagerTrainer(args.model, dtype)
    else:
        tr = Trainer(model_name=args.model, dtype=dtype, channels_last=True, report_items=False, use_graph=not args.no_graph)
    log('trainer built')
    nb = 4
    if args.multiscale:
        # BASELINE config 4: the reference's multi-scale collate draws ONE size per batch (utils/dataset.py:125-132,
        # config.py:58-60 size_list); all ranks draw the same one (shared RNG).  12 resident batches, 4 per size; the
        # first three steps visit each size once so that the warm-up captures all three graphs.
        import random as _random
        sizes = (256, 320, 384)
        rng = _random.Random(0)
        order = [0, 1, 2] + [rng.randrange(3) for _ in range(args.warmup + args.steps)]
        host = [synth_batch(1234 + rank + 100 * i, BS, sizes[k]) for k in range(3) for i in range(nb)]
        seen = [0, 0, 0]
        pick = []
        for k in order:                       # batch index of step i: next unused batch of the drawn size
            pick.append(k * nb + seen[k] % nb)
            seen[k] += 1
        mean_pixels = sum(sizes[k] ** 2 for k in order[:args.warmup + args.steps][args.warmup:]) / max(args.steps, 1)
    else:
        host = [synth_batch(1234 + rank + 100 * i, BS, SIZE) for i in range(nb)]
        pick = [i % nb for i in range(args.warmup + args.steps)]
        mean_pixels = SIZE * SIZE
    host = [(x.pin_memory(), m.pin_memory()) for x, m in host]
    dev = [(x.cuda(non_blocking=True), m.cuda(non_blocking=True)) for x, m in host]
    h2d = int(BS * mean_pixels * 16)          # 3 image planes + 1 mask plane, fp32

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync_all()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        sync_all()
        ms = torch.tensor([s.elapsed_time(e)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # -- device-resident arm ---------------------------------------------------------------------------
    clk = ClockSampler(local).__enter__()
    trace_at = 1 if args.multiscale else 0          # the 320x320 iteration (multi-scale warm-up visits 256, 320, 384)
    for i in range(args.warmup):
        if i == trace_at:
            syncbn.TRACE = []
        tr.forward_backward_update(*dev[pick[i]])
        torch.cuda.synchronize(); log(f'warmup {i} done')
        if i == trace_at:
            trace, syncbn.TRACE = syncbn.TRACE, None
    l0 = _lib.launches
    if os.environ.get("SOD_BENCH_PROFILE"):
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for i in range(2):
                tr.forward_backward_update(*dev[pick[i]])
            torch.cuda.synchronize()
        with open(os.environ["SOD_BENCH_PROFILE"], "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=90))
    rid = torch.cuda.nvtx.range_start("timed")      # start/end range: process-wide (backward runs on autograd's thread)
    clk.mark()
    w0 = args.warmup
    last = {}

    def timed_step(i):
        last["out"] = tr.forward_backward_update(*dev[pick[w0 + i]])
    ms = timed(timed_step, args.steps)
    clk.mark()
    torch.cuda.nvtx.range_end(rid)
    clk.__exit__()
    launches = _lib.launches - l0
    log(f'timed region done: {ms / args.steps:.2f} ms/step')
    if args.dump_outputs:           # before the end-to-end arm replays the graph and overwrites its output buffers
        if rank == 0:
            dump_outputs(args.dump_outputs, last["out"])
        sync_all()
    value = world * BS * args.steps / (ms * 1e-3)

    # -- end-to-end arm: pinned host batch in, loss out, every step ------------------------------------
    for i in range(min(args.warmup, 3)):
        tr.step_from_host(*host[pick[i]])
    tr.last_loss()
    ms_e2e = timed(lambda i: (tr.step_from_host(*host[pick[w0 + i]]), tr.last_loss() if i == args.steps - 1 else None), args.steps)
    e2e = world * BS * args.steps / (ms_e2e * 1e-3)
    log(f'e2e done: {ms_e2e / args.steps:.2f} ms/step')
    if args.impl == "torch":
        if rank == 0:
            print(json.dumps({"impl": "torch-eager", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
                              "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "dtype": args.dtype,
                              "config": {"workload": "stock PyTorch on the same GPUs: nn.BatchNorm2d / nn.SyncBatchNorm + "
                                                     "DistributedDataParallel over NCCL, torch losses, SGD(fused=True), bf16 autocast, "
                                                     "channels-last" + (", multi-scale {256,320,384}" if args.multiscale else "")},
                              "e2e": {"value": e2e, "unit": UNIT}, "clocks": clk.summary()}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    tr.check_errors()            # device-side barrier / packet time-outs of BOTH arenas (gradient bucket and SyncBN slots)

    # -- untimed parity leg (world > 1): the driver's GPU test box has one GPU, so the cross-rank kernels are checked here,
    #    on the very processes and parameters that were just timed; a mismatch fails the run (exit code 1) ---------------
    parity = None
    if world > 1 and not args.no_parity_check:
        try:
            parity = parity_check(tr, rank, world)
        except Exception as ex:                          # noqa: BLE001
            parity = {"ok": False, "error": repr(ex)}

    # -- measurements that ride along (BASELINE metric also names the all-reduce bus bandwidth); every rank takes part,
    #    nothing in here may prevent the line from being printed -----------------------------------------------------
    extras = {}
    try:
        opt, flat = tr.optimizer, tr.optimizer.flat
        for _ in range(3):
            opt.step()                                   # the gather + fused (all-reduce +) SGD kernels alone
        step_graph = torch.cuda.CUDAGraph()              # replayed from a graph: the host side of an eager step() costs more than the kernels
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(step_graph, stream=side):
                opt.step()
        torch.cuda.current_stream().wait_stream(side)
        us_step = timed(lambda i: step_graph.replay(), 10) / 10 * 1e3
        n_real = sum(p.numel() for p, _ in flat.slots)
        if world > 1:
            bus = 2.0 * (world - 1) / world * 4.0 * flat.numel / (us_step * 1e-6) / 1e9
            extras["fused_allreduce_sgd"] = {"us": us_step, "flat_elems": flat.numel, "params": n_real, "bus_gbs": bus,
                                             "frac_of_nvlink_900": bus / 900.0,
                                             "note": "multi-tensor gather + [reduce-scatter(grad, bf16 on the wire) + SGD + all-gather(param)] in one kernel"}
        else:
            per = 22 if flat.grad16 is not None else 24   # bf16 gradient in (2) + p, v in/out (16) + bf16 shadow out (2) + clear (2) | g, p, v + clear
            gbs = per * flat.numel / (us_step * 1e-6) / 1e9
            extras["fused_sgd"] = {"us": us_step, "flat_elems": flat.numel, "bytes_per_elem": per, "gbs": gbs,
                                   "frac_of_hbm": gbs / peaks()[0]["hbm_gbs"]}
    except Exception as ex:                              # noqa: BLE001
        extras["step_error"] = repr(ex)
    if not args.multiscale and not args.no_extras:
        # BASELINE configs 4 and 5 and the same-box comparator ride along with every default run, so that the round-end
        # 1/2/4/8-GPU runs record them too (every rank takes part; a failure here never costs the headline line)
        for name, fn in (("input_pipeline", lambda: extra_pipeline(tr, rank, world, timed)),
                         ("multiscale", lambda: extra_multiscale(tr, rank, world, timed)),
                         ("allreduce_sweep", lambda: extra_sweep(world, timed)),
                         ("syncbn_exchange", lambda: extra_syncbn_exchange(world, timed, dtype)),
                         ("torch_same_box", lambda: extra_torch_arm(args, dtype, rank, world, timed))):
            try:
                res = fn()
                if res is not None:
                    extras[name] = res
            except Exception as ex:                      # noqa: BLE001
                extras[name] = {"error": repr(ex)}
            log(f"extra {name} done")

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if parity is not None and not parity.get("ok", False):
            sys.exit(1)
        return
    pk, pk_kind = peaks()
    from distributed_sod_project_b200.syncbn import SyncBatchNorm
    n_bn = sum(isinstance(mod, SyncBatchNorm) for mod in tr.module.modules())
    bw, avg_ms, avg_bytes = bn_roofline(trace[:n_bn], dtype)   # cp_res50 traces its recompute forwards too
    log(f'roofline replay done: {bw:.0f} GB/s')
    roof = {"bound": "hbm", "kernel": "syncbn_bwd_kernel (84 launches/iteration, replayed alone on the model's layer shapes, "
                                      "L2 flushed between launches)",
            "achieved": bw, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": bw / pk["hbm_gbs"], "peak_kind": pk_kind,
            "how": "84 launches of one iteration replayed; per layer: CUDA events around 4 x [256 MB L2 flush + launch], flush time subtracted",
            "traffic": None, "avg_launch_ms": avg_ms, "algorithmic_bytes_per_launch": avg_bytes}
    try:        # dram__bytes_read + dram__bytes_write per launch, from the committed ncu pass over the same 84 launches (tools/bn_dram.py)
        dram = json.load(open(os.path.join(ROOT, "profiles", "r02_syncbn_bwd_dram.json")))
        roof["traffic"] = dram["avg_dram_bytes_per_launch"]
        roof["traffic_source"] = "profiles/r02_syncbn_bwd_dram.json (ncu dram__bytes_read.sum + dram__bytes_write.sum, each launch cold)"
    except (OSError, KeyError, ValueError):
        roof["traffic_source"] = "no committed ncu capture for this kernel revision"
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": f"TestModel {args.model} (ResNet-50 encoder) "
                                   + ("multi-scale {256,320,384} (one size per batch, rank-shared RNG; BASELINE config 4)"
                                      if args.multiscale else f"{SIZE}x{SIZE}")
                                   + f" bs={BS}/GPU, one training iteration: "
                                   "fwd (cuDNN convs NHWC + fused SyncBN kernels) + fused BCE/CEL fwd+bwd + bwd + "
                                   "fused (all-reduce+)SGD-momentum", "global_batch": BS * world,
                       "parallelism": f"dp{world}", "l2": "4 rotating input batches; per-iteration working set (>5 GB of "
                                                          "activations) far exceeds the 126 MB L2, no explicit flush"},
            "clocks": clk.summary(),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "roofline": roof}
    try:        # the loss kernel alone: at the workload shape (latency bound) and at SURVEY §8d's scaled shape
        from distributed_sod_project_b200.loss import bce_cel_fwd_bwd
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        for tag, shape in (("loss_workload", (BS, 1, SIZE, SIZE)), ("loss_scaled", (64, 1, 1024, 1024))):
            lx = torch.randn(shape, device="cuda").to(dtype)
            lt = (torch.rand(shape, device="cuda") > 0.8).float()
            ts = []
            for _ in range(7):
                flush.zero_()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                bce_cel_fwd_bwd(lx, lt)
                e.record()
                e.synchronize()
                ts.append(s.elapsed_time(e) * 1e3)
            us = sorted(ts)[len(ts) // 2]
            byts = lx.numel() * (2 * lx.element_size() + 4)      # logits in + grad out + fp32 mask in
            extras[tag] = {"shape": list(shape), "us": us, "algorithmic_bytes": byts, "gbs": byts / (us * 1e-6) / 1e9,
                           "frac_of_hbm": byts / (us * 1e-6) / 1e9 / pk["hbm_gbs"]}
            del lx, lt
    except Exception as ex:                              # noqa: BLE001
        extras["loss_error"] = repr(ex)
    line["extras"] = extras
    if parity is not None:
        line["parity_check"] = parity
    if not args.no_cpu_baseline:
        res = cpu_reference(args.model, args.cpu_batch, 6, 1)
        line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity is not None and not parity.get("ok", False):
        sys.exit(1)


def run_sweep(args):
    """BASELINE config 5: all-reduce bus bandwidth 64 KB–256 MB, peer-memory kernels vs torch NCCL, same box."""
    rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    if world < 2:
        print(json.dumps({"sweep": "needs world_size >= 2"}))
        return
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from distributed_sod_project_b200 import comm
    sizes = [64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20, 99_625_220 // 16 * 16, 256 << 20]
    arena = comm.Arena(payload_bytes=(256 << 20) + 4096)
    off = arena.alloc(256 << 20)
    rows = []
    for nbytes in sizes:
        n = nbytes // 4
        buf = arena.view(off, n, torch.float32)
        ref = torch.empty(n, device="cuda")
        res = {"bytes": nbytes}
        for name, fn in (("nccl", lambda: dist.all_reduce(ref)),
                         ("sod_multimem" if arena.has_multicast else "sod_p2p", lambda: arena.allreduce_(off, n, algo=2, force_multimem=True)),
                         ("sod_auto", lambda: arena.allreduce_(off, n, algo=0)),
                         ("sod_p2p_forced", lambda: arena.allreduce_(off, n, algo=2, no_multimem=True)),
                         ("sod_one_shot", (lambda: arena.allreduce_(off, n, algo=1)) if nbytes <= (1 << 20) else None)):
            if fn is None:
                continue
            buf.fill_(1.0); ref.fill_(1.0)
            iters = 20 if nbytes <= (16 << 20) else 8
            for _ in range(3):
                fn()
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(iters):
                fn()
            e.record(); torch.cuda.synchronize()
            t = torch.tensor([s.elapsed_time(e) / iters], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            us = float(t.item()) * 1e3
            res[name] = {"us": us, "bus_gbs": 2 * (world - 1) / world * nbytes / (us * 1e-6) / 1e9}
        rows.append(res)
    arena.check_error()
    if rank == 0:
        print(json.dumps({"sweep": "allreduce", "world": world, "multicast": arena.has_multicast, "nvlink_peak_gbs": 900,
                          "rows": rows}), flush=True)
    dist.barrier(); dist.destroy_process_group()


def log(msg):
    if os.environ.get("SOD_BENCH_VERBOSE"):
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def main():
    args = parse()
    if args.impl == "torch":
        return run_b200_arm(args)
    if os.environ.get("SOD_BENCH_VERBOSE"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ.get("SOD_BENCH_WATCHDOG", "120")), repeat=True, file=sys.stderr)
    if args.sweep:
        return run_sweep(args)
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    main()
