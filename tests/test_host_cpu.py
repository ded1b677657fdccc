"""CPU-only checks: the C-ABI library loads and exports every symbol of include/sod_b200.h, host-side layout
logic (flat parameter storage, optimizer grouping, scheduler), and the model plugins' contract."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from distributed_sod_project_b200 import _lib, build
    build.build()
    header = open(os.path.join(ROOT, "include", "sod_b200.h")).read()
    declared = set(re.findall(r"\b(sod_[a-z0-9_]+)\s*\(", header))
    assert declared, "no prototypes found"
    h = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(h, name), f"{name} declared in include/sod_b200.h but not exported"
    assert declared == set(_lib.EXPORTS)
    lib = _lib.lib()
    assert lib.sod_version() == 7
    assert lib.sod_comm_flag_bytes() == 4 * 1024 * 8 * 4
    assert lib.sod_syncbn_exchange_bytes(64) == 8 * 2 * 64 * 8
    assert b"workspace" in lib.sod_strerror(-3)
    # struct layout agrees with the header (sizes are part of the ABI)
    assert ctypes.sizeof(_lib.sod_sgd_segment) == 32 and ctypes.sizeof(_lib.sod_comm) == 8 + 64 + 8 + 8 + 8 + 8 + 8


def test_no_cpu_fallback_in_product_path():
    from distributed_sod_project_b200 import _lib
    from distributed_sod_project_b200.loss import CEL
    from distributed_sod_project_b200.syncbn import SyncBatchNorm
    with pytest.raises(_lib.SodError):
        CEL()(torch.zeros(4), torch.zeros(4))
    with pytest.raises(_lib.SodError):
        SyncBatchNorm(8)(torch.zeros(1, 8, 2, 2))
    # and nothing under the package imports the oracle
    pkg = os.path.join(ROOT, "distributed_sod_project_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f


def test_model_plugin_contract():
    from distributed_sod_project_b200 import network
    from distributed_sod_project_b200.utils import init_seed
    init_seed(0)
    m = network.res50()
    names = [n for n, _ in m.named_parameters()]
    assert len(names) == 319 and sum(p.numel() for p in m.parameters()) == 24_906_305
    assert names[0] == "div_2.0.weight" and names[-1] == "classifier.bias"
    assert sum(isinstance(x, nn.BatchNorm2d) for x in m.modules()) == 84
    backbone = [n for n in names if n.startswith("div") and not n.startswith("div_2")]
    head = [n for n in names if not n.startswith("div")]
    assert (len(backbone), len(head), len(names) - len(backbone) - len(head)) == (156, 160, 3)
    m.eval()
    with torch.no_grad():
        assert m(torch.zeros(1, 3, 64, 64)).shape == (1, 1, 64, 64)
    assert network.cp_res50.recompute and not network.res50.recompute


def test_model_plugin_is_bit_identical_to_reference(golden):
    """res50 after `init_seed(0)` against the reference's res50 (tests/golden/model_res50_init.npz, tools/make_golden.py):
    the same state_dict keys in the same order and bit-identical initial values (sha256 of every entry), and the same
    output on one seeded input.  The outputs are held to a tolerance, not to the bit: the CPU convolutions' summation
    order depends on the thread count and instruction set of the host that computes them (1 vs 8 threads moves the
    eval-mode output by 2e-6 and the train-mode output, whose deepest BN normalises 8 samples, by 1.1e-4 of its range)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from make_golden import tensor_digest
    from distributed_sod_project_b200 import network
    from distributed_sod_project_b200.utils import init_seed
    g = golden("model_res50_init.npz")
    init_seed(0)
    m = network.res50()
    sd = m.state_dict()
    assert list(sd) == list(g["names"])
    for name, want in zip(sd, g["digests"]):
        assert tensor_digest(sd[name]) == want, name
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        for mode, tol in (("eval", 1e-5), ("train", 1e-3)):
            got, want = getattr(m, mode)()(x).numpy(), g[f"out_{mode}"]
            assert np.abs(got - want).max() <= tol * np.abs(want).max(), mode


def test_flat_params_layout_cpu():
    from distributed_sod_project_b200 import network
    from distributed_sod_project_b200.optim import FusedSGD, make_optimizer
    m = network.res50().to(memory_format=torch.channels_last)
    w_before = m.div_4[1][0].conv2.weight.detach().clone()
    opt = make_optimizer(m, "f3_trick", dict(lr=0.05, momentum=0.9, weight_decay=5e-4, nesterov=False))
    assert isinstance(opt, FusedSGD)
    f = opt.flat
    (b0, e0), (b1, e1), (b2, e2) = f.ranges
    assert b0 == 0 and e0 == b1 and e1 == b2 and e2 == f.numel and f.numel % 64 == 0
    assert [g["lr"] for g in opt.param_groups] == pytest.approx([0.005, 0.05])
    # views, not copies; memory format preserved; values preserved
    w = m.div_4[1][0].conv2.weight
    assert w.data_ptr() >= f.param.data_ptr() and w.data_ptr() < f.param.data_ptr() + 4 * f.numel
    assert w.is_contiguous(memory_format=torch.channels_last) and torch.equal(w.detach(), w_before)
    assert w.grad is not None and w.grad.stride() == w.stride()
    frozen = dict(m.named_parameters())["div_2.0.weight"]
    assert frozen.data_ptr() >= f.param.data_ptr() + 4 * b2
    segs, n = opt._segments()
    assert n == 3 and segs[2].flags == 1 and abs(segs[0].lr - 0.005) < 1e-9 and abs(segs[1].weight_decay - 5e-4) < 1e-9
    # autograd accumulates INTO the flat buffer
    m.train()
    m(torch.randn(2, 3, 64, 64)).sum().backward()
    assert float(f.grad.abs().sum()) > 0
    opt.zero_grad()
    assert float(f.grad.abs().sum()) == 0
    from distributed_sod_project_b200 import _lib
    with pytest.raises(_lib.SodError):
        opt.step()          # CPU parameters: the fused step refuses instead of falling back


def test_scheduler_matches_reference_table(golden):
    from distributed_sod_project_b200.optim import CustomScheduler
    g = golden("sgd_kat.npz")

    class _Opt:
        param_groups = [{"lr": 0.005}, {"lr": 0.05}]
    for kind in ("poly", "poly_warmup", "cosine_warmup", "f3_sche"):
        opt = _Opt(); opt.param_groups = [{"lr": 0.005}, {"lr": 0.05}]
        sch = CustomScheduler(opt, total_num=30, scheduler_type=kind, scheduler_info=dict(lr_decay=0.9, warmup_epoch=3))
        for e, row in enumerate(g[f"sched/{kind}"]):
            sch.step(opt, curr_epoch=e)
            got = [gr["lr"] for gr in opt.param_groups]
            if any(isinstance(v, complex) for v in got) or np.isnan(row).any():
                break
            np.testing.assert_allclose(got, row, rtol=1e-12)


def test_exp_name_and_paths():
    import config
    from distributed_sod_project_b200.utils import construct_exp_name, construct_path_dict
    name = construct_exp_name(config.user_config)
    assert name.startswith(config.user_config["model"] + "_SIZE320_BS")
    paths = construct_path_dict(config.user_config["proj_root"], name, config.user_config["xlsx_name"])
    assert paths["final_full_net"].endswith("pth/checkpoint_final.pth.tar")


def test_shadow_weight_installation_is_structural_only():
    """amp's bf16 shadow: every managed Conv2d gets bf16 leaves that alias the flat shadow / gradient buffers; without
    autocast (eval, CPU) the patched forward still runs on the fp32 master, so outputs are unchanged."""
    from distributed_sod_project_b200 import amp, network
    from distributed_sod_project_b200.optim import make_optimizer
    from distributed_sod_project_b200.utils import init_seed
    init_seed(0)
    ref = network.res50().eval()
    init_seed(0)
    m = network.res50().eval()
    opt = make_optimizer(m, "f3_trick", dict(lr=0.05, momentum=0.9, weight_decay=5e-4, nesterov=False))
    flat = opt.flat
    flat.enable_shadow(torch.bfloat16)
    n = amp._install_shadow_weights(m, flat)
    assert n == sum(isinstance(x, nn.Conv2d) for x in m.modules()) == 105
    conv = m.sim8.h2h_1
    lo, hi = flat.shadow16.data_ptr(), flat.shadow16.data_ptr() + 2 * flat.numel
    assert lo <= conv._sod_w16.data_ptr() < hi and lo <= conv._sod_b16.data_ptr() < hi
    # weights: `.grad` stays None so that autograd hands over cuDNN's gradient tensor (gathered by the fused step);
    # biases: bound to their slot of the flat bf16 gradient buffer (the SyncBN backward adds into it)
    assert conv._sod_w16.dtype == torch.bfloat16 and conv._sod_w16.requires_grad and conv._sod_w16.grad is None
    assert conv._sod_b16.grad.data_ptr() - flat.grad16.data_ptr() == conv._sod_b16.data_ptr() - flat.shadow16.data_ptr()
    leaves = {id(t): (off, steal) for t, off, steal in flat.shadow_leaves}
    assert leaves[id(conv._sod_w16)] == (flat.offset_of(conv.weight), True)
    assert leaves[id(conv._sod_b16)] == (flat.offset_of(conv.bias), False)
    assert len(leaves) == 105 + 46
    assert torch.equal(conv._sod_w16.detach().float(), conv.weight.detach().to(torch.bfloat16).float())
    frozen = m.div_2[0]
    assert frozen._sod_w16.requires_grad                       # div_2 still receives gradients (it is only left un-optimised)
    x = torch.randn(1, 3, 64, 64)
    with torch.no_grad():
        assert torch.equal(m(x), ref(x))
    # a state_dict load refreshes the shadow
    sd = ref.state_dict()
    sd["classifier.weight"] = sd["classifier.weight"] + 1.0
    m.load_state_dict(sd)
    assert torch.equal(m.classifier._sod_w16.detach().float(), m.classifier.weight.detach().to(torch.bfloat16).float())


def test_ctypes_prototypes_match_header_argument_by_argument():
    """every prototype of include/sod_b200.h, parsed from the header text, against the ctypes binding: same number of
    arguments, same width/kind for each (a mismatch here is a silent stack/registers mix-up on the GPU box)"""
    import ctypes as C
    from distributed_sod_project_b200 import _lib
    text = open(os.path.join(ROOT, "include", "sod_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    protos = re.findall(r"\b(int|size_t|const char\s*\*)\s+(sod_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text)
    assert {name for _, name, _ in protos} == set(_lib.EXPORTS)

    def kind(ctype: str):
        t = ctype.strip()
        t = re.sub(r"\s+[A-Za-z_][A-Za-z0-9_]*(\[[0-9A-Z_]*\])?$", "", t) if not t.endswith("*") else t    # drop the name
        t = re.sub(r"\bconst\b", "", t).replace(" ", "")
        if t.endswith("*"):
            base = t[:-1]
            if base == "sod_comm":
                return C.POINTER(_lib.sod_comm)
            if base == "sod_sgd_segment":
                return C.POINTER(_lib.sod_sgd_segment)
            return "ptr"
        return {"int": C.c_int, "int64_t": C.c_int64, "uint64_t": C.c_uint64, "uint32_t": C.c_uint32, "float": C.c_float,
                "size_t": C.c_size_t, "int32_t": C.c_int32}[t]

    ret = {"int": C.c_int, "size_t": C.c_size_t}
    for r, name, args in protos:
        res, bound = _lib._PROTOTYPES[name]
        assert res == ret.get(r, C.c_char_p), name
        params = [] if args.strip() in ("", "void") else [a for a in args.split(",")]
        # "type* name" → split the name off pointers too
        kinds = [kind(re.sub(r"\*\s*[A-Za-z_][A-Za-z0-9_]*\s*$", "*", p.strip())) for p in params]
        assert len(kinds) == len(bound), f"{name}: header has {len(kinds)} parameters, binding {len(bound)}"
        for i, (k, b) in enumerate(zip(kinds, bound)):
            if k == "ptr":
                assert b is C.c_void_p or (isinstance(b, type) and issubclass(b, C._Pointer)), f"{name} arg {i}: {b} for a pointer"
            else:
                assert k is b or k == b, f"{name} arg {i}: header {k}, binding {b}"


def test_amp_seam_call_shapes():
    """apex-amp call shapes the reference uses (train.py:183, 299; utils/pipeline_ops.py:74,121)"""
    from distributed_sod_project_b200 import _lib, amp
    saved = dict(amp._cfg)
    try:
        net = nn.Conv2d(3, 4, 1)
        opt = torch.optim.SGD(net.parameters(), lr=0.1)
        m, o = amp.initialize(net, opt, opt_level="O1")                 # (model, optimizer) like apex
        assert m is net and o is opt
        assert amp.initialize(nn.Conv2d(3, 4, 1), opt_level="O0") is not None          # model only → model only
        with pytest.raises(_lib.SodError):
            amp.initialize(net, opt, opt_level="O2")
        loss = torch.tensor(2.0, requires_grad=True)
        with amp.scale_loss(loss, opt) as scaled:                      # bf16: static scale 1 → the loss itself
            assert scaled is loss
        amp.load_state_dict({"loss_scaler0": {"loss_scale": 1024.0, "unskipped": 7}})
        assert amp.state_dict() == {"loss_scaler0": {"loss_scale": 1024.0, "unskipped": 7}}
    finally:
        amp._cfg.clear(); amp._cfg.update(saved)
