"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/mmd.h declares, the ctypes
mirrors match the compiled structs, the drop-in modules keep the reference's state_dict contract, the op-list
builder produces a consistent plan, error behaviour, and the N>1 gradient exchange on gloo (world size 2)."""
import ctypes
import os
import re
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import mm_distillnet_b200 as mmd
from mm_distillnet_b200 import _lib, bifpn
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "mmd.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(mmd_[a-z0-9_]+)\s*\(", hdr))
    assert declared >= {"mmd_mta_fwd", "mmd_mta_bwd", "mmd_bifpn_run", "mmd_last_error", "mmd_version"}
    L = _lib.lib()
    for name in sorted(declared):
        assert hasattr(L, name), "libmmd_b200.so does not export %s" % name
    assert set(_lib.EXPORTS) == declared
    assert L.mmd_version() >= 102


def test_struct_mirrors_match():
    L = _lib.lib()
    assert L.mmd_sizeof_op() == ctypes.sizeof(_lib.Op)
    assert L.mmd_sizeof_mta_args() == ctypes.sizeof(_lib.MtaArgs)


@pytest.mark.parametrize("fixture,first", [("cell_c112", False), ("stack2_c112", True)])
def test_state_dict_contract_matches_reference(fixture, first):
    """Keys recorded from the real reference (golden fixture) == keys / shapes of our modules; init values too."""
    g = H.golden(fixture)
    C, cc, n_cells = H.STACK_CASES[fixture][:3]
    ref_keys = {k[len("buf_"):] for k in g if k.startswith("buf_")} | {k[len("pgsum_"):] for k in g if k.startswith("pgsum_")}
    stack = mmd.BiFPNStack(*[mmd.BiFPN(C, cc, first_time=(i == 0 and first)) for i in range(n_cells)])
    sd = stack.state_dict()
    assert set(sd.keys()) == ref_keys
    params, _ = H.stack_case_inputs(fixture)
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in params.items()}
    stack.load_state_dict(params, strict=True)
    # fusion weights start at one (fast-attention init), BN momentum / eps as the reference
    cell = mmd.BiFPN(C, cc)
    assert torch.equal(cell.p4_w2.data, torch.ones(3)) and cell.conv3_up.bn.momentum == 0.01 and cell.conv3_up.bn.eps == 1e-3


def test_plan_structure():
    cells = [mmd.BiFPN(112, [48, 120, 352], first_time=(i == 0)) for i in range(5)]
    shapes = [(16, 48, 96, 96), (16, 120, 48, 48), (16, 352, 24, 24)]
    plan = bifpn._Plan(cells, "cells", shapes, torch.float32, True, True, [True] * 3)
    kinds = [o.kind for o in plan.fwd_ops]
    assert kinds.count(_lib.OP_NODE_FWD) == 40 and kinds.count(_lib.OP_PROJ_FWD) == 6
    assert kinds.count(_lib.OP_BNAPPLY) == 2 + 5
    assert plan.out_shapes == [(16, 112, 96 >> i, 96 >> i) for i in range(5)]
    n_par = sum(p.numel() for c in cells for p in c.parameters())
    assert n_par == 708159
    # one flat fp32 buffer, parameter order, each gradient 16-byte aligned (<= 3 floats of padding per tensor)
    assert n_par <= plan.grad_floats <= n_par + 3 * len(plan.params)
    assert all(off % 16 == 0 for off, _, _ in plan.grad_off.values())
    bk = [o.kind for o in plan.bwd_ops]
    assert bk.count(_lib.OP_NODE_BWD) == 40 and bk.count(_lib.OP_PROJ_BWD) == 6
    assert all(0 <= o.n_cons <= 3 for o in plan.bwd_ops)
    # every NODE_BWD gathers from at least one consumer and owns storage
    for o in plan.bwd_ops:
        if o.kind == _lib.OP_NODE_BWD:
            assert o.n_cons >= 1 and o.du.base == bifpn.B_BWD and o.g_pw.base == bifpn.B_ZERO
    # forward arena allocations do not overlap
    spans = []
    for op in plan.ops:
        if op.out.base == bifpn.B_FWD:
            spans.append((op.out.off, op.out.off + plan.B * op.out.H * op.out.W * 112 * 4))
    spans.sort()
    assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:]))
    # regression: references that an op does not use must be NULL (base -1), never "forward arena + 0";
    # with inputs that need no gradient the projection backward must not get a dx destination
    ng = bifpn._Plan(cells, "cells", shapes, torch.float32, True, True, [False] * 3)
    for o in ng.bwd_ops:
        if o.kind == _lib.OP_PROJ_BWD:
            assert o.dx.base == -1 and o.du.base == -1 and o.g_dw.base == -1
        if o.kind == _lib.OP_NODE_BWD:
            assert o.dx.base == -1
        for c in range(o.n_cons, 3):
            assert o.cons[c].slot.base == -1 and o.cons[c].du.data.base == -1
    assert all(o.dx.base == -1 and o.du.base == -1 for o in ng.fwd_ops)
    # eval plan: no deferred BatchNorm, outputs written in place by the last cell
    ev = bifpn._Plan(cells, "cells", shapes, torch.float32, False, False, [False] * 3)
    assert all(o.out.bn.base < 0 for o in ev.fwd_ops) and ev.bwd_ops is None
    assert [o.kind for o in ev.fwd_ops].count(_lib.OP_BNAPPLY) == 2


def test_bf16_plan_splits_pooled_nodes():
    """bf16 plans run every node with a pooled input as POOLFUSE + NODE_FWD(input 0, aux): 4 such nodes per cell; the
    backward ops keep the node's original three inputs and get the pre-pass outputs (aux, raw arg-max values)."""
    cells = [mmd.BiFPN(112, [48, 120, 352], first_time=(i == 0)) for i in range(5)]
    shapes = [(16, 48, 96, 96), (16, 120, 48, 48), (16, 352, 24, 24)]
    plan = bifpn._Plan(cells, "cells", shapes, torch.bfloat16, True, True, [True] * 3)
    kinds = [o.kind for o in plan.fwd_ops]
    assert kinds.count(_lib.OP_POOLFUSE) == 20 and kinds.count(_lib.OP_NODE_FWD) == 40
    for i, o in enumerate(plan.fwd_ops):
        if o.kind == _lib.OP_POOLFUSE:
            nxt = plan.fwd_ops[i + 1]
            assert nxt.kind == _lib.OP_NODE_FWD and nxt.n_in == 2 and nxt.fw_idx[1] == -1 and nxt.fw_n == o.fw_n
            assert o.mode[0] == _lib.IN_POOL and o.pidx[0].base == bifpn.B_FWD and o.save_d.base == bifpn.B_FWD
            assert (nxt.inp[1].data.base, nxt.inp[1].data.off) == (o.out.data.base, o.out.data.off)
            assert o.out.bn.base == -1                       # final values: no deferred BatchNorm on the operand
    for o in plan.fwd_ops:
        if o.kind == _lib.OP_NODE_FWD:
            assert all(o.mode[k] != _lib.IN_POOL for k in range(o.n_in)) and o.packed.base == bifpn.B_PERSIST
    pooled_bwd = [o for o in plan.bwd_ops if o.kind == _lib.OP_NODE_BWD and _lib.IN_POOL in list(o.mode)[:o.n_in]]
    assert len(pooled_bwd) == 20 and all(o.aux.base == bifpn.B_FWD and o.praw.base == bifpn.B_FWD for o in pooled_bwd)
    # fp32 (parity) plans keep the single fused node
    p32 = bifpn._Plan(cells, "cells", shapes, torch.float32, True, True, [True] * 3)
    assert [o.kind for o in p32.fwd_ops].count(_lib.OP_POOLFUSE) == 0
    # eval bf16 plan: pre-pass without arg-max / raw outputs
    ev = bifpn._Plan(cells, "cells", shapes, torch.bfloat16, False, False, [False] * 3)
    assert all(o.pidx[0].base == -1 and o.save_d.base == -1 for o in ev.fwd_ops if o.kind == _lib.OP_POOLFUSE)


def test_shape_validation_and_errors():
    cells = [mmd.BiFPN(112, [48, 120, 352], first_time=True)]
    with pytest.raises(ValueError):   # P4 is not exactly half of P3
        bifpn._Plan(cells, "cells", [(1, 48, 20, 20), (1, 120, 9, 9), (1, 352, 5, 5)], torch.float32, False, False, [False] * 3)
    with pytest.raises(ValueError):
        bifpn._Plan(cells, "cells", [(1, 48, 16, 16)] * 5, torch.float32, False, False, [False] * 5)
    with pytest.raises(RuntimeError):   # CPU tensors: the product path has no CPU fallback
        cells[0](tuple(torch.randn(1, c, 16 >> i, 16 >> i) for i, c in enumerate([48, 120, 352])))
    with pytest.raises(RuntimeError):
        mmd.MTALoss()([torch.randn(1, 112, 4, 4)], [torch.randn(1, 112, 4, 4)])
    with pytest.raises(NotImplementedError):   # a norm=False block is a parameter holder of the heads, not runnable alone
        mmd.SeparableConvBlock(112, 36, norm=False)(torch.randn(1, 112, 4, 4))
    crit = mmd.MTALoss(T="9", p="2")     # config passes strings (src/utils/utils.py:1603-1604)
    assert crit.T == 9.0 and crit.p == 2.0


def test_patch_reference_rebinds_globals():
    import types
    det = types.ModuleType("fake_det")

    class FakeDet(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.bifpn = torch.nn.Sequential(*[det.BiFPN(112, [48, 120, 352], first_time=(i == 0)) for i in range(2)])

    det.BiFPN = object
    det.YetAnotherEfficientDet = FakeDet
    loss = types.ModuleType("fake_loss")
    loss.MTALoss = object
    utils = types.ModuleType("fake_utils")
    utils.MTALoss = object
    mmd.patch_reference(det, loss, utils)
    assert det.BiFPN is mmd.BiFPN and loss.MTALoss is mmd.MTALoss and utils.MTALoss is mmd.MTALoss
    m = det.YetAnotherEfficientDet()
    assert isinstance(m.bifpn, mmd.BiFPNStack) and list(m.state_dict())[0].startswith("bifpn.0.")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        student = mmd.BiFPNStack(mmd.BiFPN(112, [48, 120, 352], first_time=True))
        step = mmd.DistillStep(student, [], device=torch.device("cpu"))
        n = sum(p.numel() for p in student.parameters())
        flat = torch.full((n,), float(rank + 1))
        flat[:3] = torch.tensor([1.0, 2.0, 3.0]) * (rank + 1)
        step._on_flat_grad(flat)                      # the N>1 exchange: one all-reduce (sum) then 1/world
        out[rank] = (step.flat_grad[:4].tolist(), step.world)
    finally:
        dist.destroy_process_group()


def test_flat_gradient_allreduce_gloo_world2():
    world, port = 2, _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_gloo_worker, args=(world, port, out), nprocs=world, join=True)
        res = dict(out)
    for r in range(world):
        vals, w = res[r]
        assert w == 2
        assert vals == [1.5, 3.0, 4.5, 1.5]    # mean over ranks (DDP semantics, train_methods.py:957-961)


def test_header_constants_match_python_mirrors():
    """Constants shared between include/mmd.h and the ctypes side (array extents, accumulator replicas, version)."""
    hdr = open(os.path.join(ROOT, "include", "mmd.h")).read()
    defs = dict(re.findall(r"#define\s+(MMD_[A-Z_]+)\s+(\d+)", hdr))
    assert int(defs["MMD_MTA_MAX_LEVELS"]) == _lib.MTA_MAX_LEVELS
    assert int(defs["MMD_MTA_MAX_TEACHERS"]) == _lib.MTA_MAX_TEACHERS
    assert int(defs["MMD_STATS_REPLICAS"]) == _lib.STATS_REPLICAS
    assert _lib.lib().mmd_version() == int(defs["MMD_VERSION"])
    # the per-teacher batching flag of the MTA call is part of the mirrored struct
    assert "separate" in [f[0] for f in _lib.MtaArgs._fields_]


def test_mta_forward_each_rejects_cpu_tensors_and_bad_shapes():
    """No CPU fallback on the batched per-teacher entry either; argument checks happen before any launch."""
    crit = mmd.MTALoss()
    fs = [torch.randn(2, 112, 4, 4), torch.randn(2, 112, 2, 2)]
    ts = [[torch.randn(2, 112, 4, 4), torch.randn(2, 112, 2, 2)] for _ in range(3)]
    with pytest.raises(RuntimeError):
        crit.forward_each(fs, ts)
    with pytest.raises(ValueError):
        crit.forward_each(fs, [ts[0]] * 5)          # more teachers than one call takes


def test_distill_step_rejects_foreign_modules():
    with pytest.raises(TypeError):
        mmd.DistillStep(torch.nn.Linear(2, 2), [])


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs first): ONE JSON line with the contract keys, same metric /
    unit / config as the CUDA arm, impl = reference, e2e = the line's own value with zero copy bytes."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "distill samples/s" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]


def test_flat_channels_last_views():
    """DistillStep's static / staging input sets: channels_last views of ONE allocation with identical layouts, so a
    whole set moves with a single copy of the flat buffer."""
    from mm_distillnet_b200.distill import _flat_channels_last
    xs = [torch.randn(2, 48, 8, 8).to(torch.bfloat16), torch.randn(2, 120, 4, 4).to(torch.bfloat16), torch.randn(2, 352, 2, 2)]
    flat_a, va = _flat_channels_last(xs, torch.device("cpu"))
    flat_b, vb = _flat_channels_last(xs, torch.device("cpu"))
    assert flat_a.numel() == flat_b.numel() and flat_a.dtype == torch.uint8
    for v, x in zip(va, xs):
        assert v.shape == x.shape and v.dtype == x.dtype and v.is_contiguous(memory_format=torch.channels_last)
        assert v.data_ptr() % 16 == 0          # bulk copies / 16-byte vector loads of the kernels
        v.copy_(x)
    flat_b.copy_(flat_a)
    assert all(torch.equal(b, x) for b, x in zip(vb, xs))
    leaf = va[0].requires_grad_(True)
    assert leaf.is_leaf and leaf.requires_grad


def test_other_channel_counts_fail_at_construction():
    """The reference builds D0..D7 (64/88/112/160.. channels, src/YetAnotherEfficientDet.py:611-629); the kernels exist for
    D2 only, and a drop-in must say so when the model is built, not at its first forward."""
    with pytest.raises(NotImplementedError):
        mmd.BiFPN(64, [40, 112, 320], first_time=True)
    with pytest.raises(NotImplementedError):
        mmd.BiFPN(160, [48, 136, 384])


def test_modules_with_cached_plans_deepcopy_and_pickle():
    """A runner that holds plans (ctypes op lists full of device pointers) must not break copy.deepcopy / pickling of the
    module (EMA copies, best-model snapshots, spawn-based workers): the copy gets a fresh, empty runner."""
    import copy
    import pickle
    stack = mmd.BiFPNStack(*[mmd.BiFPN(112, [48, 120, 352], first_time=(i == 0)) for i in range(2)])
    shapes = [(2, 48, 16, 16), (2, 120, 8, 8), (2, 352, 4, 4)]
    plan = bifpn._Plan(list(stack), "cells", shapes, torch.bfloat16, True, True, [False] * 3)
    stack._runner.plans["k"] = plan
    stack[0]._runner.plans["k"] = plan
    stack._runner.grad_sink = lambda flat: None
    dup = copy.deepcopy(stack)
    assert dup._runner is not stack._runner and dup._runner.plans == {} and dup._runner.grad_sink is None
    assert dup[0]._runner.plans == {} and len(stack._runner.plans) == 1
    assert all(torch.equal(a, b) for a, b in zip(dup.state_dict().values(), stack.state_dict().values()))
    stack._runner.grad_sink = None
    back = pickle.loads(pickle.dumps(stack))
    assert back._runner.plans == {} and set(back.state_dict()) == set(stack.state_dict())


def test_library_staleness_is_a_content_hash():
    """_lib.lib() rebuilds when the .so was built from other sources (hash of the sources, not mtimes)."""
    assert os.path.exists(_lib.LIB_PATH) and not _lib.is_stale()
    with open(_lib.HASH_PATH) as f:
        saved = f.read()
    try:
        with open(_lib.HASH_PATH, "w") as f:
            f.write("0" * 64 + "\n")
        assert _lib.is_stale()
    finally:
        with open(_lib.HASH_PATH, "w") as f:
            f.write(saved)
    assert not _lib.is_stale() and saved.strip() == _lib.source_hash()


def _reference_d2_state():
    """(parameters, buffers) of the reference D2 model's bifpn / regressor / classifier as recorded from the reference
    modules in the golden fixtures (oracle/make_golden.py loads each module strictly, then stores every parameter's
    gradient in named_parameters order and every BatchNorm buffer): [(key, array)], parameter arrays shaped like the
    parameters.  stack2_c112 holds a first cell ("0.") and a later one ("1."), reg_c112 / cls_c112 the D2 heads (112
    channels, 9 anchors, 3 layers, 20 classes)."""
    fixtures = {n: H.golden(n) for n in ("stack2_c112", "reg_c112", "cls_c112")}
    parts = [("bifpn.%d." % i, "stack2_c112", "0." if i == 0 else "1.") for i in range(5)] + \
        [("regressor.", "reg_c112", ""), ("classifier.", "cls_c112", "")]
    params, bufs = [], []
    for prefix, fixture, src in parts:
        for k, v in fixtures[fixture].items():
            for tag, out in (("pgrad_" + src, params), ("buf_" + src, bufs)):
                if k.startswith(tag):
                    out.append((prefix + k[len(tag):], v))
    return params, bufs


def test_d2_model_matches_the_reference_state_dict():
    """patch_reference(heads=True) on a stand-in YetAnotherEfficientDet that builds the BiFPN and the heads as the
    reference's constructor does (src/YetAnotherEfficientDet.py:611-629 sizes, :639-652 modules): the D2 model has the
    reference's parameter names in the reference's order, its shapes and its buffers (golden fixtures), loads a state_dict
    with exactly those keys strictly, and other compound coefficients / too wide headers fail at construction."""
    import types
    det = types.ModuleType("det")

    class YetAnotherEfficientDet(torch.nn.Module):
        def __init__(self, num_classes=20, compound_coef=2):
            super().__init__()
            C = [64, 88, 112][compound_coef]
            cc = [[40, 112, 320], [40, 112, 320], [48, 120, 352]][compound_coef]
            self.bifpn = torch.nn.Sequential(*[det.BiFPN(C, cc, True if i == 0 else False) for i in range([3, 4, 5][compound_coef])])
            self.regressor = det.Regressor(in_channels=C, num_anchors=9, num_layers=3)
            self.classifier = det.Classifier(in_channels=C, num_anchors=9, num_classes=num_classes, num_layers=3)

    det.YetAnotherEfficientDet = YetAnotherEfficientDet
    det.BiFPN = det.Regressor = det.Classifier = object
    loss = types.ModuleType("loss")
    loss.MTALoss = object
    mmd.patch_reference(det, loss, types.ModuleType("utils"), heads=True)
    params, bufs = _reference_d2_state()
    assert len(params) == 72 + 4 * 48 + 2 * 42 and len(bufs) == 42 + 4 * 24 + 2 * 45
    m = det.YetAnotherEfficientDet(num_classes=20, compound_coef=2)
    assert isinstance(m.bifpn, mmd.BiFPNStack) and len(m.bifpn) == 5
    assert isinstance(m.regressor, mmd.Regressor) and isinstance(m.classifier, mmd.Classifier)
    assert [(k, tuple(p.shape)) for k, p in m.named_parameters()] == [(k, v.shape) for k, v in params]
    sd = m.state_dict()
    pkeys = {k for k, _ in params}
    assert {(k, tuple(v.shape)) for k, v in sd.items() if k not in pkeys} == {(k, v.shape) for k, v in bufs}
    ref_sd = {k: torch.from_numpy(v) for k, v in params + bufs}
    assert set(sd) == set(ref_sd)
    m.load_state_dict(ref_sd, strict=True)
    assert all(torch.equal(v, ref_sd[k]) for k, v in m.state_dict().items())
    with pytest.raises(NotImplementedError):   # D0: 64 channels
        det.YetAnotherEfficientDet(num_classes=20, compound_coef=0)
    with pytest.raises(NotImplementedError):   # 9 x 90 = 810 header channels: more than two C-row halves
        det.YetAnotherEfficientDet(num_classes=90, compound_coef=2)


# a checkout of the reference (robot-learning-freiburg/MM-DistillNet) and its Python dependencies; not part of this repository
REF = os.environ.get("MMD_REFERENCE_SRC", "")


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "src"))),
                    reason="set MMD_REFERENCE_SRC to a checkout of the reference MM-DistillNet to run this test")
def test_patch_reference_on_the_real_modules():
    """patch_reference() on the REAL src.* modules (not fakes): the patched YetAnotherEfficientDet(D2) has the same
    state_dict keys / shapes as the unpatched one, loads its state_dict strictly, holds a fused BiFPNStack, refuses CPU
    tensors (no fallback), and other compound coefficients fail at construction."""
    import importlib
    import sys
    sys.path.insert(0, REF)
    try:
        det = importlib.import_module("src.YetAnotherEfficientDet")
        loss = importlib.import_module("src.loss.MTALoss")
        orig_bifpn, orig_mta, orig_init = det.BiFPN, loss.MTALoss, det.YetAnotherEfficientDet.__init__
        orig_heads = det.Regressor, det.Classifier
        torch.manual_seed(0)
        ref_model = det.YetAnotherEfficientDet(num_classes=20, compound_coef=2)
        ref_sd = ref_model.state_dict()
        try:
            mmd.patch_reference()
            assert det.BiFPN is mmd.BiFPN and loss.MTALoss is mmd.MTALoss
            torch.manual_seed(0)
            ours = det.YetAnotherEfficientDet(num_classes=20, compound_coef=2)
            assert isinstance(ours.bifpn, mmd.BiFPNStack) and len(ours.bifpn) == 5
            sd = ours.state_dict()
            assert list(sd.keys()) == list(ref_sd.keys())
            assert all(tuple(sd[k].shape) == tuple(ref_sd[k].shape) for k in sd)
            # same construction order under the same seed -> identical initial weights
            assert all(torch.equal(sd[k], ref_sd[k]) for k in sd if k.startswith("bifpn."))
            ours.load_state_dict(ref_sd, strict=True)
            with pytest.raises(RuntimeError):          # CPU tensors: the product path has no CPU fallback
                ours.eval()(torch.zeros(1, 3, 768, 768))
            with pytest.raises(NotImplementedError):   # D0: 64 channels
                det.YetAnotherEfficientDet(num_classes=20, compound_coef=0)
            crit = loss.MTALoss(T="9", p="2")
            assert isinstance(crit, mmd.MTALoss)
            assert det.Regressor is orig_heads[0]      # the heads are rebound on request only
            # heads=True: the detection heads become ours too, with the same keys, shapes and initial weights
            mmd.patch_reference(heads=True)
            assert det.Regressor is mmd.Regressor and det.Classifier is mmd.Classifier
            torch.manual_seed(0)
            ours = det.YetAnotherEfficientDet(num_classes=20, compound_coef=2)
            assert isinstance(ours.regressor, mmd.Regressor) and isinstance(ours.classifier, mmd.Classifier)
            sd = ours.state_dict()
            assert list(sd.keys()) == list(ref_sd.keys())
            assert all(torch.equal(sd[k], ref_sd[k]) for k in sd if k.startswith(("bifpn.", "regressor.", "classifier.")))
            ours.load_state_dict(ref_sd, strict=True)
            with pytest.raises(NotImplementedError):   # 9 x 90 = 810 header channels: more than two C-row halves
                det.YetAnotherEfficientDet(num_classes=90, compound_coef=2)
        finally:
            det.BiFPN, loss.MTALoss = orig_bifpn, orig_mta
            det.Regressor, det.Classifier = orig_heads
            det.YetAnotherEfficientDet.__init__ = orig_init
            det.YetAnotherEfficientDet._mmd_patched = False
    finally:
        sys.path.remove(REF)


def test_set_option_switches_exist_and_reject_unknown_names():
    """mmd_set_option (include/mmd.h): the documented A/B switches are accepted without a GPU (they only set flags), an
    unknown name is an argument error with a message."""
    for name, default in (("chain_fwd", 0), ("mta_fast", 1), ("proj_tma", 1)):
        _lib.set_option(name, 1 - default)
        _lib.set_option(name, default)
    with pytest.raises(RuntimeError, match="unknown option"):
        _lib.set_option("definitely_not_an_option", 1)
    hdr = open(os.path.join(ROOT, "include", "mmd.h")).read()
    for name in ("chain_fwd", "mta_fast", "proj_tma"):
        assert '"%s"' % name in hdr, "include/mmd.h does not document option %s" % name


def test_plan_records_pool_tags_for_the_argmax_hook():
    """The parity tests force the oracle's max-pool arg-max to the CUDA forward's own choice (bifpn.debug_pool_argmax):
    every op that pools carries a (cell, name) tag and arg-max storage in a training plan with gradients."""
    cells = [mmd.BiFPN(112, [48, 120, 352], first_time=(i == 0)) for i in range(2)]
    shapes = [(2, 48, 32, 32), (2, 120, 16, 16), (2, 352, 8, 8)]
    for dt in (torch.float32, torch.bfloat16):
        plan = bifpn._Plan(cells, "cells", shapes, dt, True, True, [True] * 3)
        tags = sorted(op.tag for op in plan.ops if op.tag is not None)
        assert tags == sorted([(0, "p6_in"), (0, "p7_in")] + [(c, n) for c in range(2) for n in ("p3_out", "p4_out", "p5_out", "p6_out")])
        assert all(any(r is not None for r in op.pidx) for op in plan.ops if op.tag is not None)
    with pytest.raises(RuntimeError):
        bifpn.debug_pool_argmax(torch.zeros(1, requires_grad=True) * 2)     # not an output of a BiFPN forward


def test_product_never_touches_the_oracle_or_the_reference_tree():
    """The oracle is test infrastructure: nothing under mm_distillnet_b200/ (Python or CUDA) may import, open or mention
    oracle/ or /root/reference at run time; bench.py may use oracle/ only in its CPU legs (cpu_step / time_cpu /
    run_reference)."""
    pkg = os.path.join(ROOT, "mm_distillnet_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if not fn.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            txt = open(os.path.join(dirpath, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), fn
            assert "mmd_oracle" not in txt and "/root/reference" not in txt, fn
    bench = open(os.path.join(ROOT, "bench.py")).read()
    uses = [m.start() for m in re.finditer(r"from oracle import", bench)]
    assert len(uses) == 2                                     # cpu_state() and cpu_step() only
    gpu_arm = bench[bench.index("def measure("):bench.index("def main(")]
    assert "oracle" not in gpu_arm.replace("oracle port", "")  # the CUDA arm only NAMES the port in its cpu_baseline text


def test_head_modules_mirror_reference_state_dict_and_plan():
    """Regressor / Classifier (SURVEY 8 f1): the reference's state_dict names and shapes, and the op list a head plan is
    made of — towers and header halves as NODE ops, one HEAD_GATHER per level, COPY ops for the zero-padded header."""
    import collections
    from oracle import mmd_oracle as O
    from mm_distillnet_b200 import bifpn as bf
    for cls, args, kout in ((mmd.Regressor, (112, 9, 3), 36), (mmd.Classifier, (112, 9, 20, 3), 180)):
        m = cls(*args)
        ref = O.synth_head_params(112, kout, 3, 1)       # names recorded from the reference modules (make_golden.py)
        sd = m.state_dict()
        assert set(sd) == set(ref) and all(tuple(sd[k].shape) == tuple(ref[k].shape) for k in ref)
        m.load_state_dict(ref, strict=True)
        halves = (kout + 111) // 112
        shapes = [(2, 112, s, s) for s in (16, 8, 4, 2, 1)]
        for dt in (torch.float32, torch.bfloat16):
            pl = bf._Plan([m], "head", shapes, dt, True, True, [True] * 5)
            kf = collections.Counter(o.kind for o in pl.fwd_ops)
            kb = collections.Counter(o.kind for o in pl.bwd_ops)
            assert kf == {_lib.OP_COPY: 2, _lib.OP_NODE_FWD: 5 * (3 + halves), _lib.OP_HEAD_GATHER: 5, _lib.OP_BNAPPLY: 1,
                          _lib.OP_ACT_FWD: 1}
            assert kb == {_lib.OP_ACT_BWD: 1, _lib.OP_SLOT: 1, _lib.OP_HEAD_SCATTER: 5, _lib.OP_NODE_BWD: 5 * (3 + halves),
                          _lib.OP_PULL: 5}
            assert pl.out_shapes == [(2, 341 * 9, kout // 9), (2, 112, 1, 1)]
            hdr = [o for o in pl.fwd_ops if o.kind == _lib.OP_NODE_FWD and o.train == 0]
            assert len(hdr) == 5 * halves and all(o.save_d.base >= 0 and o.out.bn.base == -1 for o in hdr)
            ev = bf._Plan([m], "head", shapes, dt, False, False, [False] * 5)
            assert ev.bwd_ops is None and all(o.train == 0 for o in ev.fwd_ops)
    with pytest.raises(NotImplementedError):
        mmd.Regressor(64, 9, 3)
    with pytest.raises(NotImplementedError):
        mmd.Classifier(112, 9, 90, 3)
    blk = mmd.SeparableConvBlock(112, 36, norm=False)
    assert "bn.weight" not in blk.state_dict()
    with pytest.raises(NotImplementedError):
        blk(torch.zeros(1, 112, 4, 4))


def test_focal_loss_host_side():
    """YetAnotherFocalLoss (SURVEY 8 f4): label padding as the reference's annot_padded (:35-39), the mirrored argument
    struct, no CPU fallback, and the opt-in rebinding of the reference's names."""
    import types
    import numpy as np
    from mm_distillnet_b200 import focal
    ann = [np.array([[1, 2, 3, 4, 5], [6, 7, 8, 9, 0]], dtype=np.float64), np.zeros((0, 5)), np.array([[1, 1, 2, 2, 3]])]
    p = focal.pad_annotations(ann)
    assert p.shape == (3, 2, 5) and p.dtype == np.float32
    assert (p[1] == -1).all() and (p[2, 1] == -1).all() and p[0, 1, 4] == 0 and p[2, 0, 4] == 3
    assert focal.pad_annotations([np.zeros((0, 5))] * 2).shape == (2, 0, 5)
    assert _lib.lib().mmd_sizeof_focal_args() == ctypes.sizeof(_lib.FocalArgs)
    hdr = open(os.path.join(ROOT, "include", "mmd.h")).read()
    assert int(re.search(r"#define\s+MMD_FOCAL_MAX_BOXES\s+(\d+)", hdr).group(1)) == _lib.FOCAL_MAX_BOXES
    crit = mmd.YetAnotherFocalLoss()
    with pytest.raises(RuntimeError):
        crit((torch.rand(1, 8, 3), torch.rand(1, 8, 4), torch.rand(1, 8, 4)), [np.zeros((0, 5))])
    det, loss, utils = types.ModuleType("det"), types.ModuleType("loss"), types.ModuleType("utils")

    class _Det:
        def __init__(self):
            pass
    det.YetAnotherEfficientDet, det.BiFPN = _Det, object
    loss.MTALoss = object
    utils.MTALoss, utils.YetAnotherFocalLoss = object, object
    mmd.patch_reference(det, loss, utils, detection_loss=True)
    assert utils.YetAnotherFocalLoss is mmd.YetAnotherFocalLoss and utils.MTALoss is mmd.MTALoss


def test_pseudo_label_host_side():
    """Pseudo-label generation (SURVEY 8 f3) and the step wrappers (8 f5), host logic only: the mirrored argument struct and
    constants, the class-id -> label table of logits_to_ground_truth (utils.py:197-201, :299-300), config access through a
    configparser section or a dict, no CPU fallback, wrapper construction, and the opt-in rebinding of the reference's names."""
    import configparser
    import types
    import numpy as np
    from mm_distillnet_b200 import pseudo, wrappers
    from tests import helpers as H
    assert _lib.lib().mmd_sizeof_pseudo_args() == ctypes.sizeof(_lib.PseudoArgs)
    hdr = open(os.path.join(ROOT, "include", "mmd.h")).read()
    defs = dict(re.findall(r"#define\s+(MMD_[A-Z_]+)\s+(\d+)", hdr))
    assert (int(defs["MMD_PL_MAX_TEACHERS"]), int(defs["MMD_PL_MAX_CAP"]), int(defs["MMD_PL_MAX_IGNORE"])) == \
        (_lib.PL_MAX_TEACHERS, _lib.PL_MAX_CAP, _lib.PL_MAX_IGNORE)
    assert pseudo.DEFAULT_CAP <= _lib.PL_MAX_CAP and pseudo.DEFAULT_MAX_LABELS <= _lib.FOCAL_MAX_BOXES
    vcd = H.pseudo_valid_classes_dict()
    tab = pseudo.label_table(vcd, 20)
    assert tab.dtype == np.int32 and [int(tab[i]) for i in H.PSEUDO_VALID_IDS] == list(range(len(H.PSEUDO_VALID_IDS)))
    assert (tab[[i for i in range(20) if i not in H.PSEUDO_VALID_IDS]] == -1).all()
    cp = configparser.ConfigParser()
    cp.read_dict({"s": H.pseudo_config(128)})
    for cfg in (cp["s"], H.pseudo_config(128)):
        assert pseudo._cfg_get(cfg, "conf_threshold", "float") == 0.3 and pseudo._cfg_get(cfg, "image_size", "int") == 128
        assert pseudo._cfg_get(cfg, "ignore_labels", "str", default="") == "4"
        assert pseudo._cfg_get(cfg, "missing", "str", default="") == ""
        with pytest.raises(KeyError):
            pseudo._cfg_get(cfg, "missing", "float")
    # workspace size: a pure function of the sizes (no device needed)
    a = _lib.PseudoArgs()
    a.B, a.N, a.K, a.T, a.cap = 4, 110484, 20, 3, 4096
    need = _lib.lib().mmd_pseudo_workspace_bytes(ctypes.byref(a))
    assert 12 * 110484 * 5 <= need <= 12 * 110484 * 5 + 12 * 4096 * 28 + (1 << 20)
    c, r, anchors = torch.rand(1, 8, 20), torch.rand(1, 8, 4), torch.rand(1, 8, 4)
    with pytest.raises(RuntimeError):
        pseudo.teacher_pseudo_labels([(c, r, anchors)], vcd, H.pseudo_config(128))
    with pytest.raises(NotImplementedError):
        pseudo.logits_to_ground_truth((c, r, anchors), None, vcd, H.pseudo_config(128, student="EfficientDet"))
    # the wrappers keep the reference's constructor and attribute names (train_methods.py:166-175)
    student, teachers = torch.nn.Identity(), torch.nn.ModuleDict({"rgb": torch.nn.Identity()})
    for cls in (wrappers.ModelWithNMSLoss, wrappers.ModelWithNMSKDListLoss, wrappers.ModelWithNMSLossAugmented,
                wrappers.ModelWithNMSKDListLossAugmented):
        m = cls(student, teachers, mmd.YetAnotherFocalLoss(), None, mmd.MTALoss("9", "2"), cp["s"], vcd)
        assert m.student_model is student and m.teacher_models is teachers and m.criterion_div is None
        assert {"student_model", "teacher_models", "criterion_main", "criterion_kd"} <= {n for n, _ in m.named_children()}
    assert wrappers.ModelWithNMSKDListLoss.kd_list and not wrappers.ModelWithNMSLoss.kd_list
    det, loss, utils, tm = (types.ModuleType(n) for n in ("det", "loss", "utils", "tm"))

    class _Det:
        def __init__(self):
            pass
    det.YetAnotherEfficientDet, det.BiFPN = _Det, object
    loss.MTALoss = object
    utils.MTALoss, utils.logits_to_ground_truth = object, object
    tm.ModelWithNMSLoss = tm.ModelWithNMSKDListLoss = tm.ModelWithNMSLossAugmented = tm.logits_to_ground_truth = object
    tm.ModelWithNMSKDListLossAugmented = object
    mmd.patch_reference(det, loss, utils, step_wrappers=True, train_methods_module=tm)
    assert tm.ModelWithNMSLoss is mmd.ModelWithNMSLoss and tm.ModelWithNMSKDListLoss is mmd.ModelWithNMSKDListLoss
    assert tm.ModelWithNMSKDListLossAugmented is mmd.ModelWithNMSKDListLossAugmented
    assert tm.logits_to_ground_truth is mmd.logits_to_ground_truth and utils.logits_to_ground_truth is mmd.logits_to_ground_truth


def test_flat_adam_host_side():
    """Optimizer step (SURVEY 8d cfg 3): mirrored argument struct, export, no CPU fallback, DistillStep accepts it."""
    from mm_distillnet_b200 import optim
    assert _lib.lib().mmd_sizeof_adam_args() == ctypes.sizeof(_lib.AdamArgs)
    assert "mmd_adam_step" in _lib.EXPORTS
    with pytest.raises(RuntimeError):
        optim.FlatAdam([torch.nn.Parameter(torch.zeros(4))])
    with pytest.raises(ValueError):
        optim.FlatAdam([])
    import inspect
    assert "optimizer" in inspect.signature(mmd.DistillStep.__init__).parameters


def test_step_wrapper_lockstep_eligibility():
    """wrappers._lockstep_models (host logic): YetAnotherEfficientDet-shaped models made of this package's stack and heads,
    <= 3 frozen eval-mode teachers -> the lockstep path; anything else -> None (the reference's model-by-model order)."""
    import torch.nn as nn
    from mm_distillnet_b200 import wrappers

    class Det(nn.Module):
        features_from = "efficientnet"

        def __init__(self, ours=True):
            super().__init__()
            self.backbone_net = nn.Identity()
            self.bifpn = mmd.BiFPNStack(*[mmd.BiFPN(112, [48, 120, 352], first_time=(i == 0)) for i in range(2)])
            self.regressor = mmd.Regressor(112, 9, 3) if ours else nn.Identity()
            self.classifier = mmd.Classifier(112, 9, 20, 3)
            self.anchors = nn.Identity()

    def frozen(m):
        m.eval()
        for p in m.parameters():
            p.requires_grad_(False)
        return m

    def build(teachers, student=None):
        return wrappers.ModelWithNMSLoss(student or Det(), nn.ModuleDict(teachers), mmd.YetAnotherFocalLoss(), None, mmd.MTALoss(),
                                         {"conf_threshold": "0.3"}, {})
    ok = build({"rgb": frozen(Det()), "depth": frozen(Det())})
    models = ok._lockstep_models(None)
    assert models is not None and len(models) == 3 and models[0] is ok.student_model
    assert ok._lockstep_models(torch.zeros(1)) is None                               # the kdlist `augmentation` teacher
    ok.lockstep = False
    assert ok._lockstep_models(None) is None
    assert build({"rgb": Det().eval()})._lockstep_models(None) is None                # a teacher that still requires grad
    assert build({"rgb": frozen(Det()).train()})._lockstep_models(None) is None       # a teacher in train mode
    assert build({"rgb": frozen(Det(ours=False))})._lockstep_models(None) is None     # the reference's own PyTorch head
    assert build({m: frozen(Det()) for m in ("rgb", "depth", "thermal", "audio")})._lockstep_models(None) is None   # 4 teachers
    other = frozen(Det())
    other.features_from = "header"
    assert build({"rgb": other})._lockstep_models(None) is None
    assert build({"rgb": frozen(Det())}, student=nn.Identity())._lockstep_models(None) is None
