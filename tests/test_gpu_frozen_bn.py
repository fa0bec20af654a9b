"""Frozen BatchNorm: BatchNorm layers in eval() inside a training BiFPN stack or detection head (Detectron's FrozenBN,
mmdet's norm_eval=True; in plain PyTorch `model.train()` then `m.eval()` for every nn.BatchNorm2d).  Each layer follows its
own `.training` flag: an eval-mode layer normalises with its running statistics, leaves running_mean / running_var /
num_batches_tracked bit-unchanged and back-propagates PyTorch's eval-mode BatchNorm (dx = gamma * invstd_r * G); gamma and
beta still get their gradients.

Every case runs the module through the public API and compares it with the fp64 oracle run with the same frozen prefixes
(tests/frozen_oracle.py) and the same forced max-pool arg-max (bifpn.debug_pool_argmax).  Bounds are
those of the all-train tests: fp32 <= 1e-4 rel-L2 for every gradient class (test_gpu_bifpn.check_fp32), bf16 <= 4e-2
per gradient class and never worse than eager PyTorch running the same algorithm in all-bf16 (test_stack_bf16 /
test_benchmarked_batch_bf16; at B = 32 the BatchNorm class gets a wider bound, see check_bf16); heads as
test_heads_vs_oracle / test_heads_bf16_vs_oracle."""
import copy

import pytest
import torch
import torch.nn as nn

import mm_distillnet_b200 as mmd
from mm_distillnet_b200.bifpn import debug_pool_argmax
from tests import frozen_oracle as FO
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
C, CC = 112, [48, 120, 352]


# ---- helpers ---------------------------------------------------------------------------------------------------------
def bn_names(mod):
    return [n for n, m in mod.named_modules() if isinstance(m, nn.BatchNorm2d)]


def pattern(mod, kind):
    """BatchNorm prefixes to freeze: every layer, only the first-cell projections, or every other node."""
    names = bn_names(mod)
    if kind == "all":
        return names
    if kind == "proj":
        return [n for n in names if n.startswith("0.p")]          # 0.p{3,4,5}_down_channel{,_2}.1, 0.p5_to_p6.1
    if kind == "alt":
        return [n for i, n in enumerate([n for n in names if n.endswith(".bn")]) if i % 2 == 0]
    raise ValueError(kind)


def set_modes(mod, frozen):
    mod.train()
    for n, m in mod.named_modules():
        if n in frozen:
            m.eval()
    return mod


def bn_state(mod):
    return {k: v.detach().clone().cpu() for k, v in mod.state_dict().items() if "running_" in k or "num_batches" in k}


def check_buffers(before, after, frozen, stats):
    """Frozen layers: bit-identical buffers.  Train layers: the oracle's running-statistics update, num_batches_tracked + 1."""
    worst = 0.0
    for k, v in after.items():
        prefix = k.rsplit(".", 1)[0]
        if prefix in frozen:
            assert torch.equal(v, before[k]), k
        elif "num_batches" in k:
            assert int(v) == int(before[k]) + 1, k
        else:
            worst = max(worst, H.max_rel(v, stats[k].detach()))
    return worst


def param_class(k, frozen):
    """As gpu_cases.param_class, plus "fbias": the conv biases in front of frozen BatchNorm layers.  In front of a
    train-mode BatchNorm their gradient is exactly zero (the all-train tests skip them); in front of a frozen one it is
    gamma * invstd_r * dL/dbeta, a sum over B*H*W positions that largely cancels, conditioned like the beta gradient."""
    if k[-3:-1] == "_w":
        return "fw"
    if k.endswith("conv.bias") and not k.startswith("header"):
        return "fbias"
    owner = k.rsplit(".", 1)[0]
    if owner in frozen or ".bn" in k or k.endswith((".1.weight", ".1.bias")) or "bn_list" in k:
        return "bn"
    return "dw" if "depthwise" in k else "proj" if ".0.conv" in k else "pw"


def grad_metrics(named_params, leaf_ref, frozen, m, prefix=""):
    """Worst rel-L2 per parameter class; all fusion weights as one vector (fwall).  A bias that feeds a train-mode
    BatchNorm has an exactly-zero true gradient and is skipped; in front of a frozen layer it is checked."""
    fw_num = fw_den = 0.0
    for k, p in named_params:
        r = leaf_ref[k].grad
        if r is None or r.norm().item() < 1e-6:
            continue
        g = p.grad.float().cpu()
        cls = param_class(k, frozen)
        if cls == "fw":
            fw_num += float((g.double() - r.double()).pow(2).sum())
            fw_den += float(r.double().pow(2).sum())
            continue
        e = H.rel_l2(g, r)
        if e >= m.get(prefix + "pgrad_" + cls, 0.0):
            m[prefix + "pgrad_" + cls] = e
            m[prefix + "worst_" + cls] = k
    if fw_den > 0.0:
        m[prefix + "pgrad_fwall"] = (fw_num / fw_den) ** 0.5


def random_stack(n_cells, gen):
    stack = mmd.BiFPNStack(*[mmd.BiFPN(C, CC, first_time=(i == 0)) for i in range(n_cells)])
    with torch.no_grad():
        for k, p in stack.named_parameters():
            if ".bn." in k or k.endswith((".1.weight", ".1.bias")):
                p.copy_(torch.rand(p.shape, generator=gen) + 0.5 if k.endswith("weight") else torch.randn(p.shape, generator=gen) * 0.1)
        for k, b in stack.named_buffers():
            if "running_var" in k:
                b.copy_(torch.rand(b.shape, generator=gen) * 1.5 + 0.5)
            elif "running_mean" in k:
                b.copy_(torch.randn(b.shape, generator=gen) * 0.2)
    return stack


def oracle_stack(params, xs, n_cells, frozen, hints, dt, gouts=None):
    p = {k: (v.to(dt) if v.is_floating_point() else v) for k, v in params.items()}
    leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v) for k, v in p.items()}
    xin = [x.detach().clone().to(dt).requires_grad_(gouts is not None) for x in xs]
    stats = {}
    out = FO.bifpn_stack(tuple(xin), leaf, n_cells, training=True, pool_hints=hints, stats_out=stats, frozen=set(frozen))
    if gouts is not None:
        sum((t.float() * g).sum() if dt == torch.bfloat16 else (t * g.to(dt)).sum() for t, g in zip(out, gouts)).backward()
    return out, xin, leaf, stats


def stack_case(n_cells, B, s3, dtype, kind, seed=0):
    """Training forward + backward of a stack with the `kind` layers frozen, against the fp64 oracle (and, in bf16, eager
    PyTorch in all-bf16 on the same inputs)."""
    gen = torch.Generator().manual_seed(seed)
    stack = random_stack(n_cells, gen)
    params = {k: v.clone() for k, v in stack.state_dict().items()}
    xs = [torch.randn(B, c, s3 >> i, s3 >> i, generator=gen).to(dtype).float() for i, c in enumerate(CC)]
    frozen = pattern(stack, kind)
    stack = set_modes(stack.to(DEV), frozen)
    before = bn_state(stack)
    xd = [x.to(DEV).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True) for x in xs]
    tr = stack(tuple(xd))
    hints = debug_pool_argmax(tr[0])
    gouts = [torch.randn(t.shape, generator=gen) for t in tr]
    sum((t.float() * g.to(DEV)).sum() for t, g in zip(tr, gouts)).backward()
    ref, xin, leaf, stats = oracle_stack(params, xs, n_cells, frozen, hints, torch.float64, gouts)
    m = {"fwd%d" % (3 + i): H.max_rel(t.detach().float().cpu(), r.detach()) for i, (t, r) in enumerate(zip(tr, ref))}
    m["grad_in"] = max(H.rel_l2(x.grad.float().cpu(), r.grad) for x, r in zip(xd, xin))
    grad_metrics(stack.named_parameters(), leaf, frozen, m)
    m["buf"] = check_buffers(before, bn_state(stack), frozen, stats)
    if dtype == torch.bfloat16:
        tb, xb, lb, _ = oracle_stack(params, xs, n_cells, frozen, hints, torch.bfloat16, gouts)
        m.update({"torch_fwd%d" % (3 + i): H.max_rel(t.detach().float(), r.detach()) for i, (t, r) in enumerate(zip(tb, ref))})
        m["torch_grad_in"] = max(H.rel_l2(x.grad.float(), r.grad) for x, r in zip(xb, xin))
        tmp = {}
        grad_metrics([(k, v) for k, v in lb.items() if torch.is_tensor(v) and v.requires_grad], leaf, frozen, tmp)
        m.update({"torch_" + k: v for k, v in tmp.items()})
    print("frozen=%s B=%d s3=%d %s:" % (kind, B, s3, dtype), m)
    return m


def check_bf16(m, B, s3):
    """The bounds of test_stack_bf16 / test_benchmarked_batch_bf16 (3 cells or fewer): per-level forward <= 4e-2 (7e-2 on a
    level whose BatchNorm sees fewer than 64 values per channel) and <= 1.25 x eager PyTorch in all-bf16; every gradient
    class <= 4e-2 and no worse than eager PyTorch; the biases in front of frozen layers (fbias) count as BatchNorm class.
    At B >= 16 the worst single gamma / beta / fbias tensor is a sum over 295k positions that nearly cancels once frozen
    layers stop centring the gradient: measured on B200 (1000 W), B = 32, 96^2, every other node frozen, 4.1e-2 .. 1.2e-1
    in three runs against 0.62 .. 0.86 for eager PyTorch in all-bf16 — up to 1.5x the 8e-2 of the all-train test.  Bound:
    1.5e-1 and at most 0.3 x eager PyTorch."""
    for lvl in range(3, 8):
        k = "fwd%d" % lvl
        bound = 4e-2 if B * (s3 >> (lvl - 3)) ** 2 >= 64 else 7e-2
        assert m[k] <= bound and m[k] <= 1.25 * m["torch_" + k], (k, m)
    for k in ["grad_in"] + [k for k in m if k.startswith("pgrad_")]:
        big = B >= 16 and k in ("pgrad_bn", "pgrad_fbias")
        assert m[k] <= (1.5e-1 if big else 4e-2) and m[k] <= (0.3 if big else 1.0) * m["torch_" + k], (k, m)


# ---- 1. fp32 against the fp64 oracle ------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["all", "proj", "alt"])
def test_stack_fp32_frozen(kind):
    m = stack_case(2, 2, 64, torch.float32, kind)
    assert max(m["fwd%d" % i] for i in range(3, 8)) <= 2e-5 and m["buf"] <= 2e-5, m
    for k, v in m.items():
        if k.startswith(("grad_in", "pgrad_")):
            assert v <= 1e-4, (k, m)
    assert {"pgrad_dw", "pgrad_pw", "pgrad_bn", "pgrad_proj", "pgrad_fwall"} <= set(m), m


# ---- 2. bf16 ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["all", "proj", "alt"])
def test_stack_bf16_frozen(kind):
    check_bf16(stack_case(3, 2, 64, torch.bfloat16, kind), 2, 64)


def test_benchmarked_shape_bf16_frozen():
    """B = 32, 96^2 P3, 2 cells (the shape bench.py times), every other node frozen."""
    check_bf16(stack_case(2, 32, 96, torch.bfloat16, "alt"), 32, 96)


# ---- 3. heads ----------------------------------------------------------------------------------------------------------
def head_case(kind, K, dtype, frozen_levels=(0, 3), s3=32, B=2, seed=3):
    from tests.test_gpu_heads import quad_gouts, rand_case
    A, L = 9, 3
    p, xs = rand_case(C, K, L, B, s3, seed)
    xs = [x.to(dtype).float() for x in xs]
    mod = mmd.Regressor(C, A, L) if kind == "reg" else mmd.Classifier(C, A, K // A, L)
    mod.load_state_dict({k: v.clone() for k, v in p.items()}, strict=True)
    frozen = [n for n in bn_names(mod) if int(n.split(".")[1]) in frozen_levels]
    mod = set_modes(mod.to(DEV), frozen)
    before = bn_state(mod)
    xd = [x.to(DEV).to(dtype).requires_grad_(True) for x in xs]
    y, a = mod(xd)
    gfn = quad_gouts(seed)

    def oracle(dt, device):
        q = {k: (v.to(device).to(dt) if v.is_floating_point() else v.to(device)) for k, v in p.items()}
        leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v) for k, v in q.items()}
        xin = [x.to(device).to(dt).requires_grad_(True) for x in xs]
        stats = {}
        if kind == "reg":
            ry, ra = FO.regressor(tuple(xin), leaf, num_layers=L, training=True, stats_out=stats, frozen=set(frozen))
        else:
            ry, ra = FO.classifier(tuple(xin), leaf, A, K // A, num_layers=L, training=True, stats_out=stats, frozen=set(frozen))
        return ry, ra, xin, leaf, stats

    ry, ra, xin, leaf, stats = oracle(torch.float64, "cpu")
    gy, ga = gfn(ry, ra)
    ((ry * gy).sum() + (ra * ga).sum()).backward()
    gy, ga = gy.float(), ga.float()
    ((y.float() * gy.to(DEV)).sum() + (a.float() * ga.to(DEV)).sum()).backward()
    m = {"fwd": max(H.max_rel(y.detach().float().cpu(), ry.detach()), H.max_rel(a.detach().float().cpu(), ra.detach())),
         "grad_in": max(H.rel_l2(x.grad.float().cpu(), r.grad) for x, r in zip(xd, xin))}
    grad_metrics(mod.named_parameters(), leaf, frozen, m)
    m["buf"] = check_buffers(before, bn_state(mod), frozen, stats)
    if dtype == torch.bfloat16:
        by, ba, bx, bl, _ = oracle(torch.bfloat16, DEV)
        ((by.float() * gy.to(DEV)).sum() + (ba.float() * ga.to(DEV)).sum()).backward()
        m["torch_fwd"] = max(H.max_rel(by.detach().float().cpu(), ry.detach()), H.max_rel(ba.detach().float().cpu(), ra.detach()))
        m["torch_grad_in"] = max(H.rel_l2(x.grad.float().cpu(), r.grad) for x, r in zip(bx, xin))
        tmp = {}
        grad_metrics([(k, v) for k, v in bl.items() if torch.is_tensor(v) and v.requires_grad], leaf, frozen, tmp)
        m.update({"torch_" + k: v for k, v in tmp.items()})
    print("head %s K=%d %s:" % (kind, K, dtype), m)
    return m


@pytest.mark.parametrize("kind,K", [("reg", 36), ("cls", 180)])
def test_heads_fp32_frozen(kind, K):
    m = head_case(kind, K, torch.float32)
    assert m["fwd"] <= 2e-5 and m["buf"] <= 2e-5, m
    assert m["grad_in"] <= 1e-4 and all(v <= 1e-4 for k, v in m.items() if k.startswith("pgrad_")), m
    assert "pgrad_bn" in m and "pgrad_pw" in m, m


@pytest.mark.parametrize("kind,K", [("reg", 36), ("cls", 180)])
def test_heads_bf16_frozen(kind, K):
    m = head_case(kind, K, torch.bfloat16, s3=64, B=4)
    assert m["fwd"] < 2e-2 and m["buf"] < 1e-3, m
    assert m["grad_in"] < 3e-2, m
    for k in [k for k in m if k.startswith("pgrad_")]:
        assert m[k] < 4e-2 and m[k] <= m["torch_" + k], (k, m)


def test_neck_and_heads_whole_student_frozen():
    """BiFPNStack -> Regressor + Classifier in train() with EVERY BatchNorm in eval(), fp32, against the oracle chain."""
    gen = torch.Generator().manual_seed(7)
    stack = random_stack(2, gen)
    reg, cls = mmd.Regressor(C, 9, 3), mmd.Classifier(C, 9, 20, 3)
    with torch.no_grad():
        for mod in (reg, cls):
            for k, b in mod.named_buffers():
                if "running_var" in k:
                    b.copy_(torch.rand(b.shape, generator=gen) + 0.5)
                elif "running_mean" in k:
                    b.copy_(torch.randn(b.shape, generator=gen) * 0.2)
    ps, pr, pc = ({k: v.clone() for k, v in m.state_dict().items()} for m in (stack, reg, cls))
    fz = [bn_names(m) for m in (stack, reg, cls)]
    mods = [set_modes(m.to(DEV), f) for m, f in zip((stack, reg, cls), fz)]
    before = [bn_state(m) for m in mods]
    xs = [torch.randn(2, c, 64 >> i, 64 >> i, generator=gen) for i, c in enumerate(CC)]
    xd = [x.to(DEV).requires_grad_(True) for x in xs]
    feats = mods[0](tuple(xd))
    ry, ra = mods[1](feats)
    cy, ca = mods[2](feats)
    outs = (ry, ra, cy, ca)
    gouts = [torch.randn(t.shape, generator=gen) for t in outs]
    sum((t * g.to(DEV)).sum() for t, g in zip(outs, gouts)).backward()

    def leaf_of(p):
        return {k: (v.double().requires_grad_(True) if v.is_floating_point() and "running" not in k else
                    (v.double() if v.is_floating_point() else v)) for k, v in p.items()}
    ls, lr, lc = leaf_of(ps), leaf_of(pr), leaf_of(pc)
    xin = [x.double().requires_grad_(True) for x in xs]
    f = FO.bifpn_stack(tuple(xin), ls, 2, training=True, frozen=set(fz[0]))
    o = FO.regressor(tuple(f), lr, training=True, frozen=set(fz[1])) + FO.classifier(tuple(f), lc, 9, 20, training=True, frozen=set(fz[2]))
    sum((t * g.double()).sum() for t, g in zip(o, gouts)).backward()
    for t, r in zip(outs, o):
        assert H.max_rel(t.detach().cpu(), r.detach()) <= 1e-4
    for x, r in zip(xd, xin):
        assert H.rel_l2(x.grad.cpu(), r.grad) <= 1e-4
    for mod, leaf, f_, b in zip(mods, (ls, lr, lc), fz, before):
        m = {}
        grad_metrics(mod.named_parameters(), leaf, f_, m)
        assert all(v <= 1e-4 for k, v in m.items() if k.startswith("pgrad_")), m
        assert check_buffers(b, bn_state(mod), f_, {}) == 0.0


# ---- 4. identity: every layer frozen == eval forward ------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_all_frozen_training_forward_equals_eval_forward(dtype):
    gen = torch.Generator().manual_seed(11)
    stack = random_stack(2, gen).to(DEV)
    xs = [torch.randn(4, c, 64 >> i, 64 >> i, generator=gen).to(DEV).to(dtype) for i, c in enumerate(CC)]
    stack.eval()
    with torch.no_grad():
        ev = stack(tuple(xs))
    set_modes(stack, bn_names(stack))
    before = bn_state(stack)
    tr = stack(tuple(x.clone().requires_grad_(True) for x in xs))
    for a, b in zip(tr, ev):
        if dtype == torch.float32:
            assert H.rel_l2(a.detach().cpu(), b.cpu()) <= 1e-6
        else:
            assert H.max_rel(a.detach().float().cpu(), b.float().cpu()) <= 2e-2
    assert check_buffers(before, bn_state(stack), set(bn_names(stack)), {}) == 0.0


# ---- 5. plan cache, lockstep, graph capture ----------------------------------------------------------------------------
def test_mode_toggle_follows_the_layer():
    """Toggling one layer between two calls gives the matching oracle result in both directions (a stale plan does not)."""
    gen = torch.Generator().manual_seed(5)
    stack = set_modes(random_stack(2, gen).to(DEV), [])
    xs = [torch.randn(2, c, 32 >> i, 32 >> i, generator=gen) for i, c in enumerate(CC)]
    layer = "1.conv4_down.bn"
    for frozen in ([], [layer], [], [layer]):
        set_modes(stack, frozen)
        params = {k: v.detach().clone().cpu() for k, v in stack.state_dict().items()}
        with torch.no_grad():
            out = stack(tuple(x.to(DEV) for x in xs))
            ref = FO.bifpn_stack(tuple(x.double() for x in xs), {k: (v.double() if v.is_floating_point() else v)
                                                                 for k, v in params.items()}, 2, training=True, frozen=set(frozen))
        for t, r in zip(out, ref):
            assert H.max_rel(t.cpu(), r) <= 1e-4, frozen


def _distill_models(B, seed):
    from tests.test_gpu_bifpn import _bench_like_models, _bf16_inputs
    student, teachers = _bench_like_models(n_cells=2, n_teachers=3)
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for k, b in student.named_buffers():
            if "running_var" in k:
                b.copy_((torch.rand(b.shape, generator=gen) + 0.5).to(DEV))
            elif "running_mean" in k:
                b.copy_((torch.randn(b.shape, generator=gen) * 0.2).to(DEV))
    set_modes(student, pattern(student, "alt") + pattern(student, "proj"))
    return student, teachers, _bf16_inputs(B, 96, seed, 4)


def test_distill_step_lockstep_and_capture_with_frozen_student():
    student, teachers, xs = _distill_models(8, 21)
    frozen = set(pattern(student, "alt") + pattern(student, "proj"))
    res = {}
    for batch in (True, False):
        s = copy.deepcopy(student)
        before = bn_state(s)
        step = mmd.DistillStep(s, teachers, batch_networks=batch)
        loss = step(tuple(xs[0]), [tuple(x) for x in xs[1:]])
        res[batch] = (loss.clone(), step.flat_grad.clone())
        check_buffers(before, bn_state(s), frozen, {k: v for k, v in bn_state(s).items()})
    assert H.max_rel(res[True][0].cpu(), res[False][0].cpu()) <= 1e-2, res
    assert H.rel_l2(res[True][1].cpu(), res[False][1].cpu()) <= 1e-2
    # a captured replay equals the eager step (no optimizer: parameters do not move; frozen buffers stay put)
    s = copy.deepcopy(student)
    step = mmd.DistillStep(s, teachers)
    eager = step(tuple(xs[0]), [tuple(x) for x in xs[1:]])
    eager, g_eager = eager.clone(), step.flat_grad.clone()
    step.capture(tuple(xs[0]), [tuple(x) for x in xs[1:]], warmup=2)
    before = bn_state(s)
    out = step.replay(tuple(xs[0]), [tuple(x) for x in xs[1:]])
    torch.cuda.synchronize()
    assert H.max_rel(out.cpu(), eager.cpu()) <= 1e-2
    assert H.rel_l2(step.flat_grad.cpu(), g_eager.cpu()) <= 1e-2
    after = bn_state(s)
    for k, v in after.items():
        if k.rsplit(".", 1)[0] in frozen:
            assert torch.equal(v, before[k]), k
