"""Tiled BiFPN kernels where they loop and where their tile shape changes.

Every tiled node kernel launches min(resident CTAs, tiles) CTAs and walks `tile += gridDim.x`; the code that only runs from
a CTA's second tile on (part B's double-buffered ring and its parity, part A's TMEM-resident [dW|db] flushed once per CTA,
the forward's early request of the next tile's input, the projection pipeline's double-buffered accumulator) carries the
whole step at the benchmarked batch.  pick_geom() chooses one of five tile shapes per level, or the run-time-geometry
kernels.  These tests check both against the fp64 oracle, with metrics that resolve one tile:

  A  a geometry matrix of non-square pyramids (H != W) at B = 2, bf16 and fp32 storage, that reaches every tile shape and the
     run-time-geometry kernels in the forward and the backward (the CPU tests below check the coverage claim against the
     dispatch in the .cu sources);
  B  the benchmarked regime (B = 32 and 16, 96 x 96 P3, bf16): whole-tensor metrics plus the worst per-tile rel-L2 of every
     input gradient; the lockstep student + 3 frozen teachers forward (DistillStep's configuration); bit-exact batch
     invariance of the frozen forward; batch-permutation invariance of the training step, with its noise floor measured in
     the same test and a positive control (one zeroed upstream-gradient tile on a CTA's later loop iteration) that the
     metric must flag.
"""
import os
import re

import pytest
import torch

from tests import helpers as H

DEV = "cuda:0"
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "mm_distillnet_b200", "csrc")

# Part A: P3 (H, W) -> expected (TW, TH) tile of the fusion nodes at P3 .. P7 (None: run-time-geometry kernels)
GEOM_CASES = {
    (48, 80): ((16, 8), (8, 8), None, None, None),
    (80, 48): ((16, 8), (12, 8), None, None, None),
    (96, 144): ((16, 8), (12, 8), (12, 8), (6, 6), None),
    (48, 96): ((16, 8), (16, 8), (12, 6), (12, 6), None),
    (80, 80): ((16, 8), (8, 8), None, None, None),   # square: a v4 producer next to run-time-geometry consumers, both ways
}


def levels(H3, W3):
    return [(H3 >> i, W3 >> i) for i in range(5)]


# ---- CPU: the Python mirror of pick_geom and the coverage of the case table -------------------------------------------

def _parsed_dispatch(fname, ns):
    src = open(os.path.join(CSRC, fname)).read()
    body = re.search(r"static int pick_geom\(int H, int W\) \{(.*?)\n\}", src, re.S).group(1)
    rules, optin = [], []
    for line in body.splitlines():
        r = re.search(r"if \((prefer8 && )?W % (\d+) == 0 && H % (\d+) == 0\) return (\d+);", line)
        if r:
            (optin if r.group(1) else rules).append((int(r.group(2)), int(r.group(3)), int(r.group(4))))
    assert re.search(r"return -1;", body)
    cases = {int(c): (int(tw), int(th)) for c, tw, th in
             re.findall(r"case (\d): return %s::launch_geom<(\d+), (\d+)>\(" % ns, src)}
    return rules, optin, cases


@pytest.mark.parametrize("fname,ns", [("bifpn_fwd_v4.cu", "v4"), ("bifpn_bwd_v4.cu", "b4")])
def test_pick_geom_mirror_matches_the_dispatch(fname, ns):
    """helpers.pick_geom mirrors pick_geom() of the forward and of the backward: the same divisibility rules in the same
    order, and every returned code launches the kernel of that (TW, TH).  If the dispatch changes, this fails before the
    coverage claims of the geometry matrix go stale."""
    rules, optin, cases = _parsed_dispatch(fname, ns)
    assert [(tw, th) for tw, th, _ in rules] == list(H.TILE_GEOMS)
    for tw, th, code in rules:
        assert cases[code] == (tw, th), (fname, code)
    # the backward's MMD_BWD_GEOM_8x8 A/B switch (off by default) only moves levels onto the 8x8 kernel
    assert all(cases[code] == (tw, th) == (8, 8) for tw, th, code in optin)
    assert len(optin) == (1 if ns == "b4" else 0)
    for h in range(1, 100):
        for w in range(1, 100):
            hit = next(((tw, th) for tw, th, _ in rules if w % tw == 0 and h % th == 0), None)
            assert H.pick_geom(h, w) == hit


def test_geometry_cases_reach_every_tile_shape_with_h_ne_w():
    """The part-A table reaches each of the five tile shapes and the run-time-geometry kernels on a level with H != W.
    Forward and backward share the rules (without the backward's opt-in 8x8 switch), and the backward's extra conditions
    for a pooled input or consumer (exactly twice the node's size) hold on these pyramids."""
    seen = set()
    for (H3, W3), expect in GEOM_CASES.items():
        lv = levels(H3, W3)
        assert [H.pick_geom(h, w) for h, w in lv] == list(expect), (H3, W3)
        for i in range(4):   # every level halves exactly: upsampled and pooled neighbours match in both directions
            assert lv[i] == (2 * lv[i + 1][0], 2 * lv[i + 1][1]), (H3, W3, i)
        for (h, w), g in zip(lv, expect):
            if h != w:
                seen.add(g)
    assert seen == set(H.TILE_GEOMS) | {None}
    # 80 x 80: a v4 level next to a run-time-geometry level in both directions (P4 8x8 <-> P5 generic)
    sq = GEOM_CASES[(80, 80)]
    assert sq[1] is not None and sq[2] is None


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _assert_ctas_loop(B, H3, W3, n_nets=1):
    """The test's own premise: at this batch every CTA of the P3 kernels walks several tiles.  Forward: 2 x SMs CTAs shared
    between the networks of a launch; backward part A: 2 CTAs per SM on 16-wide tiles; part B: one per SM."""
    sms = _sm_count()
    tw, th = H.pick_geom(H3, W3)
    assert (tw, th) == (16, 8)
    tiles = B * (H3 // th) * (W3 // tw)
    fwd = tiles / min(tiles, (2 * sms) // n_nets)
    part_a = tiles / min(tiles, 2 * sms)
    part_b = tiles / min(tiles, sms)
    assert fwd >= 3 and part_b >= 3 and part_a >= 2, (tiles, sms, fwd, part_a, part_b)


def _check_bf16(m, n_cells, B, H3, W3):
    """The bounds of test_stack_bf16 on any pyramid: per-level forward against an absolute cap and against PyTorch's own
    all-bf16 run of the same algorithm (same forced arg-max), every gradient class too."""
    seen = set()
    for k, v in m.items():
        if k.startswith("eval_"):
            assert v <= 1e-2, (k, v)
        elif k.startswith("train_"):
            h, w = levels(H3, W3)[int(k[-1]) - 3]
            bound = 4e-2 if (n_cells <= 3 and B * h * w >= 64) else 7e-2
            assert v <= bound and v <= 1.25 * m["torchbf16_" + k], (k, v, m["torchbf16_" + k])
        elif k.startswith("grad_in") or (k.startswith("pgrad_") and k != "pgrad_fw"):
            seen.add(k)
            cap = 4e-2 if n_cells <= 3 else 7e-2
            if k == "pgrad_bn" and B >= 16:
                # the worst single BatchNorm parameter at the benchmarked batch is ill-conditioned (a sum over 32x more
                # positions that largely cancels): measured 2.2e-2 .. 5.9e-2 for ours, 0.43 .. 0.60 for PyTorch's all-bf16 run
                cap = 8e-2
            assert v <= cap and v <= 1.0 * m["torchbf16_" + k], (k, v, m["torchbf16_" + k])
    assert {"grad_in0", "grad_in1", "grad_in2", "pgrad_dw", "pgrad_pw", "pgrad_bn", "pgrad_proj", "pgrad_fwall"} <= seen


# worst per-tile rel-L2 of an input gradient: <= max(TILE_CAP, TILE_FACTOR x PyTorch's all-bf16 run on the same case).
# Measured on B200 (1000 W), forced arg-max: ours 1.4e-2 .. 1.8e-2 on every case of this file, PyTorch's all-bf16 run
# 2.4e-2 .. 3.0e-2 (ratio 0.5 .. 0.65); one wrong or missing tile reads ~1.
TILE_CAP, TILE_FACTOR = 3e-2, 1.5


def _check_tiles(m):
    for i in range(3):
        v, ref = m["tile_grad_in%d" % i], m["torchbf16_tile_grad_in%d" % i]
        assert v <= max(TILE_CAP, TILE_FACTOR * ref), ("tile_grad_in%d" % i, v, ref)


def _report(name, m):
    print(name, {k: (round(v, 6) if isinstance(v, float) else v) for k, v in sorted(m.items())})


@pytest.mark.gpu
@pytest.mark.parametrize("hw", list(GEOM_CASES), ids=["%dx%d" % k for k in GEOM_CASES])
def test_geometry_matrix_bf16(hw):
    """bf16 storage, B = 2, 2 cells (first with projections) on the part-A pyramids, forced arg-max: the bounds of
    test_stack_bf16 (absolute cap and never worse than PyTorch's all-bf16 run)."""
    from tests import gpu_cases as G
    m = G.random_stack_case(2, True, 2, hw, dtype=torch.bfloat16, tile_metrics=True)
    _report("geom_bf16_%dx%d" % hw, m)
    _check_bf16(m, 2, 2, *hw)
    _check_tiles(m)


@pytest.mark.gpu
@pytest.mark.parametrize("hw", list(GEOM_CASES), ids=["%dx%d" % k for k in GEOM_CASES])
def test_geometry_matrix_fp32(hw):
    """fp32 storage on the part-A pyramids: the bounds of test_stack_vs_oracle_fp32 (1e-4 and 3 x the fp32 oracle)."""
    from tests import gpu_cases as G
    from tests.test_gpu_bifpn import check_fp32
    m = G.random_stack_case(2, True, 2, hw, tile_metrics=True)
    _report("geom_fp32_%dx%d" % hw, m)
    check_fp32({k: v for k, v in m.items() if "tile_" not in k})
    for i in range(3):   # per tile: the same 1e-4 bar
        v, ref = m["tile_grad_in%d" % i], m["ref32_tile_grad_in%d" % i]
        assert v <= 1e-4 and v <= max(2e-5, 3.0 * ref), ("tile_grad_in%d" % i, v, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 16])
def test_benchmarked_batch_bf16(B):
    """BiFPNStack at the benchmarked batch (bench.py: B = 32, B = 16 for cfg 2), 96 x 96 P3, bf16, 2 cells, forced
    arg-max: whole-tensor metrics as test_stack_bf16, plus the worst per-tile rel-L2 of each input gradient (tiles of the
    backward's shape at the gradient's level), which one wrong 16x8 tile would push to ~1.  Measured on B200 (1000 W):
    per-tile 1.6e-2 .. 1.8e-2 (PyTorch all-bf16 2.7e-2 .. 2.9e-2), whole-tensor gradients 1.0e-2 .. 3.7e-2."""
    from tests import gpu_cases as G
    _assert_ctas_loop(B, 96, 96)
    m = G.random_stack_case(2, True, B, 96, dtype=torch.bfloat16, ref32=False, tile_metrics=True)
    _report("bench_b%d" % B, m)
    _check_bf16(m, 2, B, 96, 96)
    _check_tiles(m)


@pytest.mark.gpu
def test_lockstep_benchmarked_batch_bf16():
    """DistillStep's configuration at B = 32: forward_multi with the student in train mode and 3 frozen eval-mode teachers
    (the student gets a quarter of the forward's CTAs), then the student's backward.  Student forward and every gradient
    class against the fp64 oracle as test_benchmarked_batch_bf16; each teacher's outputs against the fp64 eval oracle.
    Measured on B200 (1000 W): per-tile 1.7e-2 (PyTorch all-bf16 3.0e-2), teachers max-rel <= 4.3e-3 per level."""
    from tests import gpu_cases as G
    _assert_ctas_loop(32, 96, 96, n_nets=4)
    m = G.random_stack_case(2, True, 32, 96, dtype=torch.bfloat16, ref32=False, tile_metrics=True, teachers=3)
    _report("lockstep_b32", m)
    _check_bf16({k: v for k, v in m.items() if not k.startswith("teacher")}, 2, 32, 96, 96)
    _check_tiles(m)
    t = {k: v for k, v in m.items() if k.startswith("teacher")}
    assert len(t) == 15 and max(t.values()) <= 1e-2, t


def _lockstep_models(B, seed):
    from tests.test_gpu_bifpn import _bench_like_models, _bf16_inputs
    student, teachers = _bench_like_models(n_cells=2, n_teachers=3)
    return student, teachers, _bf16_inputs(B, 96, seed, 4)


@pytest.mark.gpu
def test_frozen_lockstep_forward_is_batch_invariant():
    """Eval-mode networks are sample-independent and their forward deterministic: every sample of a B = 32 lockstep
    forward (student + 3 frozen teachers, 30+ tiles per CTA at P3) equals, bit for bit, the same sample run alone (B = 1)
    through the single-network entry point."""
    from mm_distillnet_b200.bifpn import forward_multi
    B = 32
    _assert_ctas_loop(B, 96, 96, n_nets=4)
    student, teachers, xs = _lockstep_models(B, 31)
    with torch.no_grad():
        outs = forward_multi([(student, tuple(xs[0]))] + [(t, tuple(x)) for t, x in zip(teachers, xs[1:])])
        outs = [[o.clone() for o in out] for out in outs[1:]]
        bad = []
        for k, (t, x, out) in enumerate(zip(teachers, xs[1:], outs)):
            for b in range(B):
                alone = t(tuple(v[b:b + 1] for v in x))
                for lvl, (u, o) in enumerate(zip(alone, out)):
                    if not torch.equal(u[0], o[b]):
                        bad.append((k, b, lvl, float((u[0].float() - o[b].float()).abs().max())))
    assert not bad, bad[:10]


# permutation invariance: worst per-tile rel-L2 of the input gradients, worst rel-L2 of the parameter gradients
IN_TILE_CAP, PGRAD_CAP = 2e-2, 3e-2


@pytest.mark.gpu
def test_training_step_is_batch_permutation_invariant():
    """Train forward (lockstep with 3 frozen teachers, B = 32) and backward on a batch, then on a permutation of it with the
    upstream gradients permuted too.  A permutation moves each sample's tiles to other CTAs and other loop iterations.
    Metrics: input gradients per tile (worst rel-L2 over the 16x8 / 12x8 tiles of each sample, after un-permuting);
    parameter gradients as the worst rel-L2 over the depthwise, pointwise, projection and BatchNorm parameters and all
    fusion weights as one vector.

    Measured on B200 (1000 W): the unpermuted batch run twice is bit-identical in the input gradients (0) and differs by
    4e-7 in the parameter gradients (fp32 atomics).  The permuted forward is bit-identical too (outputs, running
    statistics, max-pool arg-max), but the backward's per-CTA partial sums change their grouping, and the bf16 re-rounding
    of every stored backward tensor amplifies those last-bit differences: 64 - 77 % of the input-gradient elements move by
    about one bf16 ulp, uniformly over all tiles (per-tile rel-L2 4.7e-3 .. 5.2e-3), and the parameter gradients by 0.6e-2 ..
    1.8e-2.  So the check is per-tile rel-L2, not bit equality: permuted <= 2e-2 per tile (4x the measured), parameters
    <= 3e-2.
    Positive control: the permuted run again with the upstream gradient zeroed on one 16x8 tile of the P3 output of the
    sample at batch position 31, a tile index beyond every grid of the P3 kernels (a CTA's later iteration).  The per-tile
    input-gradient metric must flag it (measured 0.78).  The parameter metric does not resolve one tile at this noise
    (measured 2.6e-2 against 1.8e-2 permuted) and is reported only."""
    from mm_distillnet_b200.bifpn import debug_pool_argmax, forward_multi
    from tests.gpu_cases import param_class
    B = 32
    _assert_ctas_loop(B, 96, 96, n_nets=4)
    student, teachers, xs = _lockstep_models(B, 41)
    sd0 = {k: v.clone() for k, v in student.state_dict().items()}
    gen = torch.Generator().manual_seed(42)
    gouts = [torch.randn(B, 112, 96 >> i, 96 >> i, generator=gen).to(DEV) for i in range(5)]
    tiles = [H.pick_geom(x.shape[2], x.shape[3]) for x in xs[0]]

    def run(perm, zero_tile=None):
        student.load_state_dict(sd0)
        student.zero_grad(set_to_none=True)
        cl = torch.channels_last
        x = [v[perm].contiguous(memory_format=cl).requires_grad_(True) for v in xs[0]]
        items = [(student, tuple(x))] + [(t, tuple(v[perm].contiguous(memory_format=cl) for v in xt))
                                         for t, xt in zip(teachers, xs[1:])]
        outs = forward_multi(items)[0]
        inv = torch.argsort(perm)
        am = [{k: v[inv.cpu()] for k, v in d.items()} for d in debug_pool_argmax(outs[0])]
        g = [go[perm].clone() for go in gouts]
        if zero_tile is not None:
            b, ty, tx = zero_tile
            g[0][b, :, ty * 8:(ty + 1) * 8, tx * 16:(tx + 1) * 16] = 0.0
        sum((o.float() * gg).sum() for o, gg in zip(outs, g)).backward()
        return ([v.grad[inv].float() for v in x], {k: p.grad.clone() for k, p in student.named_parameters()
                                                   if not k.endswith("conv.bias")}, am)

    def diff(a, b):
        gin = max(H.worst_tile_rel_l2(u, v, t) for u, v, t in zip(a[0], b[0], tiles))
        cls, fw_num, fw_den = {}, 0.0, 0.0
        for k, r in b[1].items():
            c = param_class(k)
            if c == "fw":
                fw_num += float((a[1][k].double() - r.double()).pow(2).sum())
                fw_den += float(r.double().pow(2).sum())
            elif float(r.abs().max()) > 0:
                cls[c] = max(cls.get(c, 0.0), H.rel_l2(a[1][k], r))
        cls["fwall"] = (fw_num / fw_den) ** 0.5
        flips = sum(int((u[k] != v[k]).sum()) for u, v in zip(a[2], b[2]) for k in v)
        return gin, max(cls.values()), cls, flips

    ident = torch.arange(B, device=DEV)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(43)).to(DEV)
    base = run(ident)
    floor = diff(run(ident), base)
    permuted = diff(run(perm), base)
    sms = _sm_count()
    ty, tx = 1, 2
    assert (B - 1) * 72 + ty * 6 + tx >= 2 * sms                  # beyond the first iteration of every P3 grid
    ctrl = diff(run(perm, zero_tile=(B - 1, ty, tx)), base)
    for name, d in (("floor", floor), ("permuted", permuted), ("control", ctrl)):
        print("permutation %s: input tiles %.3e, parameters %.3e %r, arg-max flips %d"
              % (name, d[0], d[1], {k: float("%.3e" % v) for k, v in d[2].items()}, d[3]))
    assert floor[0] <= 0.1 * IN_TILE_CAP and floor[3] == 0 and permuted[3] == 0, (floor, permuted)
    assert permuted[0] <= IN_TILE_CAP and permuted[1] <= PGRAD_CAP, (permuted, floor)
    assert ctrl[0] > 10 * IN_TILE_CAP, (ctrl, permuted)
