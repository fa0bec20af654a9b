"""GPU parity cases: run the CUDA path (through the public modules -> C ABI) and the CPU oracle on the same
inputs and return error metrics.  Used by the -m gpu tests (which assert) and by tests/run_gpu_diag.py (which dumps
everything to gpurun_out/ in one pass)."""
import numpy as np
import torch

import mm_distillnet_b200 as mmd
from oracle import mmd_oracle as O
from tests import helpers as H

DEV = "cuda:0"


def build_stack(name, params, dtype=torch.float32):
    C, cc, n_cells, first, B, s3, seed = H.STACK_CASES[name]
    cells = [mmd.BiFPN(C, cc, first_time=(i == 0 and first)) for i in range(n_cells)]
    stack = mmd.BiFPNStack(*cells)
    stack.load_state_dict({k: v.clone() for k, v in params.items()}, strict=True)
    return stack.to(DEV)


def to_dev(xs, dtype=torch.float32, channels_last=False):
    out = []
    for x in xs:
        x = x.detach().to(DEV).to(dtype)
        if channels_last:
            x = x.contiguous(memory_format=torch.channels_last)
        out.append(x)
    return out


def stack_golden_case(name, dtype=torch.float32):
    """CUDA stack vs the stored outputs of the real reference (tests/golden) for one fixture."""
    C, cc, n_cells, first, B, s3, seed = H.STACK_CASES[name]
    g = H.golden(name)
    params, xs = H.stack_case_inputs(name)
    m = {}
    stack = build_stack(name, params)
    stack.eval()
    with torch.no_grad():
        ev = stack(tuple(to_dev(xs, dtype)))
    for n, t in zip(H.LEVELS, ev):
        assert tuple(t.shape) == g["eval_" + n].shape
        m["eval_" + n] = H.max_rel(t.float().cpu(), g["eval_" + n])
    stack.train()
    xd = [x.requires_grad_(True) for x in to_dev(xs, dtype)]
    tr = stack(tuple(xd))
    gouts = H.stack_case_gouts(name, [t.detach().cpu().float() for t in tr])
    loss = sum((t.float() * go.to(DEV)).sum() for t, go in zip(tr, gouts))
    loss.backward()
    for n, t in zip(H.LEVELS, tr):
        m["train_" + n] = H.max_rel(t.detach().float().cpu(), g["train_" + n])
    for i, x in enumerate(xd):
        m["grad_in%d" % i] = H.rel_l2(x.grad.float().cpu(), g["grad_in%d" % i])
    sd = stack.state_dict()
    worst_buf = 0.0
    for k, v in sd.items():
        if "running_" in k:
            worst_buf = max(worst_buf, H.max_rel(v.cpu(), g["buf_" + k]))
        elif "num_batches" in k:
            assert int(v) == int(g["buf_" + k]), k
    m["running_stats"] = worst_buf
    worst = {"dw": 0.0, "pw": 0.0, "bn": 0.0, "fw": 0.0, "proj": 0.0}
    worst_el = {}
    for k, p in stack.named_parameters():
        if k.endswith("conv.bias"):
            continue  # zero gradient in exact arithmetic (bias feeding a train-mode BatchNorm)
        s, nrm = g["pgsum_" + k]
        err = abs(p.grad.double().norm().item() - nrm) / max(nrm, 1e-6)
        cls = param_class(k)
        worst[cls] = max(worst[cls], err)
        if "pgrad_" + k in g:   # the full reference tensor: element-wise (a permuted / sign-flipped gradient fails here)
            ref = torch.from_numpy(g["pgrad_" + k])
            assert tuple(ref.shape) == tuple(p.grad.shape), k
            if ref.abs().max().item() > 1e-6:
                worst_el[cls] = max(worst_el.get(cls, 0.0), H.rel_l2(p.grad.float().cpu(), ref))
    for k, v in worst.items():
        m["pgrad_norm_" + k] = v
    for k, v in worst_el.items():
        m["pgrad_" + k] = v
    return m


def param_class(k):
    return "fw" if k[-3:-1] == "_w" else "dw" if "depthwise" in k else "pw" if "pointwise" in k else \
        "proj" if ".0.conv" in k else "bn"


def input_tile(x):
    """(TW, TH) of the tiles the backward uses at x's level: the whole sample on a run-time-geometry level."""
    return H.pick_geom(x.shape[2], x.shape[3]) or (x.shape[3], x.shape[2])


def random_stack_case(n_cells, first, B, s3, dtype=torch.float32, seed=0, channels_last=False, ref64=True,
                      fw_mode="ones", force_argmax=None, attention=True, ref32=True, tile_metrics=False, teachers=0):
    """CUDA stack vs the oracle (fp64 and fp32) on D2-shaped random data.  Returns metrics for ours and, for
    calibration, for the fp32 oracle against the fp64 oracle.
    force_argmax (default on): every oracle run takes its max-pool arg-max from the window indices the CUDA forward itself
    recorded (mm_distillnet_b200.bifpn.debug_pool_argmax -> oracle.maxpool_same(hint=...)), so a near-tie resolved
    differently by two summation orders (fp32: 1e-4 .. 1e-3 jumps of every gradient; bf16 storage: the dominant part of
    the gradient error) no longer hides the arithmetic error of the kernels.  The forward comparison of the train
    outputs uses the hinted oracle too: its values differ from the true maxima by the top-2 gap of the flipped windows
    only (~1e-7 fp32); the eval forward is always compared against the plain, unhinted oracle.
    s3: the P3 side, or (H3, W3) for a non-square pyramid (level i is (H3 >> i) x (W3 >> i)).
    ref32=False skips the fp32 oracle (its metrics are then absent).
    tile_metrics: also the worst per-tile rel-L2 of every input gradient ("tile_grad_in<i>", and the same metric of the
    comparators), tiles being the backward's tile shape of the input's level (whole samples on a run-time-geometry level).
    teachers=n: the student's train forward runs in lockstep with n frozen eval-mode teachers (forward_multi, the
    configuration of DistillStep); "teacher<k>_<level>" is each teacher's output against the fp64 eval oracle (max-rel)."""
    if force_argmax is None:
        force_argmax = True
    from mm_distillnet_b200.bifpn import debug_pool_argmax
    C, cc = 112, [48, 120, 352]
    gen = torch.Generator().manual_seed(seed)
    H3, W3 = (s3, s3) if isinstance(s3, int) else s3

    def random_stack():
        cells = [mmd.BiFPN(C, cc, first_time=(i == 0 and first), attention=attention) for i in range(n_cells)]
        stack = mmd.BiFPNStack(*cells)
        with torch.no_grad():
            for k, p in stack.named_parameters():
                if k[-3:-1] == "_w":
                    if fw_mode == "mixed":
                        p.copy_(torch.rand(p.shape, generator=gen) * 2.5 - 0.5)
                elif ".bn." in k or k.endswith(".1.weight") or k.endswith(".1.bias"):
                    if k.endswith("weight"):
                        p.copy_(torch.rand(p.shape, generator=gen) + 0.5)
                    else:
                        p.copy_(torch.randn(p.shape, generator=gen) * 0.1)
            for k, b in stack.named_buffers():
                if "running_var" in k:
                    b.copy_(torch.rand(b.shape, generator=gen) * 1.5 + 0.5)
                elif "running_mean" in k:
                    b.copy_(torch.randn(b.shape, generator=gen) * 0.2)
        return stack, {k: v.clone() for k, v in stack.state_dict().items()}

    def random_inputs():
        if first:
            xs = [torch.randn(B, c, H3 >> i, W3 >> i, generator=gen) for i, c in enumerate(cc)]
        else:
            xs = [torch.randn(B, C, max(H3 >> i, 1), max(W3 >> i, 1), generator=gen) for i in range(5)]
        if dtype != torch.float32:   # compare on identical (rounded) inputs
            xs = [x.to(dtype).float() for x in xs]
        return xs

    stack, params = random_stack()
    xs = random_inputs()
    t_stacks, t_params, t_xs = [], [], []
    for _ in range(teachers):
        t, tp = random_stack()
        t_stacks.append(t.to(DEV).eval().requires_grad_(False))   # frozen, as DistillStep's teachers
        t_params.append(tp)
        t_xs.append(random_inputs())
    stack = stack.to(DEV)
    m = {}
    # CUDA first: eval forward, then the train forward whose recorded arg-max the oracle follows; its backward runs last
    stack.eval()
    with torch.no_grad():
        ev = stack(tuple(to_dev(xs, dtype, channels_last)))
    stack.train()
    xd = [x.requires_grad_(True) for x in to_dev(xs, dtype, channels_last)]
    if teachers:
        from mm_distillnet_b200.bifpn import forward_multi
        t_xd = [tuple(to_dev(x, dtype, channels_last)) for x in t_xs]
        outs = forward_multi([(stack, tuple(xd))] + list(zip(t_stacks, t_xd)))
        tr = outs[0]
        t_ev = [[o.clone() for o in out] for out in outs[1:]]
        for k, (tp, x, out) in enumerate(zip(t_params, t_xs, t_ev)):
            with torch.no_grad():
                ref = O.bifpn_stack(tuple(v.double() for v in x), {n: (v.double() if v.is_floating_point() else v)
                                                                   for n, v in tp.items()},
                                    n_cells, first_cell_first_time=first, training=False, attention=attention)
            for n, o, r in zip(H.LEVELS, out, ref):
                m["teacher%d_%s" % (k, n)] = H.max_rel(o.float().cpu(), r)
    else:
        tr = stack(tuple(xd))
    hints = debug_pool_argmax(tr[0]) if force_argmax else None

    def oracle_run(dt, training):
        p = {k: (v.to(dt) if v.is_floating_point() else v) for k, v in params.items()}
        leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v)
                for k, v in p.items()}
        xin = [x.detach().clone().to(dt).requires_grad_(training) for x in xs]
        if training:
            out = O.bifpn_stack(tuple(xin), leaf, n_cells, first_cell_first_time=first, training=True, pool_hints=hints,
                                attention=attention)
        else:
            with torch.no_grad():
                out = O.bifpn_stack(tuple(xin), leaf, n_cells, first_cell_first_time=first, training=False, attention=attention)
        return out, xin, leaf

    gout_seed = torch.Generator().manual_seed(seed + 1)
    dt_ref = torch.float64 if ref64 else torch.float32
    ev_ref, _, _ = oracle_run(dt_ref, False)
    tr_ref, xin_ref, leaf_ref = oracle_run(dt_ref, True)
    gouts = [torch.randn(t.shape, generator=gout_seed) for t in tr_ref]
    sum((t * go.to(dt_ref)).sum() for t, go in zip(tr_ref, gouts)).backward()
    ref32 = ref32 and ref64
    if ref32:
        tr32, xin32, leaf32 = oracle_run(torch.float32, True)
        sum((t * go).sum() for t, go in zip(tr32, gouts)).backward()
    if dtype == torch.bfloat16:   # calibration: the same algorithm executed by PyTorch entirely in bf16
        trb, xinb, leafb = oracle_run(torch.bfloat16, True)
        sum((t.float() * go).sum() for t, go in zip(trb, gouts)).backward()
        for i, n in enumerate(H.LEVELS):
            m["torchbf16_train_" + n] = H.max_rel(trb[i].detach().float(), tr_ref[i].detach())
        for i in range(len(xs)):
            m["torchbf16_grad_in%d" % i] = H.rel_l2(xinb[i].grad.float(), xin_ref[i].grad)
            if tile_metrics:
                m["torchbf16_tile_grad_in%d" % i] = H.worst_tile_rel_l2(xinb[i].grad.float(), xin_ref[i].grad,
                                                                        input_tile(xs[i]))
        fwn = fwd_ = 0.0
        for k, v in leafb.items():   # the all-bf16 run's parameter gradients, worst per class (same metric as ours below)
            if not (torch.is_tensor(v) and v.requires_grad) or k.endswith("conv.bias"):
                continue
            r = leaf_ref[k].grad
            if r is None or r.abs().max().item() == 0.0:
                continue
            cls = param_class(k)
            m["torchbf16_pgrad_" + cls] = max(m.get("torchbf16_pgrad_" + cls, 0.0), H.rel_l2(v.grad.float(), r))
            if cls == "fw":
                fwn += float((v.grad.double() - r.double()).pow(2).sum())
                fwd_ += float(r.double().pow(2).sum())
        if fwd_ > 0.0:
            m["torchbf16_pgrad_fwall"] = (fwn / fwd_) ** 0.5

    for n, t, r in zip(H.LEVELS, ev, ev_ref):
        assert t.shape == r.shape
        m["eval_" + n] = H.max_rel(t.float().cpu(), r)
    sum((t.float() * go.to(DEV)).sum() for t, go in zip(tr, gouts)).backward()
    for i, (n, t, r) in enumerate(zip(H.LEVELS, tr, tr_ref)):
        m["train_" + n] = H.max_rel(t.detach().float().cpu(), r.detach())
        if ref32:
            m["ref32_train_" + n] = H.max_rel(tr32[i].detach(), r.detach())
    for i, x in enumerate(xd):
        m["grad_in%d" % i] = H.rel_l2(x.grad.float().cpu(), xin_ref[i].grad)
        if ref32:
            m["ref32_grad_in%d" % i] = H.rel_l2(xin32[i].grad, xin_ref[i].grad)
        if tile_metrics:
            m["tile_grad_in%d" % i] = H.worst_tile_rel_l2(x.grad.float().cpu(), xin_ref[i].grad, input_tile(xs[i]))
            if ref32:
                m["ref32_tile_grad_in%d" % i] = H.worst_tile_rel_l2(xin32[i].grad, xin_ref[i].grad, input_tile(xs[i]))
    worst, worst32 = {}, {}
    fw_num = fw_den = fw_num32 = 0.0
    for k, p in stack.named_parameters():
        if k.endswith("conv.bias"):
            continue
        cls = param_class(k)
        r = leaf_ref[k].grad
        if r is None:   # attention=False: the fusion weights exist (state_dict contract) but take no part in _forward (:394-442)
            assert cls == "fw" and not attention
            m["zero_grad_abs"] = max(m.get("zero_grad_abs", 0.0), 0.0 if p.grad is None else p.grad.abs().max().item())
            continue
        if r.abs().max().item() == 0.0:
            # exactly-zero true gradient (e.g. both fusion weights of a node clamped by the ReLU -> constant node):
            # nothing to be relative to; require it to stay at rounding-noise level instead
            m["zero_grad_abs"] = max(m.get("zero_grad_abs", 0.0), p.grad.abs().max().item())
            continue
        e = H.rel_l2(p.grad.cpu(), r)
        if cls == "fw":   # all fusion-weight gradients of the stack as ONE vector (see check_fp32)
            fw_num += float((p.grad.cpu().double() - r.double()).pow(2).sum())
            fw_den += float(r.double().pow(2).sum())
            if ref32:
                fw_num32 += float((leaf32[k].grad.double() - r.double()).pow(2).sum())
        if e > worst.get(cls, 0.0):
            worst[cls] = e
            m["worstname_" + cls] = "%s |g|=%.3e" % (k, r.norm().item())
        worst.setdefault(cls, 0.0)
        if ref32:
            worst32[cls] = max(worst32.get(cls, 0.0), H.rel_l2(leaf32[k].grad, r))
    for k, v in worst.items():
        m["pgrad_" + k] = v
    for k, v in worst32.items():
        m["ref32_pgrad_" + k] = v
    if fw_den > 0.0:
        m["pgrad_fwall"] = (fw_num / fw_den) ** 0.5
        if ref32:
            m["ref32_pgrad_fwall"] = (fw_num32 / fw_den) ** 0.5
    return m


def mta_golden_case(name, dtype=torch.float32, channels_last=False):
    B, C, sizes, seed = H.MTA_CASES[name]
    g = H.golden(name)
    crit = mmd.MTALoss(T="9", p="2")
    go = torch.tensor([0.005 * (i + 1) for i in range(len(sizes))], device=DEV)
    teachers = [to_dev(H.structured_features(B, C, sizes, seed + 10 * (k + 1)), dtype, channels_last) for k in range(3)]
    m = {}
    for branch, g_t in (("single", teachers[0]), ("multi", teachers)):
        g_s = [f.requires_grad_(True) for f in to_dev(H.structured_features(B, C, sizes, seed), dtype, channels_last)]
        loss = crit(g_s, g_t)
        (loss * go).sum().backward()
        m["loss_abs_" + branch] = float(np.abs(loss.detach().float().cpu().numpy() - g["loss_" + branch]).max())
        m["grad_" + branch] = max(H.rel_l2(f.grad.float().cpu(), g["grad_%s_%d" % (branch, i)]) for i, f in enumerate(g_s))
    return m


def mta_random_case(B, C, sizes, n_teachers, dtype=torch.float32, channels_last=True, seed=0, structured=True, T=9.0, p=2.0):
    """CUDA MTA vs the fp64 oracle on the same (dtype-rounded) inputs; also the fp32 oracle's own error."""
    gen = torch.Generator().manual_seed(seed)

    def feats():
        fs = []
        for s in sizes:
            f = torch.randn(B, C, s, s, generator=gen)
            if structured:
                f = f * torch.exp(1.5 * torch.randn(B, 1, s, s, generator=gen))
            fs.append(f.to(dtype).float())
        return fs

    fs = feats()
    teachers = [feats() for _ in range(n_teachers)]
    go = torch.rand(len(sizes), generator=gen) * 0.01 + 0.001
    g_t64 = [[f.double() for f in t] for t in teachers]
    g_t64 = g_t64[0] if n_teachers == 1 else g_t64
    fs64 = [f.double().requires_grad_(True) for f in fs]
    l64 = O.mta_loss(fs64, g_t64, T, p)
    (l64 * go.double()).sum().backward()
    fs32 = [f.clone().requires_grad_(True) for f in fs]
    g_t32 = teachers[0] if n_teachers == 1 else teachers
    l32 = O.mta_loss(fs32, g_t32, T, p)
    (l32 * go).sum().backward()

    crit = mmd.MTALoss(T, p)
    fd = [f.requires_grad_(True) for f in to_dev(fs, dtype, channels_last)]
    td = [to_dev(t, dtype, channels_last) for t in teachers]
    loss = crit(fd, td[0] if n_teachers == 1 else td)
    (loss * go.to(DEV)).sum().backward()
    lnn = torch.tensor([np.log(s * s) for s in sizes], dtype=torch.float64)
    m = {
        "loss_abs": float((loss.detach().double().cpu() - l64.detach()).abs().max()),
        "ref32_loss_abs": float((l32.detach().double() - l64.detach()).abs().max()),
        "loss_plus_lnN_rel": float(((loss.detach().double().cpu() - l64.detach()).abs() /
                                    (l64.detach() + lnn).abs().clamp_min(1e-12)).max()),
        "grad": max(H.rel_l2(a.grad.float().cpu(), b.grad) for a, b in zip(fd, fs64)),
        "ref32_grad": max(H.rel_l2(a.grad, b.grad) for a, b in zip(fs32, fs64)),
    }
    return m


def mta_each_case(B, C, sizes, n_teachers, dtype=torch.float32, channels_last=True, seed=0):
    """MTALoss.forward_each (n_teachers single-teacher calls sharing the student, one set of launches) vs the fp64
    oracle run as the reference's step wrapper does: criterion_kd(features_s, features_t) per teacher
    (train_methods.py:351-358), stacked, with a different upstream gradient for every (teacher, level) entry."""
    gen = torch.Generator().manual_seed(seed)

    def feats():
        return [(torch.randn(B, C, s, s, generator=gen) * torch.exp(1.5 * torch.randn(B, 1, s, s, generator=gen))).to(dtype).float()
                for s in sizes]

    fs = feats()
    teachers = [feats() for _ in range(n_teachers)]
    go = torch.rand(n_teachers, len(sizes), generator=gen) * 0.01 + 0.001
    fs64 = [f.double().requires_grad_(True) for f in fs]
    l64 = torch.stack([O.mta_loss(fs64, [f.double() for f in t]) for t in teachers])
    (l64 * go.double()).sum().backward()

    crit = mmd.MTALoss()
    fd = [f.requires_grad_(True) for f in to_dev(fs, dtype, channels_last)]
    td = [to_dev(t, dtype, channels_last) for t in teachers]
    loss = crit.forward_each(fd, td)
    (loss * go.to(DEV)).sum().backward()
    g_each = [f.grad.clone() for f in fd]
    for f in fd:
        f.grad = None
    loss_loop = torch.stack([crit(fd, t) for t in td])       # the same through n_teachers ordinary calls
    (loss_loop * go.to(DEV)).sum().backward()
    return {
        "shape_ok": tuple(loss.shape) == (n_teachers, len(sizes)),
        "loss_abs": float((loss.detach().double().cpu() - l64.detach()).abs().max()),
        "grad": max(H.rel_l2(g.float().cpu(), b.grad) for g, b in zip(g_each, fs64)),
        "loss_vs_loop": float((loss.detach() - loss_loop.detach()).abs().max()),
        "grad_vs_loop": max(H.rel_l2(g.float(), f.grad.float()) for g, f in zip(g_each, fd)),
    }
