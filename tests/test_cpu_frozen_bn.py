"""CPU checks of frozen BatchNorm (BatchNorm layers in eval() inside a training module): the op-list flags, the plan key
and the MmdOp mirror.  The numerics run on the GPU (tests/test_gpu_frozen_bn.py)."""
import ctypes
import os
import re

import torch
import torch.nn as nn

import mm_distillnet_b200 as mmd
from mm_distillnet_b200 import _lib, bifpn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(2, 48, 32, 32), (2, 120, 16, 16), (2, 352, 8, 8)]


def _cells(n=2):
    torch.manual_seed(0)
    return [mmd.BiFPN(112, [48, 120, 352], first_time=(i == 0)) for i in range(n)]


def _flags(ops):
    return [o.frozen_bn for o in ops]


def test_all_train_op_lists_carry_no_frozen_flags():
    for dtype in (torch.float32, torch.bfloat16):
        plan = bifpn._Plan(_cells(), "cells", SHAPES, dtype, True, True, [True] * 3)
        assert not any(_flags(plan.fwd_ops)) and not any(_flags(plan.bwd_ops))
        ev = bifpn._Plan(_cells(), "cells", SHAPES, dtype, False, False, [False] * 3)
        assert not any(_flags(ev.fwd_ops))


def test_frozen_layers_are_flagged_on_their_producer_ops_only():
    cells = _cells()
    frozen = [cells[0].p3_down_channel[1], cells[1].conv4_down.bn]
    for dtype in (torch.float32, torch.bfloat16):
        plan = bifpn._Plan(cells, "cells", SHAPES, dtype, True, True, [True] * 3, frozen=[id(m) for m in frozen])
        ptrs = {m.weight.data_ptr() for m in frozen}
        for ops, kinds in ((plan.fwd_ops, (_lib.OP_NODE_FWD, _lib.OP_PROJ_FWD)), (plan.bwd_ops, (_lib.OP_NODE_BWD, _lib.OP_PROJ_BWD))):
            flagged = [o for o in ops if o.frozen_bn]
            assert len(flagged) == 2 and all(o.kind in kinds and o.train == 1 for o in flagged)
            assert {o.bn_w for o in flagged} == ptrs
        # an eval plan folds every BatchNorm whatever its flag: no frozen ops
        ev = bifpn._Plan(cells, "cells", SHAPES, dtype, False, False, [False] * 3, frozen=[id(m) for m in frozen])
        assert not any(_flags(ev.fwd_ops))


def test_head_tower_layers_are_flagged_headers_never():
    head = mmd.Classifier(112, 9, 20, 3)
    frozen = [head.bn_list[0][1], head.bn_list[4][2]]
    shapes = [(2, 112, 16 >> i, 16 >> i) for i in range(5)]
    plan = bifpn._Plan([head], "head", shapes, torch.float32, True, True, [True] * 5, frozen=[id(m) for m in frozen])
    flagged = [o for o in plan.fwd_ops if o.frozen_bn]
    assert len(flagged) == 2 and {o.bn_w for o in flagged} == {m.weight.data_ptr() for m in frozen}
    assert all(o.kind == _lib.OP_NODE_FWD and o.train == 1 for o in flagged)
    assert len([o for o in plan.bwd_ops if o.frozen_bn]) == 2


class _FakeCudaInput:
    """What _Runner._plan_for reads of an input tensor (the plan cache needs no device)."""
    is_cuda, requires_grad, dtype = True, False, torch.float32

    def __init__(self, shape):
        self.shape, self.device = torch.Size(shape), torch.device("cpu")

    def dim(self):
        return len(self.shape)


def test_mode_mask_is_part_of_the_plan_key():
    cells = _cells()
    stack = mmd.BiFPNStack(*cells).train()
    runner, xs = stack._runner, [_FakeCudaInput(s) for s in SHAPES]
    with torch.no_grad():
        p_train = runner._plan_for(cells, xs, True, "cells")[0]
        cells[1].conv4_down.bn.eval()
        p_frozen = runner._plan_for(cells, xs, True, "cells")[0]
        assert p_frozen is not p_train and p_frozen.frozen == {id(cells[1].conv4_down.bn)}
        assert sum(_flags(p_frozen.fwd_ops)) == 1 and not any(_flags(p_train.fwd_ops))
        cells[1].conv4_down.bn.train()
        assert runner._plan_for(cells, xs, True, "cells")[0] is p_train          # back: the matching cached plan
        cells[1].conv4_down.bn.eval()
        assert runner._plan_for(cells, xs, True, "cells")[0] is p_frozen
        # eval plans ignore the per-layer flags
        e1 = runner._plan_for(cells, xs, False, "cells")[0]
        cells[1].conv4_down.bn.train()
        assert runner._plan_for(cells, xs, False, "cells")[0] is e1 and not e1.frozen


def test_mmdop_frozen_field_is_mirrored():
    hdr = open(os.path.join(ROOT, "include", "mmd.h")).read()
    body = hdr[hdr.index("typedef struct {\n  int32_t kind;"):hdr.index("} MmdOp;")]
    assert re.search(r"int32_t frozen_bn;", body)
    names = [f[0] for f in _lib.Op._fields_]
    assert names[-2:] == ["frozen_bn", "pad2_"]
    assert _lib.Op.frozen_bn.offset == ctypes.sizeof(_lib.Op) - 8
    assert _lib.lib().mmd_sizeof_op() == ctypes.sizeof(_lib.Op)
    assert _lib.lib().mmd_version() >= 111


def test_bn_modules_of_the_key_cover_every_layer():
    """Every nn.BatchNorm2d the kernels normalise with is in the mask: 8 per cell, 6 projections in the first cell."""
    cells = _cells()
    stack = mmd.BiFPNStack(*cells)
    n = len([m for m in stack.modules() if isinstance(m, nn.BatchNorm2d)])
    assert n == 8 * 2 + 6
    plan = bifpn._Plan(cells, "cells", SHAPES, torch.float32, True, True, [True] * 3,
                       frozen=[id(m) for m in stack.modules() if isinstance(m, nn.BatchNorm2d)])
    assert sum(_flags(plan.fwd_ops)) == n and sum(_flags(plan.bwd_ops)) == n


def test_frozen_oracle_takes_the_eval_branch_for_listed_layers_only():
    """tests/frozen_oracle.py (the reference the GPU tests compare with): every layer frozen == the oracle's eval forward,
    frozen layers produce no running-statistics update, and the oracle module is left as it was."""
    from oracle import mmd_oracle as O
    from tests import frozen_oracle as FO
    torch.manual_seed(0)
    stack = mmd.BiFPNStack(*_cells(1))
    with torch.no_grad():
        for k, b in stack.named_buffers():
            if "running_var" in k:
                b.uniform_(0.5, 2.0)
            elif "running_mean" in k:
                b.normal_(0.0, 0.2)
    p = {k: (v.double() if v.is_floating_point() else v) for k, v in stack.state_dict().items()}
    xs = [torch.randn(1, c, 16 >> i, 16 >> i, dtype=torch.float64) for i, c in enumerate([48, 120, 352])]
    names = [n for n, m in stack.named_modules() if isinstance(m, nn.BatchNorm2d)]
    orig = O.batch_norm
    stats = {}
    out = FO.bifpn_stack(tuple(xs), p, 1, training=True, stats_out=stats, frozen=names)
    ev = O.bifpn_stack(tuple(xs), p, 1, training=False)
    assert O.batch_norm is orig and not stats
    assert all(torch.equal(a, b) for a, b in zip(out, ev))
    stats = {}
    FO.bifpn_stack(tuple(xs), p, 1, training=True, stats_out=stats, frozen=names[1:])
    assert {k.rsplit(".", 1)[0] for k in stats} == {names[0]}
