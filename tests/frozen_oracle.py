"""The fp64 oracle (oracle/mmd_oracle.py) with frozen BatchNorm layers: inside a training forward, the BatchNorm layers
whose prefixes are listed (e.g. "0.conv6_up.bn", "0.p3_down_channel.1", "bn_list.0.1") take the oracle's own eval branch —
running statistics, no running-statistics update — exactly what nn.BatchNorm2d in eval() does inside a train() module.

The oracle's functions call `batch_norm` through the module's globals, so each entry point here swaps in a wrapper for the
duration of the call; the oracle's arithmetic is used unchanged.  Autograd through the result gives the reference
gradients of the mixed-mode module (eval-mode BatchNorm backward for the frozen layers)."""
import contextlib

from oracle import mmd_oracle as O


@contextlib.contextmanager
def _frozen(frozen):
    frozen = frozenset(frozen)
    orig = O.batch_norm

    def batch_norm(x, p, prefix, training, stats_out=None):
        return orig(x, p, prefix, training and prefix not in frozen, stats_out)

    O.batch_norm = batch_norm
    try:
        yield
    finally:
        O.batch_norm = orig


def bifpn_stack(*args, frozen=(), **kw):
    with _frozen(frozen):
        return O.bifpn_stack(*args, **kw)


def regressor(*args, frozen=(), **kw):
    with _frozen(frozen):
        return O.regressor(*args, **kw)


def classifier(*args, frozen=(), **kw):
    with _frozen(frozen):
        return O.classifier(*args, **kw)
