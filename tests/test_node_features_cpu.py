"""node_features outside 1..8 are refused where they enter: at module construction, and by the C-ABI before any CUDA call
(so these run without a GPU).  F = 0 in regt_args means the kernels' width, 8, as for callers that zero-initialise it."""
import ctypes as C

import pytest


@pytest.mark.parametrize("F", [0, 9])
def test_constructors_refuse_node_features_outside_1_to_8(F):
    from models import RegionalTemporalGCN, TemporalGCN
    from models.utils import TGCN
    for make in (lambda: RegionalTemporalGCN(F, 10, 4, 2, hidden=32), lambda: TemporalGCN(F, 4, 2, hidden=32),
                 lambda: TGCN(F, 32)):
        with pytest.raises(ValueError, match="feature width is 8"):
            make()


def test_constructors_accept_1_to_8():
    from models import TemporalGCN
    for F in range(1, 9):
        sd = TemporalGCN(F, 4, 2, hidden=32).state_dict()
        assert tuple(sd["tgnn._base_tgcn.conv_h.lin.weight"].shape) == (32, F)
        assert tuple(sd["tgnn.conv.lins.0.weight"].shape) == (32, F)


def _args(F):
    from regt_b200 import _lib
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O = 2, 10, 4, 32, 2
    a.mode, a.precision = _lib.MODE_A3TGCN, _lib.PREC_FP32
    a.plan.N, a.plan.R = 10, 1
    a.F = F
    return a


def test_abi_refuses_more_than_8_features():
    from regt_b200 import _lib
    lib = _lib.load()
    a = _args(9)
    assert lib.regt_workspace_bytes(C.byref(a)) == 0
    msg = lib.regt_last_error().decode()
    assert "F=9" in msg and "1..8" in msg, msg
    assert lib.regt_cell_forward(C.byref(a)) != 0
    msg = lib.regt_last_error().decode()
    assert "regt_cell_forward" in msg and "F=9" in msg and "1..8" in msg, msg
    a.F = -1
    assert lib.regt_workspace_bytes(C.byref(a)) == 0


def test_abi_zero_features_means_eight():
    from regt_b200 import _lib
    lib = _lib.load()
    for prec in (_lib.PREC_FP32, _lib.PREC_TF32X3, _lib.PREC_BF16):
        a0, a8 = _args(0), _args(8)
        a0.precision = a8.precision = prec
        n0 = lib.regt_workspace_bytes(C.byref(a0))
        assert n0 > 0 and n0 == lib.regt_workspace_bytes(C.byref(a8))


def test_narrow_x_widens_only_on_the_ffma_and_unfused_paths():
    """F < 8 reserves the widened copy of x [B, x_rows, 8, T] on the fp32 and unfused tf32x3 paths only."""
    from regt_b200 import _lib
    lib = _lib.load()
    for prec, H, grows in ((_lib.PREC_FP32, 32, True), (_lib.PREC_TF32X3, 96, True), (_lib.PREC_TF32X3, 64, False),
                           (_lib.PREC_BF16, 64, False)):
        a2, a8 = _args(2), _args(8)
        for a in (a2, a8):
            a.precision, a.H = prec, H
        d = lib.regt_workspace_bytes(C.byref(a2)) - lib.regt_workspace_bytes(C.byref(a8))
        assert d == (2 * 10 * 8 * 4 * 4 + 255) // 256 * 256 if grows else d == 0, (prec, H, d)
