"""The masked / MAE loss of the fused step without a GPU: the C-ABI fields (route independence, argument checks), the
Python option checks, the oracle's masked losses on a hand-computed batch, and the masked evaluation entry point."""
import ctypes as C
import math
import os
import re

import pytest
import torch

import parity_util  # noqa: F401  (puts the repository and the package on sys.path)

HEADER = os.path.join(parity_util.ROOT, "include", "regt_b200.h")

# (precision, H, O, B*N, T, mode, fused training step): one shape per head path of the route table
_SHAPES = [(2, 64, 16, 256, 12, 1, True),      # bf16: k_head_tc
           (1, 128, 16, 256, 12, 1, True),     # tf32x3: head_f.cu
           (1, 64, 16, 127, 12, 1, True),      # k_head_fused
           (0, 128, 12, 256, 12, 1, True),     # k_head_fwd / k_head_bwd
           (2, 64, 45, 256, 12, 1, True),
           (0, 64, 12, 256, 12, 1, False)]


def _args(case):
    from regt_b200 import _lib
    prec, H, O, BN, T, mode, step = case
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O, a.mode, a.precision, a.fuse_head = 1, BN, T, H, O, mode, prec, int(step)
    a.plan.N = BN
    a.y, a.loss, a.d_out, a.out = 0x1000, 0x2000, 0x3000, 0x4000   # never dereferenced
    return a


def _route(a):
    from regt_b200 import _lib
    o = (C.c_int32 * 4)()
    _lib.check(_lib.load().regt_debug_route(C.byref(a), o), "regt_debug_route")
    return list(o)


@pytest.mark.parametrize("case", _SHAPES)
def test_route_ignores_the_loss_fields(case, monkeypatch):
    monkeypatch.delenv("REGT_UNFUSED", raising=False)
    want = _route(_args(case))
    for kind in (0, 1):
        for masked in (0, 1):
            for count in (None, 0x5000):
                a = _args(case)
                a.loss_kind, a.loss_masked, a.loss_null, a.loss_count = kind, masked, float("nan") if masked else 0.0, count
                assert _route(a) == want, (case, kind, masked, count)


def test_zeroed_loss_fields_mean_unmasked_mse():
    from regt_b200 import _lib
    a = _lib.Args()
    assert (a.loss_kind, a.loss_masked, a.loss_null, a.loss_count) == (_lib.LOSS_MSE, 0, 0.0, None)
    # appended after F: everything before them keeps its offset
    assert _lib.Args.loss_kind.offset > _lib.Args.F.offset and _lib.Args.loss_count.offset % 8 == 0


def test_bad_loss_arguments_are_refused_on_the_host():
    from regt_b200 import _lib
    lib = _lib.load()
    a = _lib.Args()
    a.B, a.N, a.T, a.H, a.O = 1, 4, 2, 8, 1
    a.plan.N = 4
    a.loss_kind = 2
    for fn in (lib.regt_cell_forward, lib.regt_head_forward, lib.regt_head_backward, lib.regt_cell_backward):
        assert fn(C.byref(a)) != 0
        assert b"loss_kind" in lib.regt_last_error()
    a.loss_kind, a.loss_masked = _lib.LOSS_MAE, 1
    assert lib.regt_head_forward(C.byref(a)) != 0 and b"loss_masked needs y" in lib.regt_last_error()
    assert lib.regt_eval_metrics_masked(None, None, 1, 4, 95.0, 0.0, None, None) != 0
    assert b"regt_eval_metrics_masked" in lib.regt_last_error()


def test_python_rejects_unknown_loss_and_null_value():
    from models import TemporalGCN
    from regt_b200 import engine
    assert engine.check_loss("mse", None) == 0 and engine.check_loss("mae", 0.0) == 1 and engine.check_loss("mae", float("nan"))
    with pytest.raises(ValueError, match=r"\['mae', 'mse'\]"):
        engine.check_loss("huber", None)
    with pytest.raises(ValueError, match="null_value"):
        engine.check_loss("mse", "0")
    m = TemporalGCN(8, 3, 2, hidden=16)
    x, y = torch.zeros(1, 4, 8, 3), torch.zeros(1, 4, 2)
    with pytest.raises(ValueError, match="loss must be one of"):     # refused before anything touches a device
        m._fused_step(x, y, None, loss="l1")


def test_loss_counts_helper():
    from regt_b200 import engine
    y = torch.tensor([[[0.0, 1.0], [float("nan"), 2.0]], [[0.0, 0.0], [0.0, float("nan")]]])
    assert engine.loss_counts(y, 0.0).tolist() == [2.0, 0.0]
    assert engine.loss_counts(y, float("nan")).tolist() == [3.0, 3.0]


def test_oracle_masked_losses_by_hand():
    from oracle.masked_loss import masked_loss
    nan = float("nan")
    # snapshot 0: 0 and NaN missing (null 0); snapshot 1 all missing; out == y tie at [0,1,0]
    y = torch.tensor([[[0.0, 2.0], [nan, 1.0]], [[0.0, 0.0], [nan, 0.0]], [[3.0, 1.0], [4.0, 2.0]]], dtype=torch.float64)
    out = torch.tensor([[[5.0, 1.0], [7.0, 3.0]], [[1.0, 2.0], [3.0, 4.0]], [[3.0, 2.0], [1.0, 2.5]]], dtype=torch.float64,
                       requires_grad=True)
    # mse, null 0: snapshot 0 = ((1-2)^2 + (3-1)^2) / 2 = 2.5; snapshot 1 adds 0; snapshot 2 = (0 + 1 + 9 + 0.25) / 4
    mse = masked_loss(out, y, "mse", 0.0)
    assert float(mse.detach()) == pytest.approx(2.5 + 10.25 / 4, abs=1e-15)
    mse.backward()
    g = out.grad
    assert not torch.isnan(g).any()
    assert g[1].abs().max() == 0                                      # empty snapshot: no gradient
    assert g[0].tolist() == [[0.0, -1.0], [0.0, 2.0]]                 # 2 (out - y) / 2 on the valid entries
    assert g[2].tolist() == [[0.0, 0.5], [-1.5, 0.25]]
    out.grad = None
    mae = masked_loss(out, y, "mae", 0.0)
    assert float(mae.detach()) == pytest.approx((1 + 2) / 2 + (0 + 1 + 3 + 0.5) / 4, abs=1e-15)
    mae.backward()
    assert out.grad[2].tolist() == [[0.0, 0.25], [-0.25, 0.25]]       # sign(0) = 0 at the tie
    assert out.grad[0].tolist() == [[0.0, -0.5], [0.0, 0.5]]
    # NaN as the null value: zeros are valid targets, only the NaNs drop out
    nanloss = masked_loss(out.detach(), y, "mae", nan)
    assert float(nanloss) == pytest.approx((5 + 1 + 2) / 3 + (1 + 2 + 4) / 3 + 4.5 / 4, abs=1e-15)
    # no mask: a NaN propagates, and the value is the plain mean otherwise
    assert math.isnan(float(masked_loss(out.detach(), y, "mse", None)))
    assert float(masked_loss(out.detach()[2:], y[2:], "mse", None)) == pytest.approx(10.25 / 4, abs=1e-15)
    # fp32 twin: same code at the other dtype
    assert float(masked_loss(out.detach().float(), y.float(), "mse", 0.0)) == pytest.approx(float(mse.detach()), rel=1e-6)


def test_masked_eval_entry_point_is_declared_and_exported():
    from regt_b200 import _lib
    src = open(HEADER).read()
    assert re.search(r"int regt_eval_metrics_masked\(", src)
    assert "regt_eval_metrics_masked" in _lib.EXPORTS
    assert hasattr(_lib.load(), "regt_eval_metrics_masked")
    assert "#define REGT_LOSS_MSE 0" in src and "#define REGT_LOSS_MAE 1" in src
