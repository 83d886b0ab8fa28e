"""Tensor-core (tcgen05) precision modes of the cell against the fp64 oracle.
tf32x3 (generic 3xTF32 GEMM path, any hidden % 32 == 0): fp32-equivalent accuracy (1e-5 normwise); bf16 (fused H=64 kernels): stated tolerance 2e-2 activations / loss,
5e-2 gradients (bf16 operands have an 8-bit mantissa; accumulation is fp32).
Every bf16 case here has one work item per CTA, one period per item and at most 12 outputs; test_gpu_bf16_edges.py
covers the rest: several items and head tiles per CTA, 1 < tp < T, the bench's shape and graph replay, every head
kernel, the autograd surface, 1 to 64 periods, many regions and one."""
import pytest
import torch

from parity_util import W, attention_limit, build_cuda, is_dead, oracle_step, relerr, to_dev

pytestmark = pytest.mark.gpu
TOL = {"tf32x3": (1e-5, 1e-5), "bf16": (2e-2, 5e-2)}


def _cases():
    return [
        (W.tiny_workload("TemporalGCN", N=150, T=12, H=64, O=12, R=0, B=1, seed=24, k_intra=5), 1),
        (W.tiny_workload("TemporalGCN", N=19, T=3, H=64, O=2, R=0, B=2, seed=21, adversarial=True), 2),
        (W.tiny_workload("RegionalTemporalGCN", N=70, T=5, H=64, O=1, R=5, B=3, seed=23, k_intra=4), 3),
        (W.tiny_workload("RegionalTemporalGCN", N=23, T=4, H=64, O=3, R=3, B=2, seed=22, adversarial=True), 2),
        (W.make_workload(2), 3),
    ]


@pytest.mark.parametrize("precision", ["tf32x3", "bf16"])
@pytest.mark.parametrize("w,B", _cases(), ids=lambda v: v.name if hasattr(v, "name") else str(v))
def test_tc_forward_matches_oracle(w, B, precision):
    ref = oracle_step(w, B)
    m = build_cuda(w, ref["state"], precision=precision)
    x, _ = w.inputs(B)
    with torch.no_grad():
        out, hid = m(x.cuda(), *to_dev(w.graph_args(), "cuda"))
    tol = TOL[precision][0]
    assert relerr(hid, ref["hid"]) <= tol, f"out_hidden {relerr(hid, ref['hid']):.3e}"
    assert relerr(out, ref["out"]) <= tol, f"out {relerr(out, ref['out']):.3e}"


@pytest.mark.parametrize("w,B", _cases(), ids=lambda v: v.name if hasattr(v, "name") else str(v))
def test_bf16_fused_step_matches_oracle(w, B):
    """forward + loss + backward with the tcgen05 bf16 kernels (all weight gradients on tensor cores)."""
    ref = oracle_step(w, B)
    m = build_cuda(w, ref["state"], precision="bf16")
    x, y = w.inputs(B)
    loss, out, hid = m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"))
    atol, gtol = TOL["bf16"]
    assert relerr(hid, ref["hid"]) <= atol and relerr(out, ref["out"]) <= atol
    assert abs(float(loss) - ref["loss"]) <= atol * abs(ref["loss"])
    worst = {}
    for k, g in ref["grads"].items():
        if is_dead(w.model, k):
            continue
        worst[k] = relerr(m.get_parameter(k).grad, g)
    # the attention gradient is a difference of nearly equal dot products <G, H'_t>: cancellation
    # amplifies the bf16 rounding of the saved planes, so it gets a looser (stated) bound
    bad = {k: v for k, v in worst.items() if v > (0.15 if k.endswith("_attention") else gtol)}
    assert not bad, f"gradient errors above {gtol}: {bad}"


def _tf32_cases():
    return [
        (W.tiny_workload("TemporalGCN", N=19, T=3, H=32, O=2, R=0, B=2, seed=21, adversarial=True), 2),
        (W.tiny_workload("RegionalTemporalGCN", N=23, T=4, H=32, O=3, R=3, B=2, seed=22, adversarial=True), 2),
        (W.tiny_workload("RegionalTemporalGCN", N=70, T=5, H=64, O=1, R=5, B=3, seed=23, k_intra=4), 3),
        (W.tiny_workload("RegionalTemporalGCN", N=300, T=6, H=128, O=12, R=7, B=2, seed=25, k_intra=4), 2),
        (W.make_workload(1), 1),      # TPIMS, reference defaults H=256 R=5
        (W.make_workload(2), 3),      # METR-LA shape
        (W.make_workload(3), 1),      # PEMS-BAY shape, H=256 R=12
    ]


@pytest.mark.parametrize("w,B", _tf32_cases(), ids=lambda v: v.name if hasattr(v, "name") else str(v))
def test_tf32x3_fused_step_matches_oracle(w, B):
    """precision tf32x3: every H x H contraction (forward, data gradients, weight gradients) on the tensor
    cores as three tf32 products -- fp32-equivalent accuracy, so the fp32 tolerance (1e-5) applies."""
    ref = oracle_step(w, B)
    m = build_cuda(w, ref["state"], precision="tf32x3")
    x, y = w.inputs(B)
    loss, out, hid = m.fused_step(x.cuda(), y.cuda(), *to_dev(w.graph_args(), "cuda"))
    assert relerr(hid, ref["hid"]) <= 1e-5 and relerr(out, ref["out"]) <= 1e-5
    assert abs(float(loss) - ref["loss"]) <= 1e-5 * abs(ref["loss"])
    # the attention gradient is a difference of nearly equal dot products <G, H'_t>: SURVEY 8(c)'s rule -- 1e-5, or within
    # 4x of the error the fp32 twin of the oracle (the reference's own arithmetic) makes on the same inputs
    att_lim, twin_err = attention_limit(w, B, ref)
    for k, g in ref["grads"].items():
        if not is_dead(w.model, k):
            e = relerr(m.get_parameter(k).grad, g)
            if k.endswith("_attention"):
                print(f"{w.name}: d_attention err {e:.3e}, fp32 twin {twin_err:.3e}, limit {att_lim:.3e}")
            assert e <= (att_lim if k.endswith("_attention") else 1e-5), f"grad {k}: {e:.3e}"


def test_tf32x3_autograd_path_and_unsupported_width():
    w = W.tiny_workload("RegionalTemporalGCN", N=70, T=5, H=64, O=1, R=5, B=3, seed=23, k_intra=4)
    ref = oracle_step(w, 3)
    m = build_cuda(w, ref["state"], precision="tf32x3")
    x, y = w.inputs(3)
    out, hid = m(x.cuda(), *to_dev(w.graph_args(), "cuda"))
    ((out - y.cuda()) ** 2).mean(dim=(1, 2)).sum().backward()
    att_lim, _ = attention_limit(w, 3, ref)
    for k, g in ref["grads"].items():
        if not is_dead(w.model, k):
            assert relerr(m.get_parameter(k).grad, g) <= (att_lim if k.endswith("_attention") else 1e-5), k
    w2 = W.tiny_workload("TemporalGCN", N=30, T=3, H=72, O=2, R=0, B=1, seed=3)
    m2 = build_cuda(w2, oracle_step(w2, 1)["state"], precision="tf32x3")
    x2, _ = w2.inputs(1)
    with pytest.raises(RuntimeError, match="hidden % 32"):
        m2(x2.cuda(), *to_dev(w2.graph_args(), "cuda"))
