"""shared helpers of the parity tests: run the oracle and the CUDA path on the same seeded inputs."""
import copy
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "regt-gcn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from regt_b200 import workloads as W  # noqa: E402

DEAD = ("_weight_att1", "_weight_att2", "_bias_att1", "_bias_att2", "tgnn.linear.weight", "tgnn.linear.bias")


def is_dead(model_name: str, key: str) -> bool:
    leaf = key.split(".")[-1]
    if leaf in DEAD[:4]:
        return True
    # A3TGCN.linear = Linear(64,H) is dead in TemporalGCN (models/TemporalGCN.py:70)
    return model_name == "TemporalGCN" and key.startswith("tgnn.linear.")


def profiled(fn):
    """run ``fn`` with the library's launch recorder on; returns (fn's result, names of the kernels it launched)."""
    from regt_b200 import _lib
    lib = _lib.load()
    torch.cuda.synchronize()
    lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
    try:
        res = fn()
        torch.cuda.synchronize()
        names = {n for n, _ in _lib.profile_read()}
    finally:
        lib.regt_profile(0, None)
    return res, names


def build_oracle(w, dtype=torch.float64, seed=1234):
    from oracle import regt_oracle as O
    torch.manual_seed(0)
    if w.model == "TemporalGCN":
        m = O.TemporalGCN(8, w.T, w.O, hidden=w.H)
    else:
        m = O.RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R)
    W.init_params_synthetic(m, seed)
    return m.to(dtype)


def build_cuda(w, state_dict, device="cuda", precision="fp32"):
    from models import RegionalTemporalGCN, TemporalGCN
    if w.model == "TemporalGCN":
        m = TemporalGCN(8, w.T, w.O, hidden=w.H, precision=precision)
    else:
        m = RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R, precision=precision)
    m.load_state_dict({k: v.float() for k, v in state_dict.items()}, strict=True)
    return m.to(device)


def oracle_step(w, B, dtype=torch.float64, seed=1234):
    """returns dict(out, hid, loss, grads{key: tensor}) from the CPU oracle."""
    from oracle import regt_oracle as O
    m = build_oracle(w, dtype, seed)
    x, y = w.inputs(B)
    out, hid, loss = O.batched_step(m, x.to(dtype), y.to(dtype), w.graph_args())
    grads = {k: (p.grad.detach().clone() if p.grad is not None else None) for k, p in m.named_parameters()}
    return dict(out=out, hid=hid, loss=loss, grads=grads, state=copy.deepcopy(m.state_dict()))


def shipped_checkpoint_state(fname, seed=0):
    """a state_dict with the tensor names, shapes and dtype of the upstream project's checkpoint ``fname``
    (pretrained/occrate/RegionalTemporalGCN/, 3 MB each, not redistributed here), filled with seeded values.  The layout is
    stored in tests/golden/shipped_checkpoints.json: it is the one the three files were loaded with, strict, into the
    oracle while they were at hand (26 float32 tensors, 766 577 parameters in model_in6_out1_epoch50.pt)."""
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "shipped_checkpoints.json")) as f:
        spec = json.load(f)[fname]
    g = torch.Generator().manual_seed(seed)
    dtype = getattr(torch, spec["dtype"])
    return spec, {k: torch.rand(s, generator=g, dtype=dtype) - 0.5 for k, s in spec["shapes"].items()}


def to_dev(args, device):
    return tuple(None if a is None else a.to(device) for a in args)


def relerr(a: torch.Tensor, ref: torch.Tensor) -> float:
    """normwise: max|a-ref| / max|ref| (SURVEY 8(c))."""
    a = a.detach().double().cpu()
    ref = ref.detach().double().cpu()
    den = float(ref.abs().max())
    num = float((a - ref).abs().max())
    if den == 0.0:
        return num
    return num / den


def attention_limit(w, B, ref, tol=1e-5, seed=1234):
    """bound for the period-attention gradient (SURVEY 8(c)): <= tol, or within 4x of the fp32 twin's own error.
    d_attention is a softmax-Jacobian difference of nearly equal dot products <G, H'_t>; the reference's own fp32
    arithmetic (restated by the fp32 twin of the oracle) loses the same digits -- 1.6e-5 at config 4."""
    twin = oracle_step(w, B, dtype=torch.float32, seed=seed)
    att = [k for k in ref["grads"] if k.endswith("_attention")]
    if not att:
        return tol, 0.0
    e = relerr(twin["grads"][att[0]], ref["grads"][att[0]])
    return max(tol, 4.0 * e), e


def twin_limits(w, B, ref, tol=1e-5, seed=1234):
    """per-gradient bound of SURVEY 8(c): tol, or 4x the fp32 twin's own error where that is larger.  The twin restates the
    reference's fp32 arithmetic; where IT deviates from the fp64 master by more than tol (a ReLU / leaky_relu unit whose
    pre-activation rounds to the other side of zero changes every upstream gradient by a discrete amount -- seen at
    R = 256, T = 2), no fp32 implementation can be asked for more."""
    twin = oracle_step(w, B, dtype=torch.float32, seed=seed)
    errs = {k: relerr(twin["grads"][k], g) for k, g in ref["grads"].items() if g is not None and twin["grads"][k] is not None}
    return {k: max(tol, 4.0 * e) for k, e in errs.items()}, errs
