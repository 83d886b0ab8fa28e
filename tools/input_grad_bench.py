"""Cost of the gradient wrt x (regt_cell_backward_x) on the B200.

For config 5 at B = 16 and config 2 (B = 64), with the default precision (fused tf32x3 cell):
  - the backward (head + cell) without and with the input gradient, CUDA events, L2 flushed (256 MB overwritten)
    before every timed pass, after warm-up;
  - each kernel of the input-gradient pass (regt_profile, one run of its own);
  - k_xg_contract's algorithmic bytes (valid rows of D read once + the F-wide rows written) over its time, against
    the 6 530 GB/s HBM peak measured in DESIGN section 5.
The card name and power limit are read in the same run and written beside the numbers.

    python tools/input_grad_bench.py [--out profiles/input_grad_b200.json] [--reps 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "regt-gcn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from regt_b200 import _lib, engine  # noqa: E402
from regt_b200 import workloads as W  # noqa: E402

HBM_PEAK_GBS = 6530.0
F = W.F_IN


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:     # the numbers stay usable; the missing context is stated
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def build(cfg, B):
    from models import RegionalTemporalGCN, TemporalGCN
    w = W.make_workload(cfg, B)
    if w.model == "TemporalGCN":
        m = TemporalGCN(8, w.T, w.O, hidden=w.H)
    else:
        m = RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R)
    W.init_params_synthetic(m, 1234)
    m = m.cuda()
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    g = tuple(None if t is None else t.cuda() for t in w.graph_args())
    plan = m._plan(x, g[0], g[1:]) if w.model == "RegionalTemporalGCN" else m._plan(x, g[0], g[1])
    return w, m, x, y, plan


def measure(cfg, B, reps, flush):
    w, m, x, y, plan = build(cfg, B)
    prec = m._prec(w.T)
    params = m._param_dict()
    grads = {k: torch.empty_like(t) for k, t in params.items()}
    plan.xgrad_struct()
    st = engine.build_state(m._mode, prec, plan, x, w.H, w.O, params)
    ws = st.workspace

    def fresh():
        s = engine.build_state(m._mode, prec, plan, x, w.H, w.O, params, workspace=ws)
        engine.run_forward(s, True)
        return s, (2.0 / (w.N * w.O)) * (s.out - y)

    def timed(with_x):
        s, d_out = fresh()
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        engine.run_backward(s, grads, d_out, None, False, True)
        if with_x:
            engine.run_backward_x(s)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    for with_x in (False, True):      # warm-up: module loads, the first allocation of the scratch
        timed(with_x)
    t = {False: [], True: []}
    for _ in range(reps):             # alternate, so that drift of the clock or of the neighbours hits both alike
        for with_x in (False, True):
            t[with_x].append(timed(with_x))
    # per-kernel times of the input-gradient pass (profiled run of its own)
    s, d_out = fresh()
    engine.run_backward(s, grads, d_out, None, False, True)
    flush.zero_()
    torch.cuda.synchronize()
    lib = _lib.load()
    lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
    try:
        engine.run_backward_x(s)
        torch.cuda.synchronize()
        kern = _lib.profile_read()
    finally:
        lib.regt_profile(0, None)
    rows = B * w.N * w.T
    nseg = plan.nseg
    contract_bytes = rows * 4 * w.H * 4 + B * (2 * w.N + nseg) * w.T * F * 4
    t_contract = sum(ms for n, ms in kern if n == "k_xg_contract")
    med0, med1 = statistics.median(t[False]), statistics.median(t[True])
    return dict(
        workload=w.name, B=B, precision={v: k for k, v in _lib.PRECISIONS.items()}[prec], reps=reps,
        backward_ms=dict(without_x_grad=med0, with_x_grad=med1, added=med1 - med0, runs_without=t[False], runs_with=t[True]),
        input_grad_kernels_ms=[[n, ms] for n, ms in kern],
        contraction=dict(algorithmic_bytes=contract_bytes, ms=t_contract,
                         gb_per_s=contract_bytes / (t_contract * 1e-3) / 1e9 if t_contract else None,
                         share_of_hbm_peak=(contract_bytes / (t_contract * 1e-3) / 1e9) / HBM_PEAK_GBS if t_contract else None,
                         hbm_peak_gbs=HBM_PEAK_GBS),
    )


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "input_grad_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU: it needs one"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = dict(card=card(), l2_flush_bytes=flush.numel(), timing="CUDA events around the backward, median of --reps",
               results=[measure("5", 16, args.reps, flush), measure("2", 64, args.reps, flush)])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in res["results"]:
        b = r["backward_ms"]
        print(f"{r['workload']} B={r['B']} [{r['precision']}]: backward {b['without_x_grad']:.2f} ms -> {b['with_x_grad']:.2f} ms "
              f"(+{b['added']:.2f}); contraction {r['contraction']['ms']:.3f} ms, "
              f"{(r['contraction']['gb_per_s'] or 0):.0f} GB/s; kernels {r['input_grad_kernels_ms']}")
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
