"""Training-step time of precision bf16 at the widths the fused bf16 cell does not cover, against tf32x3, on the B200.

Config 3 (B = 128, H = 256: both precisions on the GEMM-by-GEMM cell of cell_g.cu, 3xTF32 or single-pass bf16 GEMMs) and
config 5 (B = 64 in micro-batches of 16 as bench.py runs it, H = 128: bf16 on the GEMM-by-GEMM cell against the fused
tf32x3 cell of cell_f.cu).  One model per config whose ``precision`` switches between the two from step to step, so both
share its graph plan and workspace and the runs alternate in one call.  Step time: CUDA events around one eager
fused_step, with the L2 flushed (256 MB overwritten) before every timed step; median and spread of --reps per precision.
Per-kernel times from regt_profile in a step of their own.  The card name and power limit are read in the same run.

    python tools/bf16_widths_bench.py [--out profiles/bf16_widths_b200.json] [--reps 5]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "regt-gcn_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from input_grad_bench import card  # noqa: E402
from regt_b200 import _lib  # noqa: E402
from regt_b200 import workloads as W  # noqa: E402

SHAPES = (("3", 128, 128), ("5", 64, 16))   # (config, batch, micro-batch)
PRECISIONS = ("tf32x3", "bf16")


class Runner:
    def __init__(self, cfg, B, mb):
        from models import RegionalTemporalGCN, TemporalGCN
        w = W.make_workload(cfg, B)
        if w.model == "TemporalGCN":
            m = TemporalGCN(8, w.T, w.O, hidden=w.H)
        else:
            m = RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R)
        W.init_params_synthetic(m, 1234)
        self.w, self.m, self.mb = w, m.cuda(), mb
        x, y = w.inputs(B)
        self.x, self.y = x.cuda(), y.cuda()
        self.g = tuple(None if t is None else t.cuda() for t in w.graph_args())

    def step(self, prec):
        self.m.precision = prec
        for p in self.m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        return self.m.fused_step(self.x, self.y, *self.g, micro_batch=self.mb)

    def timed(self, prec, flush):
        self.m.precision = prec
        for p in self.m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        self.m.fused_step(self.x, self.y, *self.g, micro_batch=self.mb)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def kernels(self, prec):
        lib = _lib.load()
        torch.cuda.synchronize()
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
        try:
            self.step(prec)
            torch.cuda.synchronize()
            kern = _lib.profile_read()
        finally:
            lib.regt_profile(0, None)
        out = {}
        for n, ms in kern:
            if not n.startswith("<"):
                out[n] = out.get(n, 0.0) + ms
        return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def relerr(a, ref):
    a, ref = a.double(), ref.double()
    return float((a - ref).abs().max() / ref.abs().max())


def measure(cfg, B, mb, reps, flush):
    r = Runner(cfg, B, mb)
    outs = {}
    # warm-up (workspace, plan, modules) and the outputs of one step of each; bf16 first: its workspace (fp32 planes of
    # the GEMM-by-GEMM cell) is the larger one, and the tf32x3 steps then run in it instead of holding a second one
    for prec in reversed(PRECISIONS):
        loss, out, hid = r.step(prec)
        torch.cuda.synchronize()
        outs[prec] = (float(loss), out.clone(), hid.clone())
    t = {p: [] for p in PRECISIONS}
    for _ in range(reps):
        for prec in PRECISIONS:
            t[prec].append(r.timed(prec, flush))
    kern = {p: r.kernels(p) for p in PRECISIONS}
    gemm = {p: {k: v for k, v in kern[p].items() if k.startswith(("k_gemm", "k_pack", "k_split", "k_cell"))} for p in PRECISIONS}
    res = dict(workload=r.w.name, B=B, micro_batch=mb, reps=reps,
               path={"tf32x3": "fused tf32x3 cell (cell_f.cu)" if cfg == "5" else "GEMM-by-GEMM cell, 3xTF32 GEMMs",
                     "bf16": "GEMM-by-GEMM cell, single-pass bf16 GEMMs"},
               step_ms_median={p: statistics.median(v) for p, v in t.items()},
               step_ms_spread={p: max(v) - min(v) for p, v in t.items()},
               step_ms_runs=t,
               bf16_over_tf32x3=statistics.median(t["bf16"]) / statistics.median(t["tf32x3"]),
               kernels_ms=kern, tensor_core_kernels_ms=gemm,
               bf16_vs_tf32x3_relerr=dict(loss=abs(outs["bf16"][0] - outs["tf32x3"][0]) / abs(outs["tf32x3"][0]),
                                          out=relerr(outs["bf16"][1], outs["tf32x3"][1]),
                                          out_hidden=relerr(outs["bf16"][2], outs["tf32x3"][2])))
    del r
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bf16_widths_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU: it needs one"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = dict(card=card(), l2_flush_bytes=flush.numel(),
               timing="CUDA events around one eager fused_step, L2 flushed before each, precisions alternated, median of --reps",
               results=[measure(cfg, B, mb, args.reps, flush) for cfg, B, mb in SHAPES])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in res["results"]:
        steps = " ".join(f"{p}: {v:.2f} (spread {r['step_ms_spread'][p]:.2f})" for p, v in r["step_ms_median"].items())
        print(f"{r['workload']} B={r['B']} mb={r['micro_batch']} step ms {steps}; bf16 / tf32x3 {r['bf16_over_tf32x3']:.3f}; "
              f"bf16 vs tf32x3 {r['bf16_vs_tf32x3_relerr']}")
        for p in PRECISIONS:
            print(f"  {p}: " + ", ".join(f"{k} {v:.2f}" for k, v in r["tensor_core_kernels_ms"][p].items()))
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
