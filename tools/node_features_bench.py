"""Training-step time against the number of node features F on the B200.

For F in {1, 2, 4, 8} at three shapes -- config 2 (B = 64) and config 5 (B = 16, one micro-batch) on the fused tf32x3
cell, config 3 (B = 128, H = 256) on the unfused tf32x3 cell -- as bench.py times it: fused_step captured in a CUDA
graph, L2 flushed (256 MB overwritten) before every timed replay, CUDA events around the replay.  One model at a time,
F = 8 first and again last, so the spread of repeated F = 8 runs (drift during the call included) is measured in the same
call.  Per-kernel times come from regt_profile in an eager step of their own.
Conditions recorded: the F = 2 step is no slower than the F = 8 step beyond that spread; on the unfused path k_widen_x
costs under 1 % of the step.  The card name and power limit are read in the same run and written beside the numbers.

    python tools/node_features_bench.py [--out profiles/node_features_b200.json] [--reps 7]
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

FS = (1, 2, 4, 8)
SHAPES = (("2", 64, "fused tf32x3"), ("5", 16, "fused tf32x3"), ("3", 128, "unfused tf32x3"))


class Runner:
    """one model at F features, its fused_step captured in a CUDA graph."""

    def __init__(self, cfg, B, F):
        from models import RegionalTemporalGCN, TemporalGCN
        w = W.make_workload(cfg, B)
        w.F = F
        if w.model == "TemporalGCN":
            m = TemporalGCN(F, w.T, w.O, hidden=w.H)
        else:
            m = RegionalTemporalGCN(F, w.N, w.T, w.O, hidden=w.H, n_regions=w.R)
        W.init_params_synthetic(m, 1234)
        self.w, self.m = w, m.cuda()
        x, y = w.inputs(B)
        self.x, self.y = x.cuda(), y.cuda()
        self.g = tuple(None if t is None else t.cuda() for t in w.graph_args())
        self.step()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.step()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.step()
        torch.cuda.synchronize()

    def step(self):
        for p in self.m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        return self.m.fused_step(self.x, self.y, *self.g, micro_batch=self.w.B)

    def timed(self, flush):
        for p in self.m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        self.graph.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def kernels(self):
        lib = _lib.load()
        torch.cuda.synchronize()
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
        try:
            self.step()
            torch.cuda.synchronize()
            kern = _lib.profile_read()
        finally:
            lib.regt_profile(0, None)
        out = {}
        for n, ms in kern:
            if not n.startswith("<"):
                out[n] = out.get(n, 0.0) + ms
        return out


def measure(cfg, B, path, reps, flush):
    # one model at a time (config 5's saved planes at B = 16 take tens of GB), F = 8 first and last: the spread of its two
    # blocks of runs includes whatever drifts during the call
    order = (8,) + tuple(F for F in FS if F != 8) + (8,)
    t, kern = {}, {}
    for i, F in enumerate(order):
        r = Runner(cfg, B, F)
        name = r.w.name
        r.timed(flush)
        t.setdefault(F, []).extend(r.timed(flush) for _ in range(reps))
        if i < len(order) - 1:
            kern[F] = r.kernels()
        del r
        torch.cuda.empty_cache()
    med = {str(k): statistics.median(v) for k, v in t.items()}
    spread = max(t[8]) - min(t[8])
    res = dict(workload=name, B=B, path=path, reps=reps, step_ms_median=med, step_ms_runs={str(k): v for k, v in t.items()},
               f8_spread_ms=spread, kernels_ms={str(k): v for k, v in kern.items()},
               feat_tc_ms={str(k): kern[k].get("k_feat_tc") for k in FS})
    res["f2_no_slower_than_f8"] = med["2"] <= med["8"] + spread
    if "k_widen_x" in kern[2]:
        res["widen_x_share_of_step_f2"] = kern[2]["k_widen_x"] / sum(kern[2].values())
        res["widen_x_under_1pct"] = res["widen_x_share_of_step_f2"] < 0.01
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "node_features_b200.json"))
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU: it needs one"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = dict(card=card(), l2_flush_bytes=flush.numel(),
               timing="CUDA events around one CUDA-graph replay of fused_step, L2 flushed before each, median of --reps",
               results=[measure(cfg, B, path, args.reps, flush) for cfg, B, path in SHAPES])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in res["results"]:
        steps = " ".join(f"F={k}: {v:.2f}" for k, v in r["step_ms_median"].items())
        feat = " ".join(f"F={k}: {v:.3f}" for k, v in r["feat_tc_ms"].items() if v is not None)
        print(f"{r['workload']} B={r['B']} [{r['path']}] step ms {steps} (F=8 spread {r['f8_spread_ms']:.2f}); "
              f"k_feat_tc ms {feat}; F=2 no slower: {r['f2_no_slower_than_f8']}; "
              f"k_widen_x share: {r.get('widen_x_share_of_step_f2')}")
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
