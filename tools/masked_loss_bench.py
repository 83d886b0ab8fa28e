"""Cost of the masked / MAE loss of the fused step on the B200: step time of the unmasked MSE (the default kernels)
against the masked MAE (the LX instantiations of the head kernels plus k_loss_count / k_loss_inv) at

  config 5 in tf32x3 (B = 64 in micro-batches of 16, as bench.py runs it; head k_hf_mid),
  config 2 in bf16   (B = 64, the k_head_tc shape),
  config 3 in tf32x3 (B = 128; head k_hf_mid).

One model per config; the two losses alternate from step to step in one call, so they share its plan and workspace.  The
masked runs zero 20 % of the targets and pass null_value=0.0.  Step time: CUDA events around one eager fused_step with the
L2 flushed (256 MB overwritten) before every timed step; median and spread of --reps per loss.  Per-kernel times (the head
kernel and k_loss_count) from regt_profile in a step of their own.  The card name and power limit are read in the same run.

    python tools/masked_loss_bench.py [--out profiles/masked_loss_b200.json] [--reps 7]
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

SHAPES = (("5", 64, 16, "tf32x3"), ("2", 64, 64, "bf16"), ("3", 128, 128, "tf32x3"))   # (config, batch, micro-batch, precision)
LOSSES = {"mse": dict(loss="mse", null_value=None), "masked_mae": dict(loss="mae", null_value=0.0)}
HEADS = ("k_head_fwd", "k_head_fused", "k_hf_mid", "k_head_tc", "k_loss_count", "k_loss_inv")


class Runner:
    def __init__(self, cfg, B, mb, prec):
        from models import RegionalTemporalGCN, TemporalGCN
        w = W.make_workload(cfg, B)
        if w.model == "TemporalGCN":
            m = TemporalGCN(8, w.T, w.O, hidden=w.H, precision=prec)
        else:
            m = RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R, precision=prec)
        W.init_params_synthetic(m, 1234)
        self.w, self.m, self.mb = w, m.cuda(), mb
        x, y = w.inputs(B)
        drop = torch.rand(y.shape, generator=torch.Generator().manual_seed(7)) < 0.2
        ym = y.clone()
        ym[drop] = 0.0
        self.x = x.cuda()
        self.y = {"mse": y.cuda(), "masked_mae": ym.cuda()}
        self.g = tuple(None if t is None else t.cuda() for t in w.graph_args())

    def step(self, kind):
        for p in self.m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        return self.m.fused_step(self.x, self.y[kind], *self.g, micro_batch=self.mb, **LOSSES[kind])

    def timed(self, kind, flush):
        for p in self.m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        self.m.fused_step(self.x, self.y[kind], *self.g, micro_batch=self.mb, **LOSSES[kind])
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def kernels(self, kind):
        lib = _lib.load()
        torch.cuda.synchronize()
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
        try:
            self.step(kind)
            torch.cuda.synchronize()
            kern = _lib.profile_read()
        finally:
            lib.regt_profile(0, None)
        out = {}
        for n, ms in kern:
            if n in HEADS:
                out[n] = out.get(n, 0.0) + ms
        return out


def measure(cfg, B, mb, prec, reps, flush):
    r = Runner(cfg, B, mb, prec)
    for kind in LOSSES:       # warm-up: workspace (the masked one is B floats larger), plan, modules
        r.step(kind)
    torch.cuda.synchronize()
    t = {k: [] for k in LOSSES}
    for _ in range(reps):
        for kind in LOSSES:
            t[kind].append(r.timed(kind, flush))
    kern = {k: r.kernels(k) for k in LOSSES}
    res = dict(workload=r.w.name, precision=prec, B=B, micro_batch=mb, reps=reps,
               step_ms_median={k: statistics.median(v) for k, v in t.items()},
               step_ms_spread={k: max(v) - min(v) for k, v in t.items()},
               step_ms_runs=t,
               masked_mae_over_mse=statistics.median(t["masked_mae"]) / statistics.median(t["mse"]),
               head_kernels_ms=kern)
    del r
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "masked_loss_b200.json"))
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU: it needs one"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = dict(card=card(), l2_flush_bytes=flush.numel(),
               timing="CUDA events around one eager fused_step, L2 flushed before each, losses alternated, median of --reps",
               results=[measure(cfg, B, mb, prec, args.reps, flush) for cfg, B, mb, prec in SHAPES])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in res["results"]:
        steps = " ".join(f"{k}: {v:.2f} (spread {r['step_ms_spread'][k]:.2f})" for k, v in r["step_ms_median"].items())
        print(f"{r['workload']} {r['precision']} B={r['B']} mb={r['micro_batch']} step ms {steps}; "
              f"masked_mae / mse {r['masked_mae_over_mse']:.3f}; kernels {r['head_kernels_ms']}")
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
