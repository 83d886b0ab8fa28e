"""Epoch time with the cell shared across the sliding windows (train_epoch / evaluate with share_periods=True) against the
windowed epoch, on the B200:

  config 2's series shape (TemporalGCN, N = 207, H = 64, T = 12, O = 12, 256 windows, 64 per pass) in tf32x3 and in bf16,
  config 5's shape (RegionalTemporalGCN, 100k nodes, R = 256, H = 128, T = 12, O = 12, 256 windows) in tf32x3 (the
  windowed epoch in micro-batches of 16, as bench.py runs config 5).

64 windows per pass are asked for; a pass shrinks when its buffers do not fit beside the windowed run's cached workspace
(at config 5 it does), and the pass size that ran is recorded as windows_per_pass.

One model and one synthetic series per shape (seeded).  Epoch time: CUDA events around one train_epoch (or evaluate), the
L2 flushed (256 MB overwritten) before each; the two modes alternate in one run, median and spread of --reps.  Kernel split:
one epoch of each mode under regt_profile, every launch attributed to the entry point that issued it (cell, head, combine,
or the loop's gather / optimizer kernels).  GB/s of the combine kernels: the bytes they must move (forward (S + C) N H 4,
backward (S + C + S) N H 4) over their summed time.  Gradient difference: normwise max |g_shared - g_windowed| / max |g_windowed|
per parameter, over the accumulated gradients of one epoch from the same state.  The card name and power limit are read in
the same run.

    python tools/shared_periods_bench.py [--out profiles/shared_periods_b200.json] [--reps 5]
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
from regt_b200.loop import FlatRMSprop, SlidingWindows, evaluate, train_epoch  # noqa: E402

WINDOWS, BATCH = 256, 64
SHAPES = (("2", "tf32x3", None), ("2", "bf16", None), ("5", "tf32x3", 16))   # (config, precision, windowed micro-batch)
PHASES = {"regt_cell_forward": "cell", "regt_cell_backward": "cell", "regt_head_forward": "head", "regt_head_backward": "head",
          "regt_combine_forward": "combine", "regt_combine_backward": "combine"}


class _NoStep:
    """optimizer stand-in: the epoch's gradients stay in .grad (every timed epoch starts from the same parameters)"""

    def __init__(self, params):
        self.params = list(params)

    def zero_grad(self):
        for p in self.params:
            if p.grad is not None:
                p.grad.zero_()

    def step(self):
        pass


class Runner:
    def __init__(self, cfg, prec, mb):
        from models import RegionalTemporalGCN, TemporalGCN
        w = W.make_workload(cfg, BATCH)
        if w.model == "TemporalGCN":
            m = TemporalGCN(8, w.T, w.O, hidden=w.H, precision=prec)
        else:
            m = RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R, precision=prec)
        W.init_params_synthetic(m, 1234)
        self.w, self.m, self.mb, self.prec = w, m.cuda(), mb, prec
        g = torch.Generator().manual_seed(5)
        nd = torch.rand(w.N, 8, w.T + w.O + WINDOWS - 1, generator=g)
        self.sw = SlidingWindows(nd.cuda(), w.T, w.O)
        self.g = tuple(None if t is None else t.cuda() for t in w.graph_args())
        self.opt = _NoStep(self.m.parameters())
        FlatRMSprop(list(self.m.parameters()))       # .grad views of one flat buffer, as in run.py

    def epoch(self, share):
        return train_epoch(self.m, self.sw, self.g, self.opt, batch=BATCH, micro_batch=None if share else self.mb,
                           share_periods=share)

    def evaluate(self, share):
        return evaluate(self.m, self.sw, self.g, batch=BATCH, share_periods=share)

    def timed(self, fn, flush):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def grads(self, share):
        self.epoch(share)
        torch.cuda.synchronize()
        return {k: p.grad.detach().clone() for k, p in self.m.named_parameters() if p.grad is not None}

    def split(self, share):
        """kernel ms per phase over one epoch, attributed to the entry point that launched each kernel"""
        lib = _lib.load()
        origs = {n: getattr(lib, n) for n in PHASES}
        spans = []

        def wrap(name, fn):
            def call(*a):
                n0 = len(_lib.profile_read(1 << 16))
                rc = fn(*a)
                spans.append((n0, len(_lib.profile_read(1 << 16)), PHASES[name]))
                return rc
            return call

        torch.cuda.synchronize()
        for n, f in origs.items():
            setattr(lib, n, wrap(n, f))
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
        try:
            self.epoch(share)
            torch.cuda.synchronize()
            kern = _lib.profile_read(1 << 16)
        finally:
            lib.regt_profile(0, None)
            for n, f in origs.items():
                setattr(lib, n, f)
        phase = ["other"] * len(kern)
        for n0, n1, ph in spans:
            for i in range(n0, n1):
                phase[i] = ph
        out, comb = {}, {}
        for (name, ms), ph in zip(kern, phase):
            out[ph] = out.get(ph, 0.0) + ms
            if name.startswith("k_comb"):
                comb[name] = comb.get(name, 0.0) + ms
        return out, comb


def measure(cfg, prec, mb, reps, flush):
    r = Runner(cfg, prec, mb)
    for share in (False, True):               # warm-up: plans, workspaces, modules, every pass shape
        r.epoch(share)
        r.evaluate(share)
    torch.cuda.synchronize()
    t = {"windowed": [], "shared": []}
    e = {"windowed": [], "shared": []}
    for _ in range(reps):
        for share, k in ((False, "windowed"), (True, "shared")):
            t[k].append(r.timed(lambda: r.epoch(share), flush))
            e[k].append(r.timed(lambda: r.evaluate(share), flush))
    gw, gs = r.grads(False), r.grads(True)
    gdiff = {k: float((gs[k] - g).abs().max() / g.abs().max().clamp_min(1e-30)) for k, g in gw.items() if float(g.abs().max()) > 0}
    split = {k: r.split(s) for k, s in (("windowed", False), ("shared", True))}
    w = r.w
    C, T = r.m._shared_bufs["C"], w.T
    passes = -(-WINDOWS // C)
    S_tot, C_tot = WINDOWS + passes * (T - 1), WINDOWS                   # steps and windows over all passes of the epoch
    row = w.N * w.H * 4
    comb = split["shared"][1]
    gbs = {"k_comb_fwd": (S_tot + C_tot) * row / (comb.get("k_comb_fwd", float("nan")) * 1e-3) / 1e9,
           "k_comb_bwd": (2 * S_tot + C_tot) * row / (comb.get("k_comb_bwd", float("nan")) * 1e-3) / 1e9}
    res = dict(workload=w.name, precision=prec, windows=WINDOWS, windows_per_pass=C, windowed_micro_batch=mb, reps=reps,
               periods_per_epoch=dict(windowed=WINDOWS * T, shared=S_tot),
               train_epoch_ms_median={k: statistics.median(v) for k, v in t.items()},
               train_epoch_ms_spread={k: max(v) - min(v) for k, v in t.items()},
               train_epoch_ms_runs=t,
               evaluate_ms_median={k: statistics.median(v) for k, v in e.items()},
               evaluate_ms_spread={k: max(v) - min(v) for k, v in e.items()},
               speedup_train=statistics.median(t["windowed"]) / statistics.median(t["shared"]),
               speedup_evaluate=statistics.median(e["windowed"]) / statistics.median(e["shared"]),
               kernel_ms_by_phase={k: v[0] for k, v in split.items()},
               combine_kernel_ms=comb, combine_gb_per_s=gbs,
               grad_normwise_diff=gdiff, grad_normwise_diff_max=max(gdiff.values()))
    del r
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shared_periods_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shapes", default="0,1,2", help="indices into SHAPES")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU: it needs one"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = dict(card=card(), l2_flush_bytes=flush.numel(),
               timing="CUDA events around one train_epoch / evaluate, L2 flushed before each, modes alternated, median of --reps; "
                      "gradients accumulate over the epoch, no optimizer step",
               results=[measure(*SHAPES[int(i)], args.reps, flush) for i in args.shapes.split(",")])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in res["results"]:
        print(f"{r['workload']} {r['precision']}: train_epoch ms {r['train_epoch_ms_median']} (x{r['speedup_train']:.2f}), "
              f"evaluate ms {r['evaluate_ms_median']} (x{r['speedup_evaluate']:.2f}); phases {r['kernel_ms_by_phase']}; "
              f"combine GB/s {r['combine_gb_per_s']}; max grad diff {r['grad_normwise_diff_max']:.2e}")
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
