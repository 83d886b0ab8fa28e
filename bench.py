#!/usr/bin/env python
"""bench.py -- RegT-GCN hot path: fwd + loss + bwd samples/s on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # reference CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs to DIR/*.npy

One "step" = one pass of the hot path (forward + MSE loss + backward, all parameter gradients)
over one batch of B synthetic snapshots.  Default workload: BASELINE.json's headline config --
configs[4], the 100k-node / 256-region graph (SURVEY 8(d) config 5: B=64, N=100 000, R=256, H=128)
-- in fp32-equivalent arithmetic (3xTF32 on the tensor cores, 1e-5 parity with the fp64 oracle).
  * N = 1: the whole graph on one GPU, micro-batched inside the step (saved planes of the full
    batch do not fit 180 GB; samples/s is still B / t_step, SURVEY 8(d));
  * N > 1: each GPU owns a set of regions (LPT bin packing), reads its rows + 1-hop halo rows of x,
    and the job processes the SAME B snapshots (strong scaling, SURVEY 8(e)); the shared-weight
    gradients (+ the loss) are summed by one exchange kernel over NVLink peer memory inside the step;
  * workloads without regions (--workload 2) shard the batch instead (weak scaling).

Timing: CUDA events on the launching stream around every step, L2 flushed (256 MiB memset)
between timed steps, barrier + synchronize on both sides, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "regt-gcn_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

_REAL_STDOUT = None
METRIC = "regt_gcn_fwd_bwd_samples_per_s"
UNIT = "samples/s"
L2_NOTE = "flushed between timed steps (256 MiB memset) on the GPU arm; the CPU arm's working set exceeds its caches"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="5", help="SURVEY 8(d) config id (default 5 = the 100k-node region-sharded config the metric is quoted on)")
    ap.add_argument("--batch", type=int, default=None, help="override the batch B")
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32x3", "bf16"],
                    help="tf32x3 (default) = fp32-equivalent arithmetic on the tensor cores (three tf32 products per contraction, "
                         "1e-5 parity); fp32 = FFMA kernels; bf16 = bf16 operands / fp32 accumulate (stated tolerance, hidden 64 only)")
    ap.add_argument("--micro-batch", type=int, default=None)
    ap.add_argument("--shard", default="auto", choices=["auto", "region", "batch"],
                    help="N>1: 'region' = each GPU owns a set of regions (strong scaling, SURVEY 8(e)); "
                         "'batch' = each GPU runs its own per-GPU batch (weak scaling); auto = region when the workload has regions")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the step in a CUDA graph")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N > 1: the gradient all-reduce as one kernel over NVLink peer memory (csrc/peer.cu) or through NCCL; "
                         "auto = the peer kernels (NCCL only if CUDA IPC is unavailable)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the spmm / reference_call_pattern / cfg2 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (loss, out, hidden, every parameter "
                         "gradient; rank 0's) as DIR/<name>.npy, float32, at most 64 MB in all (see dump_outputs)")
    return ap.parse_args()


DUMP_BUDGET_BYTES = 60_000_000     # data of all .npy files together; their headers stay well inside 64 MB


def dump_outputs(dirname: str, arrays: dict) -> dict:
    """writes every tensor of ``arrays`` as ``dirname/<name>.npy`` in float32.  The smallest arrays are written whole; an array
    that would overrun what is left of DUMP_BUDGET_BYTES is written as a fixed sample of its flattened elements: one element
    drawn (seed 0) from each of k equal strides.  The sample depends only on the array's size, so two runs, or two builds,
    with the same arguments compare element for element.  Returns {name: (full shape, elements written)}."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    left = DUMP_BUDGET_BYTES // 4
    written = {}
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(items):
        a = t.detach()
        n = a.numel()
        k = min(n, max(1, left // (len(items) - i)))
        if k < n:
            idx = np.arange(k, dtype=np.int64) * n // k + np.random.default_rng(0).integers(0, n // k, size=k)
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(dirname, name + ".npy"), a.float().cpu().numpy())
        left -= k
        written[name] = (tuple(t.shape), k)
    return written


# ------------------------------------------------------------------------------------------------
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    source="measured (MEASURED_PEAKS.json; bf16 = the sustained figure, the kernels are timed inside a long step)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation cannot be imported (torch_geometric is absent and not
# installable offline, SURVEY 8(c)), so both `cpu_baseline` and `--impl reference` time the oracle's fp32
# port of it: per-call re-normalisation, per-sample and per-period Python loops, literal [N, R*H] concat.
# ------------------------------------------------------------------------------------------------
def cpu_sample_workload(w):
    """-> (workload the CPU can hold, factor, description).  The literal regional combine materialises [N, R*H] per period
    and keeps it for the backward: 13 GB per period at config 5, 164 MB at config 4.  Such workloads are timed on a PREFIX of
    their regions (same generator, same nodes per region, same edges per node, R' regional lists) and the measured rate is
    multiplied by N'/N -- an UPPER bound of the CPU path's rate at full size (each node of the full problem also pays R/R'
    times more in the combine GEMM)."""
    from regt_b200 import workloads as W
    lit = w.N * max(w.R, 1) * w.H * 4 * w.T * 3
    if w.R == 0 or lit <= (4 << 30):
        return w, 1.0, "the full workload graph"
    Rp = 8
    Np = int(round(w.N * Rp / w.R))
    full, rei, rea = W._regional_graph(Np, Rp, 6, max(1, Np // 10), w.seed)
    sub = W.Workload(f"{w.name}__prefix_R{Rp}_N{Np}", w.model, w.B, Np, w.T, w.H, w.O, Rp, w.seed, full, None, rei, rea)
    return sub, Np / w.N, (f"a prefix of {Rp} of the {w.R} regions ({Np} of {w.N} nodes, same generator); rate scaled by "
                           f"{Np}/{w.N} = an upper bound of the literal CPU path at full size")


def cpu_model(w):
    from oracle import regt_oracle as O
    from regt_b200 import workloads as W
    torch.manual_seed(0)
    if w.model == "TemporalGCN":
        m = O.TemporalGCN(8, w.T, w.O, hidden=w.H)
    else:
        m = O.RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R)
    W.init_params_synthetic(m, 1234)
    return m


def cpu_oracle_rate(w, seconds: float, min_samples: int = 4, warm: int = 1):
    """snapshots/s of the oracle's fp32 port on this box's host cores, one snapshot at a time (run.py:170)."""
    sub, scale, what = cpu_sample_workload(w)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    m = cpu_model(sub)
    x, y = sub.inputs(max(min_samples, 4))
    g = sub.graph_args()

    def one(b):
        out, _ = m(x[b % x.shape[0]], *g)
        loss = torch.mean((out - y[b % x.shape[0]]) ** 2)
        loss.backward()

    for b in range(warm):
        one(b)
    n, t0 = 0, time.perf_counter()
    while True:
        one(n); n += 1
        el = time.perf_counter() - t0
        if (el >= seconds and n >= min_samples) or n >= 4096:
            break
    return n / el * scale, n, el, torch.get_num_threads(), what


def bench_config(w) -> dict:
    """the workload-identifying keys: identical in both arms."""
    return dict(w.describe(), l2=L2_NOTE)


def run_reference(args):
    """--impl reference: times the oracle port of the reference's CPU path (see above) on the same config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from regt_b200 import workloads as W
    w = W.make_workload(args.workload, args.batch)
    sub, scale, what = cpu_sample_workload(w)
    per_step = 4  # snapshots per "step": a bounded sample of the workload's batch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    m = cpu_model(sub)
    x, y = sub.inputs(per_step)
    g = sub.graph_args()

    def step():
        for b in range(per_step):
            out, _ = m(x[b], *g)
            torch.mean((out - y[b]) ** 2).backward()

    for _ in range(max(1, min(args.warmup, 2))):
        step()
    ts = []
    budget_t0 = time.perf_counter()
    for _ in range(args.steps):
        t0 = time.perf_counter(); step(); ts.append(time.perf_counter() - t0)
        if time.perf_counter() - budget_t0 > 150:
            break
    ms = 1e3 * sum(ts) / len(ts)
    val = per_step / (ms / 1e3) * scale
    sample = (f"{per_step} of {w.B} snapshots per step, {len(ts)} steps, on {what}; oracle fp32 port of the reference "
              f"(torch_geometric is not installable here), one snapshot at a time as run.py:170")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(ts),
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if w.R > 0 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": bench_config(w),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
# rooflines
# ------------------------------------------------------------------------------------------------
def kernel_work(w, B: int, name: str):
    """(algorithmic bytes, fp32-equivalent flops) of ONE pass of a dominant kernel over B snapshots, under SURVEY 8(d)'s
    save-4-planes accounting (DESIGN.md section 5).  Per (b,n,t) row: the forward cell reads X_t,S_t (+U_t) and writes 4
    H-wide planes; the backward cell reads them back (and writes the 4H-wide gate gradients for the weight-gradient pass)."""
    rows = float(B) * w.N * w.T
    F, H = 8, w.H
    wts = (F + H) * 3 * H * 4
    fwd_b = rows * (2 * F * 4 + 4 * H * 4) + B * w.N * H * 4 + wts
    bwd_b = rows * (4 * H * 4) + B * w.N * H * 4 + wts
    gate_f = 2.0 * rows * 3 * (F + H) * H          # three gates, [S|h] x [F+H, H]
    dgrad_f = 2.0 * rows * 3 * H * H               # dHR, dhg (K = 2H)
    table = {
        "k_cell_fwd": (fwd_b, gate_f), "k_cell_bwd": (bwd_b, dgrad_f),
        "k_cell_fwd_tc": (fwd_b, gate_f), "k_cell_bwd_tc": (bwd_b, dgrad_f + 2.0 * rows * 3 * (F + H) * H),
        "k_cell_fwd_f": (fwd_b, gate_f), "k_cell_bwd_f": (bwd_b + rows * 4 * H * 4, dgrad_f),
        # the six H x H gate contractions of the unfused 3xTF32 path: A read once, C written once
        "k_gemm_nt_tma_ts": (rows * 4.0 * 11 * H, 2.0 * rows * H * H * 6),
        # weight-gradient row contraction: D [rows][4H] + h, hR + the 32-wide feature plane
        "k_gemm_tn_tma": (rows * 4.0 * (6 * H + 32), 2.0 * rows * (3 * H * H + 4 * H * 32)),
    }
    return table.get(name)


def pick_roofline(w, B, per_kernel, counts, step_sum, precision, pk, traffic_of):
    cand = [k for k in per_kernel if kernel_work(w, B, k) is not None]
    if not cand:
        return None
    dom = max(cand, key=lambda k: per_kernel[k])
    nbytes, flops = kernel_work(w, B, dom)
    t_all = per_kernel[dom] * 1e-3                    # all launches of this kernel in one step (micro-batches included)
    # fp32-equivalent tensor peak: tf32 runs at half the bf16 rate and the 3xTF32 split issues three products
    peak_tc = pk["bf16_tflops"] / (6.0 if precision == "tf32x3" else 1.0)
    tensor_kernel = precision in ("tf32x3", "bf16") and dom not in ("k_cell_fwd", "k_cell_bwd")
    t_hbm = nbytes / (pk["hbm_gbs"] * 1e9)
    t_tc = flops / (peak_tc * 1e12) if tensor_kernel else 0.0
    if t_hbm >= t_tc:
        ach, peak, unit, bound = nbytes / t_all / 1e9, pk["hbm_gbs"], "GB/s", "hbm"
    else:
        ach, peak, unit, bound = flops / t_all / 1e12, peak_tc, "TFLOP/s", "tensor"
    n = counts[dom]
    return {"kernel": dom, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
            "traffic": traffic_of(dom), "peak_source": pk["source"] + ("" if bound == "hbm" else
                                                                     "; fp32-equivalent = bf16 dense / 6 (tf32 = half the bf16 rate, 3 products per contraction)"),
            "alg_bytes_per_launch": nbytes / n, "alg_flops_per_launch": flops / n, "launch_ms": per_kernel[dom] / n,
            "launches_per_step": n, "t_hbm_ms_per_step": t_hbm * 1e3, "t_tensor_ms_per_step": t_tc * 1e3,
            "share_of_step": per_kernel[dom] / step_sum}


def time_events(fn, n, flush):
    ts = []
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return ts


def measure_spmm(w, dev, x_dev, graph_args, flush, pk):
    """BASELINE's second metric, "SpMM HBM GB/s vs peak": the stand-alone F-wide SpMM  S = A_hat X  over all (b, t) of the
    workload (GCNConv.propagate at models/utils.py:169,175,181; one pass feeds all three gates), through the C-ABI
    regt_spmm_f8_blocked (row blocks from regt_spmm_partition, built once per static graph and cached like the plan).  SpMMBytes = 2*B*T*N*F*4 + (N+1)*4 + (E+N)*8 (SURVEY 8(d))."""
    from regt_b200 import plan as P, workloads as W
    ei = graph_args[0]
    ew = graph_args[1] if w.model == "TemporalGCN" else None
    plan = P.get_plan(w.N, dev, ei, ew, [], [], need_cheb=False)
    B = x_dev.shape[0]
    t = plan.t
    for _ in range(3):
        y = P.spmm_f8(t["g_rowptr"], t["g_col"], t["g_val"], x_dev)
    ts = time_events(lambda: P.spmm_f8(t["g_rowptr"], t["g_col"], t["g_val"], x_dev), 10, flush)
    ms_wrapper = statistics.median(ts)
    # the kernel alone: CUDA events around the launch on the launching stream (regt_profile), L2 flushed before each launch
    from regt_b200 import _lib
    lib = _lib.load()
    ks = []
    for _ in range(10):
        flush.zero_()
        torch.cuda.synchronize()
        lib.regt_profile(1, torch.cuda.current_stream().cuda_stream)
        P.spmm_f8(t["g_rowptr"], t["g_col"], t["g_val"], x_dev)
        torch.cuda.synchronize()
        ks.append(sum(v for n, v in _lib.profile_read() if n.startswith("k_spmm")))
        lib.regt_profile(0, None)
    ms = statistics.median(ks) if ks and min(ks) > 0 else ms_wrapper
    nbytes = W.spmm_bytes(w, B)
    return {"kernel": "k_spmm_blk (regt_spmm_f8_blocked over the plan's regt_spmm_partition)", "bytes": nbytes, "ms": ms, "gbs": nbytes / (ms * 1e-3) / 1e9,
            "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / pk["hbm_gbs"], "peak_gbs": pk["hbm_gbs"], "B": B,
            "ms_through_wrapper": ms_wrapper, "gbs_through_wrapper": nbytes / (ms_wrapper * 1e-3) / 1e9,
            "note": "ms = the kernel launch between CUDA events on its stream (median of 10, L2 flushed before each); "
                    "ms_through_wrapper also counts the Python wrapper (allocation of y, partition cache lookup) after the flush"}


def measure_reference_call_pattern(dev, precision_note="auto"):
    """the reference's REAL call pattern (run.py:170-192) on config 1 at the reference's defaults (TPIMS graph, N=104, H=256,
    R=5, T=12): one [N,8,T] snapshot per model(...) call through the 12-tensor forward, batch.to(device) per snapshot,
    loss.cpu() per snapshot, loss.backward() through autograd.  Python + launches dominate here; reported as is."""
    from models import RegionalTemporalGCN
    from regt_b200 import workloads as W
    w = W.make_workload(1)
    model = RegionalTemporalGCN(8, w.N, w.T, w.O)          # reference ctor, reference defaults
    W.init_params_synthetic(model, 1234)
    model = model.to(dev)
    n = 40
    xs, ys = w.inputs(n)
    g_host = w.graph_args()

    def one(i):
        x = xs[i].to(dev)                                   # run.py:172  batch.to(device): x, y AND the edge lists
        y = ys[i].to(dev)
        g = tuple(a.to(dev) for a in g_host)
        out, _ = model(x, *g)                               # run.py:178
        loss = torch.mean((out - y) ** 2).cpu()             # run.py:180
        loss.backward()                                     # run.py:190
        return float(loss)

    for i in range(5):
        one(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(5, n):
        one(i)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    return {"workload": w.name, "value": (n - 5) / el, "unit": UNIT, "ms_per_snapshot": el / (n - 5) * 1e3, "snapshots": n - 5,
            "precision": model.precision,
            "note": "one snapshot per model(...) + loss.cpu() + loss.backward(), per-snapshot .to(device) of x, y and the 11 graph "
                    "tensors; the plan cache hits by content fingerprint (K1 runs once)"}


def measure_cfg2_bf16(dev, flush):
    """round 1's headline, kept as a side key: config 2 (A3TGCN, H=64, B=64) on the fused bf16 tcgen05 kernels
    (bf16 operands, fp32 accumulate -- narrower than the reference's arithmetic, stated tolerance), CUDA-graph replay."""
    from models import TemporalGCN
    from regt_b200 import workloads as W
    w = W.make_workload(2)
    model = TemporalGCN(8, w.T, w.O, hidden=w.H, precision="bf16")
    W.init_params_synthetic(model, 1234)
    model = model.to(dev)
    g = tuple(None if a is None else a.to(dev) for a in w.graph_args())
    x, y = w.inputs(w.B)
    x, y = x.to(dev), y.to(dev)
    for _ in range(3):
        model.fused_step(x, y, *g)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        model.fused_step(x, y, *g)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    with torch.cuda.graph(gr):
        model.fused_step(x, y, *g)
    torch.cuda.synchronize()
    for _ in range(3):
        gr.replay()
    ts = time_events(gr.replay, 20, flush)
    ms = sum(ts) / len(ts)
    return {"workload": w.name, "precision": "bf16", "value": w.B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": 20,
            "alg_bytes_per_step": W.alg_bytes_per_step(w), "note": "not fp32 arithmetic: side key only"}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner to stdout) are sent
    # to stderr by pointing fd 1 there; the line is written to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    from models import RegionalTemporalGCN, TemporalGCN
    from regt_b200 import _lib, workloads as W
    lib = _lib.load()

    w = W.make_workload(args.workload, args.batch)
    B = w.B
    if args.precision == "bf16" and w.H != 64:
        raise SystemExit("--precision bf16: the fused bf16 kernels are built for hidden 64 (workload 2)")
    if w.model == "TemporalGCN":
        model = TemporalGCN(8, w.T, w.O, hidden=w.H, precision=args.precision)
    else:
        model = RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R, precision=args.precision)
    W.init_params_synthetic(model, 1234)
    model = model.to(dev)
    graph_args = tuple(None if a is None else a.to(dev) for a in w.graph_args())

    from regt_b200 import shard as S
    os.environ["REGT_EXCHANGE"] = args.exchange
    sharded = world > 1 and w.R > 0 and args.shard != "batch"
    if args.shard == "region" and world > 1 and w.R == 0:
        raise SystemExit("--shard region needs a regional workload (3, 4 or 5)")

    # host (pinned) and device-resident inputs
    sm = None
    if sharded:
        # region shards: every rank sees every snapshot, owns the nodes of its regions (+ halo rows)
        sm = S.RegionShardedModel(model, graph_args[0], list(graph_args[1:1 + w.R]), list(graph_args[1 + w.R:]), rank, world)
        ex = sm.exchange
        xh, yh = w.inputs(B)
        xh = xh.index_select(1, torch.from_numpy(sm.shard.perm)).contiguous()   # the rank's loader reads its rows only
        yh = yh.index_select(1, torch.from_numpy(sm.shard.own)).contiguous()
    else:
        # one flat gradient buffer so that a single all-reduce covers every shared weight
        ex = S.GradExchange([p for n, p in model.named_parameters() if p.requires_grad], world)
        xh, yh = w.inputs(B, seed_offset=rank)     # batch shards: every rank gets its own snapshots
    xh, yh = xh.pin_memory(), yh.pin_memory()
    # two device input buffers: the end-to-end loop copies step k+1's inputs while step k computes
    bufs = [(xh.to(dev), yh.to(dev)), (xh.to(dev), yh.to(dev))]
    loss_h = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    the_model = sm.model if sharded else model
    results = [None, None]    # (loss, out, hid) of the last step on each input buffer; the graphs' static outputs once captured

    def raw_step(b=0):
        xd, yd = bufs[b]
        ex.zero()     # per-step gradients: the flat buffer holds this step's contribution only (and feeds the exchange at N > 1)
        if sharded:
            results[b] = sm.fused_step(None, None, micro_batch=args.micro_batch, local_inputs=(xd, yd), sync=False)
        else:
            results[b] = model.fused_step(xd, yd, *graph_args, micro_batch=args.micro_batch)
        return results[b][0]

    # warm-up (eager) -- also builds and caches the static-graph plan (K1), excluded from timing
    lib.regt_launch_count(1)
    loss_d = None
    nwarm = max(3, args.warmup)
    for _ in range(nwarm):
        loss_d = raw_step()
    torch.cuda.synchronize()
    launches_per_step = lib.regt_launch_count(1) // nwarm

    def exchange(loss):
        """the exchange step: shared-weight gradients + loss, ONE all-reduce of the flat buffer (peer-memory kernel or NCCL)"""
        if not sharded:
            ex.add_loss(loss)
        return ex.sync()

    def full_step(b=0):
        loss = raw_step(b)
        return exchange(loss) if dist is not None else loss

    if dist is not None:          # communicator warm-up before any capture
        for _ in range(2):
            loss_d = full_step()
        torch.cuda.synchronize()

    graphs, graph_loss, graph_has_exchange = None, [None, None], False
    if not args.no_graph:
        def capture(fn):
            gs, ls = [torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()], [None, None]   # one per input buffer
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                fn()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            for b in (0, 1):
                with torch.cuda.graph(gs[b]):
                    ls[b] = fn(b)
                torch.cuda.synchronize()
            return gs, ls
        if dist is not None:
            # the all-reduce is captured INSIDE the step's graph (one replay = compute + exchange); if capture fails on
            # any rank, every rank falls back to replay + eager all-reduce
            ok = torch.ones(1, device=dev)
            try:
                graphs, graph_loss = capture(full_step)
            except Exception as e:  # noqa: BLE001
                ok.zero_()
                print(f"[rank {rank}] exchange graph capture failed ({type(e).__name__}): eager exchange", file=sys.stderr)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            graph_has_exchange = bool(ok.item())
            if not graph_has_exchange:
                graphs, graph_loss = capture(raw_step)
        else:
            graphs, graph_loss = capture(raw_step)
    graph = graphs[0] if graphs else None

    def step(b=0):
        nonlocal loss_d
        if graphs is not None:
            graphs[b].replay()
            loss_d = graph_loss[b]
            if dist is not None and not graph_has_exchange:
                loss_d = exchange(loss_d)
        else:
            loss_d = full_step(b)

    for _ in range(3):
        step()
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput ("value") ----------------
    K = args.steps
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    align = torch.zeros(1, device=dev)
    for a, b in evs:
        flush.zero_()                      # evict L2 between timed iterations (outside the event pair)
        if dist is not None:
            dist.all_reduce(align)         # ... and re-align the ranks: the flush's skew is not part of the step
        a.record(); step(); b.record()
    barrier()
    per = [a.elapsed_time(b) for a, b in evs]
    tot_ms = torch.tensor([sum(per)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(tot_ms) / K
    clocks = sampler.stop() if sampler else None

    # ---------------- N > 1: cross-rank correctness evidence, same run ----------------
    xcheck = None
    if dist is not None:
        # after a step every rank must hold the SAME reduced gradient buffer (bit for bit: the exchange kernels sum in rank
        # order) and the reduced loss must equal the sum of the per-rank losses of that step
        xd, yd = bufs[0]
        ex.zero()
        if sharded:
            local_loss = sm.fused_step(None, None, micro_batch=args.micro_batch, local_inputs=(xd, yd), sync=False)[0].clone()
        else:
            local_loss = model.fused_step(xd, yd, *graph_args, micro_batch=args.micro_batch)[0].clone()
        red_loss = exchange(local_loss)
        torch.cuda.synchronize()
        nflat = ex.flat.numel() - 4
        bits = ex.flat[:nflat].view(torch.int32).to(torch.int64)
        wts = torch.arange(1, nflat + 1, device=dev, dtype=torch.int64)
        mine = torch.stack([bits.sum(), (bits * wts).sum()])
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        losses_all = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(losses_all, local_loss.reshape(1).float())
        red_all = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(red_all, red_loss.reshape(1).float())
        same = all(bool(torch.equal(e, every[0])) for e in every)
        lsum = float(sum(float(v) for v in losses_all))
        reds = [float(v) for v in red_all]
        finite = bool(torch.isfinite(ex.flat[:nflat]).all())
        xcheck = {"gradient_buffer_checksums_identical_on_all_ranks": same, "checksum_rank0": [int(v) for v in every[0].tolist()],
                  "gradient_floats": int(nflat), "gradients_finite": finite,
                  "reduced_loss": reds[0], "reduced_loss_identical_on_all_ranks": all(v == reds[0] for v in reds),
                  "sum_of_rank_losses": lsum, "loss_rel_diff": abs(reds[0] - lsum) / max(abs(lsum), 1e-30),
                  "peer_kernel_error_flag": int(ex.region.error()) if ex.region is not None else None}
        assert same and finite, f"cross-rank check failed: {xcheck}"
        assert xcheck["loss_rel_diff"] <= 1e-5, f"reduced loss != sum of rank losses: {xcheck}"

    # ---------------- end to end: host buffers in, loss out, every step ----------------
    # Every step's x,y are copied from pinned host memory and every step's loss is read on the host, all
    # inside the timed region.  The copies run on a second stream into the buffer the running step does
    # not use, and a step's loss is read while the next step computes (the reference reads it
    # synchronously, run.py:180; the values are the same, only one step late).
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    main_s, cs = torch.cuda.current_stream(), torch.cuda.Stream()
    ev_in = [torch.cuda.Event(), torch.cuda.Event()]
    ev_done = [torch.cuda.Event(), torch.cuda.Event()]
    ev_loss = [torch.cuda.Event(), torch.cuda.Event()]

    def h2d(b, wait_free):
        with torch.cuda.stream(cs):
            if wait_free:
                cs.wait_event(ev_done[b])       # the step that last used this buffer has finished
            bufs[b][0].copy_(xh, non_blocking=True)
            bufs[b][1].copy_(yh, non_blocking=True)
            ev_in[b].record(cs)

    barrier()
    cs.wait_stream(main_s)
    e0.record()
    h2d(0, False)
    losses = []
    for k in range(K):
        b = k & 1
        if k + 1 < K:
            h2d(1 - b, k >= 1)
        main_s.wait_event(ev_in[b])
        step(b)
        ev_done[b].record(main_s)
        loss_h[b].copy_(loss_d, non_blocking=True)
        ev_loss[b].record(main_s)
        if k >= 1:
            ev_loss[1 - b].synchronize()
            losses.append(float(loss_h[1 - b]))
    ev_loss[(K - 1) & 1].synchronize()
    losses.append(float(loss_h[(K - 1) & 1]))
    e1.record()
    barrier()
    assert len(losses) == K and all(v == v for v in losses), "end-to-end loop lost a loss value"
    e2e_ms = torch.tensor([e0.elapsed_time(e1) / K], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_ms)

    # ---------------- what the last timed step returned, before the eager steps below overwrite the gradients ----------
    if args.dump_outputs and rank == 0:
        _, out_d, hid_d = results[(K - 1) & 1]
        arrays = {"loss": loss_d, "out": out_d, "hidden": hid_d}
        arrays.update({"grad." + n: p.grad for n, p in the_model.named_parameters() if p.grad is not None})
        for name, (shape, k) in dump_outputs(args.dump_outputs, arrays).items():
            print(f"dump {name}: shape {list(shape)}, {k} elements written", file=sys.stderr)

    # ---------------- per-kernel breakdown for the roofline (rank 0, eager, events per launch) -----
    roofline, breakdown, step_roof = None, None, None
    pk = peaks()
    mb_used = min(B, args.micro_batch or getattr(the_model, "_mb", None) or B)
    if rank == 0:
        st_ptr = torch.cuda.current_stream().cuda_stream
        nprof = 3
        agg = {}
        for i in range(nprof):
            flush.zero_()
            torch.cuda.synchronize()
            lib.regt_profile(1, st_ptr)
            raw_step()
            torch.cuda.synchronize()
            for name, ms in _lib.profile_read():
                agg.setdefault(name, []).append(ms)
            lib.regt_profile(0, None)
        # launches of one kernel name within a step are summed per step
        per_kernel = {k: sum(v) / nprof for k, v in agg.items()}
        counts = {k: max(1, len(v) // nprof) for k, v in agg.items()}
        step_sum = sum(per_kernel.values())
        breakdown = {k: {"ms_per_step": round(v, 5), "launches": counts[k], "share": round(v / step_sum, 4)}
                     for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1])}

        def traffic_of(kernel):
            # DRAM bytes of that kernel per launch from the committed `ncu --set full` capture of this same command
            # (profiles/ncu_traffic.json, written by tools/ncu_summary.py, keyed "<workload>/<precision>/<kernel>"); else null
            tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
            if not os.path.exists(tpath) or world != 1 or args.batch:
                return None
            d = json.load(open(tpath))
            e = d.get(f"{args.workload}/{args.precision}/{kernel}") or (d.get(kernel) if (str(args.workload), args.precision) == ("2", "bf16") else None)
            return e.get("bytes_per_launch") if e else None

        rows_B = B if not sharded else B      # every rank sees all B snapshots for its own nodes
        wl = w
        if sharded:   # rank 0's share of the rows
            import copy
            wl = copy.copy(w)
            wl.N = int(sm.shard.n_own)
        roofline = pick_roofline(wl, rows_B, per_kernel, counts, step_sum, args.precision, pk, traffic_of)
        step_bytes = W.alg_bytes_per_step(w, B if (sharded or world == 1) else world * B)
        step_flops = 3 * W.fwd_flops_per_step(w, B if (sharded or world == 1) else world * B)
        peak_tc = pk["bf16_tflops"] / (6.0 if args.precision == "tf32x3" else 1.0) * world
        t_hbm = step_bytes / (pk["hbm_gbs"] * 1e9 * world)
        t_tc = step_flops / (peak_tc * 1e12) if args.precision != "fp32" else 0.0
        step_roof = {"alg_bytes_per_step": step_bytes, "achieved_gbs": step_bytes / (ms_per_step * 1e-3) / 1e9,
                     "frac_of_hbm_peak": t_hbm / (ms_per_step * 1e-3),
                     "fwd_bwd_flops_per_step": step_flops,
                     "achieved_tflops_fp32_equivalent": step_flops / (ms_per_step * 1e-3) / 1e12,
                     "frac_of_tensor_peak": (t_tc / (ms_per_step * 1e-3)) if t_tc else None,
                     "binding": "tensor" if t_tc > t_hbm else "hbm",
                     "frac_of_binding_roofline": max(t_hbm, t_tc) / (ms_per_step * 1e-3),
                     "t_hbm_ms": t_hbm * 1e3, "t_tensor_ms": t_tc * 1e3,
                     "note": f"whole job ({world} GPU): SURVEY 8(d) AlgBytes and 3 x collapsed FwdFlops over the step time; peaks x n_gpus"}

    # ---------------- side measurements (rank 0, N = 1) ----------------
    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            extras["spmm"] = measure_spmm(w, dev, bufs[0][0], graph_args, flush, pk)
        except Exception as e:  # noqa: BLE001
            extras["spmm"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            extras["reference_call_pattern"] = measure_reference_call_pattern(dev)
        except Exception as e:  # noqa: BLE001
            extras["reference_call_pattern"] = {"error": f"{type(e).__name__}: {e}"}
        if str(args.workload) != "2":
            try:
                extras["cfg2_bf16"] = measure_cfg2_bf16(dev, flush)
            except Exception as e:  # noqa: BLE001
                extras["cfg2_bf16"] = {"error": f"{type(e).__name__}: {e}"}

    # ---------------- CPU baseline (rank 0, N=1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, n, el, thr, what = cpu_oracle_rate(w, args.cpu_seconds)
        cpu = {"value": rate, "unit": UNIT, "cores": thr, "kind": "port",
               "sample": f"{n} snapshots in {el:.1f}s on {what} (oracle fp32 port of the reference, one snapshot at a time)"}

    if rank == 0:
        job_B = B if (sharded or world == 1) else world * B     # snapshots the whole job processes per step
        h2d_bytes = xh.numel() * 4 + yh.numel() * 4
        xport = {"peer": "one-kernel all-reduce over NVLink peer memory (CUDA IPC, csrc/peer.cu)", "nccl": "NCCL all-reduce",
                 "gloo": "gloo all-reduce"}[ex.transport] if world > 1 else ""
        out = {
            "metric": METRIC, "value": job_B / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": nwarm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak" if (world > 1 and not sharded) else "strong",
            "vs_baseline": None,
            "dtype": {"fp32": "f32", "tf32x3": "f32 (3xTF32 on the tensor cores: fp32-equivalent, 1e-5 parity)",
                      "bf16": "bf16 operands, f32 accumulate (f32 inputs, outputs, loss, gradients)"}[args.precision],
            "data": "synthetic",
            "config": bench_config(w),
            "run": dict(precision=args.precision, per_gpu_batch=B, micro_batch=mb_used,
                        cuda_graph=graph is not None, exchange_in_graph=graph_has_exchange,
                        optimizer="none: metric is fwd+bwd; the reference steps once per epoch (run.py:194)",
                        parallelism=("single GPU" if world == 1 else
                                     f"region-sharded x{world} (LPT regions->ranks, halo rows of x read locally), {xport} of the flat gradient buffer"
                                     if sharded else
                                     f"batch-sharded x{world}, {xport} of the flat gradient buffer")),
            "clocks": clocks,
            "e2e": {"value": job_B / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms, "pipeline": "double-buffered H2D on a copy stream; each step's loss read on the host one step late"},
            "gpu_launches": int(launches_per_step * K),
            "launches_per_step": int(launches_per_step),
            "roofline": roofline, "roofline_step": step_roof, "kernels": breakdown, "cpu_baseline": cpu,
            "cross_rank_check": xcheck,
        }
        out.update(extras)
        _REAL_STDOUT.write(json.dumps(out) + "\n")
        _REAL_STDOUT.flush()
    if dist is not None:
        # CUDA graphs that captured collective kernels are still alive: a regular communicator teardown can wait on them
        # forever.  Everything is measured and printed; leave without the teardown.
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
