"""phase timing of the fused 3xTF32 cell kernels: clock64 marks of CTA 0 / epilogue thread 0 over 16 consecutive steps
(REGT_F_DEBUG=<first step>), printed as mean microseconds per phase (SM clock taken as 1.9 GHz)."""
import ctypes as C, os, sys
os.environ.setdefault("REGT_F_DEBUG", "20")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "regt-gcn_b200")):
    sys.path.insert(0, p)
import torch
from models import RegionalTemporalGCN
from regt_b200 import _lib, workloads as W
B = int(os.environ.get("PB", "16"))
w = W.make_workload(os.environ.get("PW", "4"), B)
dev = torch.device("cuda:0")
m = RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R, precision="tf32x3")
W.init_params_synthetic(m, 1234)
m = m.to(dev)
g = tuple(None if a is None else a.to(dev) for a in w.graph_args())
x, y = w.inputs(B)
x, y = x.to(dev), y.to(dev)
for _ in range(2):
    m.fused_step(x, y, *g)
torch.cuda.synchronize()
buf = (C.c_longlong * (3 * 16 * 12))()
_lib.check(_lib.load().regt_debug_f_timestamps(buf), "timestamps")
names = {0: ["wait z-gate MMAs", "E1z (sigmoid, save Z, acc)", "wait r-gate MMAs", "E1r (sigmoid, save R, h*R -> A)", "Pcompute(next)",
             "wait candidate MMAs", "Pstore(next)", "E2 (tanh, save H~, acc)"],
         1: ["E0 (recompute h, planes, Dz Dc h hR out, Dc -> A)", "wait M1 (dHR)", "Dz -> A", "E1 (Dr, t1)", "wait M2z", "Dr -> A", "wait M2r",
             "E2 (d h_pre out)"]}
for which, title in ((0, "forward k_cell_fwd_f"), (1, "backward k_cell_bwd_f")):
    rows = [[buf[(which * 16 + s) * 12 + i] for i in range(12)] for s in range(16)]
    rows = [r for r in rows if r[0] > 0 and r[8] > 0]
    if not rows:
        print(title, ": no timestamps"); continue
    print(f"== {title}: {len(rows)} steps of CTA 0, thread 0")
    tot = 0.0
    for i, nm in enumerate(names[which]):
        d = sum(r[i + 1] - r[i] for r in rows) / len(rows) / 1.9e3
        tot += d
        print(f"   {nm:55s} {d:7.2f} us")
    if which == 1 and all(r[9] > 0 for r in rows):
        for nm, (i0, i1) in (("E0: feature loads + h of chunk 0", (0, 9)), ("E0: plane loads, math, stores of chunk 0", (9, 10)),
                             ("E0: Dc -> A, pGZ -> acc2 of chunk 0", (10, 11)), ("E0: all of chunk 1 + st wait + arrive", (11, 1))):
            print(f"      {nm:52s} {sum(r[i1] - r[i0] for r in rows) / len(rows) / 1.9e3:7.2f} us")
    step = sum(rows[i + 1][0] - rows[i][0] for i in range(len(rows) - 1)) / max(1, len(rows) - 1) / 1.9e3
    print(f"   {'sum of phases':55s} {tot:7.2f} us      step to step {step:7.2f} us")

# forward, MMA warp (lane 0 of CTA 0): when the gate blocks are ISSUED (the tensor pipe runs behind the issue by its queue)
rows = [[buf[(2 * 16 + s) * 12 + i] for i in range(12)] for s in range(16)]
rows = [r for r in rows if r[0] > 0 and r[7] > 0]
if rows:
    print(f"== forward, MMA warp: {len(rows)} steps")
    for nm, (i0, i1) in (("wait bar_a (h staged)", (0, 1)), ("issue z block (incl. waits for weight stages)", (1, 2)), ("wait acc_c free", (2, 3)),
                         ("issue r block", (3, 4)), ("wait bar_a2 (h*R staged)", (4, 5)), ("issue c block", (5, 6)), ("wait bar_x + issue h_pre MMAs", (6, 7))):
        print(f"   {nm:55s} {sum(r[i1] - r[i0] for r in rows) / len(rows) / 1.9e3:7.2f} us")
    print(f"   {'of which: waiting for weight stages (bar_full)':55s} {sum(r[8] for r in rows) / len(rows) / 1.9e3:7.2f} us")
