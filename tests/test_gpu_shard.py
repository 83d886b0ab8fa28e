"""GPU parity of the region-sharded path (SURVEY 8(e)): the K4 row gather/scatter kernels, and the
sum over the ranks' shards (run one after the other on ONE GPU: gradient accumulation plays the part
of the all-reduce) against the unsharded CPU oracle.  The 2-process NCCL test needs 2 GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from parity_util import W, build_cuda, is_dead, oracle_step, relerr, to_dev

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("width", [12, 1, 96, 7])
def test_gather_scatter_rows_bit_exact(width):
    from regt_b200 import shard as S
    g = torch.Generator().manual_seed(width)
    src = torch.rand(3, 50, width, generator=g).cuda()
    idx = torch.randperm(50, generator=g)[:31].cuda()
    got = S.gather_rows(src, idx)
    assert torch.equal(got, src.index_select(1, idx))
    dst = torch.zeros(3, 50, width, device="cuda")
    S.scatter_rows(got, idx, dst)
    ref = torch.zeros_like(dst).index_copy_(1, idx, got)
    assert torch.equal(dst, ref)


def _cases():
    return [
        (W.tiny_workload("RegionalTemporalGCN", N=70, T=5, H=64, O=1, R=5, B=3, seed=23, k_intra=4, n_cross=12), 3, "fp32"),
        (W.tiny_workload("RegionalTemporalGCN", N=70, T=5, H=64, O=1, R=5, B=3, seed=23, k_intra=4, n_cross=12), 3, "bf16"),
        (W.tiny_workload("RegionalTemporalGCN", N=41, T=4, H=32, O=3, R=6, B=2, seed=29, n_cross=9), 2, "fp32"),
        (W.make_workload(1), 1, "fp32"),
        (W.make_workload(3), 2, "fp32"),
    ]


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("w,B,precision", _cases(), ids=lambda v: v.name if hasattr(v, "name") else str(v))
def test_sum_of_region_shards_equals_unsharded_oracle(w, B, precision, world):
    from regt_b200 import shard as S
    ref = oracle_step(w, B)
    x, y = w.inputs(B)
    x, y = x.cuda(), y.cuda()
    ei, reis, reas = w.edge_index.cuda(), [e.cuda() for e in w.reg_edge_index], [a.cuda() for a in w.reg_edge_attr]
    tol, gtol = (1e-5, 1e-5) if precision == "fp32" else (2e-2, 5e-2)
    loss_sum, grad_sum = 0.0, {}
    out_full = torch.zeros(B, w.N, w.O, device="cuda")
    hid_full = torch.zeros(B, w.N, w.H, device="cuda")
    halo_seen = 0
    for rank in range(world):
        m = build_cuda(w, ref["state"], precision=precision)
        sm = S.RegionShardedModel(m, ei, reis, reas, rank, world)
        halo_seen += sm.shard.n_halo
        loss, out, hid = sm.fused_step(x, y, sync=False)
        loss_sum += float(loss)
        S.scatter_rows(out, sm.own, out_full)
        S.scatter_rows(hid, sm.own, hid_full)
        for k, p in m.named_parameters():
            if p.grad is not None:
                grad_sum[k] = p.grad.double().cpu() + grad_sum.get(k, 0.0)
    if w.E > w.E_reg:
        assert halo_seen > 0, "the case has cross-region edges: some rank must read halo rows"
    assert relerr(out_full, ref["out"]) <= tol and relerr(hid_full, ref["hid"]) <= tol
    assert abs(loss_sum - ref["loss"]) <= tol * abs(ref["loss"])
    for k, g in ref["grads"].items():
        if is_dead(w.model, k):
            continue
        lim = 0.15 if (precision == "bf16" and k.endswith("_attention")) else gtol
        assert relerr(grad_sum[k], g) <= lim, f"grad {k}: {relerr(grad_sum[k], g):.3e}"


def test_local_plan_rows_match_global_plan():
    """bit-exact: the rank's gcn CSR is the owned rows of the global K1 output, columns renumbered."""
    from regt_b200 import shard as S
    from regt_b200.plan import GraphPlanTensors, build_gcn
    w = W.make_workload(3)
    dev = torch.device("cuda:0")
    g = GraphPlanTensors(dev, w.N)
    build_gcn(g, w.edge_index.to(dev), None)
    rp, col, val = (g.t[k].cpu().numpy() for k in ("g_rowptr", "g_col", "g_val"))
    for rank in range(4):
        sh = S.make_shard(w.N, w.edge_index, w.reg_edge_index, rank, 4)
        lp = S.build_local_plan(sh, dev, w.edge_index.to(dev), None, [e.to(dev) for e in w.reg_edge_index],
                                [a.to(dev) for a in w.reg_edge_attr])
        lrp, lcol, lval = (lp.t[k].cpu().numpy() for k in ("g_rowptr", "g_col", "g_val"))
        perm = sh.perm
        for i, n in enumerate(sh.own):
            assert np.array_equal(perm[lcol[lrp[i]:lrp[i + 1]]], col[rp[n]:rp[n + 1]])
            assert np.array_equal(lval[lrp[i]:lrp[i + 1]], val[rp[n]:rp[n + 1]])
        assert lp.N == sh.n_own and lp.R == w.R


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_process_nccl_region_shards(tmp_path):
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "shard_nccl_worker.py")
    port = 29700 + os.getpid() % 2000
    out_path = str(tmp_path / "rank0.pt")
    procs = [subprocess.Popen([sys.executable, worker, str(r), "2", str(port), out_path]) for r in range(2)]
    try:
        for p in procs:
            assert p.wait(timeout=300) == 0
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
    got = torch.load(out_path)
    w = W.make_workload(3)
    ref = oracle_step(w, 2)
    assert abs(got["loss"] - ref["loss"]) <= 1e-5 * abs(ref["loss"])
    assert relerr(got["out"], ref["out"]) <= 1e-5 and relerr(got["hid"], ref["hid"]) <= 1e-5
    for k, g in ref["grads"].items():
        if not is_dead(w.model, k):
            assert relerr(got["grads"][k], g) <= 1e-5, k


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("world", [0, 3])
def test_peer_memory_allreduce_bit_exact_and_graph_capturable(world):
    """csrc/peer.cu: the one-kernel NVLink all-reduce sums in rank order (bit-identical to the explicit sum on every
    rank), survives repeated calls (device-side epochs) and CUDA-graph replay, and carries GradExchange's flat buffer."""
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "peer_allreduce_worker.py")
    if world == 0:
        world = min(torch.cuda.device_count(), 8)       # every GPU of the box
    elif torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")               # 3 ranks: a world size that does not divide the buffer
    port = 31700 + os.getpid() % 2000 + world
    procs = [subprocess.Popen([sys.executable, worker, str(r), str(world), str(port)]) for r in range(world)]
    try:
        for p in procs:
            assert p.wait(timeout=300) == 0
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
