"""CPU tests that pin the oracle (oracle/regt_oracle.py) as far as it can be pinned offline."""
import os

import numpy as np
import pytest
import torch

from oracle import regt_oracle as O
from oracle import dense_check as D
from regt_b200 import workloads as W


def test_laplacian_known_answer_upstream():
    """Known-answer vector of PyG's own test-suite for get_laplacian(normalization='sym')
    (test/utils/test_laplacian.py upstream, recalled; not checkable offline):
    edge_index [[0,1,1,2],[1,0,2,1]], weights [1,2,2,4] -> off-diagonal [-0.5,-1,-0.5,-1]."""
    ei = torch.tensor([[0, 1, 1, 2], [1, 0, 2, 1]])
    ew = torch.tensor([1.0, 2.0, 2.0, 4.0])
    row, col, lap = O.cheb_norm(ei, ew, 3, torch.float64)
    assert row.tolist() == [0, 1, 1, 2] and col.tolist() == [1, 0, 2, 1]
    # Cheb rescale 2L/2 - I leaves the off-diagonal untouched and zeroes the diagonal
    assert lap.tolist() == [-0.5, -1.0, -0.5, -1.0]


def test_gcn_norm_hand_computed():
    """3-node path 0->1->2 with a weighted self-loop on 1 (weight 3), unit elsewhere.
    After add_remaining_self_loops: edges (0,1,w1) (1,2,w1) + loops (1, 3, 1).
    in-degree: d0 = 1, d1 = 1+3 = 4, d2 = 1+1 = 2."""
    ei = torch.tensor([[0, 1, 1], [1, 1, 2]])
    ew = torch.tensor([1.0, 3.0, 1.0])
    row, col, w = O.gcn_norm(ei, ew, 3, torch.float64)
    assert row.tolist() == [0, 1, 0, 1, 2] and col.tolist() == [1, 2, 0, 1, 2]
    exp = [1 / (1 * 2), 1 / (2 * 2 ** 0.5), 1.0, 3 / 4, 1 / 2]
    assert np.allclose(w.numpy(), exp, rtol=1e-15)
    # edge_weight=None: an existing self-loop is replaced by one unit loop
    row, col, w = O.gcn_norm(ei, None, 3, torch.float64)
    assert w.numel() == 5 and np.allclose(w.numpy(), [1 / 2 ** 0.5, 0.5, 1.0, 0.5, 0.5])


def test_zero_degree_inf_masking():
    ei = torch.tensor([[0], [1]])
    row, col, lap = O.cheb_norm(ei, torch.tensor([2.0]), 3, torch.float64)
    # node 1 has zero out-degree -> dis = 0 -> entry is exactly 0, no nan/inf
    assert lap.tolist() == [-0.0] or lap.tolist() == [0.0]
    assert torch.isfinite(lap).all()


@pytest.mark.parametrize("adv", [False, True])
@pytest.mark.parametrize("model", ["TemporalGCN", "RegionalTemporalGCN"])
def test_scatter_formulation_matches_dense_restatement(model, adv):
    w = W.tiny_workload(model, N=14, T=3, H=8, O=2, R=3 if model != "TemporalGCN" else 0, B=1, seed=7, adversarial=adv)
    torch.manual_seed(0)
    if model == "TemporalGCN":
        m = O.TemporalGCN(8, w.T, w.O, hidden=w.H).double()
    else:
        m = O.RegionalTemporalGCN(8, w.N, w.T, w.O, hidden=w.H, n_regions=w.R).double()
    W.init_params_synthetic(m, 3)
    x, _ = w.inputs()
    out, hid = m(x[0].double(), *w.graph_args())
    sd = {k: v.detach().numpy() for k, v in m.state_dict().items()}
    o2, h2 = D.forward(sd, x[0].double().numpy(), w.edge_index.numpy(),
                       None if w.edge_attr is None else w.edge_attr.numpy(),
                       [e.numpy() for e in w.reg_edge_index], [a.numpy() for a in w.reg_edge_attr],
                       regional=(model != "TemporalGCN"))
    assert np.abs(out.detach().numpy() - o2).max() < 1e-12
    assert np.abs(hid.detach().numpy() - h2).max() < 1e-12


@pytest.mark.parametrize("fname,nn_,od", [("model_in6_out1_epoch50.pt", 104, 1), ("model_in6_out3_epoch50.pt", 105, 3),
                                          ("model_in6_out36_epoch50.pt", 105, 36)])
def test_shipped_checkpoints_load_strict(fname, nn_, od):
    """the layout of the upstream checkpoints (tensor names, shapes, dtype; tests/golden/shipped_checkpoints.json) loads strict
    into the oracle built with that checkpoint's constructor arguments."""
    from parity_util import shipped_checkpoint_state
    spec, sd = shipped_checkpoint_state(fname)
    assert (spec["num_nodes"], spec["periods"], spec["output_dim"]) == (nn_, 6, od)
    m = O.RegionalTemporalGCN(8, nn_, 6, od)
    m.load_state_dict(sd, strict=True)
    assert len(sd) == 26 and all(v.dtype == torch.float32 for v in sd.values())
    if fname == "model_in6_out1_epoch50.pt":
        assert sum(v.numel() for v in sd.values()) == 766_577
    full, rei, rea, N = W.tpims_graph()
    x = torch.rand(N, 8, 6, generator=torch.Generator().manual_seed(1))
    out, hid = m(x, full, *rei, *rea)
    assert out.shape == (N, od) and hid.shape == (N, 256) and torch.isfinite(out).all()


def test_canonical_csr_structures():
    w = W.tiny_workload("RegionalTemporalGCN", N=20, T=2, H=8, O=1, R=3, B=1, seed=11, adversarial=True)
    ei = w.edge_index.numpy()
    rowptr, col, eid = O.canonical_gcn_csr(ei, w.N)
    assert rowptr[0] == 0 and rowptr[-1] == len(col) == (ei[0] != ei[1]).sum() + w.N
    for n in range(w.N):
        seg = eid[rowptr[n]:rowptr[n + 1]]
        assert (np.diff(seg) > 0).all()          # stable: original order inside a row
    rp, c, reg, eid, segp = O.canonical_cheb_csr([e.numpy() for e in w.reg_edge_index], w.N)
    assert rp[-1] == len(c) and segp[-1] >= (np.diff(rp) > 0).sum()
    assert (segp[1:] - segp[:-1]).max() == 2     # the adversarial node with two segments
    ro = O.region_of_nodes([e.numpy() for e in w.reg_edge_index], w.N)
    assert (ro == -2).sum() == 1 and (ro == -1).sum() >= 1


def test_lpt_partition():
    own = O.lpt_partition([5, 9, 3, 9, 1, 4], 2)
    assert own.tolist() == [0, 0, 1, 1, 1, 1] or sum(s for s, o in zip([5, 9, 3, 9, 1, 4], own) if o == 0) in (15, 16)
    # deterministic tie-breaking: equal sizes go round-robin from rank 0
    assert O.lpt_partition([4, 4, 4, 4], 4).tolist() == [0, 1, 2, 3]


def test_workload_shapes_match_survey():
    w2 = W.make_workload(2)
    assert (w2.N, w2.E, w2.H, w2.B, w2.O) == (207, 1722, 64, 64, 12)
    assert (w2.edge_index[0] != w2.edge_index[1]).all() and w2.edge_attr.min() > 0
    w3 = W.make_workload(3)
    assert (w3.N, w3.E_reg, w3.E, w3.R) == (325, 2600, 2694, 12)
    w1 = W.make_workload(1)
    assert (w1.N, w1.E, [e.shape[1] for e in w1.reg_edge_index]) == (104, 348, [270, 16, 22, 26, 14])
    # SURVEY table: 344 MB / 4.23 GB algorithmic bytes, 4.98 / 209 GFLOP
    assert abs(W.alg_bytes_per_step(w2) / 344e6 - 1) < 0.02
    assert abs(W.alg_bytes_per_step(w3) / 4.23e9 - 1) < 0.02
    assert abs(W.fwd_flops_per_step(w2) / 4.98e9 - 1) < 0.02
    assert abs(W.fwd_flops_per_step(w3) / 209e9 - 1) < 0.02


def test_oracle_reproduces_committed_config1_golden():
    """drift guard: the oracle of today gives the vectors committed under tests/golden/ (config 1 = BASELINE configs[0])."""
    import os
    import numpy as np
    from parity_util import W, is_dead, oracle_step
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfg1_oracle_fp64.npz"))
    w = W.make_workload(1)
    ref = oracle_step(w, 1)
    assert np.allclose(ref["out"].numpy(), gold["out"], rtol=0, atol=1e-12)
    assert np.allclose(ref["hid"].numpy(), gold["hid"], rtol=0, atol=1e-12)
    assert abs(float(ref["loss"]) - float(gold["loss"])) <= 1e-12
    n = 0
    for k, g in ref["grads"].items():
        if g is None or is_dead(w.model, k):
            continue
        assert np.allclose(g.double().reshape(-1).numpy()[:32], gold["ghead:" + k], rtol=0, atol=1e-12 * max(1.0, float(gold["gmax:" + k]))), k
        n += 1
    assert n >= 20
