"""Synthetic workloads of SURVEY.md section 8(d) / BASELINE.json ``configs``.

Every tensor is produced on the CPU from a fixed seed (numpy ``default_rng`` for graph
structure, ``torch.Generator`` for dense data), so the GPU box, the build container and
the oracle see bit-identical inputs.  Nothing here reads ``/root/reference``; the TPIMS
topology of config 1 comes from the committed fixture ``tests/golden/tpims_links.npz``
(made by ``tests/golden/make_tpims_fixture.py`` from the reference's
``dataset/tpims_link_0322.tar.xz``).
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
import torch

F_IN = 8  # node features of the reference's data (run.py:116 ``node_features=8``), the default of every workload


@dataclass
class Workload:
    name: str
    model: str                 # "RegionalTemporalGCN" | "TemporalGCN"
    B: int
    N: int
    T: int
    H: int
    O: int
    R: int                     # 0 for TemporalGCN
    seed: int
    edge_index: torch.Tensor                     # int64 [2,E] full graph
    edge_attr: Optional[torch.Tensor]            # f32 [E] (TemporalGCN only)
    reg_edge_index: List[torch.Tensor] = field(default_factory=list)
    reg_edge_attr: List[torch.Tensor] = field(default_factory=list)
    F: int = F_IN                                # node features of x (1..8)

    @property
    def E(self) -> int:
        return int(self.edge_index.shape[1])

    @property
    def E_reg(self) -> int:
        return int(sum(e.shape[1] for e in self.reg_edge_index))

    def inputs(self, B: Optional[int] = None, seed_offset: int = 0):
        """x [B,N,F,T] ~ U[0,1), y [B,N,O] ~ U[0,1) (MinMax-scaled features, load_dataset.py:430)."""
        B = self.B if B is None else B
        g = torch.Generator().manual_seed(self.seed * 1000 + seed_offset)
        x = torch.rand(B, self.N, self.F, self.T, generator=g, dtype=torch.float32)
        y = torch.rand(B, self.N, self.O, generator=g, dtype=torch.float32)
        return x, y

    def graph_args(self):
        """positional tail of the reference forward() after ``x``."""
        if self.model == "TemporalGCN":
            return (self.edge_index, self.edge_attr)
        return (self.edge_index, *self.reg_edge_index, *self.reg_edge_attr)

    def describe(self) -> dict:
        return dict(workload=self.name, model=self.model, B=self.B, N=self.N, T=self.T, F=self.F,
                    H=self.H, O=self.O, R=self.R, E=self.E, E_reg=self.E_reg, seed=self.seed)


def init_params_synthetic(module: torch.nn.Module, seed: int) -> None:
    """SURVEY 8(d): every ``weight`` ~ U(-a,a), a = sqrt(6/(fan_in+fan_out)); every ``bias``
    ~ U(-0.05,0.05) (non-zero on purpose); ``_attention`` ~ U(0,1); dead parameters untouched.
    Drawn on the CPU in ``named_parameters`` order, then copied to the parameter's device."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            leaf = name.split(".")[-1]
            if leaf in ("_weight_att1", "_weight_att2", "_bias_att1", "_bias_att2"):
                continue
            if leaf == "_attention":
                v = torch.rand(p.shape, generator=g, dtype=torch.float64)
            elif leaf == "bias":
                v = (torch.rand(p.shape, generator=g, dtype=torch.float64) - 0.5) * 0.1
            elif p.dim() == 2:
                a = math.sqrt(6.0 / (p.shape[0] + p.shape[1]))
                v = (torch.rand(p.shape, generator=g, dtype=torch.float64) * 2 - 1) * a
            else:
                continue
            p.copy_(v.to(p.dtype))


# ------------------------------------------------------------------------------------------
# graph generators
# ------------------------------------------------------------------------------------------
def _out_neighbours(rng: np.random.Generator, nodes: np.ndarray, k_of: np.ndarray) -> np.ndarray:
    """for node nodes[i] draw k_of[i] distinct targets from ``nodes`` excluding itself."""
    src, dst = [], []
    m = len(nodes)
    for i in range(m):
        k = int(min(k_of[i], m - 1))
        if k <= 0:
            continue
        pick = rng.choice(m - 1, size=k, replace=False)
        pick = pick + (pick >= i)  # skip self
        src.append(np.full(k, nodes[i], dtype=np.int64))
        dst.append(nodes[pick].astype(np.int64))
    if not src:
        return np.zeros((2, 0), dtype=np.int64)
    return np.stack([np.concatenate(src), np.concatenate(dst)])


def _regional_graph(N: int, R: int, k_intra: int, n_cross: int, seed: int):
    rng = np.random.default_rng(seed)
    regions = np.array_split(np.arange(N), R)
    reg_ei, reg_ea = [], []
    for nodes in regions:
        ei = _out_neighbours(rng, nodes, np.full(len(nodes), k_intra))
        reg_ei.append(torch.from_numpy(ei))
        w = rng.uniform(75.0, 3057.0, size=ei.shape[1]).astype(np.float32)
        reg_ea.append(torch.from_numpy(w))
    region_of = np.concatenate([np.full(len(n), r) for r, n in enumerate(regions)])
    cs, cd = [], []
    while R > 1 and len(cs) < n_cross:     # one region: there is no cross-region edge to draw
        s, d = int(rng.integers(N)), int(rng.integers(N))
        if region_of[s] != region_of[d]:
            cs.append(s); cd.append(d)
    cross = torch.tensor([cs, cd], dtype=torch.int64).reshape(2, -1)
    full = torch.cat(reg_ei + [cross], dim=1)
    return full, reg_ei, reg_ea


def _golden_dir() -> str:
    here = os.path.dirname(os.path.abspath(__file__))
    return os.path.normpath(os.path.join(here, "..", "..", "tests", "golden"))


def tpims_graph():
    """the reference's real regional link lists IA,KS,KY,OH,WI (directed, weighted by DIST)."""
    z = np.load(os.path.join(_golden_dir(), "tpims_links.npz"))
    reg_ei, reg_ea = [], []
    for r in range(5):
        m = z["region"] == r
        reg_ei.append(torch.from_numpy(np.stack([z["src"][m], z["dst"][m]]).astype(np.int64)))
        reg_ea.append(torch.from_numpy(z["dist"][m].astype(np.float32)))
    # link_data.csv (full graph) is not shipped: the documented substitute is IA|KS|KY|OH|WI
    full = torch.cat(reg_ei, dim=1)
    return full, reg_ei, reg_ea, int(z["num_nodes"])


def make_workload(cfg: int | str, B: Optional[int] = None) -> Workload:
    cfg = str(cfg)
    if cfg in ("1", "tpims"):
        full, rei, rea, N = tpims_graph()
        w = Workload("cfg1_tpims_N104_R5_H256", "RegionalTemporalGCN", 1, N, 12, 256, 6, 5, 101, full, None, rei, rea)
    elif cfg in ("2", "metrla"):
        rng = np.random.default_rng(102)
        N = 207
        k = np.full(N, 8); k[:66] = 9
        ei = _out_neighbours(rng, np.arange(N), k)
        ea = (1.0 - rng.uniform(0.0, 1.0, size=ei.shape[1])).astype(np.float32)  # U(0,1]
        w = Workload("cfg2_a3tgcn_metrla_N207_H64_B64", "TemporalGCN", 64, N, 12, 64, 12, 0, 102,
                     torch.from_numpy(ei), torch.from_numpy(ea))
    elif cfg in ("3", "pemsbay"):
        full, rei, rea = _regional_graph(325, 12, 8, 94, 103)
        w = Workload("cfg3_regional_pemsbay_N325_R12_H256_B128", "RegionalTemporalGCN", 128, 325, 12, 256, 12, 12, 103,
                     full, None, rei, rea)
    elif cfg in ("4", "road10k"):
        full, rei, rea = _regional_graph(10_000, 32, 6, 1_000, 104)
        w = Workload("cfg4_regional_road_N10k_R32_H128_B256", "RegionalTemporalGCN", 256, 10_000, 12, 128, 12, 32, 104,
                     full, None, rei, rea)
    elif cfg in ("5", "multistate100k"):
        full, rei, rea = _regional_graph(100_000, 256, 6, 10_000, 105)
        w = Workload("cfg5_regional_multistate_N100k_R256_H128_B64", "RegionalTemporalGCN", 64, 100_000, 12, 128, 12, 256, 105,
                     full, None, rei, rea)
    else:
        raise ValueError(f"unknown workload {cfg!r}")
    if B is not None:
        w.B = B
    return w


def cfg5_shaped(N: int = 2560, T: int = 2, B: int = 2, H: int = 128, R: int = 256, O: int = 12) -> Workload:
    """config 5's generator (same seed, R = 256 regions, H = 128, 6 intra-region out-edges per node, N/10 cross-region
    edges) at a node count the literal CPU oracle can hold: its [N, R*H] regional concat is N * 256 KiB per period in fp64."""
    full, rei, rea = _regional_graph(N, R, 6, max(1, N // 10), 105)
    return Workload(f"cfg5_shaped_N{N}_R{R}_H{H}_T{T}", "RegionalTemporalGCN", B, N, T, H, O, R, 105, full, None, rei, rea)


def tiny_workload(model: str, N: int, T: int, H: int, O: int, R: int, B: int, seed: int,
                  k_intra: int = 3, n_cross: int = 4, adversarial: bool = False, F: int = F_IN) -> Workload:
    """small seeded cases for parity tests.  ``adversarial`` adds what SURVEY section 4 asks for:
    existing self-loops (with weights), duplicate edges, isolated nodes, zero out-degree
    nodes, asymmetric weights, and a node that appears in two regional lists."""
    rng = np.random.default_rng(seed)
    if model == "TemporalGCN":
        k = np.full(N, k_intra)
        ei = _out_neighbours(rng, np.arange(N), k)
        ea = (1.0 - rng.uniform(0.0, 1.0, size=ei.shape[1])).astype(np.float32)
        if adversarial and N >= 6:
            # isolate last node, self-loops (two on node 1: last wins), duplicate edge 0->2
            keep = (ei[0] != N - 1) & (ei[1] != N - 1)
            ei, ea = ei[:, keep], ea[keep]
            # node N-2: zero out-degree
            keep = ei[0] != N - 2
            ei, ea = ei[:, keep], ea[keep]
            extra = np.array([[1, 1, 0, 0, 3], [1, 1, 2, 2, 3]], dtype=np.int64)
            ew = np.array([0.3, 0.7, 0.25, 0.5, 2.0], dtype=np.float32)
            ei = np.concatenate([ei, extra], axis=1); ea = np.concatenate([ea, ew])
            perm = rng.permutation(ei.shape[1])
            ei, ea = ei[:, perm], ea[perm]
        return Workload(f"tiny_tgcn_N{N}_H{H}_s{seed}", model, B, N, T, H, O, 0, seed,
                        torch.from_numpy(ei), torch.from_numpy(ea), F=F)
    full, rei, rea = _regional_graph(N, R, k_intra, n_cross, seed)
    if adversarial and N >= 8 and R >= 2:
        # a self-loop inside list 0, a duplicate edge in list 1, and an edge of list 1 that
        # points into region 0 (so that node gets two (node, region) segments)
        n0 = int(rei[0][0, 0]); n1 = int(rei[1][0, 0]); d1 = int(rei[1][1, 0])
        rei[0] = torch.cat([rei[0], torch.tensor([[n0], [n0]])], dim=1)
        rea[0] = torch.cat([rea[0], torch.tensor([123.0])])
        rei[1] = torch.cat([rei[1], torch.tensor([[n1, n1], [d1, n0]])], dim=1)
        rea[1] = torch.cat([rea[1], torch.tensor([500.0, 900.0])])
        # full graph: self-loop + duplicates too, and make the last node isolated
        full = torch.cat([full, torch.tensor([[2, 0, 0], [2, 1, 1]])], dim=1)
        keep = (full[0] != N - 1) & (full[1] != N - 1)
        full = full[:, keep]
        last = len(rei) - 1
        keep = (rei[last][0] != N - 1) & (rei[last][1] != N - 1)
        rei[last], rea[last] = rei[last][:, keep], rea[last][keep]
    return Workload(f"tiny_regional_N{N}_R{R}_H{H}_s{seed}", model, B, N, T, H, O, R, seed, full, None, rei, rea, F=F)


# ------------------------------------------------------------------------------------------
# algorithmic work (SURVEY 8(d) formulas; "the formulas are the contract")
# ------------------------------------------------------------------------------------------
def param_count(w: Workload) -> int:
    H, F, O, T, R = w.H, w.F, w.O, w.T, w.R
    tgcn = 3 * (H * F + H) + 3 * (2 * H * H + H)
    cheb = 2 * H * F + H
    head = 128 * H + 128 + O * 128 + O
    comb = (R * H * H + H) if w.model == "RegionalTemporalGCN" else 0
    return tgcn + cheb + head + comb + T


def alg_bytes_per_step(w: Workload, B: Optional[int] = None) -> int:
    B = w.B if B is None else B
    N, T, H, O, F = w.N, w.T, w.H, w.O, w.F
    E, Er = w.E, (w.E_reg if w.R else w.E)
    G = ((N + 1) * 4 + (E + N) * 8) + ((N + 1) * 4 + Er * 8)
    return B * N * (2 * T * F * 4 + 2 * T * 4 * H * 4 + 2 * (H + O) * 4) + 3 * param_count(w) * 4 + 2 * G


def fwd_flops_per_step(w: Workload, B: Optional[int] = None) -> int:
    B = w.B if B is None else B
    N, T, H, O, F = w.N, w.T, w.H, w.O, w.F
    E, Er = w.E, (w.E_reg if w.R else w.E)
    return 2 * B * T * N * (3 * (F + H) * H + 2 * F * H) + 2 * B * N * (128 * H + 128 * O) + 2 * B * T * ((E + N) + Er) * F


def spmm_bytes(w: Workload, B: Optional[int] = None) -> int:
    B = w.B if B is None else B
    return 2 * B * w.T * w.N * w.F * 4 + (w.N + 1) * 4 + (w.E + w.N) * 8
