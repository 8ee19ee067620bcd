"""Model construction: SNN graph -> Ising vectors (+ lazily evaluated rank-1 groups) for the sampler.

Every builder restates one construction of the reference (file:line in each docstring) in vectorised
numpy; ``oracle/models_ref.py`` holds the line-by-line dict-loop restatement these are tested against,
and ``tests/golden/`` holds Q dicts captured from the reference's own functions.

Output type ``LoweredModel`` is what the annealer consumes:
    E(s) = offset + sum_v h_v s_v + sum_c J_c s_{u_c} s_{v_c} + sum_g lam_g/4 (sum_{v in g} a_v s_v + kappa_g)^2
with the caller-facing variables BINARY x = (s+1)/2.  ``structured=True`` keeps the dense all-pairs /
cluster-size terms of the reference as rank-1 groups (SURVEY.md Appendix A) instead of O(n^2) couplers.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, Hashable, List, Optional, Sequence, Tuple

import numpy as np

from .bqm import BINARY, BinaryQuadraticModel, _accumulate_rows, _seq_sum, qubo_to_ising_vectors


# ------------------------------------------------------------------------------------------------
# containers
# ------------------------------------------------------------------------------------------------
@dataclass
class Groups:
    grp: np.ndarray      # int32 [n]  group id or -1
    coef: np.ndarray     # int32 [n]  a_v
    lam: np.ndarray      # float64 [G]
    kappa: np.ndarray    # int64 [G]
    # interval groups (include/qanneal.h qa_model_set_group_bounds): lam/4 * d(u)^2 with u = sum a_v s_v + kappa and
    # d(u) = max(lo - u, 0, u - hi); int64 [G], INT64_MIN / INT64_MAX for an open side.  None: equality groups (lam/4 * u^2)
    lo: Optional[np.ndarray] = None
    hi: Optional[np.ndarray] = None

    @property
    def interval(self) -> bool:
        return self.lo is not None

    def astuple(self):
        if self.lo is None:
            return self.grp, self.coef, self.lam, self.kappa
        return self.grp, self.coef, self.lam, self.kappa, self.lo, self.hi


@dataclass
class LoweredModel:
    h: np.ndarray                 # float64 [n]   spin linear biases
    starts: np.ndarray            # int32 [m]     coupler row (larger index)   -- dimod to_numpy_vectors order
    ends: np.ndarray              # int32 [m]     coupler col (smaller index)
    weights: np.ndarray           # float64 [m]   J
    offset: float                 # spin-model offset: E_binary(x) = E_spin(s) + offset
    labels: List[Hashable]        # caller-facing label of every binary variable
    groups: Optional[Groups] = None
    meta: Dict = field(default_factory=dict)

    @property
    def num_variables(self) -> int:
        return int(len(self.h))

    @property
    def num_couplers(self) -> int:
        return int(len(self.weights))

    def materialise(self) -> "LoweredModel":
        """Expand the rank-1 groups into explicit couplers (J_ij += lam a_i a_j / 2, h_i += lam kappa a_i / 2)."""
        if self.groups is None:
            return self
        if self.groups.interval:
            raise ValueError("interval groups are not quadratic: they have no coupler form")
        n = self.num_variables
        dense = np.zeros((n, n), dtype=np.float64)
        dense[self.starts, self.ends] = self.weights
        h = self.h.copy()
        offset = self.offset
        g = self.groups
        for gi in range(len(g.lam)):
            idx = np.nonzero(g.grp == gi)[0]
            a = g.coef[idx].astype(np.float64)
            outer = np.outer(a, a) * (g.lam[gi] / 2.0)
            sub = dense[np.ix_(idx, idx)]
            sub += np.tril(outer, -1)
            dense[np.ix_(idx, idx)] = sub
            h[idx] += g.lam[gi] * float(g.kappa[gi]) * a / 2.0
            offset += g.lam[gi] / 4.0 * (float(np.sum(a * a)) + float(g.kappa[gi]) ** 2)
        r, c = np.nonzero(np.tril(dense, -1))
        order = np.lexsort((c, r))
        r, c = r[order], c[order]
        return LoweredModel(h, r.astype(np.int32), c.astype(np.int32), dense[r, c], float(offset), list(self.labels), None,
                            dict(self.meta))

    def energies(self, spins: np.ndarray) -> np.ndarray:
        """Reference energies (numpy, any summation order) of +-1 rows, including offset: for tests."""
        s = np.atleast_2d(np.asarray(spins)).astype(np.float64)
        e = s @ self.h + self.offset
        if len(self.weights):
            e = e + (s[:, self.starts] * s[:, self.ends]) @ self.weights
        if self.groups is not None:
            g = self.groups
            for gi in range(len(g.lam)):
                idx = g.grp == gi
                M = s[:, idx] @ g.coef[idx].astype(np.float64)
                u = M + float(g.kappa[gi])
                if g.interval:
                    u = np.maximum(np.maximum(float(g.lo[gi]) - u, 0.0), u - float(g.hi[gi]))
                e = e + g.lam[gi] / 4.0 * u ** 2
        return e


def graph_arrays(G) -> Tuple[List[Hashable], np.ndarray, np.ndarray, np.ndarray]:
    """(node labels in G.nodes order, edge u index, edge v index, weight) in G.edges order.

    ``G`` is a networkx graph as produced by create_graphs.py:5-18, or a tuple (n | labels, eu, ev, w).
    """
    if isinstance(G, tuple):
        nodes, eu, ev, w = G
        labels = list(range(nodes)) if isinstance(nodes, (int, np.integer)) else list(nodes)
        return labels, np.asarray(eu, dtype=np.int64), np.asarray(ev, dtype=np.int64), np.asarray(w, dtype=np.float64)
    root = getattr(G, "_graph", None)
    if root is not None:
        # A subgraph VIEW (the recursion of BQM_clustering.py:113-203 calls itself on G.subgraph(S0 / S1)): networkx iterates
        # the nodes and adjacencies of a view smaller than half its parent in SET order, i.e. in an order that depends on
        # PYTHONHASHSEED -- the reference inherits that nondeterminism.  Pinned here to the induced subgraph in the ROOT
        # graph's node and adjacency order (what a view of more than half the parent yields, and what qa_graph_split emits).
        while getattr(root, "_graph", None) is not None:
            root = root._graph
        members = set(G.nodes)
        labels = [v for v in root.nodes if v in members]
        pos = {v: i for i, v in enumerate(labels)}
        eu_l, ev_l, w_l = [], [], []
        seen = set()
        for u in labels:
            for v, d in root.adj[u].items():
                if v in members and v not in seen:
                    eu_l.append(pos[u])
                    ev_l.append(pos[v])
                    w_l.append(d["weight"])
            seen.add(u)
        return labels, np.asarray(eu_l, dtype=np.int64), np.asarray(ev_l, dtype=np.int64), np.asarray(w_l, dtype=np.float64)
    labels = list(G.nodes)
    pos = {v: i for i, v in enumerate(labels)}
    m = G.number_of_edges()
    eu = np.empty(m, dtype=np.int64)
    ev = np.empty(m, dtype=np.int64)
    w = np.empty(m, dtype=np.float64)
    for c, (u, v, d) in enumerate(G.edges(data=True)):
        eu[c], ev[c], w[c] = pos[u], pos[v], d["weight"]
    return labels, eu, ev, w


def _edge_order_sum(n: int, eu: np.ndarray, ev: np.ndarray, vals: np.ndarray) -> np.ndarray:
    """out[u] += vals[c]; out[v] += vals[c] for edges in order (the reference's ``Q[(u,u)] += ...`` loops)."""
    return _accumulate_rows(np.zeros(n), eu, ev, vals)


def _canonical(r: np.ndarray, c: np.ndarray, q: np.ndarray):
    """Sort couplers by (row=larger index, col=smaller index): dimod ``to_numpy_vectors`` order."""
    lo = np.minimum(r, c)
    hi = np.maximum(r, c)
    order = np.lexsort((lo, hi))
    return hi[order].astype(np.int32), lo[order].astype(np.int32), np.asarray(q, dtype=np.float64)[order]


def _total_weight(G, n: int, eu: np.ndarray, ev: np.ndarray, w: np.ndarray) -> float:
    """``G.size(weight='weight')`` exactly as networkx computes it: sum of the weighted degrees (node order, each degree
    summed in adjacency order) divided by 2 -- NOT the plain sum of edge weights (differs in the last bits)."""
    if not isinstance(G, tuple) and getattr(G, "_graph", None) is None:
        return float(G.size(weight="weight"))      # (Python >= 3.12: sum() is compensated; bit-pinned by the golden fixtures)
    # arrays and subgraph views: plain left-to-right adds in the canonical order (graph_arrays), like the device builders
    deg = _edge_order_sum(n, eu, ev, np.asarray(w, dtype=np.float64))  # adjacency order of a graph built edge by edge
    return _seq_sum(deg) / 2


# ------------------------------------------------------------------------------------------------
# 2-way models (BQM_clustering.py) and the pruning QUBO (QA_subsampling.py)
# ------------------------------------------------------------------------------------------------
def cut_balance_model(G, gamma_factor: float, k: float = 8.0, structured: bool = True) -> LoweredModel:
    """``clustering_bqm`` QUBO (BQM_clustering.py:29-47; same Q in other_tools.py:28-46).

    Q_ii = k*d_i + gamma*(1-n), Q_ij = -2*k*w_ij + 2*gamma on edges and 2*gamma on every other pair,
    gamma = gamma_factor*W/n, k = 8 (hard-coded at :33).  E(x) = k*cut_w(x) + gamma*S*(S-n).
    """
    labels, eu, ev, w = graph_arrays(G)
    n = len(labels)
    W = _total_weight(G, n, eu, ev, w)
    gamma = gamma_factor * W / n
    diag = _edge_order_sum(n, eu, ev, k * w)
    meta = {"kind": "bqm", "builder": "cut_balance", "gamma": gamma, "k": k, "W": W}
    if structured:
        r, c, q = _canonical(eu, ev, k * -2 * w)
        h, J, off = qubo_to_ising_vectors(diag, r, c, q)
        groups = Groups(np.zeros(n, dtype=np.int32), np.ones(n, dtype=np.int32), np.array([gamma]), np.array([0], dtype=np.int64))
        return LoweredModel(h, r, c, J, off - gamma * n * n / 4.0, labels, groups, meta)
    diag = diag + gamma * (1 - n)
    dense = np.full((n, n), 2 * gamma)
    lo, hi = np.minimum(eu, ev), np.maximum(eu, ev)
    dense[hi, lo] = k * -2 * w + 2 * gamma
    r, c = np.tril_indices(n, -1)
    h, J, off = qubo_to_ising_vectors(diag, r.astype(np.int32), c.astype(np.int32), dense[r, c])
    return LoweredModel(h, r.astype(np.int32), c.astype(np.int32), J, off, labels, None, meta)


def cut_linear_model(G, gamma_factor: float, k: float) -> LoweredModel:
    """``clustering_bqm_2`` QUBO (BQM_clustering.py:210-236): Q_ii = k*d_i + gamma, Q_uv = -2*k*w, gamma = (W/n)*gamma_factor."""
    labels, eu, ev, w = graph_arrays(G)
    n = len(labels)
    W = _total_weight(G, n, eu, ev, w)
    gamma = (W / n) * gamma_factor
    diag = _edge_order_sum(n, eu, ev, k * w) + gamma
    r, c, q = _canonical(eu, ev, k * -2 * w)
    h, J, off = qubo_to_ising_vectors(diag, r, c, q)
    return LoweredModel(h, r, c, J, off, labels, None, {"kind": "bqm", "builder": "cut_linear", "gamma": gamma, "k": k})


def cut_inequality_bqm(G, gamma_factor: float, size_limit: int, k: float = 8.0) -> BinaryQuadraticModel:
    """``clustering_bqm_3`` model (BQM_clustering.py:364-380): k*cut QUBO + size_limit <= sum x <= n/6 as a slack penalty."""
    labels, eu, ev, w = graph_arrays(G)
    n = len(labels)
    W = _total_weight(G, n, eu, ev, w)
    gamma = gamma_factor * W / n
    Q = {}
    for c in range(len(w)):
        u, v = labels[eu[c]], labels[ev[c]]
        Q[(u, u)] = Q.get((u, u), 0) + k * w[c]
        Q[(v, v)] = Q.get((v, v), 0) + k * w[c]
        Q[(u, v)] = Q.get((u, v), 0) + k * -2 * w[c]
    bqm = BinaryQuadraticModel.from_qubo(Q)
    x = [str(v) for v in labels]
    c1 = [(x[int(v)], 1) for v in labels]  # reference indexes x by int(node label): labels must be '0'..'n-1'
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        bqm.add_linear_inequality_constraint(c1, lb=size_limit, ub=n / 6, lagrange_multiplier=gamma, label="c1_constraint")
    return bqm


def subsampling_model(G, gamma: float, P: float = 1.0) -> LoweredModel:
    """``graph_subsampling`` QUBO (QA_subsampling.py:26-35): Q_ii = gamma - sum_j P(1-w_ij), Q_uv = P(1-w_uv)."""
    labels, eu, ev, w = graph_arrays(G)
    n = len(labels)
    diag = _edge_order_sum(n, eu, ev, -P * (1 - w)) + gamma
    r, c, q = _canonical(eu, ev, P * (1 - w))
    h, J, off = qubo_to_ising_vectors(diag, r, c, q)
    return LoweredModel(h, r, c, J, off, labels, None, {"kind": "bqm", "builder": "subsampling", "gamma": gamma})


# ------------------------------------------------------------------------------------------------
# k-way models
# ------------------------------------------------------------------------------------------------
def _onehot_couplers(n: int, K: int, A: float):
    """Intra-cell quadratic +2A between the K bits of each cell (variable index i*K + c)."""
    ca, cb = np.triu_indices(K, 1)
    base = (np.arange(n, dtype=np.int64) * K)[:, None]
    lo = (base + ca[None, :]).ravel()
    hi = (base + cb[None, :]).ravel()
    return hi, lo, np.full(lo.shape, 2.0 * A)


def default_onehot_penalty(n: int, K: int, eu, ev, quad_edge: np.ndarray, lin: np.ndarray, gamma_pair: float) -> float:
    """A larger than the most any single bit can gain: |linear| + sum of |edge couplings| + all-pairs term."""
    gain = np.abs(lin).astype(np.float64)
    gain = gain + _accumulate_rows(np.zeros(n), eu, ev, np.abs(quad_edge))
    return float(gain.max() + 2.0 * abs(gamma_pair) * n / max(K, 1) + 1.0)


def dqm_model(G, num_of_clusters: int, gamma: float, penalty: Optional[float] = None, semantics: str = "as_written",
              structured: bool = True) -> LoweredModel:
    """``clustering_dqm`` model (DQM_clustering.py:29-43) expanded one-hot: binary variable (cell i, case c) -> i*K + c.

    as_written (``set_*`` overwrite each other, comment at :39): linear_i = weight of the last edge touching i
    (gamma*(1-n/K) for isolated cells), same-case quadratic = -2*w on edges and 2*gamma on every other pair.
    intended: linear_i = gamma*(1-n/K) + d_i, same-case quadratic = 2*gamma - 2*w on edges.
    One-hot is enforced by ``penalty``*(sum_c x_ic - 1)^2 (LeapHybridDQMSampler enforces it natively; the
    penalty value is ours and is reported in ``meta``).
    """
    if semantics not in ("as_written", "intended"):
        raise ValueError("semantics must be 'as_written' or 'intended'")
    labels, eu, ev, w = graph_arrays(G)
    n, K = len(labels), int(num_of_clusters)
    base_lin = gamma * (1 - n / K)
    if semantics == "as_written":
        lin = np.full(n, base_lin)
        for c in range(len(w)):  # last set_linear wins (DQM_clustering.py:42-43)
            lin[eu[c]] = w[c]
            lin[ev[c]] = w[c]
        # edges overwrite the all-pairs 2*gamma (:41); written relative to the all-pairs term that stays rank-1
        edge_q_total = -2 * w
    else:
        lin = base_lin + _edge_order_sum(n, eu, ev, w)
        edge_q_total = 2 * gamma - 2 * w
    A = default_onehot_penalty(n, K, eu, ev, edge_q_total, lin, gamma) if penalty is None else float(penalty)
    meta = {"kind": "dqm", "builder": "dqm", "num_cases": K, "cells": labels, "penalty": A, "gamma": gamma,
            "semantics": semantics}
    var_labels = [(v, c) for v in labels for c in range(K)]
    cases = np.arange(K, dtype=np.int64)
    oh_r, oh_c, oh_q = _onehot_couplers(n, K, A)
    lin_x = np.repeat(lin, K) - A
    offset_onehot = A * n
    if structured:
        edge_q = edge_q_total - 2 * gamma  # minus the pair term carried by the group
        er = (eu[:, None] * K + cases[None, :]).ravel()
        ec = (ev[:, None] * K + cases[None, :]).ravel()
        eq = np.repeat(edge_q, K)
        r, c, q = _canonical(np.concatenate([er, oh_r]), np.concatenate([ec, oh_c]), np.concatenate([eq, oh_q]))
        h, J, off = qubo_to_ising_vectors(lin_x, r, c, q)
        # gamma * sum_c (N_c^2 - N_c) = gamma * sum_c [(N_c - 1/2)^2 - 1/4]  ->  lam=gamma, kappa = n - 1
        grp = np.tile(np.arange(K, dtype=np.int32), n)
        groups = Groups(grp, np.ones(n * K, dtype=np.int32), np.full(K, float(gamma)), np.full(K, n - 1, dtype=np.int64))
        return LoweredModel(h, r, c, J, off + offset_onehot - gamma * K / 4.0, var_labels, groups, meta)
    dense = np.full((n, n), 2 * gamma)
    lo, hi = np.minimum(eu, ev), np.maximum(eu, ev)
    dense[hi, lo] = edge_q_total
    pr, pc = np.tril_indices(n, -1)
    er = (pr[:, None] * K + cases[None, :]).ravel()
    ec = (pc[:, None] * K + cases[None, :]).ravel()
    eq = np.repeat(dense[pr, pc], K)
    r, c, q = _canonical(np.concatenate([er, oh_r]), np.concatenate([ec, oh_c]), np.concatenate([eq, oh_q]))
    h, J, off = qubo_to_ising_vectors(lin_x, r, c, q)
    return LoweredModel(h, r, c, J, off + offset_onehot, var_labels, None, meta)


def dense_kway_model(A: np.ndarray, num_of_clusters: int, gamma: float, penalty: Optional[float] = None,
                     labels: Optional[List[Hashable]] = None) -> LoweredModel:
    """BASELINE.json config 5: the DQM-style k-way model of ``clustering_dqm`` (DQM_clustering.py:29-43, "intended" semantics)
    on a DENSE symmetric affinity ``A`` (zero diagonal) instead of a sparse SNN graph: every pair of cells is an edge, so
    same-case quadratic = 2*gamma - 2*A_ij for all i != j, linear_i = gamma*(1 - n/K) + sum_j A_ij, one-hot penalty as in
    ``dqm_model``.  Built without a networkx round trip (n^2 K / 2 couplers, emitted directly in dimod's vector order:
    row = larger index, ascending columns).  ``meta['num_cases']`` lets the sampler enable the tensor-core form."""
    A = np.asarray(A, dtype=np.float64)
    n, K = A.shape[0], int(num_of_clusters)
    if A.shape != (n, n):
        raise ValueError("A must be square")
    labels = list(range(n)) if labels is None else list(labels)
    lin = gamma * (1 - n / K) + A.sum(axis=1)
    pair_q = 2 * gamma - 2 * A                       # QUBO coefficient of x_ic x_jc
    Apen = float(np.abs(lin).max() + np.abs(pair_q).sum(axis=1).max() + 1.0) if penalty is None else float(penalty)
    meta = {"kind": "dqm", "builder": "dense_kway", "num_cases": K, "cells": labels, "penalty": Apen, "gamma": gamma,
            "semantics": "intended", "dense": True}
    # row v = i*K + c holds, ascending: (j*K + c) for j < i, then (i*K + c2) for c2 < c
    cnt = (np.arange(n)[:, None] + np.arange(K)[None, :]).ravel()             # couplers per row
    rows = np.repeat(np.arange(n * K, dtype=np.int64), cnt)
    first = np.cumsum(cnt) - cnt
    pos = np.arange(rows.shape[0], dtype=np.int64) - first[rows]             # position inside the row
    i, c = rows // K, rows % K
    inter = pos < i
    cols = np.where(inter, pos * K + c, i * K + (pos - i))
    q = np.where(inter, pair_q[i, np.minimum(pos, n - 1)], 2.0 * Apen)
    lin_x = np.repeat(lin, K) - Apen
    h, J, off = qubo_to_ising_vectors(lin_x, rows.astype(np.int32), cols.astype(np.int32), q)
    var_labels = [(v, cc) for v in labels for cc in range(K)]
    return LoweredModel(h, rows.astype(np.int32), cols.astype(np.int32), J, off + Apen * n, var_labels, None, meta)


def slack_coefficients(upper: int) -> List[int]:
    """Binary-encoded slack spanning exactly 0..upper (dimod add_linear_inequality_constraint; SURVEY.md A3)."""
    if upper <= 0:
        return []
    nbits = int(math.floor(math.log2(upper)))
    coeffs = [2 ** j for j in range(nbits)]
    if upper - 2 ** nbits >= 0:
        coeffs.append(upper - 2 ** nbits + 1)
    return coeffs


SIZE_LOWERINGS = ("slack", "interval")
INT64_MIN, INT64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max


def _cqm_size_penalty(A: float, n: int, size_lowering: str) -> float:
    """Default B.  slack: B = A / n (see cqm_model).  interval: B = A -- a single flip gains less than A in objective (A is
    above every cell's objective scale by construction), so one unit of size violation costs more than any flip can gain;
    A / n was a workaround for frozen slack bits, which the interval form does not have."""
    if size_lowering not in SIZE_LOWERINGS:
        raise ValueError(f"size_lowering must be one of {SIZE_LOWERINGS}, not {size_lowering!r}")
    return A if size_lowering == "interval" else A / max(n, 1)


def cqm_model(G, num_of_clusters: int, min_size: int = 20, onehot_penalty: Optional[float] = None,
              size_penalty: Optional[float] = None, subindex: Optional[Sequence[int]] = None,
              structured: bool = True, size_lowering: str = "slack") -> LoweredModel:
    """``clustering_cqm`` / ``clustering_cqm_2`` model (CQM_clustering.py:30-48, 62-84) lowered to penalties.

    objective  sum_edges sum_p (x_ip + x_jp - 2*w_ij*x_ip*x_jp)            (:40-44; linear coefficient is 1, not w)
    one-hot    add_discrete per cell (:36-37)      ->  A * (sum_p x_ip - 1)^2
    size       sum_i x_ij >= min_size per cluster (:47-48, min_size = 20)
                                                   ->  B * (N_j - min_size - sum_b c_b*sigma_jb)^2, binary slack sigma
    Variable (cell i, cluster p) -> i*K + p with label 'v_{i},{p}' (i = node label, or ``subindex`` for cqm_2);
    slack sigma_jb -> n*K + j*nb + b with label 'slack_cluster_size{j}_{b}'.  A and B are ours (Leap's CQM solver
    handles constraints natively; defaults A = max degree + max sum |2w| + 1, B = A / n) and are reported in ``meta``.

    ``size_lowering="interval"``: no slack bits; each size constraint is an interval group with bounds [0, +inf) on
    u = 2 (N_j - min_size), i.e. the term  B * max(0, min_size - N_j)^2, evaluated by the kernels from the group counter.
    The cell part (h, couplers, offset) is the slack model's, bit for bit.  Default B = A (see ``_cqm_size_penalty``).
    """
    labels, eu, ev, w = graph_arrays(G)
    n, K = len(labels), int(num_of_clusters)
    cases = np.arange(K, dtype=np.int64)
    deg = _edge_order_sum(n, eu, ev, np.ones(len(w)))
    wdeg = _edge_order_sum(n, eu, ev, np.abs(2 * w))
    A = float(deg.max() + wdeg.max() + 1.0) if onehot_penalty is None else float(onehot_penalty)
    # size penalty: scaled so that one cell changing cluster moves it by at most 2*B*n = 2*A, the one-hot scale.  With B = 1
    # the binary slack bits (coefficients up to ~n/2) freeze at every temperature the objective cares about, the cell bits are
    # slaved to them and no read ends one-hot (measured: 0 of 100 000 reads on config 3); with B = A/n every read of the same
    # job is feasible.  The reference never meets this: Leap's CQM solver handles constraints natively.
    B = _cqm_size_penalty(A, n, size_lowering) if size_penalty is None else float(size_penalty)
    interval = size_lowering == "interval"
    coeffs = [] if interval else slack_coefficients(n - min_size)
    nb = len(coeffs)
    names = labels if subindex is None else list(subindex)
    var_labels: List[Hashable] = [f"v_{names[i]},{p}" for i in range(n) for p in range(K)]
    var_labels += [f"slack_cluster_size{j}_{b}" for j in range(K) for b in range(nb)]
    nx_ = n * K
    nvar = nx_ + K * nb
    lin = np.zeros(nvar)
    lin[:nx_] = np.repeat(deg, K) - A
    oh_r, oh_c, oh_q = _onehot_couplers(n, K, A)
    er = (eu[:, None] * K + cases[None, :]).ravel()
    ec = (ev[:, None] * K + cases[None, :]).ravel()
    eq = np.repeat(-2 * w, K)
    r, c, q = _canonical(np.concatenate([er, oh_r]), np.concatenate([ec, oh_c]), np.concatenate([eq, oh_q]))
    h, J, off = qubo_to_ising_vectors(lin, r, c, q)
    # B * (sum a x - min_size)^2 with a = +1 (cells), -c_b (slack):  lam = B, kappa = sum(a) - 2*min_size
    grp = np.full(nvar, -1, dtype=np.int32)
    coef = np.zeros(nvar, dtype=np.int32)
    grp[:nx_] = np.tile(np.arange(K, dtype=np.int32), n)
    coef[:nx_] = 1
    for j in range(K):
        sl = slice(nx_ + j * nb, nx_ + (j + 1) * nb)
        grp[sl] = j
        coef[sl] = -np.asarray(coeffs, dtype=np.int32)
    kappa = np.full(K, n - sum(coeffs) - 2 * min_size, dtype=np.int64)
    groups = Groups(grp, coef, np.full(K, B), kappa)
    if interval:
        groups.lo, groups.hi = np.zeros(K, dtype=np.int64), np.full(K, INT64_MAX, dtype=np.int64)
    meta = {"kind": "cqm", "builder": "cqm", "num_cases": K, "cells": labels, "names": list(names), "min_size": min_size,
            "onehot_penalty": A, "size_penalty": B, "num_cell_variables": nx_, "size_lowering": size_lowering}
    if not interval:
        meta["slack_coefficients"] = coeffs
    model = LoweredModel(h, r, c, J, off + A * n, var_labels, groups, meta)
    return model if structured else model.materialise()


def consistent_slack(states: np.ndarray, meta: Dict) -> np.ndarray:
    """Set the slack bits of +-1 CQM states (in place) to the binary encoding of ``max(N_j - min_size, 0)``, N_j = number of
    cells whose bit for cluster j is set, so that the size penalty B*(N_j - min_size - slack_j)^2 starts at zero.

    Why: with uniformly random slack bits the penalty starts at ~(n/2)^2 per cluster and the high slack bits (a flip moves it by
    ~c_b * n) are frozen at every temperature the objective cares about; the cell bits are then slaved to the random slack values
    and no read ends one-hot (measured on config 3: 0 of 100 000 reads).  The reference never meets this -- it hands the CQM to
    Leap's hybrid solver, which treats constraints natively.  Used by ``sample_cqm`` for generated initial states."""
    K = int(meta["num_cases"])
    nx = int(meta["num_cell_variables"])
    coeffs = np.asarray(meta["slack_coefficients"], dtype=np.int64)
    nb = len(coeffs)
    if nb == 0:
        return states
    cells = nx // K
    counts = (states[:, :nx].reshape(len(states), cells, K) > 0).sum(axis=1).astype(np.int64)          # [R][K]
    v = np.clip(counts - int(meta["min_size"]), 0, int(coeffs.sum()))
    for b in np.argsort(-coeffs, kind="stable"):          # greedy from the largest coefficient: exact for dimod's encoding
        take = v >= coeffs[b]
        v = v - coeffs[b] * take
        states[:, nx + np.arange(K) * nb + b] = np.where(take, 1, -1).astype(states.dtype)
    return states


# ------------------------------------------------------------------------------------------------
# everything about a model EXCEPT its vectors: what the host needs when the vectors are built on the device (qa_build_*)
# ------------------------------------------------------------------------------------------------
def device_spec(kind: str, G, **p) -> Dict:
    """Graph arrays, variable labels, penalties and ``meta`` of the model ``kind`` ('cut_balance', 'cut_linear', 'subsampling',
    'dqm', 'cqm') -- O(n + m) numpy, no O(n^2) term, no Python loop over pairs.  The vectors come from ``Context.build_*``; they
    are bit-identical to the host builders above (tests/test_gpu_builders.py)."""
    labels, eu, ev, w = graph_arrays(G)
    n = len(labels)
    graph = (n, eu.astype(np.int32), ev.astype(np.int32), w)
    if kind == "cut_balance":
        return {"graph": graph, "labels": labels, "meta": {"kind": "bqm", "builder": "cut_balance", "k": p.get("k", 8.0)}}
    if kind == "cut_linear":
        return {"graph": graph, "labels": labels, "meta": {"kind": "bqm", "builder": "cut_linear", "k": p.get("k", 1.0)}}
    if kind == "subsampling":
        return {"graph": graph, "labels": labels, "meta": {"kind": "bqm", "builder": "subsampling", "gamma": p["gamma"]}}
    K = int(p["num_of_clusters"])
    if kind == "dqm":
        gamma, semantics = p["gamma"], p.get("semantics", "as_written")
        if semantics not in ("as_written", "intended"):
            raise ValueError("semantics must be 'as_written' or 'intended'")
        base_lin = gamma * (1 - n / K)
        if semantics == "as_written":
            lin = np.full(n, base_lin)
            last = np.full(n, -1, dtype=np.int64)           # last edge touching every cell (DQM_clustering.py:42-43)
            idx = np.arange(len(w), dtype=np.int64)
            np.maximum.at(last, eu, idx)
            np.maximum.at(last, ev, idx)
            lin[last >= 0] = w[last[last >= 0]]
            edge_q_total = -2 * w
        else:
            lin = base_lin + _edge_order_sum(n, eu, ev, w)
            edge_q_total = 2 * gamma - 2 * w
        A = default_onehot_penalty(n, K, eu, ev, edge_q_total, lin, gamma) if p.get("penalty") is None else float(p["penalty"])
        meta = {"kind": "dqm", "builder": "dqm", "num_cases": K, "cells": labels, "penalty": A, "gamma": gamma,
                "semantics": semantics}
        return {"graph": graph, "labels": [(v, c) for v in labels for c in range(K)], "meta": meta, "penalty": A}
    if kind == "cqm":
        min_size = int(p.get("min_size", 20))
        deg = _edge_order_sum(n, eu, ev, np.ones(len(w)))
        wdeg = _edge_order_sum(n, eu, ev, np.abs(2 * w))
        A = float(deg.max() + wdeg.max() + 1.0) if p.get("onehot_penalty") is None else float(p["onehot_penalty"])
        size_lowering = p.get("size_lowering", "slack")
        B = _cqm_size_penalty(A, n, size_lowering) if p.get("size_penalty") is None else float(p["size_penalty"])  # see cqm_model
        coeffs = [] if size_lowering == "interval" else slack_coefficients(n - min_size)
        names = labels if p.get("subindex") is None else list(p["subindex"])
        var_labels: List[Hashable] = [f"v_{names[i]},{q}" for i in range(n) for q in range(K)]
        var_labels += [f"slack_cluster_size{j}_{b}" for j in range(K) for b in range(len(coeffs))]
        meta = {"kind": "cqm", "builder": "cqm", "num_cases": K, "cells": labels, "names": list(names), "min_size": min_size,
                "onehot_penalty": A, "size_penalty": B, "num_cell_variables": n * K, "size_lowering": size_lowering}
        if size_lowering != "interval":
            meta["slack_coefficients"] = coeffs
        return {"graph": graph, "labels": var_labels, "meta": meta, "onehot_penalty": A, "size_penalty": B, "min_size": min_size,
                "size_lowering": size_lowering}
    raise ValueError(f"unknown model kind {kind!r}")


# ------------------------------------------------------------------------------------------------
# decoding (plot_and_save.py:36-63 read `.first.sample` this way)
# ------------------------------------------------------------------------------------------------
def decode_onehot(bits: np.ndarray, n: int, K: int) -> Tuple[np.ndarray, np.ndarray]:
    """bits [R][>= n*K] in {0,1} -> (case index [R][n], feasible [R][n]); infeasible cells take their first set bit (or 0)."""
    x = np.asarray(bits)[:, : n * K].reshape(-1, n, K)
    count = x.sum(axis=2)
    case = np.argmax(x, axis=2)
    return case.astype(np.int32), count == 1


def lowered_from_bqm(bqm: BinaryQuadraticModel) -> LoweredModel:
    """What neal does with a BQM: change_vartype(SPIN) then to_numpy_vectors (SURVEY.md row a7)."""
    spin = bqm.change_vartype("SPIN", inplace=False)
    ldata, (irow, icol, qdata), offset, labels = spin.to_numpy_vectors(return_labels=True)
    return LoweredModel(np.ascontiguousarray(ldata), np.ascontiguousarray(irow), np.ascontiguousarray(icol),
                        np.ascontiguousarray(qdata), float(offset), labels, None,
                        {"kind": "bqm", "vartype": bqm.vartype.name})
