"""Interval rank-1 groups on the CPU: the reference loop against the oracle and against exact arithmetic, and the host-side
lowerings (models.cqm_model(size_lowering="interval"), ConstrainedQuadraticModel.to_lowered(lowering="interval"))."""
import itertools
import math
from fractions import Fraction as Fr

import numpy as np
import pytest

import interval_reference as iref
from oracle import oracle
from scrna_seq_qannealing_clustering_b200 import models, schedule, snn
from scrna_seq_qannealing_clustering_b200.cqm import Binary, ConstrainedQuadraticModel

I64 = np.iinfo(np.int64)


@pytest.fixture(scope="module")
def graph256():
    return snn.synthetic_snn(256, k=5, seed=3)[0]


def _exact_energy(h, starts, ends, w, groups, s):
    grp, coef, lam, kap = groups[:4]
    lo, hi = (groups[4], groups[5]) if len(groups) == 6 else (None, None)
    e = sum(Fr(float(h[v])) * s[v] for v in range(len(h)))
    e += sum(Fr(float(x)) * s[u] * s[v] for u, v, x in zip(starts, ends, w))
    for g in range(len(lam)):
        u = sum(int(coef[v]) * s[v] for v in range(len(s)) if grp[v] == g) + int(kap[g])
        d = u if lo is None else max(int(lo[g]) - u, 0, u - int(hi[g]))
        e += Fr(float(lam[g])) * d * d / 4
    return e


def _small_model(n=12, seed=0):
    rng = np.random.default_rng(seed)
    pairs = [(u, v) for u in range(n) for v in range(u) if rng.random() < 0.3]
    starts = np.array([p[0] for p in pairs], dtype=np.int32)
    ends = np.array([p[1] for p in pairs], dtype=np.int32)
    w = rng.normal(size=len(pairs)).round(3)
    h = rng.normal(size=n).round(3)
    # one-sided (>=), one-sided (<=), two-sided with mixed signs, negative kappa
    grp = np.array([0, 0, 0, 1, 1, 1, 2, 2, 2, 2, 3, -1][:n], dtype=np.int32)
    coef = np.array([1, 2, 1, 1, 1, 3, 2, -1, 3, -2, 5, 0][:n], dtype=np.int32)
    lam = np.array([0.75, 1.3, 0.4, 2.1])
    kap = np.array([-1, 2, -3, -4], dtype=np.int64)
    lo = np.array([0, I64.min, -2, 1], dtype=np.int64)
    hi = np.array([I64.max, 0, 3, 1], dtype=np.int64)
    return h, starts, ends, w, (grp, coef, lam, kap, lo, hi)


def test_zero_bounds_reproduce_equality_groups_bitwise(graph256):
    model = models.cqm_model(graph256, 4)
    eq = model.groups.astuple()
    G = len(eq[2])
    ivl = eq + (np.zeros(G, dtype=np.int64), np.zeros(G, dtype=np.int64))
    R, n = 24, model.num_variables
    betas, spb = schedule.make_beta_schedule((0.05, 6.0), 40, 1, "geometric")
    seeds = schedule.per_read_seeds(5, R)
    init = schedule.random_spin_states(R, n, 5)
    runs = []
    for fn, g in ((oracle.sample_ising, eq), (iref.sample_ising, eq), (iref.sample_ising, ivl)):
        st = init.copy()
        e, c = fn(model.h, model.starts, model.ends, model.weights, st, betas, spb, seeds, groups=g)
        runs.append((st, e, c))
    for st, e, c in runs[1:]:
        assert np.array_equal(st, runs[0][0])
        assert np.array_equal(e.view(np.uint64), runs[0][1].view(np.uint64))
        assert c == runs[0][2]
    assert runs[0][2]["accepted"] > 0


def test_flip_cost_and_energy_exact_brute_force():
    h, starts, ends, w, groups = _small_model()
    n = len(h)
    lam = groups[2]
    for bits in itertools.product((-1, 1), repeat=n):
        s = np.array(bits, dtype=np.int8)
        e0 = _exact_energy(h, starts, ends, w, groups, bits)
        got = iref.state_energies(h, starts, ends, w, s[None, :], groups)[0]
        assert abs(Fr(got) - e0) <= Fr(1, 10 ** 9) * (1 + abs(e0))
        if sum(bits) % 3:   # every third state: all flips (keeps the brute force quick)
            continue
        for v in range(n):
            g = groups[0][v]
            s2 = list(bits)
            s2[v] = -s2[v]
            zero_h = np.zeros(n)
            exact = (_exact_energy(zero_h, [], [], [], groups, s2) - _exact_energy(zero_h, [], [], [], groups, bits))
            got = iref.group_flip_cost(s, v, groups)
            # integers exact, one rounding: lambda * (integer difference * 0.25)
            if g < 0:
                assert got == 0.0 and exact == 0
            else:
                delta = exact * 4 / Fr(float(lam[g]))
                assert delta.denominator == 1
                assert got == float(lam[g]) * (float(delta) * 0.25)
                assert abs(Fr(got) - exact) <= abs(exact) * Fr(1, 2 ** 52)


def _py_anneal_interval(h, starts, ends, w, groups, state, betas, spb, seed):
    """Pure-Python restatement of the Metropolis loop with interval groups (neal's loop + the lazy group term)."""
    grp, coef, lam, kap, lo, hi = (np.asarray(a).tolist() for a in groups)
    n = len(h)
    adj = [[] for _ in range(n)]
    for u, v, x in zip(starts.tolist(), ends.tolist(), w.tolist()):
        adj[u].append((v, x))
        adj[v].append((u, x))
    mask = (1 << 64) - 1
    s0, s1 = (seed if seed else mask), 0

    def rnd():
        nonlocal s0, s1
        x, y = s0, s1
        s0 = y
        x = (x ^ (x << 23)) & mask
        s1 = x ^ y ^ (x >> 17) ^ (y >> 26)
        return (s1 + y) & mask

    def dist(u, g):
        return max(lo[g] - u, 0, u - hi[g])

    s = [int(x) for x in state]
    dE = [-2 * s[v] * (h[v] + sum(s[j] * x for j, x in adj[v])) for v in range(n)]
    M = [0] * len(lam)
    for v in range(n):
        if grp[v] >= 0:
            M[grp[v]] += coef[v] * s[v]
    draws = acc = 0
    for beta in betas:
        for _ in range(spb):
            thr = 44.36142 / beta
            for v in range(n):
                d = dE[v]
                g = grp[v]
                if g >= 0:
                    u = M[g] + kap[g]
                    d1, d0 = dist(u - 2 * coef[v] * s[v], g), dist(u, g)
                    d = d + lam[g] * (float(d1 * d1 - d0 * d0) * 0.25)
                if d >= thr:
                    continue
                flip = d <= 0.0
                if not flip:
                    draws += 1
                    flip = math.exp(-d * beta) * 18446744073709551616.0 > float(rnd())
                if flip:
                    acc += 1
                    for j, x in adj[v]:
                        dE[j] += 4 * s[v] * x * s[j]
                    if g >= 0:
                        M[g] -= 2 * coef[v] * s[v]
                    s[v] = -s[v]
                    dE[v] = -dE[v]
    return np.array(s, dtype=np.int8), draws, acc


def test_python_restatement_matches_reference():
    h, starts, ends, w, groups = _small_model(12, seed=4)
    R = 6
    betas, spb = schedule.make_beta_schedule((0.1, 5.0), 30, 2, "geometric")
    seeds = schedule.per_read_seeds(9, R)
    init = schedule.random_spin_states(R, len(h), 9)
    st = init.copy()
    e, c = iref.sample_ising(h, starts, ends, w, st, betas, spb, seeds, groups=groups)
    draws = acc = 0
    for r in range(R):
        ps, d, a = _py_anneal_interval(h, starts, ends, w, groups, init[r], betas, spb, int(seeds[r]))
        assert np.array_equal(ps, st[r])
        draws, acc = draws + d, acc + a
    assert (draws, acc) == (c["draws"], c["accepted"])
    assert np.array_equal(e.view(np.uint64), iref.state_energies(h, starts, ends, w, st, groups).view(np.uint64))


def test_cqm_interval_model(graph256):
    slack = models.cqm_model(graph256, 4, min_size=40)
    ivl = models.cqm_model(graph256, 4, min_size=40, size_lowering="interval")
    nx = slack.meta["num_cell_variables"]
    assert ivl.num_variables == nx and not any(str(l).startswith("slack_") for l in ivl.labels)
    assert ivl.labels == slack.labels[:nx]
    assert np.array_equal(ivl.h.view(np.uint64), slack.h[:nx].view(np.uint64))
    cell = (slack.starts < nx) & (slack.ends < nx)
    assert cell.all()   # slack bits have no couplers: they live in the groups only
    assert np.array_equal(ivl.starts, slack.starts) and np.array_equal(ivl.ends, slack.ends)
    assert np.array_equal(ivl.weights.view(np.uint64), slack.weights.view(np.uint64))
    assert ivl.offset == slack.offset
    assert "slack_coefficients" not in ivl.meta and ivl.meta["size_lowering"] == "interval"
    A, B = ivl.meta["onehot_penalty"], ivl.meta["size_penalty"]
    assert B == A
    with pytest.raises(ValueError):
        ivl.materialise()
    # energies = objective + A * sum (onehot - 1)^2 + B * sum max(0, min_size - N_j)^2
    n, K = 256, 4
    _, eu, ev, w = models.graph_arrays(graph256)
    rng = np.random.default_rng(1)
    S = rng.choice([-1, 1], size=(8, nx)).astype(np.int8)
    x = ((S + 1) // 2).reshape(8, n, K).astype(np.float64)
    obj = sum(x[:, eu, p] + x[:, ev, p] - 2 * w * x[:, eu, p] * x[:, ev, p] for p in range(K)).sum(axis=1)
    want = obj + A * ((x.sum(axis=2) - 1) ** 2).sum(axis=1) + B * (np.maximum(0, 40 - x.sum(axis=1)) ** 2).sum(axis=1)
    assert np.allclose(ivl.energies(S), want, rtol=1e-12, atol=1e-9)
    ref = iref.state_energies(ivl.h, ivl.starts, ivl.ends, ivl.weights, S, ivl.groups.astuple()) + ivl.offset
    assert np.allclose(ref, want, rtol=1e-12, atol=1e-9)


def test_cqm_interval_tiny_ground_state_is_constrained_optimum():
    eu, ev, w = np.array([0, 1, 2, 3, 0]), np.array([1, 2, 3, 4, 4]), np.array([0.9, 0.2, 0.8, 0.1, 0.5])
    n, K, min_size = 5, 2, 2
    m = models.cqm_model((n, eu, ev, w), K, min_size=min_size, size_lowering="interval")
    S = np.array(list(itertools.product((-1, 1), repeat=n * K)), dtype=np.int8)
    E = m.energies(S)
    best = S[np.argmin(E)]
    x = ((best + 1) // 2).reshape(n, K)
    assert (x.sum(axis=1) == 1).all() and (x.sum(axis=0) >= min_size).all()
    # the CQM's constrained optimum by enumeration of feasible assignments
    opt = math.inf
    for assign in itertools.product(range(K), repeat=n):
        sizes = np.bincount(assign, minlength=K)
        if (sizes < min_size).any():
            continue
        xx = np.zeros((n, K))
        xx[np.arange(n), assign] = 1
        opt = min(opt, sum((xx[eu, p] + xx[ev, p] - 2 * w * xx[eu, p] * xx[ev, p]).sum() for p in range(K)))
    assert E.min() == pytest.approx(opt, abs=1e-9)


def _cqm_three_senses():
    cqm = ConstrainedQuadraticModel()
    xs = [Binary(f"x{i}") for i in range(9)]
    cqm.set_objective(xs[0] * xs[1] + 2 * xs[2] - xs[3] + xs[4] * xs[5] - 0.5 * xs[8])
    cqm.add_constraint(xs[0] + 2 * xs[1] + xs[2] >= 2, label="ge")
    cqm.add_constraint(xs[3] + xs[4] - xs[5] <= 0, label="le")
    cqm.add_constraint(xs[6] + xs[7] + xs[8] == 1, label="eq")
    return cqm


def test_to_lowered_interval_bounds_and_penalties():
    cqm = _cqm_three_senses()
    B = 3.0
    m = cqm.to_lowered(onehot_penalty=5.0, constraint_penalty=B, lowering="interval")
    g = m.groups
    assert m.num_variables == 9 and sorted(m.labels) == [f"x{i}" for i in range(9)]
    assert list(g.lo) == [0, I64.min, 0] and list(g.hi) == [I64.max, 0, 0]
    assert list(g.kappa) == [4 - 4, 1 + 0, 3 - 2]
    S = np.array(list(itertools.product((-1, 1), repeat=9)), dtype=np.int8)
    X = ((S + 1) // 2)[:, [list(m.labels).index(f"x{i}") for i in range(9)]]
    obj = X[:, 0] * X[:, 1] + 2 * X[:, 2] - X[:, 3] + X[:, 4] * X[:, 5] - 0.5 * X[:, 8]
    viol = (np.maximum(0, 2 - (X[:, 0] + 2 * X[:, 1] + X[:, 2])) ** 2 + np.maximum(0, X[:, 3] + X[:, 4] - X[:, 5]) ** 2
            + (X[:, 6] + X[:, 7] + X[:, 8] - 1) ** 2)
    assert np.allclose(m.energies(S), obj + B * viol, atol=1e-12)
    ref = iref.state_energies(m.h, m.starts, m.ends, m.weights, S, g.astuple()) + m.offset
    assert np.allclose(ref, obj + B * viol, atol=1e-12)
    with pytest.raises(ValueError):
        m.materialise()


def test_to_lowered_interval_rejects():
    cqm = _cqm_three_senses()
    cqm.add_constraint(Binary("x0") + Binary("y") >= 1, label="overlap")
    with pytest.raises(ValueError, match="x0"):
        cqm.to_lowered(lowering="interval")
    cqm = ConstrainedQuadraticModel()
    cqm.add_constraint(0.5 * Binary("a") + Binary("b") >= 1, label="frac")
    with pytest.raises(ValueError, match="frac"):
        cqm.to_lowered(lowering="interval")
    cqm = ConstrainedQuadraticModel()
    for i in range(65):
        cqm.add_constraint(Binary(f"a{i}") + Binary(f"b{i}") >= 1, label=f"c{i}")
    with pytest.raises(ValueError, match="at most"):
        cqm.to_lowered(lowering="interval")
    assert cqm.to_lowered().num_variables > 130   # the slack lowering is unchanged


def test_device_spec_interval():
    g = snn.synthetic_snn(64, k=4, seed=2)[0]
    spec = models.device_spec("cqm", g, num_of_clusters=3, min_size=10, size_lowering="interval")
    assert len(spec["labels"]) == 64 * 3 and "slack_coefficients" not in spec["meta"]
    assert spec["size_penalty"] == spec["onehot_penalty"]
    with pytest.raises(ValueError):
        models.cqm_model(g, 3, size_lowering="bogus")
