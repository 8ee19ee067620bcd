"""dwave-samplers' sample options on the CPU: random variable order and Gibbs acceptance in the test reference
(tests/native/proposals_sa_ref.cpp), tied to the oracle and the interval reference where the options are at their defaults,
pinned to a pure-Python restatement of the rules, checked for the Boltzmann distribution at a fixed beta, and the sampler's
argument handling without a device."""
import itertools
import math
import warnings

import numpy as np
import pytest

import interval_reference as iref
import proposals_reference as pref
from oracle import oracle
from scrna_seq_qannealing_clustering_b200 import models, schedule, snn
from scrna_seq_qannealing_clustering_b200.bqm import BinaryQuadraticModel
from scrna_seq_qannealing_clustering_b200.sampler import B200SimulatedAnnealingSampler

COMBOS = [(o, p) for o in (pref.SEQUENTIAL, pref.RANDOM) for p in (pref.METROPOLIS, pref.GIBBS)]
TWO64 = 18446744073709551616.0


def _tiny_model(n, seed, groups=True):
    rng = np.random.default_rng(seed)
    pairs = [(u, v) for u in range(n) for v in range(u) if rng.random() < 0.4]
    starts = np.array([p[0] for p in pairs], dtype=np.int32)
    ends = np.array([p[1] for p in pairs], dtype=np.int32)
    w = rng.normal(size=len(pairs)).round(3)
    h = rng.normal(size=n).round(3)
    g = None
    if groups:
        grp = np.where(np.arange(n) < n // 2, 0, np.where(np.arange(n) < n - 1, 1, -1)).astype(np.int32)
        coef = rng.integers(1, 4, size=n).astype(np.int32)
        g = (grp, coef, np.array([0.6, 1.1]), np.array([-2, 1], dtype=np.int64))
    return h, starts, ends, w, g


# ---- 1. at the defaults (sequential, Metropolis) the reference is the oracle and the interval reference -----------------------
@pytest.mark.parametrize("with_groups", [False, True])
@pytest.mark.parametrize("seed_mode", [0, 1])
def test_defaults_reproduce_the_oracle(with_groups, seed_mode):
    graph = snn.synthetic_snn(200, k=5, seed=4)[0]
    model = models.cqm_model(graph, 4) if with_groups else models.subsampling_model(graph, 7.0)
    groups = model.groups.astuple() if with_groups else None
    R, n = 16, model.num_variables
    betas, spb = schedule.make_beta_schedule((0.05, 6.0), 30, 1, "geometric")
    seeds = schedule.per_read_seeds(9, R)
    init = schedule.random_spin_states(R, n, 9)
    a, b = init.copy(), init.copy()
    ea, sa = oracle.sample_ising(model.h, model.starts, model.ends, model.weights, a, betas, spb, seeds, seed_mode=seed_mode,
                                 groups=groups)
    eb, sb = pref.sample_ising(model.h, model.starts, model.ends, model.weights, b, betas, spb, seeds, seed_mode=seed_mode,
                               groups=groups)
    assert np.array_equal(a, b)
    assert np.array_equal(ea.view(np.uint64), eb.view(np.uint64))
    assert sa == sb


def test_defaults_reproduce_the_interval_reference():
    model = models.cqm_model(snn.synthetic_snn(256, k=5, seed=3)[0], 4, min_size=60, size_lowering="interval")
    groups = model.groups.astuple()
    R, n = 12, model.num_variables
    betas, spb = schedule.make_beta_schedule((0.05, 8.0), 30, 1, "geometric")
    seeds = schedule.per_read_seeds(6, R)
    init = schedule.random_spin_states(R, n, 6)
    a, b = init.copy(), init.copy()
    ea, sa = iref.sample_ising(model.h, model.starts, model.ends, model.weights, a, betas, spb, seeds, groups=groups)
    eb, sb = pref.sample_ising(model.h, model.starts, model.ends, model.weights, b, betas, spb, seeds, groups=groups)
    assert np.array_equal(a, b)
    assert np.array_equal(ea.view(np.uint64), eb.view(np.uint64))
    assert sa == sb


def test_rejects_unknown_options():
    h, s, e, w, _ = _tiny_model(6, 1, groups=False)
    st = schedule.random_spin_states(2, 6, 1)
    with pytest.raises(RuntimeError):
        pref.sample_ising(h, s, e, w, st, [1.0], 1, [1, 2], var_order=2)
    with pytest.raises(RuntimeError):
        pref.sample_ising(h, s, e, w, st, [1.0], 1, [1, 2], proposal=-1)


# ---- 2. the written contract, restated in Python, reproduces the oracle -----------------------------------------------------
def _restated_read(h, starts, ends, w, groups, state, betas, spb, rnd, var_order, proposal):
    """include/qanneal.h's rules for one read; ``rnd`` yields the read's xorshift128+ outputs.  -> (state, draws)"""
    n = len(h)
    adj = [[] for _ in range(n)]
    for u, v, x in zip(starts.tolist(), ends.tolist(), w.tolist()):   # neal's push_back order
        adj[u].append((v, x))
        adj[v].append((u, x))
    s = [int(x) for x in state]
    dE = []
    for v in range(n):
        f = float(h[v])
        for j, x in adj[v]:
            f += s[j] * x
        dE.append(-2 * s[v] * f)
    if groups is not None:
        grp, coef, lam, kap = (g.tolist() for g in groups)
        M = [0] * len(lam)
        for v in range(n):
            if grp[v] >= 0:
                M[grp[v]] += coef[v] * s[v]
    draws = 0
    for beta in betas.tolist():
        for _ in range(spb):
            thr = 44.36142 / beta
            for k in range(n):
                v = k
                if var_order == 1:
                    v = next(rnd) % n
                    draws += 1
                d = dE[v]
                if groups is not None and grp[v] >= 0:
                    a = coef[v]
                    d = d + lam[grp[v]] * float(a * (a - s[v] * (M[grp[v]] + kap[grp[v]])))
                if d >= thr:
                    continue
                if (d <= -thr) if proposal == 1 else (d <= 0.0):
                    flip = True
                else:
                    r = float(next(rnd))
                    draws += 1
                    flip = (TWO64 > r * (1.0 + math.exp(d * beta))) if proposal == 1 else (math.exp(-d * beta) * TWO64 > r)
                if not flip:
                    continue
                mul = 4 * s[v]
                for j, x in adj[v]:
                    dE[j] += mul * x * s[j]
                if groups is not None and grp[v] >= 0:
                    M[grp[v]] -= 2 * coef[v] * s[v]
                s[v] = -s[v]
                dE[v] = -dE[v]
    return np.array(s, dtype=np.int8), draws


@pytest.mark.parametrize("var_order,proposal", COMBOS)
@pytest.mark.parametrize("n,with_groups", [(5, False), (9, True), (12, True)])
def test_restated_contract_reproduces_the_oracle(var_order, proposal, n, with_groups):
    h, starts, ends, w, groups = _tiny_model(n, 10 + n, with_groups)
    R = 6
    betas = np.array([0.2, 0.7, 1.5, 3.0])
    spb = 2
    seeds = schedule.per_read_seeds(n, R)
    init = schedule.random_spin_states(R, n, n)
    got = init.copy()
    e, st = pref.sample_ising(h, starts, ends, w, got, betas, spb, seeds, groups=groups, var_order=var_order,
                              proposal=proposal)
    total = 0
    for r in range(R):
        rnd = iter(oracle.rng_stream(int(seeds[r]), 4 * n * len(betas) * spb + 8).tolist())
        want, draws = _restated_read(h, starts, ends, w, groups, init[r], betas, spb, rnd, var_order, proposal)
        assert np.array_equal(got[r], want), f"read {r}"
        total += draws
    assert st["draws"] == total
    assert st["attempts"] == R * n * len(betas) * spb
    chk = oracle.state_energies(h, starts, ends, w, got, groups=groups)
    assert np.array_equal(e.view(np.uint64), chk.view(np.uint64))


def test_restated_contract_stream_seeding():
    """stream seeding: one xorshift128+ stream across reads, order draws included"""
    h, starts, ends, w, groups = _tiny_model(10, 3, True)
    R, betas, spb = 4, np.array([0.3, 1.0, 2.5]), 3
    init = schedule.random_spin_states(R, 10, 3)
    for var_order, proposal in COMBOS:
        got = init.copy()
        _, st = pref.sample_ising(h, starts, ends, w, got, betas, spb, [77], seed_mode=1, groups=groups,
                                  var_order=var_order, proposal=proposal)
        rnd = iter(oracle.rng_stream(77, 4 * R * 10 * len(betas) * spb).tolist())
        total = 0
        for r in range(R):
            want, draws = _restated_read(h, starts, ends, w, groups, init[r], betas, spb, rnd, var_order, proposal)
            assert np.array_equal(got[r], want)
            total += draws
        assert st["draws"] == total


# ---- 3. every combination samples the Boltzmann distribution at a fixed beta --------------------------------------------------
@pytest.mark.parametrize("var_order,proposal", COMBOS)
def test_stationary_distribution_is_boltzmann(var_order, proposal):
    """n = 7 with fields, couplers and one equality group; 60 000 independent seeded chains of 40 sweeps at beta = 0.7 from
    random states, final states against exact enumeration.  Total variation below 0.02: the multinomial noise of 60 000 exact
    draws is 0.011 here (all four combinations measure 0.009-0.014), and the same samples are 0.13 away from the
    distribution at beta * 1.3 or beta / 1.3."""
    n, beta, R, sweeps = 7, 0.7, 60000, 40
    h, starts, ends, w, _ = _tiny_model(n, 21, groups=False)
    groups = (np.array([0, 0, 0, 0, -1, -1, -1], dtype=np.int32), np.array([1, 2, 1, 1, 0, 0, 0], dtype=np.int32),
              np.array([0.35]), np.array([-1], dtype=np.int64))
    states = schedule.random_spin_states(R, n, 5)
    pref.sample_ising(h, starts, ends, w, states, np.full(sweeps, beta), 1, schedule.per_read_seeds(5, R), groups=groups,
                      var_order=var_order, proposal=proposal)
    allst = np.array(list(itertools.product([-1, 1], repeat=n)), dtype=np.int8)
    E = oracle.state_energies(h, starts, ends, w, allst, groups=groups)
    p = np.exp(-beta * (E - E.min()))
    p /= p.sum()
    idx = ((states + 1) // 2).astype(np.int64) @ (1 << np.arange(n - 1, -1, -1))
    q = np.bincount(idx, minlength=1 << n) / R
    tv = 0.5 * np.abs(p - q).sum()
    assert tv < 0.02, tv


# ---- 4. interval groups with lo = hi = 0 are the equality groups, under both options ----------------------------------------
@pytest.mark.parametrize("var_order,proposal", COMBOS)
def test_zero_interval_bounds_equal_equality_groups(var_order, proposal):
    model = models.cqm_model(snn.synthetic_snn(160, k=5, seed=2)[0], 4)
    eq = model.groups.astuple()
    G = len(eq[2])
    ivl = eq + (np.zeros(G, dtype=np.int64), np.zeros(G, dtype=np.int64))
    R, n = 12, model.num_variables
    betas, spb = schedule.make_beta_schedule((0.05, 6.0), 30, 1, "geometric")
    seeds = schedule.per_read_seeds(8, R)
    init = schedule.random_spin_states(R, n, 8)
    a, b = init.copy(), init.copy()
    ea, sa = pref.sample_ising(model.h, model.starts, model.ends, model.weights, a, betas, spb, seeds, groups=eq,
                               var_order=var_order, proposal=proposal)
    eb, sb = pref.sample_ising(model.h, model.starts, model.ends, model.weights, b, betas, spb, seeds, groups=ivl,
                               var_order=var_order, proposal=proposal)
    assert np.array_equal(a, b)
    assert np.array_equal(ea.view(np.uint64), eb.view(np.uint64))
    assert sa == sb


# ---- 5. the sampler's handling of the two arguments, before any device work -------------------------------------------------
def _bqm():
    return BinaryQuadraticModel.from_ising({0: 0.5, 1: -0.25}, {(0, 1): -1.0})


def test_sampler_rejects_unknown_acceptance_criterion():
    with pytest.raises(ValueError, match="proposal_acceptance_criteria"):
        B200SimulatedAnnealingSampler().sample(_bqm(), proposal_acceptance_criteria="Glauber", num_reads=2)


def test_sampler_takes_both_options_as_known_parameters():
    sampler = B200SimulatedAnnealingSampler()
    assert "randomize_order" in sampler.parameters and "proposal_acceptance_criteria" in sampler.parameters
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        try:   # without a device the run itself fails after argument handling; with one it completes
            sampler.sample(_bqm(), randomize_order=True, proposal_acceptance_criteria="Gibbs", num_reads=2, seed=1)
        except Exception as e:   # noqa: BLE001
            assert not isinstance(e, ValueError), e
        finally:
            sampler.close()
    assert not [w for w in caught if "unknown kwarg" in str(w.message)]
