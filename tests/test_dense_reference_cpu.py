"""The yardsticks of the dense tensor-core tests (tests/dense_reference.py) checked on the CPU: exact energies against rational
arithmetic and the oracle, the dense-form specification against the k-way builder and against each structural mutation, and the
dyadic models on which summation order cannot matter."""
from fractions import Fraction as Fr

import numpy as np
import pytest

import dense_reference as dref
from oracle import oracle
from scrna_seq_qannealing_clustering_b200 import models, schedule, snn

U = 2.0 ** -53


def _random_model(n, density, seed):
    rng = np.random.default_rng(seed)
    pairs = [(u, v) for u in range(n) for v in range(u) if rng.random() < density]
    starts = np.array([p[0] for p in pairs], dtype=np.int32)
    ends = np.array([p[1] for p in pairs], dtype=np.int32)
    # generic reals of mixed magnitude: roundings happen in any fixed-order sum
    w = rng.normal(size=len(pairs)) * 10.0 ** rng.integers(-6, 7, size=len(pairs))
    h = rng.normal(size=n) * 10.0 ** rng.integers(-6, 7, size=n)
    return h, starts, ends, w


def _fraction_energy(h, starts, ends, w, s):
    e = sum((Fr(float(h[v])) * int(s[v]) for v in range(len(h))), Fr(0))
    e += sum((Fr(float(x)) * int(s[u]) * int(s[v]) for u, v, x in zip(starts, ends, w)), Fr(0))
    return float(e)          # float(Fraction) rounds to nearest


@pytest.mark.parametrize("n,density,seed", [(1, 0.0, 0), (2, 1.0, 1), (9, 0.5, 2), (24, 0.3, 3), (40, 0.9, 4)])
def test_exact_energies_equal_rational_arithmetic(n, density, seed):
    h, st, en, w = _random_model(n, density, seed)
    states = schedule.random_spin_states(6, n, seed)
    got = dref.exact_energies(h, st, en, w, states)
    want = np.array([_fraction_energy(h, st, en, w, s) for s in states])
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))


def test_exact_energies_against_the_oracle():
    """neal's sequential sum is within n * u * sum|terms| of the exact value (and not always equal to it on these weights)."""
    h, st, en, w = _random_model(300, 0.2, 7)
    states = schedule.random_spin_states(32, 300, 7)
    exact = dref.exact_energies(h, st, en, w, states)
    neal = oracle.state_energies(h, st, en, w, states)
    mag = np.abs(h).sum() + np.abs(w).sum()
    assert np.all(np.abs(neal - exact) <= (len(h) + len(w)) * U * mag)
    assert np.any(neal != exact)


@pytest.mark.parametrize("K", [1, 2, 4, 8])
def test_dense_form_of_the_kway_builder(K):
    cells = 23
    X, _ = snn.gaussian_mixture_embedding(cells, dim=6, centres=max(K, 2), seed=K)
    A = snn.gaussian_affinity(X, k=5)
    m = models.dense_kway_model(A, K, 0.05)
    form = dref.dense_form(m.h, m.starts, m.ends, m.weights, K)
    assert form is not None
    W, P = form
    assert np.array_equal(W, W.T) and np.all(np.diag(W) == 0)
    # the dense form reproduces the model: E = s.h + sum_c 1/2 s_c^T W s_c + P * sum_{c < c'} s_c s_c'
    states = schedule.random_spin_states(8, m.num_variables, 3)
    s = states.astype(np.float64).reshape(8, cells, K)
    e = states.astype(np.float64) @ m.h + 0.5 * np.einsum("rjc,ij,ric->r", s, W, s)
    e += P * 0.5 * ((s.sum(axis=2) ** 2).sum(axis=1) - cells * K)
    exact = dref.exact_energies(m.h, m.starts, m.ends, m.weights, states)
    assert np.allclose(e, exact, rtol=1e-12, atol=0)
    if K > 1:      # read with the wrong number of cases the one-hot couplers join different cells (or cut a cell in two)
        assert dref.dense_form(m.h, m.starts, m.ends, m.weights, 2 * K if 2 * K <= 8 else K // 2) is None


@pytest.mark.parametrize("K", [2, 4, 8])
def test_dense_form_verdict_on_structure_mutations(K):
    for name, (h, st, en, w, expect) in dref.structure_mutations(cells=40, K=K).items():
        assert (dref.dense_form(h, st, en, w, K) is not None) is expect, name


def test_dense_form_k1_is_any_ising_model_without_repeated_pairs():
    h, st, en, w = _random_model(30, 0.4, 9)
    W, P = dref.dense_form(h, st, en, w, 1)
    assert P == 0.0 and W[st[0], en[0]] == w[0] and W[en[0], st[0]] == w[0]
    assert dref.dense_form(h, np.append(st, en[0]), np.append(en, st[0]), np.append(w, 1.0), 1) is None


@pytest.mark.parametrize("cells,K,zero_frac,shuffle", [(1, 1, 0.0, False), (1, 8, 0.0, True), (9, 2, 0.4, True),
                                                      (33, 4, 0.0, False), (65, 8, 0.4, True), (100, 1, 0.4, False)])
def test_dyadic_models_are_exact_in_every_order(cells, K, zero_frac, shuffle):
    h, st, en, w, W, P = dref.dyadic_dense_model(cells, K, seed=cells + K, zero_frac=zero_frac, shuffle=shuffle)
    assert len(h) == cells * K
    form = dref.dense_form(h, st, en, w, K)
    assert form is not None and np.array_equal(form[0], W) and form[1] == P
    if zero_frac:
        assert (W[np.tril_indices(cells, -1)] == 0).mean() > zero_frac / 2
        assert len(w) < K * cells * (cells - 1) // 2 + cells * K * (K - 1) // 2
    states = schedule.random_spin_states(16, len(h), 5)
    exact = dref.exact_energies(h, st, en, w, states)
    neal = oracle.state_energies(h, st, en, w, states)
    assert np.array_equal(neal.view(np.uint64), exact.view(np.uint64))
    # reversed coupler order: still bit for bit
    rev = oracle.state_energies(h, st[::-1].copy(), en[::-1].copy(), w[::-1].copy(), states)
    assert np.array_equal(rev.view(np.uint64), exact.view(np.uint64))
