"""k_anneal_dense (csrc/dense.cuh) in exact arithmetic, its structure check, and its real-valued results against exact energies.

On dyadic models (tests/dense_reference.py: h, W, P integers times 2^-8) every field, dE and energy is exact in fp64 in any
summation order, so the tensor-core kernel and the oracle must take the same decisions: states equal byte for byte, energies
bit for bit (and equal to the correctly rounded energy), all five counters equal.  Every run asserts that the dense kernel ran,
so a fall-back to a reference-order kernel cannot pass as parity.  The shapes cover one cell, a single padded spin word,
ragged 8-cell blocks and 32-cell words, one to 96 reads, and more tiles than resident warps (re-packed spin words, reset
per-tile statistics, a ragged later tile)."""
import numpy as np
import pytest

import dense_reference as dref
import scrna_seq_qannealing_clustering_b200 as qa
from oracle import oracle
from scrna_seq_qannealing_clustering_b200 import _lib, models, schedule, snn
from scrna_seq_qannealing_clustering_b200.engine import Context, IsingModel

pytestmark = pytest.mark.gpu

COUNTERS = ("attempts", "candidates", "draws", "accepted", "nbr_updates")


@pytest.fixture(scope="module")
def ctx(built):
    c = Context(0)
    yield c
    c.close()


def _schedule(h, st, en, w, sweeps, spb=1):
    beta_range = schedule.default_ising_beta_range(h, st, en, w, None)
    return schedule.make_beta_schedule(beta_range, sweeps, spb, "geometric")


def _dense_sample(ctx, h, st, en, w, K, init, betas, spb, seeds):
    gm = IsingModel(ctx, h, st, en, w)
    try:
        assert gm.enable_dense(K) is True
        states = init.copy()
        e, stats, done = gm.sample(states, betas, spb, seeds, mode=_lib.QA_MODE_THROUGHPUT)
        assert ctx.last_kernel == _lib.QA_KERNEL_DENSE
    finally:
        gm.close()
    assert done == len(init)
    return states, e, stats


def _assert_exact_parity(ctx, h, st, en, w, K, init, betas, spb, seeds, exact_rows=256):
    states, e, stats = _dense_sample(ctx, h, st, en, w, K, init, betas, spb, seeds)
    ref = init.copy()
    ref_e, ref_stats = oracle.sample_ising(h, st, en, w, ref, betas, spb, seeds)
    assert np.array_equal(states, ref), f"{(states != ref).any(axis=1).sum()} of {len(ref)} reads left the oracle's trajectory"
    assert np.array_equal(e.view(np.uint64), ref_e.view(np.uint64))
    rows = np.unique(np.linspace(0, len(init) - 1, min(exact_rows, len(init))).astype(np.int64))
    exact = dref.exact_energies(h, st, en, w, states[rows])
    assert np.array_equal(e[rows].view(np.uint64), exact.view(np.uint64))
    for key in COUNTERS:
        assert getattr(stats, key) == ref_stats[key], (key, getattr(stats, key), ref_stats[key])
    return states, stats


# ---- B. exact regime -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cells", [1, 3, 7, 8, 9, 31, 32, 33, 63, 65, 100])
@pytest.mark.parametrize("K", [1, 2, 4, 8])
def test_dyadic_parity_at_edge_shapes(ctx, K, cells):
    """40 reads: a full tile and a ragged one; odd cell counts also shuffle the coupler list (neal's row order changes)."""
    h, st, en, w, _, _ = dref.dyadic_dense_model(cells, K, seed=100 * K + cells, shuffle=cells % 2 == 1)
    R = 40
    betas, spb = _schedule(h, st, en, w, 6)
    _assert_exact_parity(ctx, h, st, en, w, K, schedule.random_spin_states(R, cells * K, cells), betas, spb,
                         schedule.per_read_seeds(K + cells, R))


@pytest.mark.parametrize("R", [1, 31, 33, 96])
def test_dyadic_parity_read_counts(ctx, R):
    h, st, en, w, _, _ = dref.dyadic_dense_model(33, 4, seed=7)
    betas, spb = _schedule(h, st, en, w, 8)
    _assert_exact_parity(ctx, h, st, en, w, 4, schedule.random_spin_states(R, 132, R), betas, spb, schedule.per_read_seeds(R, R))


def test_dyadic_parity_several_tiles_per_warp(ctx):
    """3 tiles for every resident warp (launch_dense: at most 2 CTAs of 4 warps per SM) plus a ragged 17-read tile."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    R = 3 * 8 * sms * 32 + 17
    h, st, en, w, _, _ = dref.dyadic_dense_model(45, 2, seed=11, shuffle=True)
    betas, spb = _schedule(h, st, en, w, 2)
    _assert_exact_parity(ctx, h, st, en, w, 2, schedule.random_spin_states(R, 90, 4), betas, spb,
                         schedule.per_read_seeds(12, R), exact_rows=64)


def test_dyadic_parity_sweeps_per_beta(ctx):
    h, st, en, w, _, _ = dref.dyadic_dense_model(31, 4, seed=3)
    betas, spb = _schedule(h, st, en, w, 9, spb=3)
    assert spb == 3 and len(betas) == 3
    _assert_exact_parity(ctx, h, st, en, w, 4, schedule.random_spin_states(64, 124, 3), betas, spb, schedule.per_read_seeds(3, 64))


def test_dyadic_zero_sweeps_return_the_input(ctx):
    h, st, en, w, _, _ = dref.dyadic_dense_model(37, 8, seed=5)
    init = schedule.random_spin_states(45, 296, 5)
    states, e, stats = _dense_sample(ctx, h, st, en, w, 8, init, np.zeros(0), 1, schedule.per_read_seeds(5, 45))
    assert np.array_equal(states, init)
    assert np.array_equal(e.view(np.uint64), dref.exact_energies(h, st, en, w, init).view(np.uint64))
    assert stats.attempts == stats.accepted == stats.nbr_updates == 0


def test_dyadic_parity_seed_zero(ctx):
    """An explicit seed vector with zeros: xorshift128+ maps seed 0 to ~0 (neal), on every read that has it."""
    h, st, en, w, _, _ = dref.dyadic_dense_model(20, 4, seed=9)
    R = 40
    seeds = schedule.per_read_seeds(9, R)
    seeds[[0, 5, 33, 39]] = 0
    betas, spb = _schedule(h, st, en, w, 10)
    init = np.repeat(schedule.random_spin_states(1, 80, 9), R, axis=0)    # identical starts: the seeds alone tell reads apart
    states, _ = _assert_exact_parity(ctx, h, st, en, w, 4, init, betas, spb, seeds)
    assert np.array_equal(states[0], states[5]) and np.array_equal(states[0], states[39])


@pytest.mark.parametrize("cells,K", [(100, 1), (33, 4), (17, 8)])
def test_dyadic_parity_with_zeros_in_W(ctx, cells, K):
    """About 40 % of the cell pairs uncoupled: a flip updates only the variable's CSR neighbours, and nbr_updates counts them."""
    h, st, en, w, W, _ = dref.dyadic_dense_model(cells, K, seed=cells, zero_frac=0.4, shuffle=True)
    assert (W[np.tril_indices(cells, -1)] == 0).mean() > 0.3
    betas, spb = _schedule(h, st, en, w, 8)
    _, stats = _assert_exact_parity(ctx, h, st, en, w, K, schedule.random_spin_states(64, cells * K, 1), betas, spb,
                                    schedule.per_read_seeds(1, 64))
    assert stats.nbr_updates < stats.accepted * (cells - 1 + K - 1)


def test_invalid_input_state(ctx):
    """A 0 spin in a later tile: QA_ERR_STATE, as on the reference-order kernels."""
    h, st, en, w, _, _ = dref.dyadic_dense_model(9, 4, seed=1)
    bad = schedule.random_spin_states(40, 36, 1)
    bad[35, 17] = 0
    betas, spb = _schedule(h, st, en, w, 2)
    gm = IsingModel(ctx, h, st, en, w)
    try:
        assert gm.enable_dense(4)
        codes = []
        for mode in (_lib.QA_MODE_THROUGHPUT, _lib.QA_MODE_REFERENCE):
            with pytest.raises(_lib.QAnnealError) as ei:
                gm.sample(bad.copy(), betas, spb, schedule.per_read_seeds(1, 40), mode=mode)
            codes.append((ei.value.code, ctx.last_kernel))
    finally:
        gm.close()
    assert codes[0] == (-3, _lib.QA_KERNEL_DENSE) and codes[1][0] == -3


# ---- C. structure check ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [2, 4, 8])
def test_structure_check_matches_the_specification(ctx, K):
    """The device check accepts exactly the models that have the dense form; in every case mode=THROUGHPUT returns the energies of
    the given model (whichever kernel runs)."""
    R = 40
    for name, (h, st, en, w, expect) in dref.structure_mutations(cells=40, K=K).items():
        assert (dref.dense_form(h, st, en, w, K) is not None) is expect, name
        betas, spb = _schedule(h, st, en, w, 4)
        init = schedule.random_spin_states(R, len(h), K)
        gm = IsingModel(ctx, h, st, en, w)
        try:
            assert gm.enable_dense(K) is expect, name
            states = init.copy()
            e, _, done = gm.sample(states, betas, spb, schedule.per_read_seeds(K, R), mode=_lib.QA_MODE_THROUGHPUT)
            assert (ctx.last_kernel == _lib.QA_KERNEL_DENSE) is expect, name
        finally:
            gm.close()
        exact = dref.exact_energies(h, st, en, w, states)
        assert np.all(np.abs(e - exact) <= 1e-12 * np.maximum(np.abs(exact), 1.0)), (name, np.abs(e - exact).max())


def test_sampler_throughput_keeps_incomplete_onehot_models_off_the_dense_kernel(ctx):
    """sampler.sample(mode='throughput') on a LoweredModel with meta['num_cases'] (what _try_dense looks at): one cell without its
    one-hot couplers must not be annealed as if it had them."""
    K, cells = 4, 72
    h, st, en, w, _, _ = dref.dyadic_dense_model(cells, K, seed=21)
    lo, hi = np.minimum(st, en), np.maximum(st, en)
    keep = ~((lo // K == hi // K) & (lo // K == 30))
    sampler = qa.B200SimulatedAnnealingSampler(context=ctx)
    for cpl, dense in ((np.ones(len(st), bool), True), (keep, False)):
        labels = [(i, c) for i in range(cells) for c in range(K)]
        m = models.LoweredModel(h, st[cpl], en[cpl], w[cpl], 0.0, labels, None, {"num_cases": K})
        ss = sampler.sample(m, num_reads=64, num_sweeps=10, seed=5, mode="throughput")
        assert (ctx.last_kernel == _lib.QA_KERNEL_DENSE) is dense
        spins = 2 * ss.record.sample.astype(np.int8) - 1
        exact = dref.exact_energies(m.h, m.starts, m.ends, m.weights, spins)
        assert np.all(np.abs(ss.record.energy - exact) <= 1e-12 * np.maximum(np.abs(exact), 1.0))


# ---- E. real-valued regime ---------------------------------------------------------------------------------------------------
def _affinity_model(cells, K, seed=2, gamma=0.05):
    X, _ = snn.gaussian_mixture_embedding(cells, dim=15, centres=max(K, 2), sep=4.0, seed=seed)
    return models.dense_kway_model(snn.gaussian_affinity(X, k=min(10, cells - 1)), K, gamma)


def _rel_dev(e, exact):
    return float(np.max(np.abs(e - exact) / np.maximum(np.abs(exact), 1.0)))


@pytest.mark.parametrize("cells,K", [(100, 8), (37, 1), (20, 4), (13, 2)])
def test_affinity_models_against_exact_energies(ctx, cells, K):
    m = _affinity_model(cells, K)
    hot = schedule.default_ising_beta_range(m.h, m.starts, m.ends, m.weights, None)[0]
    betas, spb = schedule.make_beta_schedule((hot, 30.0), 25, 1, "geometric")
    R = 96
    init = schedule.random_spin_states(R, m.num_variables, 11)
    seeds = schedule.per_read_seeds(11, R)
    states, e, _ = _dense_sample(ctx, m.h, m.starts, m.ends, m.weights, K, init, betas, spb, seeds)
    assert _rel_dev(e, dref.exact_energies(m.h, m.starts, m.ends, m.weights, states)) <= 1e-12
    ref = init.copy()
    oracle.sample_ising(m.h, m.starts, m.ends, m.weights, ref, betas, spb, seeds)
    assert (states == ref).all(axis=1).mean() >= 0.95


def test_config5_size_against_exact_energies(ctx):
    """4096 cells x 4 (33.5 M couplers), 8 reads: the kernel's energies against the correctly rounded ones."""
    m = _affinity_model(4096, 4)
    hot = schedule.default_ising_beta_range(m.h, m.starts, m.ends, m.weights, None)[0]
    betas, spb = schedule.make_beta_schedule((hot, 10 * hot), 3, 1, "geometric")
    init = schedule.random_spin_states(8, m.num_variables, 3)
    states, e, _ = _dense_sample(ctx, m.h, m.starts, m.ends, m.weights, 4, init, betas, spb, schedule.per_read_seeds(3, 8))
    dev = _rel_dev(e, dref.exact_energies(m.h, m.starts, m.ends, m.weights, states))
    print(f"config-5 size: max relative deviation from the exact energy {dev:.3e}")
    assert dev <= 1e-12, dev
