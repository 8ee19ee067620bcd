"""The replay kernel's k-way batch phase (csrc/replay.cuh rp_kway_batch; slab section built by anneal_replay.cu): one-hot
models whose K cases per cell share one neighbour-cell list run the K rows of a cell in lockstep.  Same bar as
test_gpu_replay.py -- states bytewise, energies bitwise, all five counters equal to the CPU reference -- with the k-way form
asserted to have run, against forced-generic runs (QA_REPLAY_KWAY=0), and on mutated models that must fall back."""
import os

import numpy as np
import pytest

import interval_reference as iref
from oracle import oracle
from scrna_seq_qannealing_clustering_b200 import _lib, models, schedule, snn
from scrna_seq_qannealing_clustering_b200.engine import Context, IsingModel

pytestmark = pytest.mark.gpu


def _ctx(kway=True, permille=None):
    old = {k: os.environ.get(k) for k in ("QA_REPLAY_KWAY", "QA_REPLAY_SWITCH_PERMILLE")}
    os.environ["QA_REPLAY_KWAY"] = "1" if kway else "0"
    if permille is not None:
        os.environ["QA_REPLAY_SWITCH_PERMILLE"] = str(permille)
    try:   # development knobs are read when the context is created
        ctx = Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    ctx.set_kernel(_lib.QA_KERNEL_REPLAY)
    return ctx


def _sample(ctx, model, R, sweeps, seed, spb=1, beta_range=(0.05, 8.0)):
    groups = model.groups.astuple() if model.groups is not None else None
    betas, spb = schedule.make_beta_schedule(beta_range, sweeps, spb, "geometric")
    seeds = schedule.per_read_seeds(seed, R)
    init = schedule.random_spin_states(R, model.num_variables, seed)
    gm = IsingModel(ctx, model.h, model.starts, model.ends, model.weights)
    if groups is not None:
        gm.set_groups(*groups)
    states = init.copy()
    e, st, done = gm.sample(states, betas, spb, seeds)
    kway = gm.replay_kway
    gm.close()
    assert done == R and ctx.last_kernel == _lib.QA_KERNEL_REPLAY
    ref = init.copy()
    interval = model.groups is not None and getattr(model.groups, "lo", None) is not None
    ref_e, ref_st = (iref if interval else oracle).sample_ising(model.h, model.starts, model.ends, model.weights, ref, betas,
                                                                 spb, seeds, groups=groups)
    bad = np.nonzero((states != ref).any(axis=1))[0]
    assert bad.size == 0, f"{bad.size} of {R} reads differ, first {bad[:8]}"
    assert np.array_equal(e.view(np.uint64), ref_e.view(np.uint64))
    for key in ("attempts", "candidates", "draws", "accepted", "nbr_updates"):
        assert getattr(st, key) == ref_st[key], key
    assert st.near_ties == 0
    return states, e, kway


@pytest.fixture(scope="module")
def graph101():
    return snn.synthetic_snn(101, k=5, seed=11)[0]   # odd cell count: the last half-words mix cells, slack and padding


@pytest.mark.parametrize("K", [2, 4, 8, 16])
@pytest.mark.parametrize("lowering", ["slack", "interval"])
def test_kway_cqm_matches_reference_and_generic(built, graph101, K, lowering):
    model = models.cqm_model(graph101, K, min_size=5, size_lowering=lowering)
    ctx, gen = _ctx(), _ctx(kway=False)
    try:
        s1, e1, (blocks, k) = _sample(ctx, model, 96, 40, 3 + K, beta_range=(0.02, 6.0))
        assert blocks > 0 and k == K
        s0, e0, (blocks0, _) = _sample(gen, model, 96, 40, 3 + K, beta_range=(0.02, 6.0))
        assert blocks0 == 0
        assert np.array_equal(s0, s1) and np.array_equal(e0.view(np.uint64), e1.view(np.uint64))
    finally:
        ctx.close()
        gen.close()


@pytest.mark.parametrize("permille", [0, 20, 300, 1000])
@pytest.mark.parametrize("spb", [1, 3])
def test_kway_hand_over_points_and_sweeps_per_beta(built, permille, spb):
    g = snn.synthetic_snn(257, k=5, seed=2)[0]
    model = models.cqm_model(g, 8, min_size=20)
    ctx = _ctx(permille=permille)
    try:
        _, _, (blocks, k) = _sample(ctx, model, 160, 30, 17, spb=spb, beta_range=(0.02, 6.0))
        assert blocks > 0 and k == 8
    finally:
        ctx.close()


def test_kway_dqm_and_ungrouped_model(built, graph101):
    ctx = _ctx()
    try:
        m = models.cqm_model(graph101, 4, min_size=5)
        bare = models.LoweredModel(m.h, m.starts, m.ends, m.weights, 0.0, list(range(m.num_variables)))
        _, _, (blocks, k) = _sample(ctx, bare, 64, 40, 5)
        assert blocks > 0 and k == 4
        _, _, (blocks, k) = _sample(ctx, models.dqm_model(graph101, 4, 0.005, semantics="intended"), 64, 40, 9,
                                    beta_range=(0.02, 6.0))
        if blocks:
            assert k == 4
    finally:
        ctx.close()


def _coupler(model, u, v):
    a, b = max(u, v), min(u, v)
    idx = np.nonzero((model.starts == a) & (model.ends == b))[0]
    assert idx.size == 1
    return int(idx[0])


def _mutated(model, kind):
    st, en, w = model.starts.copy(), model.ends.copy(), model.weights.copy()
    K = 8
    if kind == "missing_case_coupler":          # cell 3 loses one one-hot coupler
        k = _coupler(model, 3 * K + 1, 3 * K + 5)
        st, en, w = np.delete(st, k), np.delete(en, k), np.delete(w, k)
    elif kind == "per_case_weight":             # one case of one inter-cell coupler gets its own weight
        k = int(np.nonzero(model.starts // K != model.ends // K)[0][0])
        w[k] = w[k] * 1.5 + 0.125
    elif kind == "duplicated_coupler":          # the same inter-cell coupler twice
        k = int(np.nonzero(model.starts // K != model.ends // K)[0][3])
        st, en, w = np.append(st, st[k]), np.append(en, en[k]), np.append(w, 0.25)
    else:                                       # non-one-hot row: a cross-case inter-cell coupler
        k = int(np.nonzero(model.starts // K != model.ends // K)[0][5])
        a, b = int(model.starts[k]), int(model.ends[k])
        st, en, w = np.append(st, a), np.append(en, b - b % K + (b % K + 1) % K), np.append(w, -0.3)
    return models.LoweredModel(model.h, st.astype(np.int32), en.astype(np.int32), w, model.offset, model.labels, model.groups,
                               model.meta)


@pytest.mark.parametrize("kind", ["missing_case_coupler", "per_case_weight", "duplicated_coupler", "cross_case_coupler"])
def test_mutations_fall_back_to_the_generic_form(built, graph101, kind):
    base = models.cqm_model(graph101, 8, min_size=5)
    ctx = _ctx()
    try:
        _, _, (b0, _) = _sample(ctx, base, 64, 30, 21, beta_range=(0.02, 6.0))
        _, _, (b1, k) = _sample(ctx, _mutated(base, kind), 64, 30, 21, beta_range=(0.02, 6.0))
        assert 0 < b1 < b0 and k == 8
    finally:
        ctx.close()


def test_batched_problems(built):
    """qa_model_concat of ungrouped k-way models (batched models with groups run on the warp-per-read kernel)."""
    ctx = _ctx()
    try:
        ms = []
        for s, K in ((1, 8), (2, 4), (3, 8)):
            m = models.cqm_model(snn.synthetic_snn(64 + 7 * s, k=5, seed=s)[0], K, min_size=3)
            ms.append(models.LoweredModel(m.h, m.starts, m.ends, m.weights, 0.0, list(range(m.num_variables))))
        parts = [IsingModel(ctx, m.h, m.starts, m.ends, m.weights) for m in ms]
        bm = ctx.concat_models(parts)
        R = 64
        betas, spb = schedule.make_beta_schedule((0.05, 6.0), 30, 1, "geometric")
        seeds = schedule.per_read_seeds(40, R * len(ms))
        inits = [schedule.random_spin_states(R, m.num_variables, 40 + p) for p, m in enumerate(ms)]
        states = np.concatenate([x.ravel() for x in inits]).copy()
        e, st, done = ctx.sample_model_batch(bm, R, states, betas, spb, seeds)
        assert done == R and ctx.last_kernel == _lib.QA_KERNEL_REPLAY and bm.replay_kway[0] > 0
        o = 0
        for p, m in enumerate(ms):
            ref = inits[p].copy()
            ref_e, _ = oracle.sample_ising(m.h, m.starts, m.ends, m.weights, ref, betas, spb, seeds[p * R:(p + 1) * R])
            got = states[o:o + R * m.num_variables].reshape(R, m.num_variables)
            o += R * m.num_variables
            assert np.array_equal(got, ref)
            assert np.array_equal(e[p * R:(p + 1) * R].view(np.uint64), ref_e.view(np.uint64))
        for x in parts + [bm]:
            x.close()
    finally:
        ctx.close()
