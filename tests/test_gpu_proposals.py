"""dwave-samplers' sample options on the B200: sequential Gibbs on every reference-order kernel and random variable order
(Metropolis and Gibbs) on the warp-per-read kernel, bit-exact against the CPU reference (tests/native/proposals_sa_ref.cpp,
which at the default options is the oracle and the interval reference bit for bit); the kernel that ran is asserted every
time, so that a silent fall-back cannot pass."""
import numpy as np
import pytest

import proposals_reference as pref
import scrna_seq_qannealing_clustering_b200 as qa
from scrna_seq_qannealing_clustering_b200 import _lib, models, schedule, snn
from scrna_seq_qannealing_clustering_b200.engine import Context, IsingModel

pytestmark = pytest.mark.gpu

SEQ, RND = _lib.QA_ORDER_SEQUENTIAL, _lib.QA_ORDER_RANDOM
MET, GIB = _lib.QA_PROPOSAL_METROPOLIS, _lib.QA_PROPOSAL_GIBBS
KERNELS = {"warp_per_read": _lib.QA_KERNEL_WARP_PER_READ, "lockstep_push": _lib.QA_KERNEL_LOCKSTEP_PUSH,
           "replay": _lib.QA_KERNEL_REPLAY}


@pytest.fixture(scope="module")
def graph256():
    return snn.synthetic_snn(256, k=5, seed=3)[0]


@pytest.fixture(scope="module")
def graph200():
    return snn.synthetic_snn(200, k=5, seed=8)[0]   # n = 200: the last 32-variable chunk is ragged


@pytest.fixture(params=list(KERNELS))
def kctx(request, built):
    ctx = Context(0)
    ctx.set_kernel(KERNELS[request.param])
    ctx.requested_kernel = KERNELS[request.param]
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def pctx(built):
    ctx = Context(0)
    yield ctx
    ctx.close()


def _model(name, g256, g200):
    if name == "cut_balance":
        return models.cut_balance_model(g256, 0.05)                              # one equality group
    if name == "dqm_onehot":
        return models.dqm_model(g256, 4, 0.005, semantics="intended")           # k-way section of the replay slabs
    if name == "cqm_slack":
        return models.cqm_model(g256, 4)                                         # equality groups with slack bits
    if name == "cqm_interval":
        return models.cqm_model(g256, 4, min_size=60, size_lowering="interval")  # interval groups
    if name == "subsampling":
        return models.subsampling_model(g200, 7.0)                               # no groups, ragged n
    if name == "dense_rows":
        return models.cut_balance_model(g256, 0.05, structured=False)            # K_256: replay falls back to lockstep
    raise KeyError(name)


def _run(ctx, m, R, sweeps, seed, var_order, proposal, seed_mode=_lib.QA_SEED_PER_READ, mode=_lib.QA_MODE_REFERENCE,
         interrupt=None, dense_k=None, beta_range=(0.05, 8.0)):
    """GPU run and reference run on the same inputs; asserts bit-exactness of the completed reads.  -> (kernel, kway, stats)"""
    n = m.num_variables
    groups = m.groups.astuple() if m.groups is not None else None
    betas, spb = schedule.make_beta_schedule(beta_range, sweeps, 1, "geometric")
    stream = seed_mode == _lib.QA_SEED_STREAM
    seeds = np.array([seed], dtype=np.uint64) if stream else schedule.per_read_seeds(seed, R)
    init = schedule.random_spin_states(R, n, seed)
    gm = IsingModel(ctx, m.h, m.starts, m.ends, m.weights)
    try:
        if groups is not None:
            gm.set_groups(*groups)
        if dense_k is not None:
            assert gm.enable_dense(dense_k)
        states = init.copy()
        e, st, done = gm.sample(states, betas, spb, seeds, seed_mode=seed_mode, mode=mode, interrupt_function=interrupt,
                                var_order=var_order, proposal=proposal)
        kernel, kway = ctx.last_kernel, gm.replay_kway
    finally:
        gm.close()
    assert 0 < done <= R
    ref = init[:done].copy()
    ref_e, ref_st = pref.sample_ising(m.h, m.starts, m.ends, m.weights, ref, betas, spb, seeds if stream else seeds[:done],
                                      seed_mode=1 if stream else 0, groups=groups, var_order=var_order, proposal=proposal)
    assert np.array_equal(states[:done], ref)
    assert np.array_equal(states[done:], init[done:])   # reads not handed out keep their initial states
    assert np.array_equal(e[:done].view(np.uint64), ref_e.view(np.uint64))
    if done == R:
        assert st.attempts == ref_st["attempts"]
        for key in ("candidates", "draws", "accepted", "nbr_updates"):
            assert getattr(st, key) == ref_st[key], key
    if var_order == RND:
        assert st.chunks == 0 and st.active_chunks == 0
    return kernel, kway, st


# ---- 1. sequential Gibbs on every reference-order kernel ----------------------------------------------------------------
@pytest.mark.parametrize("name", ["cut_balance", "dqm_onehot", "cqm_slack", "cqm_interval", "subsampling", "dense_rows"])
def test_sequential_gibbs_bit_exact(kctx, graph256, graph200, name):
    m = _model(name, graph256, graph200)
    kernel, kway, st = _run(kctx, m, 96, 40, 7, SEQ, GIB, beta_range=(0.02, 6.0) if name == "dqm_onehot" else (0.05, 8.0))
    want = kctx.requested_kernel
    if want == _lib.QA_KERNEL_REPLAY and name == "dense_rows":
        want = _lib.QA_KERNEL_LOCKSTEP_PUSH
    assert kernel == want
    if kernel == _lib.QA_KERNEL_REPLAY and name == "dqm_onehot":
        assert kway[0] > 0 and kway[1] == 4
    assert st.draws > 0 and st.accepted > 0


def test_sequential_gibbs_stream_seeding(kctx, graph256, graph200):
    kernel, _, _ = _run(kctx, _model("cqm_slack", graph256, graph200), 12, 30, 11, SEQ, GIB, seed_mode=_lib.QA_SEED_STREAM)
    assert kernel == _lib.QA_KERNEL_WARP_PER_READ


def test_sequential_gibbs_replay_interrupt(graph256, graph200, built, monkeypatch):
    """an interrupt callback stops a replay run when CTAs pull their next group of reads (one-warp CTAs: many groups); the
    completed reads are exact"""
    monkeypatch.setenv("QA_REPLAY_WARPS", "1")
    ctx = Context(0)
    try:
        ctx.set_kernel(_lib.QA_KERNEL_REPLAY)
        calls = []
        kernel, _, _ = _run(ctx, _model("subsampling", graph256, graph200), 60000, 20, 5, SEQ, GIB,
                            interrupt=lambda: calls.append(1) or True)
        assert kernel == _lib.QA_KERNEL_REPLAY and calls
    finally:
        ctx.close()


# ---- 2. random order: always the warp-per-read kernel ---------------------------------------------------------------------
@pytest.mark.parametrize("proposal", [MET, GIB])
@pytest.mark.parametrize("name", ["subsampling", "cut_balance", "cqm_slack", "cqm_interval", "dqm_onehot"])
def test_random_order_bit_exact(kctx, graph256, graph200, name, proposal):
    m = _model(name, graph256, graph200)
    kernel, _, st = _run(kctx, m, 64, 20, 3, RND, proposal)
    assert kernel == _lib.QA_KERNEL_WARP_PER_READ
    assert st.draws >= st.attempts   # one order draw per attempt


@pytest.mark.parametrize("proposal", [MET, GIB])
def test_random_order_stream_seeding(pctx, graph256, graph200, proposal):
    kernel, _, _ = _run(pctx, _model("cut_balance", graph256, graph200), 10, 20, 21, RND, proposal,
                        seed_mode=_lib.QA_SEED_STREAM)
    assert kernel == _lib.QA_KERNEL_WARP_PER_READ


def test_random_order_interrupt(pctx, graph256, graph200):
    """read waves of the warp-per-read kernel: the callback stops the run after the first wave, completed reads are exact"""
    R = pctx.resident_reads + 500
    kernel, _, _ = _run(pctx, _model("subsampling", graph256, graph200), R, 10, 9, RND, GIB, interrupt=lambda: True)
    assert kernel == _lib.QA_KERNEL_WARP_PER_READ


# ---- 3. throughput mode on a dense k-way model runs a reference-order kernel with either option -----------------------------
@pytest.mark.parametrize("var_order,proposal", [(SEQ, GIB), (RND, MET)])
def test_throughput_mode_with_options_runs_reference_order(pctx, var_order, proposal):
    X, _ = snn.gaussian_mixture_embedding(64, dim=15, centres=4, sep=4.0, seed=2)
    m = models.dense_kway_model(snn.gaussian_affinity(X, k=10), 4, 0.05)
    kernel, _, _ = _run(pctx, m, 64, 30, 4, var_order, proposal, mode=_lib.QA_MODE_THROUGHPUT, dense_k=4,
                        beta_range=(0.1, 20.0))
    assert kernel != _lib.QA_KERNEL_DENSE
    if var_order == RND:
        assert kernel == _lib.QA_KERNEL_WARP_PER_READ


# ---- 4. through the sampler ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sampler(built):
    s = qa.B200SimulatedAnnealingSampler(device=0)
    yield s
    s.close()


def test_sampler_random_order_gibbs_equals_the_oracle(sampler, graph200):
    model = models.subsampling_model(graph200, 0.8)
    R, sweeps, seed = 40, 60, 13
    kw = dict(num_reads=R, num_sweeps=sweeps, beta_range=(0.05, 8.0), seed=seed, randomize_order=True,
              proposal_acceptance_criteria="Gibbs")
    ss = sampler.sample(model, **kw)
    betas, spb = schedule.make_beta_schedule((0.05, 8.0), sweeps, 1, "geometric")
    ref = schedule.random_spin_states(R, model.num_variables, seed)
    ref_e, _ = pref.sample_ising(model.h, model.starts, model.ends, model.weights, ref, betas, spb,
                                 schedule.per_read_seeds(seed, R), var_order=RND, proposal=GIB)
    assert np.array_equal(ss.record.sample, (ref + 1) // 2)
    assert np.array_equal(ss.record.energy, ref_e + model.offset)
    b = ss.info["b200"]
    assert b["randomize_order"] is True and b["proposal_acceptance_criteria"] == "Gibbs"
    assert b["kernel"] == _lib.QA_KERNEL_WARP_PER_READ
    # the k best rows, ranked on the device
    k = 5
    best = sampler.sample(model, return_samples="best_k", num_best=k, **kw)
    order = np.argsort(ref_e, kind="stable")[:k]
    assert np.array_equal(best.record.energy, ref_e[order] + model.offset)
    for row, e in zip(best.record.sample, best.record.energy):
        match = np.flatnonzero(ref_e + model.offset == e)
        assert any(np.array_equal(row, (ref[i] + 1) // 2) for i in match)


def test_clustering_dqm_reaches_the_gibbs_kernel(sampler, graph256):
    ss = qa.clustering_dqm(graph256, 4, 0.005, sampler=sampler, num_reads=64, num_sweeps=50, seed=3,
                           proposal_acceptance_criteria="Gibbs")
    b = ss.info["b200"]
    assert b["proposal_acceptance_criteria"] == "Gibbs" and b["randomize_order"] is False
    assert b["kernel"] in (_lib.QA_KERNEL_WARP_PER_READ, _lib.QA_KERNEL_LOCKSTEP_PUSH, _lib.QA_KERNEL_REPLAY)
    assert sampler.last_stats["draws"] > 0
