"""Interval rank-1 groups on the B200: every reference-mode kernel bit-exact against the CPU reference
(tests/native/interval_sa_ref.cpp), the device builder, batching, the sampler path and the error codes."""
import numpy as np
import pytest

import interval_reference as iref
from scrna_seq_qannealing_clustering_b200 import _lib, models, schedule, snn
from scrna_seq_qannealing_clustering_b200._lib import QAnnealError
from scrna_seq_qannealing_clustering_b200.cqm import Binary, ConstrainedQuadraticModel
from scrna_seq_qannealing_clustering_b200.engine import Context, IsingModel

pytestmark = pytest.mark.gpu

KERNELS = {"warp_per_read": _lib.QA_KERNEL_WARP_PER_READ, "lockstep_push": _lib.QA_KERNEL_LOCKSTEP_PUSH,
           "replay": _lib.QA_KERNEL_REPLAY}
I64 = np.iinfo(np.int64)


@pytest.fixture(params=list(KERNELS))
def kctx(request, built):
    ctx = Context(0)
    ctx.set_kernel(KERNELS[request.param])
    ctx.requested_kernel = KERNELS[request.param]
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def graph256():
    return snn.synthetic_snn(256, k=5, seed=3)[0]


def _run(ctx, h, starts, ends, w, groups, R, sweeps, seed, beta_range=(0.05, 8.0), ref_groups=None):
    n = len(h)
    betas, spb = schedule.make_beta_schedule(beta_range, sweeps, 1, "geometric")
    seeds = schedule.per_read_seeds(seed, R)
    init = schedule.random_spin_states(R, n, seed)
    ref_states = init.copy()
    ref_e, ref_st = iref.sample_ising(h, starts, ends, w, ref_states, betas, spb, seeds,
                                      groups=groups if ref_groups is None else ref_groups)
    gm = IsingModel(ctx, h, starts, ends, w)
    gm.set_groups(*groups)
    states = init.copy()
    e, st, done = gm.sample(states, betas, spb, seeds)
    gm.close()
    assert done == R
    return states, e, st, ref_states, ref_e, ref_st


def _assert_exact(states, e, st, ref_states, ref_e, ref_st):
    assert np.array_equal(states, ref_states)
    assert np.array_equal(e.view(np.uint64), ref_e.view(np.uint64))
    for key in ("attempts", "candidates", "draws", "accepted", "nbr_updates"):
        assert getattr(st, key) == ref_st[key], key
    assert st.near_ties == 0


def test_binding_cqm_interval(kctx, graph256):
    m = models.cqm_model(graph256, 4, min_size=60, size_lowering="interval")   # n/K = 64: the bound binds
    r = _run(kctx, m.h, m.starts, m.ends, m.weights, m.groups.astuple(), 96, 40, 7)
    _assert_exact(*r)
    if kctx.requested_kernel == _lib.QA_KERNEL_REPLAY:
        assert kctx.last_kernel == _lib.QA_KERNEL_REPLAY


def _two_sided_mixed(graph):
    m = models.subsampling_model(graph, 7.0)
    n = m.num_variables
    rng = np.random.default_rng(3)
    grp = rng.integers(-1, 5, size=n).astype(np.int32)
    coef = rng.choice([-3, -2, -1, 1, 2, 3], size=n).astype(np.int32)
    lam = np.array([0.3, 1.1, 0.05, 2.0, 0.7])
    kap = np.array([-5, 12, 0, -30, 3], dtype=np.int64)
    lo = np.array([-4, 0, I64.min, -10, 2], dtype=np.int64)
    hi = np.array([6, 0, -3, 10, I64.max], dtype=np.int64)
    return m, (grp, coef, lam, kap, lo, hi)


def test_two_sided_mixed_sign(kctx, graph256):
    m, g = _two_sided_mixed(graph256)
    _assert_exact(*_run(kctx, m.h, m.starts, m.ends, m.weights, g, 64, 30, 11))


@pytest.mark.parametrize("bounds", ["equality", "interval"])
def test_max_groups_wide_coefficients(kctx, graph256, bounds):
    """QA_MAX_GROUPS = 64 groups (the size of the per-read group sums in every kernel), holes (grp = -1) and coefficients of
    2^19 .. 2^20: the 64-bit integer path.  Interval bounds two-sided, lower only and upper only."""
    m = models.subsampling_model(graph256, 7.0)
    n, G = m.num_variables, 64
    rng = np.random.default_rng(64)
    grp = np.where(rng.random(n) < 0.2, -1, rng.integers(0, G, size=n)).astype(np.int32)
    coef = (rng.choice([-1, 1], size=n) * rng.integers(1 << 19, 1 << 20, size=n)).astype(np.int32)
    lam = rng.uniform(2e-14, 2e-13, size=G)           # flip costs of order 1 at |u| ~ 2^22
    kap = rng.integers(-(1 << 21), 1 << 21, size=G).astype(np.int64)
    g = (grp, coef, lam, kap)
    if bounds == "interval":
        lo = rng.integers(-(1 << 22), 1 << 22, size=G).astype(np.int64)
        hi = lo + rng.integers(0, 1 << 22, size=G)
        side = np.arange(G) % 3
        g += (np.where(side == 2, I64.min, lo), np.where(side == 1, I64.max, hi))
    _assert_exact(*_run(kctx, m.h, m.starts, m.ends, m.weights, g, 64, 30, 19))
    assert kctx.last_kernel == kctx.requested_kernel


def test_le_constraint_model(kctx):
    cqm = ConstrainedQuadraticModel()
    x = [Binary(f"x{i}") for i in range(200)]
    obj = x[0] * 0
    for i in range(199):
        obj = obj - x[i] * x[i + 1] - 0.1 * x[i]
    cqm.set_objective(obj)
    tot = x[0]
    for i in range(1, 120):
        tot = tot + x[i]
    cqm.add_constraint(tot <= 30, label="cap")
    m = cqm.to_lowered(lowering="interval", constraint_penalty=2.0)
    _assert_exact(*_run(kctx, m.h, m.starts, m.ends, m.weights, m.groups.astuple(), 64, 30, 13))


def test_zero_bounds_equal_equality_run(kctx, graph256):
    m = models.cqm_model(graph256, 4)
    eq = m.groups.astuple()
    G = len(eq[2])
    ivl = eq + (np.zeros(G, dtype=np.int64), np.zeros(G, dtype=np.int64))
    # both against the same reference run of the equality groups: bitwise the same trajectories
    _assert_exact(*_run(kctx, m.h, m.starts, m.ends, m.weights, ivl, 64, 30, 17, ref_groups=eq))
    _assert_exact(*_run(kctx, m.h, m.starts, m.ends, m.weights, eq, 64, 30, 17))


def test_device_builder_matches_host(built, graph256):
    n, K, ms, A, B = 256, 4, 50, 9.0, 2.5
    host = models.cqm_model(graph256, K, min_size=ms, onehot_penalty=A, size_penalty=B, size_lowering="interval")
    slack = models.cqm_model(graph256, K, min_size=ms, onehot_penalty=A, size_penalty=B)
    spec = models.device_spec("cqm", graph256, num_of_clusters=K, min_size=ms)
    with Context(0) as ctx:
        gm, off = ctx.build_cqm_interval(spec["graph"], K, ms, A, B)
        h, st, en, w = gm.get_ising()
        gs, off_s = ctx.build_cqm_penalty(spec["graph"], K, ms, A, B)
        hs = gs.get_ising()[0]
        gm.close()
        gs.close()
    assert np.array_equal(h.view(np.uint64), host.h.view(np.uint64)) and off == host.offset + 0.0
    assert np.array_equal(st, host.starts) and np.array_equal(en, host.ends)
    assert np.array_equal(w.view(np.uint64), host.weights.view(np.uint64))
    assert np.array_equal(h.view(np.uint64), hs[: n * K].view(np.uint64)) and off == off_s
    assert slack.offset == host.offset


def test_config3_size_replay_auto(built):
    graph = snn.synthetic_snn(16384, k=5, dim=15, centres=8, seed=0)[0]   # bench.py's config-3 graph
    m = models.cqm_model(graph, 8, min_size=1900, size_lowering="interval")
    R, n = 6144, m.num_variables
    betas, spb = schedule.make_beta_schedule((0.05, 8.0), 6, 1, "geometric")
    seeds = schedule.per_read_seeds(21, R)
    init = schedule.random_spin_states(R, n, 21)
    with Context(0) as ctx:
        gm = IsingModel(ctx, m.h, m.starts, m.ends, m.weights)
        gm.set_groups(*m.groups.astuple())
        states = init.copy()
        e, st, done = gm.sample(states, betas, spb, seeds)
        assert ctx.last_kernel == _lib.QA_KERNEL_REPLAY
        gm.close()
    pick = np.array([0, 1, 2, R // 2, R // 2 + 1, R - 3, R - 2, R - 1])
    ref = init[pick].copy()
    ref_e, _ = iref.sample_ising(m.h, m.starts, m.ends, m.weights, ref, betas, spb, seeds[pick], groups=m.groups.astuple())
    assert np.array_equal(states[pick], ref)
    assert np.array_equal(e[pick].view(np.uint64), ref_e.view(np.uint64))


def test_concat_interval_models(built, graph256):
    g2 = snn.synthetic_snn(200, k=5, seed=8)[0]
    ms = [models.cqm_model(graph256, 4, min_size=60, size_lowering="interval"),
          models.cqm_model(g2, 3, min_size=60, size_lowering="interval")]
    R = 64
    betas, spb = schedule.make_beta_schedule((0.05, 8.0), 20, 1, "geometric")
    with Context(0) as ctx:
        gms, sep = [], []
        for p, m in enumerate(ms):
            gm = IsingModel(ctx, m.h, m.starts, m.ends, m.weights)
            gm.set_groups(*m.groups.astuple())
            gms.append(gm)
            seeds = schedule.per_read_seeds(30 + p, R)
            st = schedule.random_spin_states(R, m.num_variables, 30 + p)
            init = st.copy()
            e, _, _ = gm.sample(st, betas, spb, seeds)
            sep.append((init, seeds, st, e))
        batch = ctx.concat_models(gms)
        states = np.concatenate([s[0].ravel() for s in sep]).astype(np.int8)
        seeds = np.concatenate([s[1] for s in sep])
        e, _, done = ctx.sample_model_batch(batch, R, states, betas, spb, seeds)
        assert done == R   # reads per problem
        assert ctx.last_kernel == _lib.QA_KERNEL_WARP_PER_READ
        off = 0
        for p, m in enumerate(ms):
            got = states[off: off + R * m.num_variables].reshape(R, m.num_variables)
            assert np.array_equal(got, sep[p][2])
            assert np.array_equal(e[p * R:(p + 1) * R].view(np.uint64), sep[p][3].view(np.uint64))
            off += R * m.num_variables
        batch.close()
        for gm in gms:
            gm.close()


def test_sample_cqm_interval_end_to_end(built, capsys):
    from scrna_seq_qannealing_clustering_b200.sampler import B200SimulatedAnnealingSampler
    nc = 120
    graph = snn.synthetic_snn(nc, k=6, seed=4)[0]
    K, ms = 4, 27                                   # 30 cells per cluster on average: the size bound binds
    _, eu, ev, w = models.graph_arrays(graph)
    cqm = ConstrainedQuadraticModel()
    x = {(i, p): Binary(f"v_{i},{p}") for i in range(nc) for p in range(K)}
    obj = x[(0, 0)] * 0
    for u, v, wt in zip(eu.tolist(), ev.tolist(), w.tolist()):
        for p in range(K):
            obj = obj + x[(u, p)] + x[(v, p)] - 2 * wt * x[(u, p)] * x[(v, p)]
    cqm.set_objective(obj)
    for i in range(nc):
        cqm.add_discrete([f"v_{i},{p}" for p in range(K)], label=f"one_hot_{i}")
    for p in range(K):
        tot = x[(0, p)]
        for i in range(1, nc):
            tot = tot + x[(i, p)]
        cqm.add_constraint(tot >= ms, label=f"size_{p}")
    smp = B200SimulatedAnnealingSampler()
    m = models.cqm_model(graph, K, min_size=ms, size_lowering="interval")
    ss = smp.sample_cqm(m, num_reads=200, num_sweeps=400, seed=5)
    fs = np.asarray(ss.record.is_feasible)
    sl = smp.sample_cqm(models.cqm_model(graph, K, min_size=ms), num_reads=200, num_sweeps=400, seed=5)
    with capsys.disabled():
        print(f"\n[interval] feasible {fs.mean():.3f}  [slack, same instance] feasible {np.asarray(sl.record.is_feasible).mean():.3f}")
    assert fs.mean() >= 0.9
    gen = smp.sample_cqm(cqm, size_lowering="interval", onehot_penalty=m.meta["onehot_penalty"],
                         constraint_penalty=m.meta["onehot_penalty"], num_reads=50, num_sweeps=200, seed=6)
    assert set(gen.variables) == set(cqm.variables)
    chk = cqm.check_feasible(np.asarray(gen.record.sample), list(gen.variables))
    assert np.array_equal(np.asarray(gen.record.is_feasible), chk)
    smp.close()


def test_error_paths(built, graph256):
    m = models.cqm_model(graph256, 4, size_lowering="interval")
    with Context(0) as ctx:
        gm = IsingModel(ctx, m.h, m.starts, m.ends, m.weights)
        grp, coef, lam, kap, lo, hi = m.groups.astuple()
        gm.set_groups(grp, coef, lam, kap)
        with pytest.raises(QAnnealError) as e:
            gm.set_group_bounds(np.array([1, 0, 0, 0]), np.array([0, 0, 0, 0]))
        assert e.value.code == -1
        with pytest.raises(QAnnealError) as e:
            gm.set_group_bounds(np.full(4, 10 ** 9), np.full(4, I64.max))
        assert e.value.code == -5
        # set_groups after set_group_bounds: equality semantics again (== the reference's equality run)
        gm.set_group_bounds(lo, hi)
        gm.set_groups(grp, coef, lam, kap)
        R = 32
        betas, spb = schedule.make_beta_schedule((0.05, 8.0), 20, 1, "geometric")
        seeds = schedule.per_read_seeds(3, R)
        init = schedule.random_spin_states(R, m.num_variables, 3)
        st = init.copy()
        e_gpu, _, _ = gm.sample(st, betas, spb, seeds)
        ref = init.copy()
        ref_e, _ = iref.sample_ising(m.h, m.starts, m.ends, m.weights, ref, betas, spb, seeds, groups=(grp, coef, lam, kap))
        assert np.array_equal(st, ref) and np.array_equal(e_gpu.view(np.uint64), ref_e.view(np.uint64))
        gm.close()
