"""The output-stage kernels at their edges, exactly against tests/output_reference.py: energies (k_energy / k_pack_states),
argmin (k_argmin, k_argmin_pack), ranking (k_energy_keys + radix sort), aggregation (k_hash_rows / k_mark_heads), the top-k
gather (k_gather_rows) and the one-hot decode (k_decode_onehot / k_count_small_clusters).

Indices must be equal, doubles equal as uint64 bit patterns, error codes equal by value.  Every entry point runs with host
numpy inputs and with CUDA torch tensors."""
import numpy as np
import pytest

import output_reference as ref
from scrna_seq_qannealing_clustering_b200 import schedule
from scrna_seq_qannealing_clustering_b200._lib import QAnnealError
from scrna_seq_qannealing_clustering_b200.engine import IsingModel

pytestmark = pytest.mark.gpu

I64 = np.iinfo(np.int64)


def f64(bits):
    return np.array([bits], dtype=np.uint64).view(np.float64)[0]


def bits(x):
    return int(np.float64(x).view(np.uint64))


def u64(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


# quiet NaNs, signalling-pattern payload NaNs and all-ones NaNs, both signs; 0xfff8... is what x86 makes of inf - inf
NANS = [f64(0x7FF8000000000000), f64(0xFFF8000000000000), f64(0x7FF0000000000001), f64(0xFFF0000000000123),
        f64(0x7FF4000000000abc), f64(0xFFFFFFFFFFFFFFFF)]
TINY = 2.2250738585072014e-308


# ---- ranking: qa_sort_reads -----------------------------------------------------------------------------------------
def _ulp_pool():
    up = [1.0]
    for _ in range(4):
        up.append(np.nextafter(up[-1], 2.0))
    down = [np.nextafter(1.0, 0.0)]
    for _ in range(3):
        down.append(np.nextafter(down[-1], 0.0))
    return up + down + [-x for x in up]


VALUE_SETS = {
    "all_equal": [-3.75],
    "one_ulp": _ulp_pool(),
    "signed_zero": [0.0, -0.0],
    "subnormal": [0.0, -0.0, 5e-324, -5e-324, 1e-310, -1e-310, TINY, -TINY],
    "infinite": [np.inf, -np.inf, 0.0, -1.0, 1.0],
    "nan": None,            # normal values with NaNs of every pattern scattered through them
    "nan_specials": [np.inf, -np.inf, 0.0, -0.0, 5e-324, -5e-324] + NANS,
}


def _values(kind, R, rng):
    if kind == "nan":
        v = rng.normal(size=R)
        hit = rng.random(R) < 0.1
        v[hit] = rng.choice(np.array(NANS), size=int(hit.sum()))
        if R > 1:
            v[0], v[-1] = NANS[1], NANS[0]
        return v
    return rng.choice(np.array(VALUE_SETS[kind], dtype=np.float64), size=R)


@pytest.mark.parametrize("kind", list(VALUE_SETS))
@pytest.mark.parametrize("R", [1, 2, 31, 255, 256, 257, 4097, 300_000])
def test_sort_reads(gpu_ctx, R, kind):
    v = _values(kind, R, np.random.default_rng(R + len(kind)))
    want = ref.sort_order(v)
    assert np.array_equal(gpu_ctx.sort_reads(v), want)
    assert np.array_equal(gpu_ctx.sort_reads(dev(v)), want)


# ---- argmin: qa_argmin, qa_argmin_device ------------------------------------------------------------------------------
ARGMIN_COUNTS = [1, 31, 32, 33, 1023, 1024, 1025, 2049, 1_000_007]


def _argmin_cases(count, rng):
    base = rng.uniform(1.0, 2.0, size=count)

    def put(at):
        v = base.copy()
        for i, x in at.items():
            v[i] = x
        return v

    yield "first", put({0: 0.5})
    yield "last", put({count - 1: 0.5})
    # ties: different warps, the same thread's stride (i and i + 1024), different lanes of one warp
    for a, b in ((3, 3 + 32 * 5), (7, 7 + 1024), (2, 29), (count - 2, count - 1)):
        if 0 <= a < b < count:
            yield f"tie_{a}_{b}", put({a: 0.25, b: 0.25})
            yield f"zero_{a}_{b}", put({a: 0.0, b: -0.0})
            yield f"negzero_{a}_{b}", put({a: -0.0, b: 0.0})
    yield "all_inf", np.full(count, np.inf)
    yield "all_nan", rng.choice(np.array(NANS), size=count)
    yield "all_neg_nan", np.full(count, NANS[1])
    v = base.copy()
    hit = rng.random(count) < 0.2
    v[hit] = rng.choice(np.array(NANS), size=int(hit.sum()))
    v[0] = NANS[1]
    yield "nan_mixed", v
    if count > 1:
        v = rng.choice(np.array(NANS), size=count)
        v[count // 2] = np.inf
        yield "nan_and_one_inf", v
        v = np.full(count, NANS[3])
        v[-1] = -np.inf
        yield "neg_nan_then_neg_inf", v


def _check_argmin(ctx, v, what):
    wv, wi = ref.argmin(v)
    for vals in (v, dev(v)):
        bv, bi = ctx.argmin(vals)
        assert bi == wi and bits(bv) == bits(wv), what
    for off in (0, 1 << 40):
        import torch
        out = torch.full((2,), -7.0, dtype=torch.float64, device="cuda")
        for vals in (v, dev(v)):
            ctx.argmin_into(vals, off, out)
            o = host(out)
            assert bits(o[0]) == bits(wv), what
            assert o[1] == float(off + wi) and int(o[1]) == off + wi, what
    # the best read is the first one of the ranking
    assert int(ctx.sort_reads(v)[0]) == wi, what


@pytest.mark.parametrize("count", ARGMIN_COUNTS)
def test_argmin(gpu_ctx, count):
    for what, v in _argmin_cases(count, np.random.default_rng(count)):
        _check_argmin(gpu_ctx, v, what)


def test_argmin_empty(gpu_ctx):
    assert gpu_ctx.argmin(np.zeros(0)) == (np.inf, -1)
    import torch
    out = torch.zeros(2, dtype=torch.float64, device="cuda")
    with pytest.raises(QAnnealError) as ei:
        gpu_ctx.argmin_into(np.zeros(0), 0, out)
    assert ei.value.code == -1


def test_energies_best_pair_ties(gpu_ctx):
    """The best pair of IsingModel.energies (k_energy then k_argmin): a model with 8 distinct energies, the lowest state
    planted at two reads in different warps / strides / lanes."""
    h = np.array([1.0, 2.0, 4.0])
    gm = IsingModel(gpu_ctx, h, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0))
    rng = np.random.default_rng(5)
    for R in ARGMIN_COUNTS[:-1]:
        for a, b in ((0, R - 1), (3, 163), (7, 1031), (2, 29), (R - 1, R - 1)):
            if not (0 <= a <= b < R):
                continue
            s = np.where(rng.random((R, 3)) < 0.5, 1, -1).astype(np.int8)
            s[:, 2] = 1                                   # every other read has E >= -3
            s[a] = s[b] = -1                              # E = -7
            want = ref.energies(h, [], [], [], s)
            e, be, bi, _ = gm.energies(s)
            assert np.array_equal(u64(e), u64(want))
            wv, wi = ref.argmin(want)
            assert (bi, bits(be)) == (wi, bits(wv)) and wi == a
            de = dev(np.zeros(R))
            _, be, bi, _ = gm.energies(dev(s), de)
            assert np.array_equal(u64(host(de)), u64(want)) and (bi, bits(be)) == (wi, bits(wv))
    gm.close()


# ---- aggregation: qa_aggregate_reads ----------------------------------------------------------------------------------
AGG_R = [1, 2, 255, 256, 257, 70_000]
AGG_N = [0, 1, 2, 31, 300, 100_003]


def _agg_cases(R, n, rng):
    pm = np.array([-1, 1], dtype=np.int8)
    base = rng.choice(pm, size=n)
    yield "equal", np.tile(base, (R, 1))
    yield "distinct", rng.choice(pm, size=(R, n))
    if n:
        s = np.tile(base, (R, 1))
        s[:, -1] = rng.integers(-4, 4, size=R)
        yield "last_byte", s
        s = np.tile(base, (R, 1))
        s[:, 0] = rng.integers(-4, 4, size=R)
        yield "first_byte", s
    uniq = rng.choice(pm, size=(max(1, R // 7), n))
    yield "shuffled_duplicates", uniq[rng.integers(0, len(uniq), size=R)]


@pytest.mark.parametrize("n", AGG_N)
@pytest.mark.parametrize("R", AGG_R)
def test_aggregate_reads(gpu_ctx, R, n):
    if R * n > 1 << 26:
        pytest.skip("state matrix above 64 MB: the 257-read and 300-variable cases cover both extents")
    rng = np.random.default_rng(R * 7 + n)
    for what, s in _agg_cases(R, n, rng):
        s = np.ascontiguousarray(s, dtype=np.int8)
        wf, wc = ref.aggregate(s)
        for states in (s, dev(s)):
            f, c = gpu_ctx.aggregate_reads(states)
            assert np.array_equal(f, wf) and np.array_equal(c, wc), what


# ---- top-k gather: qa_gather_samples ----------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 15, 16, 17, 4097])
@pytest.mark.parametrize("R", [1, 37])
def test_gather_samples(gpu_ctx, R, n):
    rng = np.random.default_rng(R * 31 + n)
    s = rng.integers(-128, 128, size=(R, n)).astype(np.int8)
    for k in (1, R, 3 * R):
        order = rng.integers(0, R, size=k).astype(np.int32)        # 3R: every read repeated
        want = ref.gather(s, order)
        for states in (s, dev(s)):
            assert np.array_equal(gpu_ctx.gather_samples(states, order), want)
    for bad in (-1, R):
        order = np.array([0, bad], dtype=np.int32)
        for states in (s, dev(s)):
            with pytest.raises(QAnnealError) as ei:
                gpu_ctx.gather_samples(states, order)
            assert ei.value.code == -2


# ---- one-hot decode: qa_decode_onehot ---------------------------------------------------------------------------------
def _onehot_states(R, cells, K, stride, on, rng):
    core = np.full((R, cells, K), -on, dtype=np.int8)
    lab = rng.integers(0, K, size=(R, cells))
    np.put_along_axis(core, lab[:, :, None], on, axis=2)
    core[rng.random((R, cells)) < 0.05] = -on                 # cells with no case set
    if K > 1:
        two = rng.random((R, cells)) < 0.05                   # cells with two cases set
        core[two, (lab[two] + 1) % K] = on
    s = np.empty((R, stride), dtype=np.int8)
    s[:, : cells * K] = core.reshape(R, cells * K)
    if stride > cells * K:                                    # slack: on_value and values other than +-1
        s[:, cells * K:] = rng.choice(np.array([on, 0, 2, -128, 127], dtype=np.int8), size=(R, stride - cells * K))
    return s


@pytest.mark.parametrize("cells", [1, 31, 1000])
@pytest.mark.parametrize("K", [1, 2, 3, 8, 16, 64])
def test_decode_onehot(gpu_ctx, K, cells):
    rng = np.random.default_rng(K * 1000 + cells)
    for R in (1, 255, 256, 257, 5000):
        for stride in (cells * K, cells * K + 13):
            if R * stride > 1 << 26:
                continue    # 5000 reads of 16 or 64 cases x 1000 cells: the 257-read matrices cover those widths
            for on in (1, -1):
                s = _onehot_states(R, cells, K, stride, on, rng)
                d = dev(s)
                for min_size in (0, 1, cells // K, cells + 1):
                    wl, wv = ref.decode_onehot(s, cells, K, stride, on, min_size)
                    for states in (s, d):
                        labels, viol = gpu_ctx.decode_onehot(states, cells, K, on_value=on, min_size=min_size)
                        assert np.array_equal(labels, wl) and np.array_equal(viol, wv), (R, stride, on, min_size)
                        none, viol = gpu_ctx.decode_onehot(states, cells, K, on_value=on, min_size=min_size, want_labels=False)
                        assert none is None and np.array_equal(viol, wv), (R, stride, on, min_size)


def test_decode_onehot_geometry_errors(gpu_ctx):
    s = np.ones((4, 12), dtype=np.int8)
    for cells, K in ((3, 0), (3, -2), (4, 4), (13, 1)):       # K < 1, and stride 12 < cells * K
        with pytest.raises(QAnnealError) as ei:
            gpu_ctx.decode_onehot(s, cells, K)
        assert ei.value.code == -1


# ---- energies: qa_energy_argmin and the post-anneal k_energy ---------------------------------------------------------
def _couplers(n, m, rng):
    """m couplers among the first n - n // 8 variables (the rest isolated), unsorted, in both orientations, with duplicates."""
    act = n - n // 8
    if m == 0 or act < 2:
        return np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0)
    u = rng.integers(0, act, size=m)
    v = rng.integers(0, act - 1, size=m)
    v = v + (v >= u)
    if m >= 4:
        u[-1], v[-1] = v[0], u[0]          # the first coupler again, the other way round
        u[-2], v[-2] = u[1], v[1]          # and the second one again as it was
    return u.astype(np.int32), v.astype(np.int32), rng.normal(size=m)


def _groups(kind, n, rng):
    """None, or the (grp, coef, lam, kappa[, lo, hi]) tuple of ``kind``: one group or QA_MAX_GROUPS = 64 groups with holes
    (grp = -1) and coefficients of 2^19 .. 2^20 (the 64-bit integer path), equality or interval bounds (one-sided ones too)."""
    if kind == "none":
        return None
    G = 1 if kind.endswith("1") else 64
    grp = np.where(rng.random(n) < 0.2, -1, rng.integers(0, G, size=n)).astype(np.int32)
    if G == 1:
        coef = rng.choice([-3, -1, 1, 2, 5], size=n).astype(np.int32)
        kappa = np.array([-2], dtype=np.int64)
    else:
        coef = (rng.choice([-1, 1], size=n) * rng.integers(1 << 19, 1 << 20, size=n)).astype(np.int32)
        kappa = rng.integers(-(1 << 21), 1 << 21, size=G).astype(np.int64)
    lam = rng.uniform(0.1, 3.0, size=G)
    if kind.startswith("eq"):
        return grp, coef, lam, kappa
    scale = 4 if G == 1 else 1 << 22
    lo = rng.integers(-scale, scale, size=G).astype(np.int64)
    hi = lo + rng.integers(0, scale, size=G)
    side = np.arange(G) % 3                                  # two-sided, lower bound only, upper bound only
    lo = np.where(side == 2, I64.min, lo)
    hi = np.where(side == 1, I64.max, hi)
    if G == 1:
        hi[:] = I64.max
    return grp, coef, lam, kappa, lo, hi


ENERGY_M = [0, 1, 15, 16, 17, 31, 160, 161, 175]


@pytest.mark.parametrize("groups", ["none", "eq1", "ivl1", "eq64", "ivl64"])
@pytest.mark.parametrize("n", [1, 31, 32, 33, 1000])
def test_energies(gpu_ctx, n, groups):
    rng = np.random.default_rng(n * 10 + len(groups))
    h = rng.normal(size=n)
    h[n - n // 8:] *= 3.0
    for m in ENERGY_M if n > 1 else [0]:
        u, v, w = _couplers(n, m, rng)
        g = _groups(groups, n, rng)
        gm = IsingModel(gpu_ctx, h, u, v, w)
        if g is not None:
            gm.set_groups(*g)
        for R in (1, 127, 128, 129, 1000):
            s = np.where(rng.random((R, n)) < 0.5, 1, -1).astype(np.int8)
            want = ref.energies(h, u, v, w, s, groups=g)
            wv, wi = ref.argmin(want)
            e, be, bi, _ = gm.energies(s)
            assert np.array_equal(u64(e), u64(want)), (m, R)
            assert (bi, bits(be)) == (wi, bits(wv)), (m, R)
            # zero sweeps: the energies of the post-anneal k_energy launch
            st = s.copy()
            e2, _, done = gm.sample(st, np.zeros(0), 1, schedule.per_read_seeds(R, R))
            assert done == R and np.array_equal(st, s)
            assert np.array_equal(u64(e2), u64(want)), (m, R)
            if R == 129:
                de = dev(np.zeros(R))
                _, be, bi, _ = gm.energies(dev(s), de)
                assert np.array_equal(u64(host(de)), u64(want)) and (bi, bits(be)) == (wi, bits(wv)), m
                ds, de = dev(s), dev(np.zeros(R))
                gm.sample(ds, np.zeros(0), 1, schedule.per_read_seeds(R, R), energies=de)
                assert np.array_equal(host(ds), s) and np.array_equal(u64(host(de)), u64(want)), m
        gm.close()


def test_energies_concatenated_mixed_groups(gpu_ctx):
    """One k_energy<true> launch over an interval-group, an equality-group (64 groups) and a group-free problem."""
    rng = np.random.default_rng(77)
    R = 129
    probs = []
    for n, kind in ((70, "ivl1"), (45, "eq64"), (33, "none")):
        h = rng.normal(size=n)
        u, v, w = _couplers(n, 3 * n + 1, rng)
        probs.append((h, u, v, w, _groups(kind, n, rng)))
    gms = []
    for h, u, v, w, g in probs:
        gm = IsingModel(gpu_ctx, h, u, v, w)
        if g is not None:
            gm.set_groups(*g)
        gms.append(gm)
    batch = gpu_ctx.concat_models(gms)
    inits = [np.where(rng.random((R, len(p[0]))) < 0.5, 1, -1).astype(np.int8) for p in probs]
    states = np.concatenate([s.ravel() for s in inits])
    e, _, done = gpu_ctx.sample_model_batch(batch, R, states, np.zeros(0), 1, schedule.per_read_seeds(3, 3 * R))
    assert done == R
    for p, (prob, s) in enumerate(zip(probs, inits)):
        want = ref.energies(*prob[:4], s, groups=prob[4])
        assert np.array_equal(u64(e[p * R:(p + 1) * R]), u64(want)), p
    batch.close()
    for gm in gms:
        gm.close()


def test_energies_reject_a_zero_state(gpu_ctx):
    h = np.ones(40)
    gm = IsingModel(gpu_ctx, h, np.array([1], np.int32), np.array([0], np.int32), np.ones(1))
    s = np.ones((130, 40), dtype=np.int8)
    s[129, 39] = 0
    for states in (s, dev(s)):
        with pytest.raises(QAnnealError) as ei:
            gm.energies(states)
        assert ei.value.code == -3
    # a clean call afterwards is not affected by the flag of the failed one
    e, _, _, _ = gm.energies(np.ones((3, 40), dtype=np.int8))
    assert np.array_equal(u64(e), u64(ref.energies(h, [1], [0], [1.0], np.ones((3, 40), dtype=np.int8))))
    gm.close()
