"""CPU checks of tests/output_reference.py: every function against a slow, obviously correct loop, on small random and
hand-built inputs (NaN bit patterns of both signs, signed zeros, subnormals, infinities, all-equal rows, n = 0)."""
import math

import numpy as np
import pytest

import output_reference as ref


def f64(bits):
    return np.array([bits], dtype=np.uint64).view(np.float64)[0]


NANS = [f64(0x7FF8000000000000), f64(0xFFF8000000000000), f64(0x7FF0000000000001), f64(0xFFF0000000000123),
        f64(0x7FFFFFFFFFFFFFFF), f64(0xFFFFFFFFFFFFFFFF)]
SPECIAL = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, -2.2250738585072014e-308, np.inf, -np.inf, 1.0,
           np.nextafter(1.0, 2.0), np.nextafter(1.0, 0.0), -1.0, 1e308, -1e308]


def slow_sort(e):
    """Insertion sort with the contract's comparison written out: a NaN is greater than every number, two NaNs are equal,
    -0.0 == +0.0; an element moves left only past a strictly greater one (stable)."""
    def greater(a, b):
        if math.isnan(a):
            return not math.isnan(b)
        return not math.isnan(b) and a > b
    out = []
    for i, x in enumerate(e):
        j = len(out)
        while j > 0 and greater(e[out[j - 1]], x):
            j -= 1
        out.insert(j, i)
    return np.array(out, dtype=np.int64)


def slow_argmin(v):
    best = None
    for i, x in enumerate(v):
        if best is None:
            best = i
        elif math.isnan(v[best]) and not math.isnan(x):
            best = i
        elif not math.isnan(x) and x < v[best]:
            best = i
    return (np.float64(np.inf), -1) if best is None else (v[best], best)


def slow_aggregate(states):
    seen = {}
    for r, row in enumerate(states):
        k = bytes(np.asarray(row, dtype=np.int8).tobytes())
        if k in seen:
            seen[k][1] += 1
        else:
            seen[k] = [r, 1]
    return [tuple(x) for x in seen.values()]


def slow_decode(states, cells, K, stride, on, min_size):
    R = states.shape[0]
    labels = np.full((R, cells), -1, dtype=np.int32)
    viol = np.zeros((R, 2), dtype=np.int32)
    for r in range(R):
        sizes = [0] * K
        for c in range(cells):
            hits = [k for k in range(K) if states[r, c * K + k] == on]
            if len(hits) == 1:
                labels[r, c] = hits[0]
                sizes[hits[0]] += 1
            else:
                viol[r, 0] += 1
        viol[r, 1] = sum(s < min_size for s in sizes)
    return labels, viol


def edge_vectors(rng):
    pool = np.array(SPECIAL + NANS)
    yield np.array([])
    yield np.array([NANS[1]])
    yield np.array(NANS)
    yield np.array(NANS[::-1] + [np.inf])
    yield np.array([-0.0, 0.0, -0.0, 0.0])
    yield np.array([0.0, -0.0])
    yield np.array([np.inf] * 5)
    yield np.array([NANS[1], -np.inf, NANS[0], np.inf])          # x86 inf - inf is the sign-set NaN 0xfff8...
    yield np.full(9, 3.25)
    for size in (1, 2, 7, 40, 200):
        yield rng.choice(pool, size=size)
        yield rng.normal(size=size)
        yield np.nextafter(np.full(size, 1.5), rng.choice([0.0, 3.0], size=size)) * rng.choice([1, 1, -1], size=size)


def test_sort_order_and_key_match_the_slow_loop():
    rng = np.random.default_rng(0)
    for v in edge_vectors(rng):
        want = slow_sort(list(v))
        assert np.array_equal(ref.sort_order(v), want), v
        # the device's radix key: a stable ascending sort of the keys is the same order
        assert np.array_equal(np.argsort(ref.sort_key(v), kind="stable"), want), v


def test_sort_key_separates_nan_from_everything():
    v = np.array(SPECIAL + NANS)
    k = ref.sort_key(v)
    nan = np.isnan(v)
    assert (k[nan] == ref.NAN_KEY).all()
    assert (k[~nan] < ref.NAN_KEY).all()
    assert ref.sort_key(np.array([0.0]))[0] == ref.sort_key(np.array([-0.0]))[0]
    # the mapping the parent used (~bits for every sign-set pattern) put 0xfff8... below -inf: the case that must not recur
    assert ref.sort_key(np.array([NANS[1]]))[0] > ref.sort_key(np.array([-np.inf]))[0]


def test_argmin_matches_the_slow_loop_bit_for_bit():
    rng = np.random.default_rng(1)
    for v in edge_vectors(rng):
        bv, bi = ref.argmin(v)
        wv, wi = slow_argmin(list(v))
        assert bi == wi, v
        assert np.float64(bv).view(np.uint64) == np.float64(wv).view(np.uint64), v
        if len(v):
            assert bi == ref.sort_order(v)[0]


def test_argmin_hand_cases():
    assert ref.argmin(np.array([])) == (np.inf, -1)
    bv, bi = ref.argmin(np.array(NANS))
    assert bi == 0 and np.float64(bv).view(np.uint64) == 0x7FF8000000000000
    bv, bi = ref.argmin(np.array([0.0, -0.0]))
    assert bi == 0 and not math.copysign(1.0, bv) < 0
    bv, bi = ref.argmin(np.array([-0.0, 0.0]))
    assert bi == 0 and math.copysign(1.0, bv) < 0
    assert ref.argmin(np.array([NANS[1], np.inf]))[1] == 1
    assert ref.argmin(np.array([np.inf, np.inf]))[1] == 0
    assert ref.argmin(np.array([5e-324, 0.0, -5e-324]))[1] == 2


@pytest.mark.parametrize("n", [0, 1, 2, 5, 33])
def test_aggregate_matches_the_slow_loop(n):
    rng = np.random.default_rng(n)
    cases = [np.ones((6, n), dtype=np.int8), np.zeros((0, n), dtype=np.int8)]
    base = rng.choice(np.array([-1, 1], dtype=np.int8), size=(4, n))
    cases.append(base[rng.integers(0, 4, size=50)])
    cases.append(rng.integers(-128, 128, size=(30, n)).astype(np.int8))
    if n:
        last = np.repeat(base[:1], 40, axis=0)
        last[:, -1] = rng.integers(-3, 3, size=40)
        first = last.copy()
        first[:, -1] = base[0, -1]
        first[:, 0] = rng.integers(-3, 3, size=40)
        cases += [last, first]
    for s in cases:
        f, c = ref.aggregate(s)
        want = slow_aggregate(s)
        assert list(zip(f.tolist(), c.tolist())) == want
        assert c.sum() == s.shape[0]


def test_aggregate_without_variables_is_one_group():
    f, c = ref.aggregate(np.zeros((7, 0), dtype=np.int8))
    assert f.tolist() == [0] and c.tolist() == [7]


def test_gather():
    s = np.arange(12, dtype=np.int8).reshape(4, 3)
    assert np.array_equal(ref.gather(s, [3, 3, 0]), s[[3, 3, 0]])
    for bad in ([-1], [4]):
        with pytest.raises(IndexError):
            ref.gather(s, bad)


@pytest.mark.parametrize("K", [1, 2, 3, 8])
@pytest.mark.parametrize("cells", [1, 5, 13])
def test_decode_onehot_matches_the_slow_loop(K, cells):
    rng = np.random.default_rng(K * 100 + cells)
    for on in (1, -1):
        for slack in (0, 3):
            stride = cells * K + slack
            R = 6
            s = np.full((R, stride), -on, dtype=np.int8)
            lab = rng.integers(0, K, size=(R, cells))
            for r in range(R):
                for c in range(cells):
                    s[r, c * K + lab[r, c]] = on
            # break some cells: none set, two set; slack holds on_value and values other than +-1
            s[0, : cells * K] = -on
            if K > 1:
                s[1, :2] = on
            s[2, : min(K, cells * K)] = on
            s[:, cells * K:] = rng.choice(np.array([on, 0, 7, -100], dtype=np.int8), size=(R, slack))
            for min_size in (0, 1, cells // K, cells + 1):
                labels, viol = ref.decode_onehot(s, cells, K, stride, on, min_size)
                wl, wv = slow_decode(s, cells, K, stride, on, min_size)
                assert np.array_equal(labels, wl) and np.array_equal(viol, wv)


def test_decode_onehot_geometry_errors():
    s = np.ones((2, 6), dtype=np.int8)
    with pytest.raises(ValueError):
        ref.decode_onehot(s, 3, 0, 6, 1, 0)
    with pytest.raises(ValueError):
        ref.decode_onehot(s, 4, 2, 6, 1, 0)
