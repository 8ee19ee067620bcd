"""Reference helpers for the dense k-way tensor-core path (csrc/dense.cuh): exact energies, the specification of when a model
has the dense form, and dyadic dense models on which every kernel and the oracle compute in exact arithmetic.

No repository code is used here: these helpers are the yardstick, not the thing measured."""
import math

import numpy as np


def exact_energies(h, starts, ends, weights, states):
    """Correctly rounded Ising energy of every row of ``states`` (+-1).  Each term h_v s_v and J s_u s_v is an exact double
    (s = +-1 only flips the sign), so ``math.fsum`` of the term vector is the exact sum rounded once."""
    h = np.asarray(h, dtype=np.float64)
    starts = np.asarray(starts, dtype=np.int64)
    ends = np.asarray(ends, dtype=np.int64)
    weights = np.asarray(weights, dtype=np.float64)
    states = np.atleast_2d(np.asarray(states))
    out = np.empty(len(states), dtype=np.float64)
    for r, row in enumerate(states):
        s = row.astype(np.float64)
        terms = np.concatenate([h * s, weights * (s[starts] * s[ends])])
        out[r] = math.fsum(terms.tolist())
    return out


def dense_form(h, starts, ends, weights, K):
    """The dense k-way form (W, P) of an Ising model with variable v = cell * K + case, or None when the model does not have it.

    (W, P) exists exactly when
      * every inter-cell coupler joins equal cases, each pair of variables appears at most once, and a pair of cells is coupled
        in all K cases with one weight or in none (an absent pair is a zero of W), and
      * every cell has all K(K-1)/2 intra-cell pairs exactly once, each with weight P -- or no cell has any intra-cell coupler
        and P = 0."""
    n = len(h)
    if n == 0 or n % K:
        return None
    cells = n // K
    u = np.asarray(starts, dtype=np.int64)
    v = np.asarray(ends, dtype=np.int64)
    w = np.asarray(weights, dtype=np.float64)
    lo, hi = np.minimum(u, v), np.maximum(u, v)
    if len(np.unique(lo * n + hi)) != len(lo):
        return None                                                    # a pair listed twice
    ci, cj, ki, kj = lo // K, hi // K, lo % K, hi % K
    intra = ci == cj
    inter = ~intra
    if np.any(ki[inter] != kj[inter]):
        return None                                                    # cross-case inter-cell coupler
    W = np.zeros((cells, cells))
    count = np.zeros((cells, cells), dtype=np.int64)
    a, b, x = ci[inter], cj[inter], w[inter]
    first = ki[inter] == 0
    W[a[first], b[first]] = x[first]
    np.add.at(count, (a, b), 1)
    if np.any((count != 0) & (count != K)):
        return None                                                    # a cell pair coupled in some cases only
    if np.any(W[a, b] != x):
        return None                                                    # case-dependent weight
    W = W + W.T
    nintra = int(intra.sum())
    if nintra == 0:
        return W, 0.0
    if nintra != cells * K * (K - 1) // 2:                             # (pairs are distinct, so this means every cell is complete)
        return None
    P = w[intra]
    if np.any(P.view(np.uint64) != P[0].view(np.uint64)):
        return None
    return W, float(P[0])


def dyadic_dense_model(cells, K, seed, zero_frac=0.0, shuffle=False):
    """A dense k-way Ising model whose h, W and P are random integers in [-2^16, 2^16] times 2^-8.  Every partial sum any kernel
    or the oracle forms is then exact in fp64 (far below 2^53 units of 2^-9), so summation order cannot matter.

    ``zero_frac``: that fraction of the cell pairs get W = 0 and are left out of the coupler list (the CSR degree of a variable
    is then below ncells - 1 + K - 1).  ``shuffle``: couplers in random order with random orientation.
    Returns (h, starts, ends, weights, W, P)."""
    rng = np.random.default_rng(seed)
    q = lambda size: rng.integers(-(1 << 16), (1 << 16) + 1, size=size).astype(np.float64) * 2.0 ** -8   # noqa: E731
    n = cells * K
    h = q(n)
    W = np.zeros((cells, cells))
    pi, pj = np.tril_indices(cells, -1)                                # pi > pj
    wv = q(len(pi))
    if zero_frac > 0:
        wv[rng.random(len(pi)) < zero_frac] = 0.0
    W[pi, pj] = wv
    W = W + W.T
    P = float(q(1)[0]) if K > 1 else 0.0
    keep = wv != 0.0
    pi, pj, wv = pi[keep], pj[keep], wv[keep]
    cases = np.arange(K)
    st = [(pi[:, None] * K + cases).ravel()]
    en = [(pj[:, None] * K + cases).ravel()]
    wt = [np.repeat(wv, K)]
    if K > 1:
        c1, c2 = np.tril_indices(K, -1)
        base = np.arange(cells)[:, None] * K
        st.append((base + c1).ravel())
        en.append((base + c2).ravel())
        wt.append(np.full(cells * len(c1), P))
    starts, ends, weights = np.concatenate(st), np.concatenate(en), np.concatenate(wt)
    if shuffle:
        order = rng.permutation(len(starts))
        starts, ends, weights = starts[order], ends[order], weights[order]
        flip = rng.random(len(starts)) < 0.5
        starts, ends = np.where(flip, ends, starts), np.where(flip, starts, ends)
    return h, starts.astype(np.int32), ends.astype(np.int32), weights, W, P


def structure_mutations(cells=40, K=4, seed=0):
    """Variants of one dyadic k-way model, each breaking (or keeping) the dense form in one way: name -> (h, starts, ends,
    weights, has_dense_form).  The last element is what ``dense_form`` must say; the structure check on the device must agree."""
    h, st, en, w, _, P = dyadic_dense_model(cells, K, seed)
    lo, hi = np.minimum(st, en), np.maximum(st, en)
    intra = lo // K == hi // K
    inter_idx = np.nonzero(~intra)[0]
    case = lo % K

    def drop(mask):
        return h, st[~mask], en[~mask], w[~mask]

    def dup(i):
        return h, np.append(st, st[i]), np.append(en, en[i]), np.append(w, w[i])

    out = {"unchanged": (h, st, en, w, True)}
    out["cell_without_onehot"] = (*drop(intra & (lo // K == 5)), False)
    out["one_intra_pair_missing"] = (*drop(np.arange(len(st)) == np.nonzero(intra)[0][7]), False)
    out["intra_pair_twice"] = (*dup(np.nonzero(intra)[0][3]), False)
    out["inter_coupler_twice"] = (*dup(inter_idx[11]), False)
    # a case-1 coupler listed twice and another case-1 coupler missing: the per-case totals still match
    c1 = inter_idx[case[inter_idx] == 1]
    hh, s2, e2, w2 = dup(c1[2])
    keep = np.arange(len(s2)) != c1[9]
    out["inter_twice_and_one_missing"] = (hh, s2[keep], e2[keep], w2[keep], False)
    out["inter_pair_missing_in_one_case"] = (*drop(np.arange(len(st)) == c1[4]), False)
    wc = w.copy()
    wc[c1[6]] += 0.5
    out["inter_weight_depends_on_case"] = (h, st, en, wc, False)
    # a coupler between different cells and different cases, (cell 2, case 0) - (cell 9, case 1)
    out["cross_case_inter_coupler"] = (h, np.append(st, 9 * K + 1).astype(np.int32), np.append(en, 2 * K).astype(np.int32),
                                       np.append(w, 1.5), False)
    out["no_onehot_P0"] = (*drop(intra), True)
    w0 = w.copy()
    w0[intra & (lo == 0)] = 0.0                                        # variable 0's intra couplers 0, the others P != 0
    out["var0_intra_zero"] = (h, st, en, w0, P == 0.0)
    return out
