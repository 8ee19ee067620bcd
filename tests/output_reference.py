"""Plain numpy restatement of the output-stage entry points (csrc/postprocess.cu, csrc/energy.cu).

TEST INFRASTRUCTURE.  One function per entry point; each states the contract the GPU tests hold the kernels to, exactly
(indices equal, doubles bit for bit).  tests/test_output_reference_cpu.py checks every function against a slow loop.

- ``sort_order``     qa_sort_reads        ascending energy, stable; -0.0 == +0.0; every NaN after +inf, in read order
- ``sort_key``       k_energy_keys        the uint64 radix key whose stable ascending order is ``sort_order``
- ``argmin``         qa_argmin / qa_argmin_device / the best pair of qa_energy_argmin: the first read of ``sort_order``
- ``aggregate``      qa_aggregate_reads   (first read, count) of every distinct row, in order of first occurrence
- ``gather``         qa_gather_samples    ``states[order]``, an order entry outside [0, R) is QA_ERR_INDEX
- ``decode_onehot``  qa_decode_onehot     labels, per-read violation counts
- ``energies``       k_energy             ``oracle.state_energies`` (no groups, equality groups) or
                                          ``interval_reference.state_energies`` (interval groups): no third implementation
"""
from __future__ import annotations

import numpy as np

NAN_KEY = np.uint64(0xFFFFFFFFFFFFFFFF)
SIGN = np.uint64(0x8000000000000000)


def sort_order(e) -> np.ndarray:
    """Read indices by ascending value, ties in read order.  numpy's sort treats -0.0 and +0.0 as equal and puts every NaN,
    whatever its sign bit and payload, after +inf; the stable kind keeps read order among equal values and among NaNs."""
    return np.argsort(np.asarray(e, dtype=np.float64), kind="stable")


def sort_key(e) -> np.ndarray:
    """The radix key of each value: a stable ascending sort of these keys is ``sort_order``.  Non-NaN values map
    order-preservingly (x + 0.0 first, so -0.0 becomes +0.0 and the two tie); every NaN maps to the largest key."""
    e = np.asarray(e, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        b = (e + 0.0).view(np.uint64)
    key = np.where(b & SIGN, ~b, b | SIGN)
    return np.where(np.isnan(e), NAN_KEY, key).astype(np.uint64)


def argmin(v):
    """(v[i], i) with i the first entry of ``sort_order(v)``: the lowest non-NaN value, the lower index on a tie (-0.0 and +0.0
    tie), and (v[0], 0) when every value is NaN.  ``(inf, -1)`` for an empty input.  The value is v[i] bit for bit."""
    v = np.asarray(v, dtype=np.float64)
    if v.shape[0] == 0:
        return np.float64(np.inf), -1
    i = int(sort_order(v)[0])
    return v[i], i


def aggregate(states):
    """(first read index, count) of every distinct row of ``states`` [R][n], in order of first occurrence.  With n = 0 every
    row is the empty row: one group (0, R)."""
    states = np.asarray(states)
    R = states.shape[0]
    if R == 0:
        return np.empty(0, dtype=np.int32), np.empty(0, dtype=np.int32)
    _, first, count = np.unique(states, axis=0, return_index=True, return_counts=True)
    o = np.argsort(first, kind="stable")
    return first[o].astype(np.int32), count[o].astype(np.int32)


def gather(states, order):
    """``states[order]``; every order entry must lie in [0, R) (the library returns QA_ERR_INDEX otherwise)."""
    states = np.asarray(states)
    order = np.asarray(order, dtype=np.int64)
    if order.size and (order.min() < 0 or order.max() >= states.shape[0]):
        raise IndexError("order entry out of range")
    return states[order]


def decode_onehot(states, cells: int, K: int, stride: int, on_value: int, min_size: int):
    """One-hot decode of ``states`` [R][stride] (only the first cells * K columns count; cell c holds columns c*K .. c*K+K-1).
    -> (labels [R][cells]: the case whose entry equals ``on_value`` when exactly one does, else -1;
        violations [R][2]: cells that are not one-hot, cases with fewer than ``min_size`` cells)."""
    if K < 1 or stride < cells * K:
        raise ValueError("bad one-hot geometry")
    states = np.asarray(states, dtype=np.int8).reshape(-1, stride)
    R = states.shape[0]
    on = states[:, : cells * K].reshape(R, cells, K) == on_value
    cnt = on.sum(axis=2)
    labels = np.where(cnt == 1, on.argmax(axis=2), -1).astype(np.int32)
    sizes = np.zeros((R, K), dtype=np.int64)
    rr, cc = np.nonzero(labels >= 0)
    np.add.at(sizes, (rr, labels[rr, cc]), 1)
    viol = np.stack([(cnt != 1).sum(axis=1), (sizes < min_size).sum(axis=1)], axis=1).astype(np.int32)
    return labels, viol


def energies(h, starts, ends, weights, states, groups=None):
    """neal's get_state_energy of every row, plus the rank-1 group terms: the oracle for no groups and equality groups
    (4-tuple), the interval reference for interval groups (6-tuple, ``models.Groups.astuple()``)."""
    if groups is not None and len(groups) == 6:
        import interval_reference
        return interval_reference.state_energies(h, starts, ends, weights, states, groups=groups)
    from oracle import oracle
    return oracle.state_energies(h, starts, ends, weights, states, groups=groups)
