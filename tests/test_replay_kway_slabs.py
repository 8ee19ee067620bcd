"""CPU tests of the replay slabs' k-way section (csrc/anneal_replay.cu, through the host-only hook qa_debug_pack_slabs):
a Python specification of the cell detector and of the section, checked against the packed slabs block by block."""
import ctypes as C
import os

import numpy as np
import pytest

from scrna_seq_qannealing_clustering_b200 import _lib, models, snn

RP_D, RP_SLOTS, RP_CAP = 16, 64, 448
HDR = np.dtype([("nent", "<i4"), ("nbw", "<i4"), ("v0", "<i4"), ("nv", "<i4"), ("prev_slot", "<i4"), ("seq_off", "<i4"),
                ("nbw_next", "<i4"), ("kway", "<i4"), ("rowa", "<u4", RP_D), ("rowb", "<u4", RP_D), ("ga", "<i4", RP_D),
                ("bw", "<i4", RP_SLOTS), ("bw_next", "<i4", RP_SLOTS)])
ENT = np.dtype([("J", "<f8"), ("zero", "<u4"), ("B", "<u4")])


def _adjacency(model):
    n = model.num_variables
    rows = [[] for _ in range(n)]
    for a, b, w in zip(model.starts, model.ends, model.weights):
        rows[a].append((int(b), float(w)))
        rows[b].append((int(a), float(w)))
    rowptr = np.zeros(n + 1, dtype=np.int32)
    rowptr[1:] = np.cumsum([len(r) for r in rows])
    col = np.array([j for r in rows for j, _ in r] or [0], dtype=np.int32)
    val = np.array([w for r in rows for _, w in r] or [0.0], dtype=np.float64)
    return rows, rowptr, col, val


def pack(model, kway=True):
    rows, rowptr, col, val = _adjacency(model)
    lib = _lib.load()
    ns, nb, uni = C.c_int64(), C.c_int64(), C.c_int32()
    grp = coef = None
    ng = 0
    if model.groups is not None:
        grp = np.ascontiguousarray(model.groups.grp, dtype=np.int32)
        coef = np.ascontiguousarray(model.groups.coef, dtype=np.int32)
        ng = len(model.groups.lam)
    args = [model.num_variables, _lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(val), ng, _lib.ptr(grp), _lib.ptr(coef), C.byref(ns),
            C.byref(nb), C.byref(uni)]
    old = os.environ.get("QA_REPLAY_KWAY")
    os.environ["QA_REPLAY_KWAY"] = "1" if kway else "0"
    try:
        assert lib.qa_debug_pack_slabs(*args, None, None) == 1
        slabs = np.zeros(nb.value, dtype=np.uint8)
        off = np.zeros(ns.value + 1, dtype=np.uint32)
        assert lib.qa_debug_pack_slabs(*args, _lib.ptr(slabs), _lib.ptr(off)) == 1
    finally:
        if old is None:
            os.environ.pop("QA_REPLAY_KWAY")
        else:
            os.environ["QA_REPLAY_KWAY"] = old
    blocks = []
    for b in range(ns.value):
        o = int(off[b]) * 16
        hdr = np.frombuffer(slabs, dtype=HDR, count=1, offset=o)[0]
        ent = np.frombuffer(slabs, dtype=ENT, count=int(hdr["nent"]), offset=o + HDR.itemsize)
        assert int(off[b + 1]) * 16 == o + HDR.itemsize + ENT.itemsize * int(hdr["nent"])
        blocks.append((hdr, ent))
    return rows, blocks, slabs


def conforming_cells(rows, n, K):
    """Specification of the detector: cell i conforms when every case has exactly the other K - 1 cases of its cell once
    each, and otherwise only same-case neighbours of distinct cells, the same cells with bitwise the same J in every case."""
    conf = []
    for i in range(n // K):
        lists, ok = [], True
        for p in range(K):
            v = i * K + p
            intra = [j for j, _ in rows[v] if i * K <= j < (i + 1) * K]
            inter = sorted((j // K, np.float64(J).tobytes()) for j, J in rows[v] if not i * K <= j < (i + 1) * K)
            same_case = all(j % K == p for j, _ in rows[v] if not i * K <= j < (i + 1) * K)
            ok = ok and sorted(intra) == [i * K + q for q in range(K) if q != p] and same_case
            ok = ok and len({c for c, _ in inter}) == len(inter)
            lists.append(inter)
        conf.append(ok and all(x == lists[0] for x in lists))
    return conf


def expected_section(rows, hdr, K):
    """(J, B) of the section: per cell, neighbour cells j > i ascending, then j < v0 / K ascending."""
    v0, nv = int(hdr["v0"]), int(hdr["nv"])
    words = list(hdr["bw"][: int(hdr["nbw"])])
    out = []
    for i in range(v0 // K, (v0 + nv) // K):
        nbrs = sorted((j // K, J) for j, J in rows[i * K] if not i * K <= j < (i + 1) * K)
        for c, J in [x for x in nbrs if x[0] > i] + [x for x in nbrs if x[0] * K < v0]:
            hw = (c * K) >> 4
            slot = 0 if hw == v0 >> 4 else words.index(hw) + 1
            out.append((J, (30 - 2 * ((c * K + K - 1) & 15)) | (slot << 7) | ((c * K) << 13)))
    return out


def check_sections(model, K):
    rows, blocks, _ = pack(model)
    n = model.num_variables
    conf = conforming_cells(rows, n, K)
    nk = 0
    for hdr, ent in blocks:
        v0, nv, kw = int(hdr["v0"]), int(hdr["nv"]), int(hdr["kway"])
        whole = v0 % K == 0 and nv % K == 0 and v0 + nv <= n and all(conf[c] for c in range(v0 // K, (v0 + nv) // K))
        if kw == 0:
            # generic: not whole conforming cells, or the section would not fit the stage
            assert not whole or int(hdr["nent"]) + len(expected_section(rows, hdr, K)) > RP_CAP
            continue
        nk += 1
        assert whole and kw >> 16 == K and int(hdr["nent"]) <= RP_CAP
        sec = ent[kw & 0xFFFF:]
        assert [(float(e["J"]), int(e["B"])) for e in sec] == expected_section(rows, hdr, K)
        assert all(int(e["zero"]) == 0 for e in sec)
        # the kernel takes a cell's neighbour count from the pre part of its last case
        for c in range(nv // K):
            i = v0 // K + c
            cells = [j // K for j, _ in rows[i * K] if not i * K <= j < (i + 1) * K]
            nn = sum(1 for j in cells if j > i or j * K < v0)
            assert int(hdr["rowb"][c * K + K - 1]) >> 16 == nn
    return nk, len(blocks), blocks


@pytest.fixture(scope="module")
def graph101():
    return snn.synthetic_snn(101, k=5, seed=11)[0]


@pytest.mark.parametrize("K", [2, 4, 8, 16])
def test_cqm_sections_match_the_specification(graph101, K):
    model = models.cqm_model(graph101, K, min_size=5)
    nk, nb, _ = check_sections(model, K)
    assert nk > 0


def test_flagship_shape_every_cell_block_is_kway():
    g = snn.synthetic_snn(2048, k=5, seed=0)[0]
    model = models.cqm_model(g, 8, min_size=20)
    nk, nb, blocks = check_sections(model, 8)
    cell_blocks = sum(1 for h, _ in blocks if int(h["v0"]) + int(h["nv"]) <= 2048 * 8)
    assert nk == cell_blocks


def test_forced_generic_packs_the_parent_format(graph101):
    model = models.cqm_model(graph101, 8, min_size=5)
    _, blocks, slabs = pack(model, kway=False)
    assert all(int(h["kway"]) == 0 for h, _ in blocks)
    _, blocks_kw, _ = pack(model)
    for (h0, e0), (h1, e1) in zip(blocks, blocks_kw):   # the generic entries are the same; the section only follows them
        k = int(h1["kway"]) & 0xFFFF or int(h1["nent"])
        assert int(h0["nent"]) == k and np.array_equal(e0, e1[:k])


def _cell_couplers(model, K, kind):
    st, en, w = model.starts.copy(), model.ends.copy(), model.weights.copy()
    inter = np.nonzero(st // K != en // K)[0]
    if kind == "missing":
        k = int(np.nonzero((st == 3 * K + 5) & (en == 3 * K + 1))[0][0])
        st, en, w = np.delete(st, k), np.delete(en, k), np.delete(w, k)
    elif kind == "weight":
        w[inter[0]] += 0.125
    elif kind == "duplicate":
        k = inter[3]
        st, en, w = np.append(st, st[k]), np.append(en, en[k]), np.append(w, 0.25)
    else:
        k = inter[5]
        b = int(en[k])
        st, en, w = np.append(st, st[k]), np.append(en, b - b % K + (b % K + 1) % K), np.append(w, -0.3)
    return models.LoweredModel(model.h, st.astype(np.int32), en.astype(np.int32), w, model.offset, model.labels, model.groups,
                               model.meta)


@pytest.mark.parametrize("kind", ["missing", "weight", "duplicate", "cross_case"])
def test_mutations_leave_their_cells_generic(graph101, kind):
    base = models.cqm_model(graph101, 8, min_size=5)
    nk0, _, _ = check_sections(base, 8)
    nk1, _, _ = check_sections(_cell_couplers(base, 8, kind), 8)
    assert 0 < nk1 < nk0
