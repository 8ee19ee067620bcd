"""Thin object layer over the C ABI (include/qanneal.h): ``Context`` (one GPU) and ``IsingModel``.

Host buffers are numpy arrays; device buffers may be passed as torch CUDA tensors (used purely as
memory) -- the library detects device pointers itself.  Nothing here computes: every number comes
out of libqanneal.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from ._lib import QAStats, check, ptr


def _is_tensor(x) -> bool:
    return hasattr(x, "data_ptr") and not isinstance(x, np.ndarray)


def _as(x, dtype, name):
    """numpy view with the dtype/contiguity the ABI expects (torch tensors are passed through)."""
    if x is None or _is_tensor(x):
        return x
    a = np.ascontiguousarray(x, dtype=dtype)
    return a


def _check_states(states):
    """The library updates ``states`` in place through a raw pointer: a host array must already be C-contiguous int8 (a silent
    conversion would anneal a temporary copy, a wrong dtype would corrupt memory); a device tensor must be int8 and contiguous."""
    if _is_tensor(states):
        dt = str(getattr(states, "dtype", "int8"))
        if "int8" not in dt or "uint8" in dt:
            raise ValueError("states must be an int8 tensor")
        if hasattr(states, "is_contiguous") and not states.is_contiguous():
            raise ValueError("states must be contiguous")
    elif states.dtype != np.int8 or not states.flags.c_contiguous:
        raise ValueError("states must be a C-contiguous int8 array (it is updated in place)")


class DeviceBuffer:
    """A device allocation of the library (``qa_dev_alloc``) with a shape: lets the host layer keep a state matrix on the
    GPU from creation to the top-k export without depending on a tensor library.  Quacks like a tensor for ``_lib.ptr``."""

    def __init__(self, ctx: "Context", shape, dtype=np.int8):
        self.ctx = ctx
        self.shape = tuple(int(x) for x in shape)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = C.c_void_p()
        check(_lib.load().qa_dev_alloc(ctx._h, self.nbytes, C.byref(p)))
        self._p = p

    def data_ptr(self) -> int:
        return int(self._p.value or 0)

    def upload(self, host: np.ndarray):
        host = np.ascontiguousarray(host, dtype=self.dtype)
        if host.nbytes != self.nbytes:
            raise ValueError("size mismatch")
        check(_lib.load().qa_dev_copy(self.ctx._h, self._p, ptr(host), self.nbytes))
        return self

    def download(self) -> np.ndarray:
        out = np.empty(self.shape, dtype=self.dtype)
        check(_lib.load().qa_dev_copy(self.ctx._h, ptr(out), self._p, self.nbytes))
        return out

    def close(self):
        if getattr(self, "_p", None) is not None and self._p.value and getattr(self.ctx, "_h", None):
            _lib.load().qa_dev_free(self.ctx._h, self._p)
        self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One GPU + one CUDA stream + reusable scratch (``qa_ctx``)."""

    def __init__(self, device: int = 0):
        lib = _lib.load()
        h = C.c_void_p()
        check(lib.qa_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().qa_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_kernel(self, kernel: int):
        """Reference-mode kernel: _lib.QA_KERNEL_AUTO / QA_KERNEL_WARP_PER_READ / QA_KERNEL_LOCKSTEP_PUSH / QA_KERNEL_REPLAY."""
        check(_lib.load().qa_ctx_set_kernel(self._h, int(kernel)))

    @property
    def last_kernel(self) -> int:
        """QA_KERNEL_* the last sampling call actually ran on (after automatic selection / fall-back)."""
        return check(_lib.load().qa_ctx_last_kernel(self._h))

    @property
    def resident_reads(self) -> int:
        return check(_lib.load().qa_ctx_resident_reads(self._h))

    def synchronize(self):
        check(_lib.load().qa_ctx_synchronize(self._h))

    # -- SampleSet post-processing on the device (include/qanneal.h; reference consumption: BQM_clustering.py:93-146,
    #    plot_and_save.py:46-63, 105-126).  Arrays may be numpy (host) or torch CUDA tensors. ---
    def sort_reads(self, energies):
        """Read indices by ascending energy, ties in read order (what ``SampleSet.data(sorted_by='energy')`` iterates)."""
        num_reads = int(energies.shape[0])
        if not _is_tensor(energies):
            energies = np.ascontiguousarray(energies, dtype=np.float64)
        order = np.empty(num_reads, dtype=np.int32)
        check(_lib.load().qa_sort_reads(self._h, num_reads, ptr(energies), ptr(order)))
        return order

    def gather_samples(self, states, order):
        """``states[order]`` as a host array: only the selected rows leave the device."""
        num_reads, n = int(states.shape[0]), int(states.shape[1])
        if not _is_tensor(states):
            states = np.ascontiguousarray(states, dtype=np.int8)
        order = np.ascontiguousarray(order, dtype=np.int32)
        out = np.empty((len(order), n), dtype=np.int8)
        check(_lib.load().qa_gather_samples(self._h, n, num_reads, ptr(states), len(order), ptr(order), ptr(out)))
        return out

    def decode_onehot(self, states, cells: int, num_cases: int, on_value: int = 1, min_size: int = 0, want_labels: bool = True):
        """Labels of a DQM / CQM sample matrix: ``labels[read][cell]`` (-1: the cell is not one-hot) and per read the number of
        cells that are not one-hot and of cases with fewer than ``min_size`` cells (CQM_clustering.py:44-48).
        ``want_labels=False`` returns ``(None, violations)``: only the 8 bytes per read leave the device."""
        num_reads, stride = int(states.shape[0]), int(states.shape[1])
        if not _is_tensor(states):
            states = np.ascontiguousarray(states, dtype=np.int8)
        labels = np.empty((num_reads, cells), dtype=np.int32) if want_labels else None
        violations = np.empty((num_reads, 2), dtype=np.int32)
        check(_lib.load().qa_decode_onehot(self._h, int(cells), int(num_cases), stride, num_reads, ptr(states), int(on_value),
                                           int(min_size), ptr(labels), ptr(violations)))
        return labels, violations

    def random_states(self, seed: int, first_read: int, num_reads: int, n: int, out=None):
        """+-1 states of the counter-based generator (``schedule.counter_spin_states`` on the host), written to ``out`` (a
        ``DeviceBuffer`` / CUDA tensor / numpy array; default: a new ``DeviceBuffer``) without crossing PCIe."""
        if out is None:
            out = DeviceBuffer(self, (num_reads, n), np.int8)
        check(_lib.load().qa_random_states(self._h, int(seed), int(first_read), int(num_reads), int(n), ptr(out)))
        return out

    def aggregate_reads(self, states):
        """``SampleSet.aggregate()`` on the device: (first read index of every distinct sample in order of first occurrence,
        its number of occurrences)."""
        num_reads, n = int(states.shape[0]), int(states.shape[1])
        if not _is_tensor(states):
            states = np.ascontiguousarray(states, dtype=np.int8)
        first = np.empty(num_reads, dtype=np.int32)
        count = np.empty(num_reads, dtype=np.int32)
        nu = C.c_int32()
        check(_lib.load().qa_aggregate_reads(self._h, n, num_reads, ptr(states), C.byref(nu), ptr(first), ptr(count)))
        return first[: nu.value].copy(), count[: nu.value].copy()

    def argmin(self, values):
        """(lowest value, its first index) by the warp-shuffle reduction kernel; ``values`` numpy or a CUDA tensor (fp64)."""
        count = int(values.shape[0])
        if not _is_tensor(values):
            values = np.ascontiguousarray(values, dtype=np.float64)
        bv, bi = C.c_double(), C.c_int64()
        check(_lib.load().qa_argmin(self._h, count, ptr(values), C.byref(bv), C.byref(bi)))
        return float(bv.value), int(bi.value)

    def argmin_into(self, values, index_offset: int, out):
        """``argmin`` with the result left on the device: ``out`` (2 fp64, device) = (lowest value, index_offset + its first index) --
        the send buffer of the per-rank all_gather (SURVEY 8e)."""
        count = int(values.shape[0])
        if not _is_tensor(values):
            values = np.ascontiguousarray(values, dtype=np.float64)
        check(_lib.load().qa_argmin_device(self._h, count, ptr(values), int(index_offset), ptr(out)))

    # -- SNN graphs on the device (qa_snn_build): the step before the path ------------------------
    def build_snn(self, X, k: int = 5, prune: float = 1.0 / 15.0, max_degree: Optional[int] = 15, offsets=None) -> "DeviceGraph":
        """Seurat-style SNN graph(s) of the rows of ``X`` ([points][dim] fp64, host array or device tensor) built by the
        ``k_snn_*`` kernels (R/pbmc3k/Pbmc3k_general_data_preparation.Rmd:47-75): identical to ``snn.snn_graph``.  ``offsets``
        ([P + 1]) splits the rows into P independent point sets, each with its own graph (config 4)."""
        if not _is_tensor(X):
            X = np.ascontiguousarray(X, dtype=np.float64)
        total, dim = int(X.shape[0]), int(X.shape[1])
        off = np.array([0, total], dtype=np.int64) if offsets is None else np.ascontiguousarray(offsets, dtype=np.int64)
        if off[0] != 0 or off[-1] != total:
            raise ValueError("offsets must start at 0 and end at the number of points")
        hg = C.c_void_p()
        check(_lib.load().qa_snn_build(self._h, int(off.shape[0] - 1), ptr(off), dim, ptr(X), int(k), float(prune),
                                       int(max_degree) if max_degree else 0, C.byref(hg)))
        return DeviceGraph(self, hg, int(off.shape[0] - 1))

    # -- recursion driver on the device (csrc/recursion.cu) --------------------------------------
    def split_graph(self, graph, part, num_parts: int) -> "DeviceGraph":
        """``G.subgraph(part)`` for every part of a node partition at once (``qa_graph_split``): ``part[v]`` in [0, num_parts) or -1.
        ``graph`` is a host tuple ``(n, eu, ev, w)`` or ``DeviceGraph.device_graph(p)``."""
        n, m, eu, ev, w = self._graph_args(graph)
        part = np.ascontiguousarray(part, dtype=np.int32)
        if part.shape[0] != n:
            raise ValueError("part must have one entry per node")
        hg = C.c_void_p()
        check(_lib.load().qa_graph_split(self._h, n, m, ptr(eu), ptr(ev), ptr(w), ptr(part), int(num_parts), C.byref(hg)))
        return DeviceGraph(self, hg, int(num_parts))

    def concat_models(self, models) -> "IsingModel":
        """Single-problem resident models -> one batched model (``qa_model_concat``); the inputs stay valid."""
        arr = (C.c_void_p * len(models))(*[m._h for m in models])
        hm = C.c_void_p()
        check(_lib.load().qa_model_concat(self._h, len(models), arr, C.byref(hm)))
        out = IsingModel._from_handle(self, hm)
        out.sizes = [m.num_variables for m in models]
        return out

    def sample_model_batch(self, model: "IsingModel", reads_per_problem: int, states, beta_schedules, sweeps_per_beta: int, seeds,
                           energies=None):
        """Anneal every problem of a batched resident model in one launch.  ``beta_schedules``: [num_betas] shared, or
        [num_problems][num_betas] -- one schedule per problem."""
        beta_schedules = np.ascontiguousarray(beta_schedules, dtype=np.float64)
        per_problem = beta_schedules.ndim == 2
        num_betas = int(beta_schedules.shape[-1])
        seeds = _as(seeds, np.uint64, "seeds")
        P = len(model.sizes)
        if per_problem and beta_schedules.shape[0] != P:
            raise ValueError("one beta schedule per problem expected")
        _check_states(states)
        if energies is None:
            energies = np.empty(P * int(reads_per_problem), dtype=np.float64)
        st = QAStats()
        done = check(_lib.load().qa_sa_sample_model_batch(self._h, model._h, int(reads_per_problem), ptr(states), ptr(energies), num_betas,
                                                          ptr(beta_schedules), 1 if per_problem else 0, int(sweeps_per_beta), ptr(seeds),
                                                          C.byref(st)))
        return energies, st, done

    # -- model construction on the device (qa_build_*): graph = (n, eu, ev, w) in G.edges order ---
    def _graph_args(self, graph):
        if len(graph) == 5:                # raw device addresses (DeviceGraph.device_graph): (n, eu, ev, w, m)
            n, eu, ev, w, m = graph
            return int(n), int(m), int(eu), int(ev), int(w)
        n, eu, ev, w = graph
        if not _is_tensor(eu):
            eu = np.ascontiguousarray(eu, dtype=np.int32)
            ev = np.ascontiguousarray(ev, dtype=np.int32)
            w = np.ascontiguousarray(w, dtype=np.float64)
        return int(n), int(eu.shape[0]), eu, ev, w

    def build_cut_balance(self, graph, gamma_factor: float, k: float = 8.0):
        """``clustering_bqm`` model (BQM_clustering.py:29-47), balance term as a rank-1 group.  -> (IsingModel, offset, gamma)"""
        n, m, eu, ev, w = self._graph_args(graph)
        hm, off, gam = C.c_void_p(), C.c_double(), C.c_double()
        check(_lib.load().qa_build_cut_balance(self._h, n, m, ptr(eu), ptr(ev), ptr(w), float(gamma_factor), float(k), C.byref(hm),
                                               C.byref(off), C.byref(gam)))
        return IsingModel._from_handle(self, hm), float(off.value), float(gam.value)

    def build_cut_linear(self, graph, gamma_factor: float, k: float):
        """``clustering_bqm_2`` model (BQM_clustering.py:210-236): k * cut + gamma * sum x.  -> (IsingModel, offset, gamma)"""
        n, m, eu, ev, w = self._graph_args(graph)
        hm, off, gam = C.c_void_p(), C.c_double(), C.c_double()
        check(_lib.load().qa_build_cut_linear(self._h, n, m, ptr(eu), ptr(ev), ptr(w), float(gamma_factor), float(k), C.byref(hm),
                                              C.byref(off), C.byref(gam)))
        return IsingModel._from_handle(self, hm), float(off.value), float(gam.value)

    def build_subsampling(self, graph, gamma: float, P: float = 1.0):
        """``graph_subsampling`` model (QA_subsampling.py:26-35).  -> (IsingModel, offset)"""
        n, m, eu, ev, w = self._graph_args(graph)
        hm, off = C.c_void_p(), C.c_double()
        check(_lib.load().qa_build_subsampling(self._h, n, m, ptr(eu), ptr(ev), ptr(w), float(gamma), float(P), C.byref(hm),
                                               C.byref(off)))
        return IsingModel._from_handle(self, hm), float(off.value)

    def build_cqm_interval(self, graph, num_clusters: int, min_size: int, onehot_penalty: float, size_penalty: float):
        """``clustering_cqm`` model with the size constraints as interval groups, no slack variables
        (``qa_build_cqm_interval``: B * max(0, min_size - N_j)^2).  -> (IsingModel, offset)"""
        n, m, eu, ev, w = self._graph_args(graph)
        hm, off = C.c_void_p(), C.c_double()
        check(_lib.load().qa_build_cqm_interval(self._h, n, m, ptr(eu), ptr(ev), ptr(w), int(num_clusters), int(min_size),
                                                float(onehot_penalty), float(size_penalty), C.byref(hm), C.byref(off)))
        return IsingModel._from_handle(self, hm), float(off.value)

    def build_dqm_onehot(self, graph, num_cases: int, gamma: float, penalty: float, semantics: str = "as_written"):
        """``clustering_dqm`` model (DQM_clustering.py:29-43), one-hot expanded and structured.  -> (IsingModel, offset)"""
        n, m, eu, ev, w = self._graph_args(graph)
        hm, off = C.c_void_p(), C.c_double()
        check(_lib.load().qa_build_dqm_onehot(self._h, n, m, ptr(eu), ptr(ev), ptr(w), int(num_cases), float(gamma), float(penalty),
                                              1 if semantics == "intended" else 0, C.byref(hm), C.byref(off)))
        return IsingModel._from_handle(self, hm), float(off.value)

    def build_cqm_penalty(self, graph, num_clusters: int, min_size: int, onehot_penalty: float, size_penalty: float):
        """``clustering_cqm`` model (CQM_clustering.py:30-48) lowered to penalties.  -> (IsingModel, offset)"""
        n, m, eu, ev, w = self._graph_args(graph)
        hm, off = C.c_void_p(), C.c_double()
        check(_lib.load().qa_build_cqm_penalty(self._h, n, m, ptr(eu), ptr(ev), ptr(w), int(num_clusters), int(min_size),
                                               float(onehot_penalty), float(size_penalty), C.byref(hm), C.byref(off)))
        return IsingModel._from_handle(self, hm), float(off.value)

    # -- neal's general_simulated_annealing, one shot, host or device buffers --------------------
    def sample_ising(self, h, starts, ends, weights, states, beta_schedule, sweeps_per_beta, seeds,
                     seed_mode=_lib.QA_SEED_PER_READ, mode=_lib.QA_MODE_REFERENCE, energies=None, interrupt_function=None):
        h = _as(h, np.float64, "h")
        starts = _as(starts, np.int32, "starts")
        ends = _as(ends, np.int32, "ends")
        weights = _as(weights, np.float64, "weights")
        beta_schedule = _as(beta_schedule, np.float64, "beta_schedule")
        seeds = _as(seeds, np.uint64, "seeds")
        n = int(h.shape[0])
        m = int(starts.shape[0])
        _check_states(states)
        num_reads = int(states.shape[0]) if n else 0
        if energies is None:
            energies = np.empty(num_reads, dtype=np.float64)
        cb = None
        if interrupt_function is not None:
            cb = _lib.INTERRUPT_FN(lambda _u: 1 if interrupt_function() else 0)
        st = QAStats()
        done = check(_lib.load().qa_sa_sample_ising(
            self._h, n, ptr(h), m, ptr(starts), ptr(ends), ptr(weights), num_reads, ptr(states), ptr(energies),
            int(beta_schedule.shape[0]), ptr(beta_schedule), int(sweeps_per_beta), ptr(seeds), int(seed_mode), int(mode),
            C.cast(cb, C.c_void_p) if cb is not None else None, None, C.byref(st)))
        return energies, st, done

    def sample_ising_batch(self, var_offsets, coupler_offsets, h, starts, ends, weights, reads_per_problem, states,
                           beta_schedule, sweeps_per_beta, seeds, energies=None):
        var_offsets = np.ascontiguousarray(var_offsets, dtype=np.int64)
        coupler_offsets = np.ascontiguousarray(coupler_offsets, dtype=np.int64)
        h = _as(h, np.float64, "h")
        starts = _as(starts, np.int32, "starts")
        ends = _as(ends, np.int32, "ends")
        weights = _as(weights, np.float64, "weights")
        beta_schedule = _as(beta_schedule, np.float64, "beta_schedule")
        seeds = _as(seeds, np.uint64, "seeds")
        num_problems = int(var_offsets.shape[0]) - 1
        _check_states(states)
        if energies is None:
            energies = np.empty(num_problems * int(reads_per_problem), dtype=np.float64)
        st = QAStats()
        done = check(_lib.load().qa_sa_sample_ising_batch(
            self._h, num_problems, ptr(var_offsets), ptr(coupler_offsets), ptr(h), ptr(starts), ptr(ends), ptr(weights),
            int(reads_per_problem), ptr(states), ptr(energies), int(beta_schedule.shape[0]), ptr(beta_schedule),
            int(sweeps_per_beta), ptr(seeds), C.byref(st)))
        return energies, st, done


class DeviceGraph:
    """Edge lists that live on the GPU (``qa_graph``), one per point set; ``graph(p)`` copies one out as the host tuple
    ``(n, eu, ev, w)`` of snn.py, ``device_graph(p)`` names it by device addresses for ``Context.build_*``."""

    def __init__(self, ctx: Context, handle, num_problems: int):
        self.ctx = ctx
        self._h = handle
        self.num_problems = num_problems

    def num_nodes(self, problem: int = 0) -> int:
        return check(_lib.load().qa_graph_num_nodes(self._h, int(problem)))

    def num_edges(self, problem: int = -1) -> int:
        return int(check(_lib.load().qa_graph_num_edges(self._h, int(problem))))

    def graph(self, problem: int = 0):
        m = self.num_edges(problem)
        eu, ev, w = np.empty(m, dtype=np.int32), np.empty(m, dtype=np.int32), np.empty(m, dtype=np.float64)
        check(_lib.load().qa_graph_get_edges(self._h, int(problem), ptr(eu), ptr(ev), ptr(w)))
        return self.num_nodes(problem), eu.astype(np.int64), ev.astype(np.int64), w

    def nodes(self, problem: int = 0) -> np.ndarray:
        """Parent node index of every node of child ``problem`` (graphs made by ``Context.split_graph``)."""
        n = self.num_nodes(problem)
        out = np.empty(n, dtype=np.int32)
        check(_lib.load().qa_graph_get_nodes(self._h, int(problem), ptr(out)))
        return out

    def device_graph(self, problem: int = 0):
        eu, ev, w = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(_lib.load().qa_graph_device_edges(self._h, int(problem), C.byref(eu), C.byref(ev), C.byref(w)))
        return self.num_nodes(problem), int(eu.value or 0), int(ev.value or 0), int(w.value or 0), self.num_edges(problem)

    def close(self):
        # the native object points at its context: once that is gone (interpreter shutdown order) leak rather than touch it
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            _lib.load().qa_graph_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class IsingModel:
    """A model resident on the GPU (``qa_model``): CSR adjacency in neal's push_back order + h."""

    def __init__(self, ctx: Context, h, starts, ends, weights):
        self.ctx = ctx
        h = _as(h, np.float64, "h")
        starts = _as(starts, np.int32, "starts")
        ends = _as(ends, np.int32, "ends")
        weights = _as(weights, np.float64, "weights")
        hm = C.c_void_p()
        check(_lib.load().qa_model_from_ising(ctx._h, int(h.shape[0]), ptr(h), int(starts.shape[0]), ptr(starts), ptr(ends),
                                              ptr(weights), C.byref(hm)))
        self._h = hm
        self.num_variables = int(h.shape[0])
        self.num_couplers = int(starts.shape[0])
        self.num_groups = 0

    @classmethod
    def _from_handle(cls, ctx: Context, handle) -> "IsingModel":
        self = cls.__new__(cls)
        self.ctx = ctx
        self._h = handle
        lib = _lib.load()
        self.num_variables = check(lib.qa_model_num_variables(handle))
        self.num_couplers = int(lib.qa_model_num_couplers(handle))
        self.num_groups = 0
        return self

    def set_groups(self, grp, coef, lam, kappa, lo=None, hi=None):
        """Rank-1 groups (``qa_model_set_groups``); with ``lo`` / ``hi`` (int64 [G]) interval groups
        (``qa_model_set_group_bounds``): lam/4 * max(lo - u, 0, u - hi)^2 instead of lam/4 * u^2."""
        if (lo is None) != (hi is None):
            raise ValueError("give both lo and hi, or neither")
        grp = np.ascontiguousarray(grp, dtype=np.int32)
        coef = np.ascontiguousarray(coef, dtype=np.int32)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        kappa = np.ascontiguousarray(kappa, dtype=np.int64)
        if grp.shape[0] != self.num_variables or coef.shape[0] != self.num_variables:
            raise ValueError("grp/coef must have one entry per variable")
        check(_lib.load().qa_model_set_groups(self._h, int(lam.shape[0]), ptr(grp), ptr(coef), ptr(lam), ptr(kappa)))
        self.num_groups = int(lam.shape[0])
        if lo is not None:
            self.set_group_bounds(lo, hi)

    def set_group_bounds(self, lo, hi):
        """Interval bounds of the groups set last (``qa_model_set_group_bounds``); ``None, None``: equality groups again."""
        if lo is None and hi is None:
            check(_lib.load().qa_model_set_group_bounds(self._h, None, None))
            return
        lo = np.ascontiguousarray(lo, dtype=np.int64)
        hi = np.ascontiguousarray(hi, dtype=np.int64)
        if lo.shape != (self.num_groups,) or hi.shape != (self.num_groups,):
            raise ValueError("lo/hi must have one entry per group")
        check(_lib.load().qa_model_set_group_bounds(self._h, ptr(lo), ptr(hi)))

    def enable_dense(self, cases_per_cell: int = 1) -> bool:
        """Derive the dense k-way form (W, P) on the device; True when the model has it: ``mode=QA_MODE_THROUGHPUT`` then runs the
        fp64 tensor-core kernel (``qa_model_enable_dense``)."""
        return bool(check(_lib.load().qa_model_enable_dense(self._h, int(cases_per_cell))))

    @property
    def replay_kway(self):
        """(blocks with a k-way section, their K) of the replay kernel's slabs, (0, 0) before the first replay call."""
        k = C.c_int32(0)
        blocks = _lib.load().qa_model_replay_kway(self._h, C.byref(k))
        return int(check(blocks)), int(k.value)

    @property
    def max_degree(self) -> int:
        return check(_lib.load().qa_model_max_degree(self._h))

    def get_ising(self):
        h = np.empty(self.num_variables, dtype=np.float64)
        s = np.empty(self.num_couplers, dtype=np.int32)
        e = np.empty(self.num_couplers, dtype=np.int32)
        w = np.empty(self.num_couplers, dtype=np.float64)
        check(_lib.load().qa_model_get_ising(self._h, ptr(h), ptr(s), ptr(e), ptr(w)))
        return h, s, e, w

    def sample(self, states, beta_schedule, sweeps_per_beta, seeds, seed_mode=_lib.QA_SEED_PER_READ,
               mode=_lib.QA_MODE_REFERENCE, energies=None, interrupt_function=None, var_order=_lib.QA_ORDER_SEQUENTIAL,
               proposal=_lib.QA_PROPOSAL_METROPOLIS):
        """Anneal ``states`` ([R][n] int8 +-1, in/out).  Returns (energies, QAStats, reads_completed).  ``var_order`` /
        ``proposal``: dwave-samplers' random variable order and Gibbs acceptance (QA_ORDER_*, QA_PROPOSAL_*)."""
        beta_schedule = _as(beta_schedule, np.float64, "beta_schedule")
        seeds = _as(seeds, np.uint64, "seeds")
        num_reads = int(states.shape[0])
        _check_states(states)
        if energies is None:
            energies = np.empty(num_reads, dtype=np.float64)
        cb = None
        if interrupt_function is not None:
            cb = _lib.INTERRUPT_FN(lambda _u: 1 if interrupt_function() else 0)
        st = QAStats()
        done = check(_lib.load().qa_sa_sample_model_ex(
            self.ctx._h, self._h, num_reads, ptr(states), ptr(energies), int(beta_schedule.shape[0]), ptr(beta_schedule),
            int(sweeps_per_beta), ptr(seeds), int(seed_mode), int(mode), int(var_order), int(proposal),
            C.cast(cb, C.c_void_p) if cb is not None else None, None, C.byref(st)))
        return energies, st, done

    def energies(self, states, energies=None):
        """neal get_state_energy of each row + (best_energy, best_index) by the warp-shuffle argmin kernel."""
        num_reads = int(states.shape[0])
        if not _is_tensor(states):
            states = np.ascontiguousarray(states, dtype=np.int8)
        if energies is None:
            energies = np.empty(num_reads, dtype=np.float64)
        be = C.c_double()
        bi = C.c_int64()
        st = QAStats()
        check(_lib.load().qa_energy_argmin(self.ctx._h, self._h, num_reads, ptr(states), ptr(energies), C.byref(be),
                                           C.byref(bi), C.byref(st)))
        return energies, float(be.value), int(bi.value), st

    def close(self):
        # the native object points at its context: once that is gone (interpreter shutdown order) leak rather than touch it
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            _lib.load().qa_model_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
