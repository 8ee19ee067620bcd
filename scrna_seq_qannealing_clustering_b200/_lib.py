"""ctypes binding of libqanneal.so (C ABI declared in include/qanneal.h).

The library is the product: there is NO CPU fallback.  Importing this module works without a GPU
(so symbols can be inspected), but creating a context on a machine without a CUDA device raises
``QAnnealError`` -- loudly, by design.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("QA_LIB_PATH", _HERE / "csrc" / "libqanneal.so"))   # QA_LIB_PATH: development builds

QA_OK = 0
QA_SEED_PER_READ = 0
QA_SEED_STREAM = 1
QA_MODE_REFERENCE = 0
QA_MODE_THROUGHPUT = 1
QA_KERNEL_AUTO = 0
QA_KERNEL_WARP_PER_READ = 1
QA_KERNEL_LOCKSTEP_PUSH = 2
QA_KERNEL_LOCKSTEP_PULL = 3
QA_KERNEL_REPLAY = 4
QA_KERNEL_DENSE = 5
QA_ORDER_SEQUENTIAL = 0
QA_ORDER_RANDOM = 1
QA_PROPOSAL_METROPOLIS = 0
QA_PROPOSAL_GIBBS = 1
QA_MAX_GROUPS = 64

ERROR_NAMES = {
    -1: "QA_ERR_ARG",
    -2: "QA_ERR_INDEX",
    -3: "QA_ERR_STATE",
    -4: "QA_ERR_CUDA",
    -5: "QA_ERR_LIMIT",
    -6: "QA_ERR_INTERRUPTED",
}


class QAnnealError(RuntimeError):
    def __init__(self, code: int, message: str):
        self.code = code
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {message}")


class QAStats(C.Structure):
    """Mirror of ``qa_stats`` (include/qanneal.h)."""

    _fields_ = [
        ("attempts", C.c_uint64),
        ("candidates", C.c_uint64),
        ("draws", C.c_uint64),
        ("accepted", C.c_uint64),
        ("nbr_updates", C.c_uint64),
        ("active_chunks", C.c_uint64),
        ("chunks", C.c_uint64),
        ("near_ties", C.c_uint64),
        ("ms_h2d", C.c_double),
        ("ms_build", C.c_double),
        ("ms_anneal", C.c_double),
        ("ms_energy", C.c_double),
        ("ms_d2h", C.c_double),
        ("anneal_launches", C.c_uint32),
        ("total_launches", C.c_uint32),
        ("ms_total", C.c_double),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


INTERRUPT_FN = C.CFUNCTYPE(C.c_int, C.c_void_p)

_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64

# name -> (restype, argtypes); kept in one table so tests can check it against include/qanneal.h
SIGNATURES = {
    "qa_last_error": (C.c_char_p, []),
    "qa_version": (C.c_int, []),
    "qa_device_count": (C.c_int, []),
    "qa_ctx_create": (C.c_int, [C.c_int, C.POINTER(_p)]),
    "qa_ctx_destroy": (C.c_int, [_p]),
    "qa_ctx_synchronize": (C.c_int, [_p]),
    "qa_ctx_set_kernel": (C.c_int, [_p, C.c_int]),
    "qa_ctx_resident_reads": (C.c_int, [_p]),
    "qa_ctx_last_kernel": (C.c_int, [_p]),
    "qa_model_from_ising": (C.c_int, [_p, _i32, _p, _i64, _p, _p, _p, C.POINTER(_p)]),
    "qa_model_set_groups": (C.c_int, [_p, _i32, _p, _p, _p, _p]),
    "qa_model_set_group_bounds": (C.c_int, [_p, _p, _p]),
    "qa_model_enable_dense": (C.c_int, [_p, _i32]),
    "qa_model_replay_kway": (_i64, [_p, _p]),
    "qa_model_num_variables": (C.c_int, [_p]),
    "qa_model_num_couplers": (_i64, [_p]),
    "qa_model_max_degree": (C.c_int, [_p]),
    "qa_model_get_ising": (C.c_int, [_p, _p, _p, _p, _p]),
    "qa_model_destroy": (C.c_int, [_p]),
    "qa_sa_sample_model": (C.c_int, [_p, _p, _i32, _p, _p, _i32, _p, _i32, _p, _i32, _i32, _p, _p, C.POINTER(QAStats)]),
    "qa_sa_sample_model_ex": (C.c_int, [_p, _p, _i32, _p, _p, _i32, _p, _i32, _p, _i32, _i32, _i32, _i32, _p, _p, C.POINTER(QAStats)]),
    "qa_sa_sample_ising": (C.c_int, [_p, _i32, _p, _i64, _p, _p, _p, _i32, _p, _p, _i32, _p, _i32, _p, _i32, _i32, _p, _p, C.POINTER(QAStats)]),
    "qa_sa_sample_ising_ex": (C.c_int, [_p, _i32, _p, _i64, _p, _p, _p, _i32, _p, _p, _i32, _p, _i32, _p, _i32, _i32, _i32, _i32, _p, _p,
                                        C.POINTER(QAStats)]),
    "qa_sa_sample_ising_batch": (C.c_int, [_p, _i32, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _i32, _p, _i32, _p, C.POINTER(QAStats)]),
    "qa_build_cut_balance": (C.c_int, [_p, _i32, _i64, _p, _p, _p, C.c_double, C.c_double, C.POINTER(_p), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "qa_build_cut_linear": (C.c_int, [_p, _i32, _i64, _p, _p, _p, C.c_double, C.c_double, C.POINTER(_p), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "qa_build_subsampling": (C.c_int, [_p, _i32, _i64, _p, _p, _p, C.c_double, C.c_double, C.POINTER(_p), C.POINTER(C.c_double)]),
    "qa_build_dqm_onehot": (C.c_int, [_p, _i32, _i64, _p, _p, _p, _i32, C.c_double, C.c_double, _i32, C.POINTER(_p), C.POINTER(C.c_double)]),
    "qa_build_cqm_penalty": (C.c_int, [_p, _i32, _i64, _p, _p, _p, _i32, _i32, C.c_double, C.c_double, C.POINTER(_p), C.POINTER(C.c_double)]),
    "qa_build_cqm_interval": (C.c_int, [_p, _i32, _i64, _p, _p, _p, _i32, _i32, C.c_double, C.c_double, C.POINTER(_p), C.POINTER(C.c_double)]),
    "qa_energy_argmin": (C.c_int, [_p, _p, _i32, _p, _p, C.POINTER(C.c_double), C.POINTER(_i64), C.POINTER(QAStats)]),
    "qa_aggregate_reads": (C.c_int, [_p, _i32, _i32, _p, C.POINTER(_i32), _p, _p]),
    "qa_dev_alloc": (C.c_int, [_p, _i64, C.POINTER(_p)]),
    "qa_dev_free": (C.c_int, [_p, _p]),
    "qa_dev_copy": (C.c_int, [_p, _p, _p, _i64]),
    "qa_random_states": (C.c_int, [_p, C.c_uint64, _i64, _i32, _i32, _p]),
    "qa_argmin": (C.c_int, [_p, _i64, _p, C.POINTER(C.c_double), C.POINTER(_i64)]),
    "qa_argmin_device": (C.c_int, [_p, _i64, _p, _i64, _p]),
    "qa_debug_pack_slabs": (C.c_int, [_i32, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p]),
    "qa_snn_build": (C.c_int, [_p, _i32, _p, _i32, _p, _i32, C.c_double, _i32, C.POINTER(_p)]),
    "qa_graph_num_edges": (_i64, [_p, _i32]),
    "qa_graph_num_nodes": (C.c_int, [_p, _i32]),
    "qa_graph_get_edges": (C.c_int, [_p, _i32, _p, _p, _p]),
    "qa_graph_device_edges": (C.c_int, [_p, _i32, C.POINTER(_p), C.POINTER(_p), C.POINTER(_p)]),
    "qa_graph_destroy": (C.c_int, [_p]),
    "qa_graph_split": (C.c_int, [_p, _i32, _i64, _p, _p, _p, _p, _i32, C.POINTER(_p)]),
    "qa_graph_get_nodes": (C.c_int, [_p, _i32, _p]),
    "qa_model_concat": (C.c_int, [_p, _i32, C.POINTER(_p), C.POINTER(_p)]),
    "qa_sa_sample_model_batch": (C.c_int, [_p, _p, _i32, _p, _p, _i32, _p, _i32, _i32, _p, C.POINTER(QAStats)]),
    "qa_sort_reads": (C.c_int, [_p, _i32, _p, _p]),
    "qa_gather_samples": (C.c_int, [_p, _i32, _i32, _p, _i32, _p, _p]),
    "qa_decode_onehot": (C.c_int, [_p, _i32, _i32, _i64, _i32, _p, _i32, _i32, _p, _p]),
}

_lib = None


def load() -> C.CDLL:
    """Load libqanneal.so (built in-tree by ``__graft_entry__.build()``); raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("QANNEAL_LIB", LIB_PATH))
    if not path.exists():
        raise QAnnealError(-4, f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().qa_last_error()
    return msg.decode() if msg else ""


def check(rc: int) -> int:
    if rc < 0:
        raise QAnnealError(rc, last_error())
    return rc


def ptr(x):
    """Raw address of a numpy array / torch tensor / int / None as a ``c_void_p``."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data_as(C.c_void_p)
    if isinstance(x, int):
        return C.c_void_p(x)
    if hasattr(x, "data_ptr"):  # torch.Tensor used purely as a buffer
        return C.c_void_p(x.data_ptr())
    raise TypeError(f"cannot take the address of {type(x)!r}")
