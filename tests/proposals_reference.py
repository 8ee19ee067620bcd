"""ctypes wrapper of tests/native/proposals_sa_ref.cpp: the CPU annealing reference for dwave-samplers' sample options
(random variable order, Gibbs acceptance), equality and interval rank-1 groups, per-read and stream seeding.

TEST INFRASTRUCTURE.  The library is compiled on first use into the temporary directory (keyed by the source's hash), with
the oracle's flags (no FMA contraction, no fast math), so the repository tree is never written.  ``groups`` is the oracle's
4-tuple (grp, coef, lam, kappa) or a 6-tuple (grp, coef, lam, kappa, lo, hi) as ``models.Groups.astuple()`` returns it.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

SRC = Path(__file__).resolve().parent / "native" / "proposals_sa_ref.cpp"
SEQUENTIAL, RANDOM = 0, 1
METROPOLIS, GIBBS = 0, 1
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    digest = hashlib.sha1(SRC.read_bytes()).hexdigest()[:16]
    out = Path(tempfile.gettempdir()) / f"qa_proposals_ref_{os.getuid()}_{digest}.so"
    if not out.exists():
        cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else shutil.which("g++")
        tmp = out.with_suffix(f".{os.getpid()}.tmp")
        subprocess.run([cxx, "-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fopenmp", "-shared", "-o", str(tmp),
                        str(SRC)], check=True, capture_output=True)
        os.replace(tmp, out)
    lib = C.CDLL(str(out))
    p = C.c_void_p
    lib.pref_sample_ising.restype = C.c_int
    lib.pref_sample_ising.argtypes = [C.c_int32, p, C.c_int64, p, p, p, C.c_int32, p, p, C.c_int32, p, C.c_int32, p,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_int32, p, p, p, p, p, p, p]
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def sample_ising(h, starts, ends, weights, states, beta_schedule, sweeps_per_beta, seeds, seed_mode=0, groups=None,
                 var_order=SEQUENTIAL, proposal=METROPOLIS):
    """``states`` int8 [R][n] updated in place.  -> (energies, stats dict with the oracle's counter names)"""
    h = np.ascontiguousarray(h, dtype=np.float64)
    starts = np.ascontiguousarray(starts, dtype=np.int32)
    ends = np.ascontiguousarray(ends, dtype=np.int32)
    weights = np.ascontiguousarray(weights, dtype=np.float64)
    betas = np.ascontiguousarray(beta_schedule, dtype=np.float64)
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
    if states.dtype != np.int8 or not states.flags.c_contiguous:
        raise ValueError("states must be C-contiguous int8")
    R, n = states.shape
    e = np.empty(R, dtype=np.float64)
    st = np.zeros(5, dtype=np.uint64)
    if groups is None:
        g = (0, None, None, None, None, None, None)
    else:
        cv = lambda a, t: None if a is None else np.ascontiguousarray(a, dtype=t)
        lo, hi = (groups[4], groups[5]) if len(groups) == 6 else (None, None)
        g = (len(groups[2]), cv(groups[0], np.int32), cv(groups[1], np.int32), cv(groups[2], np.float64),
             cv(groups[3], np.int64), cv(lo, np.int64), cv(hi, np.int64))
    rc = load().pref_sample_ising(n, _ptr(h), len(starts), _ptr(starts), _ptr(ends), _ptr(weights), R, _ptr(states), _ptr(e),
                                  len(betas), _ptr(betas), int(sweeps_per_beta), _ptr(seeds), int(seed_mode), int(var_order),
                                  int(proposal), g[0], *map(_ptr, g[1:]), _ptr(st))
    if rc < 0:
        raise RuntimeError(f"proposals reference error {rc}")
    return e, dict(zip(("attempts", "candidates", "draws", "accepted", "nbr_updates"), map(int, st)))
