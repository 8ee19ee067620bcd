"""Host-side argument handling of the sampler: beta schedule, default beta range, seeds, initial states.

Restates dwave-neal ``neal/sampler.py`` (``SimulatedAnnealingSampler.sample`` and
``_default_ising_beta_range``) and dimod ``core/initialized.py::parse_initial_states`` -- SURVEY.md
row a12, from the upstream description (parity unpinned; neither package is installable offline).
"""
from __future__ import annotations

import warnings
from typing import Optional, Sequence, Tuple

import numpy as np

BETA_SCHEDULE_OPTIONS = ("linear", "geometric", "custom")


def default_ising_beta_range(h: np.ndarray, irow: np.ndarray, icol: np.ndarray, qdata: np.ndarray,
                             groups=None) -> Tuple[float, float]:
    """neal ``_default_ising_beta_range``: hot = ln2 / max_v(|h_v| + sum_j |J_vj|), cold = ln100 / min nonzero |bias|.

    ``groups`` = (grp, coef, lam, kappa) adds the couplings a rank-1 term would contribute if it were
    materialised (J_ij += lam*a_i*a_j/2, h_i += lam*kappa*a_i/2), so both forms get the same range.  Interval groups
    (grp, coef, lam, kappa, lo, hi) get the range of their equality form: the same scale of flip costs.
    """
    h = np.asarray(h, dtype=np.float64)
    q = np.asarray(qdata, dtype=np.float64)
    abs_h = np.abs(h)
    field = abs_h.copy()
    if len(q):
        np.add.at(field, irow, np.abs(q))
        np.add.at(field, icol, np.abs(q))
    nz = [abs_h[abs_h != 0], np.abs(q[q != 0])]
    if groups is not None:
        grp, coef, lam, kappa = groups[:4]
        grp = np.asarray(grp)
        coef = np.abs(np.asarray(coef, dtype=np.float64))
        for g in range(len(lam)):
            sel = grp == g
            if not sel.any() or lam[g] == 0:
                continue
            a = coef[sel]
            tot = a.sum()
            field[sel] += abs(lam[g]) * a * (tot - a) / 2.0 + abs(lam[g] * kappa[g]) * a / 2.0
            amin = a[a != 0]
            if len(amin) > 1:
                two = np.sort(amin)[:2]
                nz.append(np.array([abs(lam[g]) * two[0] * two[1] / 2.0]))
            if kappa[g] != 0 and len(amin):
                nz.append(np.array([abs(lam[g] * kappa[g]) * amin.min() / 2.0]))
    nz = np.concatenate(nz) if nz else np.zeros(0)
    if len(nz) == 0:
        return 0.1, 1.0
    min_delta = float(nz.min())
    max_delta = float(field.max())
    if max_delta == 0:
        return 0.1, 1.0
    return float(np.log(2) / max_delta), float(np.log(100) / min_delta)


def default_ising_beta_range_samplers(h: np.ndarray, irow: np.ndarray, icol: np.ndarray, qdata: np.ndarray,
                                      max_single_qubit_excitation_rate: float = 0.01, scale_T_with_N: bool = True) -> Tuple[float, float]:
    """The default range of dwave-samplers >= 1.0 (the package behind ``neal`` from Ocean 6 on; SURVEY.md row a12, restated
    from the upstream description -- unpinned like the rest of the third-party behaviour):

        hot  = ln 2 / (2 * max_v (|h_v| + sum_j |J_vj|))           (1 when the model has no bias at all)
        cold = ln(N_min / rate) / (2 * f_min),   f_min = min_v (smallest non-zero |bias| touching v),
               N_min = number of variables attaining f_min (1 when ``scale_T_with_N`` is false), rate = 0.01

    ``default_ising_beta_range`` above is the dwave-neal 0.5.x rule, which the sampler uses unless a range is passed."""
    h = np.asarray(h, dtype=np.float64)
    q = np.asarray(qdata, dtype=np.float64)
    n = len(h)
    abs_h = np.abs(h)
    field = abs_h.copy()
    fmin = np.where(abs_h != 0, abs_h, np.inf)
    if len(q):
        aq = np.abs(q)
        np.add.at(field, irow, aq)
        np.add.at(field, icol, aq)
        nzq = aq != 0
        np.minimum.at(fmin, np.asarray(irow)[nzq], aq[nzq])
        np.minimum.at(fmin, np.asarray(icol)[nzq], aq[nzq])
    max_field = float(field.max()) if n else 0.0
    hot = 1.0 if max_field == 0 else float(np.log(2) / (2 * max_field))
    finite = fmin[np.isfinite(fmin)]
    if len(finite) == 0:
        return hot, hot
    f = float(finite.min())
    n_min = int(np.sum(finite == f)) if scale_T_with_N else 1
    return hot, float(np.log(n_min / max_single_qubit_excitation_rate) / (2 * f))


def make_beta_schedule(beta_range: Optional[Sequence[float]], num_sweeps: int, num_sweeps_per_beta: int,
                       beta_schedule_type: str, beta_schedule: Optional[Sequence[float]] = None) -> Tuple[np.ndarray, int]:
    """Returns (beta_schedule, num_sweeps_per_beta) with neal's validation rules."""
    if beta_schedule_type not in BETA_SCHEDULE_OPTIONS:
        raise ValueError(f"Beta schedule type {beta_schedule_type} not implemented")
    if not isinstance(num_sweeps_per_beta, (int, np.integer)) or num_sweeps_per_beta < 1:
        raise ValueError("'num_sweeps_per_beta' should be a positive integer")
    if beta_schedule_type == "custom":
        if beta_schedule is None:
            raise ValueError("'beta_schedule' must be provided for beta_schedule_type = 'custom'")
        sched = np.array(beta_schedule, dtype=np.float64)
        if num_sweeps is not None and num_sweeps != len(sched) * num_sweeps_per_beta:
            raise ValueError("'num_sweeps' should be set to None, or a value consistent with 'beta_schedule' and "
                             "'num_sweeps_per_beta' for 'beta_schedule_type' = 'custom'")
        if sched.size and sched.min() < 0:
            raise ValueError("'beta_schedule' cannot include negative values.")
        return sched, int(num_sweeps_per_beta)
    if beta_schedule is not None:
        raise ValueError("'beta_schedule' must be set to None for 'beta_schedule_type' not equal to 'custom'")
    if num_sweeps is None:
        num_sweeps = 1000
    if not isinstance(num_sweeps, (int, np.integer)) or num_sweeps < 0:
        raise ValueError("'num_sweeps' should be a non-negative integer")
    num_betas, rem = divmod(int(num_sweeps), int(num_sweeps_per_beta))
    if rem > 0 or num_betas < 0:
        raise ValueError("'num_sweeps' must be divisible by 'num_sweeps_per_beta'")
    if beta_range is None:
        raise ValueError("beta_range must be resolved before building the schedule")
    b0, b1 = float(beta_range[0]), float(beta_range[1])
    if b0 < 0 or b1 < 0:
        raise ValueError("beta range must be non-negative")
    if num_betas == 1:
        sched = np.array([b1], dtype=np.float64)  # neal: one beta -> the final (cold) value
    elif beta_schedule_type == "linear":
        sched = np.linspace(b0, b1, num=num_betas)
    else:
        if min(b0, b1) == 0:
            raise ValueError("'beta_range' must contain non-zero values for 'beta_schedule_type' = 'geometric'")
        sched = np.geomspace(b0, b1, num=num_betas)
    return np.asarray(sched, dtype=np.float64), int(num_sweeps_per_beta)


def resolve_seed(seed) -> int:
    """neal: ``seed`` None -> random 32-bit; otherwise an int in [0, 2^32 - 1]."""
    if seed is None:
        return int(np.random.randint(2 ** 32, dtype=np.uint32))
    if not isinstance(seed, (int, np.integer)):
        raise TypeError("'seed' should be None or a positive 32-bit integer")
    if not 0 <= int(seed) <= 2 ** 32 - 1:
        raise ValueError("'seed' should be an integer between 0 and 2^32 - 1 inclusive")
    return int(seed)


def per_read_seeds(seed: int, num_reads: int, first_read: int = 0) -> np.ndarray:
    """Deterministic 32-bit seed for every read (splitmix64 of ``seed`` and the global read index).

    Read r of a per-read run equals ``neal.sample(num_reads=1, seed=seeds[r], initial_states=init[r])``;
    the seeds depend only on (seed, r), so the result is the same for any sharding over GPUs.
    """
    r = np.arange(first_read, first_read + num_reads, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) + np.uint64(1)) * np.uint64(0xD1342543DE82EF95) + r * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z & np.uint64(0xFFFFFFFF)).astype(np.uint64)


def random_spin_states(num_reads: int, n: int, seed: int) -> np.ndarray:
    """dimod ``Initialized._random``-style +-1 states: RandomState(seed).choice([1, -1], (R, n)) as int8."""
    rs = np.random.RandomState(seed)
    values = np.asarray([1, -1], dtype=np.int8)  # list(dimod.SPIN.value) == [1, -1] in CPython
    if num_reads * n == 0:
        return np.empty((num_reads, n), dtype=np.int8)
    return values[rs.randint(0, 2, size=(num_reads, n))]


def counter_spin_states(num_reads: int, n: int, seed: int, first_read: int = 0) -> np.ndarray:
    """+-1 states from the library's counter-based generator (``qa_random_states``, csrc/postprocess.cu::k_random_states):
    spin (r, v) = bit (v & 63) of splitmix64-mix(seed, first_read + r, v >> 6), 1 -> -1.  A function of the GLOBAL read index:
    any sharding of the reads over GPUs draws the same states, and the device draws them without a host copy
    (``initial_states_generator='counter'``, an extension next to dimod's 'none' / 'tile' / 'random')."""
    if num_reads * n == 0:
        return np.empty((num_reads, n), dtype=np.int8)
    words = (n + 63) // 64
    r = np.arange(first_read, first_read + num_reads, dtype=np.uint64)[:, None]
    w = np.arange(words, dtype=np.uint64)[None, :]
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) + np.uint64(1)) * np.uint64(0xD1342543DE82EF95) + r * np.uint64(0x9E3779B97F4A7C15) \
            + w * np.uint64(0xC2B2AE3D27D4EB4F)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    bits = np.unpackbits(z.view(np.uint8).reshape(num_reads, words, 8), axis=2, bitorder="little").reshape(num_reads, words * 64)
    return np.ascontiguousarray(1 - 2 * bits[:, :n].astype(np.int8))


def parse_initial_states(n: int, labels: Sequence, vartype_is_spin: bool, initial_states, initial_states_generator: str,
                         num_reads: Optional[int], seed: int) -> np.ndarray:
    """dimod ``parse_initial_states`` for the three generators ('none', 'tile', 'random') plus the library's 'counter'
    generator (random states as a function of the global read index); returns int8 +-1 [R][n]."""
    if initial_states_generator not in ("none", "tile", "random", "counter"):
        raise ValueError("unknown value for 'initial_states_generator'")
    given = None
    if initial_states is not None:
        if hasattr(initial_states, "record") and hasattr(initial_states, "variables"):  # a SampleSet
            arr = np.asarray(initial_states.record.sample)
            lab = list(initial_states.variables)
            spin_in = getattr(initial_states.vartype, "name", str(initial_states.vartype)) == "SPIN"
        elif isinstance(initial_states, tuple) and len(initial_states) == 2:
            arr, lab = np.atleast_2d(np.asarray(initial_states[0])), list(initial_states[1])
            spin_in = bool((arr == -1).any()) or vartype_is_spin
        elif isinstance(initial_states, dict):
            lab = list(initial_states.keys())
            arr = np.array([[initial_states[v] for v in lab]])
            spin_in = bool((arr == -1).any()) or vartype_is_spin
        else:
            arr = np.atleast_2d(np.asarray(initial_states))
            lab = list(labels)
            spin_in = bool((arr == -1).any()) or vartype_is_spin
        if arr.shape[1] != n or set(lab) != set(labels):
            raise ValueError("mismatch between variables in 'initial_states' and 'bqm'")
        pos = {v: i for i, v in enumerate(lab)}
        arr = arr[:, [pos[v] for v in labels]]
        given = (arr if spin_in else 2 * arr - 1).astype(np.int8)
        if not np.isin(given, (-1, 1)).all():
            raise ValueError("initial states must be +-1 (SPIN) or 0/1 (BINARY)")
    if num_reads is None:
        num_reads = 1 if given is None else len(given)
    if not isinstance(num_reads, (int, np.integer)) or num_reads < 1:
        raise ValueError("'num_reads' should be a positive integer")
    num_reads = int(num_reads)
    if given is None:
        if initial_states_generator == "none":
            raise ValueError("no initial states provided and 'initial_states_generator' is 'none'")
        if initial_states_generator == "counter":
            return counter_spin_states(num_reads, n, seed)
        return np.ascontiguousarray(random_spin_states(num_reads, n, seed))
    if len(given) > num_reads:
        given = given[:num_reads]
    missing = num_reads - len(given)
    if missing == 0:
        return np.ascontiguousarray(given)
    if initial_states_generator == "none":
        raise ValueError("initial states fewer than 'num_reads' and 'initial_states_generator' is 'none'")
    if initial_states_generator == "tile":
        reps = -(-num_reads // len(given))
        return np.ascontiguousarray(np.tile(given, (reps, 1))[:num_reads])
    extra = random_spin_states(missing, n, seed)
    return np.ascontiguousarray(np.vstack([given, extra]))


def warn_unknown_kwargs(sampler_name: str, kwargs: dict):
    """neal ``remove_unknown_kwargs``: QPU-only arguments (label, chain_strength, ...) are dropped with a warning."""
    for kw in kwargs:
        warnings.warn(f"Ignoring unknown kwarg: {kw!r} ({sampler_name} is a simulated-annealing sampler)",
                      UserWarning, stacklevel=3)
