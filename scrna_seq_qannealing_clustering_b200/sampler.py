"""``B200SimulatedAnnealingSampler``: dimod ``Sampler`` surface over libqanneal.so.

Drop-in for the sampler objects the reference constructs (``LeapHybridSampler``, ``EmbeddingComposite(DWaveSampler())``,
``LeapHybridDQMSampler``, ``LeapHybridCQMSampler``, ``hybrid.KerberosSampler``; BQM_clustering.py:56-85,386;
DQM_clustering.py:45; CQM_clustering.py:52-53,88-89; QA_subsampling.py:40-65) with the argument semantics of
dwave-neal's ``SimulatedAnnealingSampler.sample`` (SURVEY.md row a12):

    sample(bqm, beta_range=None, num_reads=None, num_sweeps=None, num_sweeps_per_beta=1,
           beta_schedule_type='geometric', seed=None, interrupt_function=None, beta_schedule=None,
           initial_states=None, initial_states_generator='random', **kwargs) -> SampleSet

and dwave-samplers >= 1.0's two further options, with its names and defaults: ``randomize_order=False`` and
``proposal_acceptance_criteria='Metropolis'`` (or ``'Gibbs'``).

All annealing, energy evaluation and argmin run in the CUDA library; this file only parses arguments,
lowers models to vectors and wraps results.  There is no CPU path: without the library or a GPU it raises.
"""
from __future__ import annotations

import time
import warnings
from typing import Mapping, Optional

import numpy as np

from . import _lib, schedule
from .bqm import BINARY, SPIN, BinaryQuadraticModel, as_vartype
from .engine import Context, DeviceBuffer, IsingModel
from .models import LoweredModel, decode_onehot, lowered_from_bqm
from .sampleset import SampleSet

_KNOWN_QPU_KWARGS = ("label", "chain_strength", "return_embedding", "time_limit", "max_iter", "qpu_reads", "tabu_timeout",
                     "qpu_params", "annealing_time", "answer_mode")


class DeviceModel:
    """A model that was BUILT ON THE DEVICE by one of the ``qa_build_*`` entry points (``Context.build_*``): the sampler anneals
    it in place -- the O(n + m) vectors never exist on the host unless a default beta range has to be derived from them."""

    def __init__(self, gm: IsingModel, labels, offset: float, meta: Optional[dict] = None):
        self.gm = gm
        self.labels = list(labels)
        self.offset = float(offset)
        self.meta = dict(meta or {})
        self.groups = None            # already resident (qa_build_* set them)
        self._vec = None

    @property
    def num_variables(self) -> int:
        return self.gm.num_variables

    def vectors(self):
        if self._vec is None:
            self._vec = self.gm.get_ising()
        return self._vec

    def close(self):
        self.gm.close()


class B200SimulatedAnnealingSampler:
    """Simulated annealing on one B200 (reads shard over ranks when torch.distributed is initialised)."""

    parameters = None
    properties = None

    def __init__(self, device: Optional[int] = None, context: Optional[Context] = None):
        self.parameters = {
            "beta_range": [], "num_reads": [], "num_sweeps": [], "num_sweeps_per_beta": [],
            "beta_schedule_type": ["beta_schedule_options"], "seed": [], "interrupt_function": [], "beta_schedule": [],
            "initial_states": [], "initial_states_generator": [],
            # dwave-samplers >= 1.0
            "randomize_order": [], "proposal_acceptance_criteria": [],
            # extensions
            "mode": [], "seed_mode": [], "sorted": [], "aggregate": [], "return_samples": [], "num_best": [],
        }
        self.properties = {"beta_schedule_options": schedule.BETA_SCHEDULE_OPTIONS}
        self._ctx = context
        self._device = device
        self.last_stats: Optional[dict] = None

    # ---- plumbing -------------------------------------------------------------------------------
    @property
    def context(self) -> Context:
        if self._ctx is None:
            dev = self._device
            if dev is None:
                import os
                dev = int(os.environ.get("LOCAL_RANK", "0"))
                if dev >= max(_lib.load().qa_device_count(), 1):
                    dev = 0
            self._ctx = Context(dev)
        return self._ctx

    def close(self):
        if self._ctx is not None:
            self._ctx.close()
            self._ctx = None

    # ---- dimod Sampler API ----------------------------------------------------------------------
    def sample(self, bqm, beta_range=None, num_reads=None, num_sweeps=None, num_sweeps_per_beta=1,
               beta_schedule_type="geometric", seed=None, interrupt_function=None, beta_schedule=None,
               initial_states=None, initial_states_generator="random", mode="reference", seed_mode="per_read",
               sorted=False, aggregate=False, return_samples="all", num_best=16, randomize_order=False,
               proposal_acceptance_criteria="Metropolis", **kwargs) -> SampleSet:
        """Anneal a ``BinaryQuadraticModel`` (ours or dimod's), a ``LoweredModel`` or a ``DeviceModel``.

        Extensions to neal's signature: ``sorted`` / ``aggregate`` (QPU-like energy-sorted, duplicate-merged record);
        ``return_samples='best_k'`` with ``num_best=k``: the state matrix lives on the device from creation to ranking and only
        the k lowest-energy samples plus all R energies (``info['energies']``) come back -- with
        ``initial_states_generator='counter'`` nothing of size R x n ever crosses PCIe (SURVEY.md hard part 7).

        dwave-samplers' options: ``randomize_order=True`` visits a random variable at each of the n attempts of a sweep
        (runs on the warp-per-read kernel); ``proposal_acceptance_criteria='Gibbs'`` accepts a flip with probability
        1 / (1 + exp(beta dE)) instead of Metropolis' min(1, exp(-beta dE)).  Both are bit-exact against the CPU oracle."""
        if proposal_acceptance_criteria not in ("Metropolis", "Gibbs"):
            raise ValueError("proposal_acceptance_criteria must be 'Metropolis' or 'Gibbs'")
        self._options = (bool(randomize_order), proposal_acceptance_criteria)
        schedule.warn_unknown_kwargs(type(self).__name__, kwargs)
        t0 = time.perf_counter_ns()
        if return_samples not in ("all", "best_k"):
            raise ValueError("return_samples must be 'all' or 'best_k'")
        self._return = (return_samples, int(num_best))
        if isinstance(bqm, (LoweredModel, DeviceModel)):
            model, vartype = bqm, BINARY
        else:
            if not isinstance(bqm, BinaryQuadraticModel):
                bqm = _coerce_bqm(bqm)
            model, vartype = lowered_from_bqm(bqm), bqm.vartype
        return self._run(model, vartype, t0, beta_range, num_reads, num_sweeps, num_sweeps_per_beta, beta_schedule_type, seed,
                         interrupt_function, beta_schedule, initial_states, initial_states_generator, mode, seed_mode,
                         sorted, aggregate)

    def sample_qubo(self, Q: Mapping, **parameters) -> SampleSet:
        """dimod ``Sampler.sample_qubo``: ``BQM.from_qubo(Q)`` then ``sample``."""
        return self.sample(BinaryQuadraticModel.from_qubo(Q), **parameters)

    def sample_ising(self, h, J, **parameters) -> SampleSet:
        return self.sample(BinaryQuadraticModel.from_ising(h, J), **parameters)

    def sample_dqm(self, dqm, penalty: Optional[float] = None, **parameters) -> SampleSet:
        """``LeapHybridDQMSampler().sample_dqm`` stand-in (DQM_clustering.py:45): one-hot expansion + anneal.

        Returns one row per read with a case index per discrete variable; ``energy`` is the DQM energy of the
        decoded assignment and the extra record field ``is_feasible`` says whether every cell was one-hot.
        """
        from .dqm import DiscreteQuadraticModel
        if isinstance(dqm, (LoweredModel, DeviceModel)):
            model = dqm
        elif isinstance(dqm, DiscreteQuadraticModel):
            model = dqm.to_lowered(penalty)
        else:
            raise TypeError("sample_dqm expects a DiscreteQuadraticModel or a LoweredModel built by models.dqm_model")
        ss = self.sample(model, **parameters)
        return _decode_discrete(ss, model, dqm if isinstance(dqm, DiscreteQuadraticModel) else None)

    def sample_cqm(self, cqm, onehot_penalty: Optional[float] = None, constraint_penalty: Optional[float] = None,
                   slack_init: str = "consistent", size_lowering: str = "slack", **parameters) -> SampleSet:
        """``LeapHybridCQMSampler().sample_cqm`` stand-in (CQM_clustering.py:53,89): constraints lowered to penalties.

        Rows keep the binary variables ('v_{i},{k}' and slack bits); record fields ``is_feasible`` (one-hot and
        minimum-size constraints satisfied by the cell variables) and ``objective`` are added.
        ``slack_init='consistent'`` (default): generated initial states get slack bits that encode their own cluster sizes, so
        the size penalty starts at zero (``models.consistent_slack``); ``'random'``: dimod's uniformly random states.
        ``size_lowering`` ('slack' or 'interval') lowers a ConstrainedQuadraticModel's linear constraints
        (``ConstrainedQuadraticModel.to_lowered(lowering=)``); an already lowered model keeps its own lowering (models built
        with ``size_lowering='interval'`` have no slack bits, and ``slack_init`` does not apply to them).
        """
        from .cqm import ConstrainedQuadraticModel
        if isinstance(cqm, (LoweredModel, DeviceModel)):
            model = cqm
        elif isinstance(cqm, ConstrainedQuadraticModel):
            model = cqm.to_lowered(onehot_penalty, constraint_penalty, lowering=size_lowering)
        else:
            raise TypeError("sample_cqm expects a ConstrainedQuadraticModel or a LoweredModel built by models.cqm_model")
        meta = getattr(model, "meta", {})
        if (slack_init == "consistent" and parameters.get("initial_states") is None and "slack_coefficients" in meta
                and parameters.get("initial_states_generator", "random") == "random"):
            # generated initial states: random cell bits, slack bits encoding max(N_j - min_size, 0) (models.consistent_slack)
            from .models import consistent_slack
            seed = schedule.resolve_seed(parameters.get("seed"))
            parameters["seed"] = seed
            init = schedule.random_spin_states(int(parameters.get("num_reads") or 1), model.num_variables, seed)
            parameters["initial_states"] = ((consistent_slack(init, meta) + 1) // 2, model.labels)
            parameters["num_reads"] = None
        ss = self.sample(model, **parameters)
        ss.info["slack_init"] = slack_init
        return _annotate_cqm(ss, model)

    def build_on_device(self, kind: str, G, **params) -> DeviceModel:
        """The reference's model ``kind`` ('cut_balance' BQM_clustering.py:29-47, 'cut_linear' BQM_clustering.py:210-236,
        'subsampling' QA_subsampling.py:26-35, 'dqm' DQM_clustering.py:29-43, 'cqm' CQM_clustering.py:30-48) built by the ``qa_build_*`` kernels from the edge list: the
        all-pairs / one-hot / slack terms never exist as host arrays.  The caller closes the returned model."""
        from . import models
        spec = models.device_spec(kind, G, **params)
        ctx = self.context
        if kind == "cut_balance":
            gm, off, gamma = ctx.build_cut_balance(spec["graph"], params["gamma_factor"], params.get("k", 8.0))
            spec["meta"]["gamma"] = gamma
        elif kind == "cut_linear":
            gm, off, gamma = ctx.build_cut_linear(spec["graph"], params["gamma_factor"], params.get("k", 1.0))
            spec["meta"]["gamma"] = gamma
        elif kind == "subsampling":
            gm, off = ctx.build_subsampling(spec["graph"], params["gamma"], params.get("P", 1.0))
        elif kind == "dqm":
            gm, off = ctx.build_dqm_onehot(spec["graph"], params["num_of_clusters"], params["gamma"], spec["penalty"],
                                           params.get("semantics", "as_written"))
        elif spec["size_lowering"] == "interval":
            gm, off = ctx.build_cqm_interval(spec["graph"], params["num_of_clusters"], spec["min_size"], spec["onehot_penalty"],
                                             spec["size_penalty"])
        else:
            gm, off = ctx.build_cqm_penalty(spec["graph"], params["num_of_clusters"], spec["min_size"], spec["onehot_penalty"],
                                            spec["size_penalty"])
        return DeviceModel(gm, spec["labels"], off, spec["meta"])

    # ---- core -----------------------------------------------------------------------------------
    def _run(self, model, vartype, t0, beta_range, num_reads, num_sweeps, num_sweeps_per_beta,
             beta_schedule_type, seed, interrupt_function, beta_schedule, initial_states, initial_states_generator, mode,
             seed_mode, sort_result, aggregate) -> SampleSet:
        if mode not in ("reference", "throughput"):
            raise ValueError("mode must be 'reference' (bit-exact neal order) or 'throughput' (fields recomputed from spins)")
        if seed_mode not in ("per_read", "stream"):
            raise ValueError("seed_mode must be 'per_read' or 'stream'")
        if interrupt_function is not None and not callable(interrupt_function):
            raise TypeError("'interrupt_function' should be a callable")
        return_samples, num_best = getattr(self, "_return", ("all", 16))
        randomize_order, criteria = getattr(self, "_options", (False, "Metropolis"))
        rank, world = _dist_rank_world()
        seed = schedule.resolve_seed(seed)
        if world > 1:
            seed = _broadcast_int(seed)       # seed=None draws a random seed: every rank must anneal with rank 0's
        n = model.num_variables
        labels = model.labels
        vartype = as_vartype(vartype)
        info = {"beta_schedule_type": beta_schedule_type}
        if n == 0:
            ss = SampleSet.from_samples((np.empty((0, 0), dtype=np.int8), []), energy=[], vartype=vartype, info=info)
            return ss
        on_device = isinstance(model, DeviceModel)
        groups = model.groups.astuple() if model.groups is not None else None
        if beta_schedule_type != "custom":
            if beta_range is None:
                h, st_, en_, w_ = model.vectors() if on_device else (model.h, model.starts, model.ends, model.weights)
                beta_range = schedule.default_ising_beta_range(h, st_, en_, w_, groups)
            elif len(beta_range) != 2 or min(beta_range) < 0:
                raise ValueError("'beta_range' should be a 2-tuple of positive numbers")
            info["beta_range"] = [float(beta_range[0]), float(beta_range[1])]
        betas, spb = schedule.make_beta_schedule(beta_range, num_sweeps, num_sweeps_per_beta, beta_schedule_type, beta_schedule)

        # initial states: on the host (dimod's generators), or -- 'counter' generator with nothing given -- described only
        device_states = return_samples == "best_k"
        draw_on_device = device_states and initial_states is None and initial_states_generator == "counter"
        if draw_on_device:
            if num_reads is None:
                num_reads = 1
            if not isinstance(num_reads, (int, np.integer)) or num_reads < 1:
                raise ValueError("'num_reads' should be a positive integer")
            num_reads = int(num_reads)
            states = None
        else:
            states = schedule.parse_initial_states(n, labels, vartype is SPIN, initial_states, initial_states_generator,
                                                   num_reads, seed)
            num_reads = states.shape[0]

        # read sharding over ranks (one process per GPU); seeds depend on the global read index only
        lo, hi = _shard(num_reads, rank, world)
        if seed_mode == "stream":
            if world > 1:
                raise ValueError("seed_mode='stream' is one serial RNG chain and cannot shard over GPUs")
            seeds = np.array([seed], dtype=np.uint64)
        else:
            seeds = schedule.per_read_seeds(seed, hi - lo, first_read=lo)

        ctx = self.context
        gm = model.gm if on_device else IsingModel(ctx, model.h, model.starts, model.ends, model.weights)
        dev_buf = None
        try:
            if groups is not None:
                gm.set_groups(*groups)
            elif mode == "throughput":
                _try_dense(gm, model)
            if device_states:
                if draw_on_device:
                    dev_buf = ctx.random_states(seed, lo, hi - lo, n)
                else:
                    dev_buf = DeviceBuffer(ctx, (hi - lo, n), np.int8).upload(states[lo:hi])
                local_states = dev_buf
            else:
                local_states = np.ascontiguousarray(states[lo:hi])
            t1 = time.perf_counter_ns()
            energies, st, done = gm.sample(local_states, betas, spb, seeds,
                                           seed_mode=_lib.QA_SEED_STREAM if seed_mode == "stream" else _lib.QA_SEED_PER_READ,
                                           mode=_lib.QA_MODE_THROUGHPUT if mode == "throughput" else _lib.QA_MODE_REFERENCE,
                                           interrupt_function=interrupt_function,
                                           var_order=_lib.QA_ORDER_RANDOM if randomize_order else _lib.QA_ORDER_SEQUENTIAL,
                                           proposal=_lib.QA_PROPOSAL_GIBBS if criteria == "Gibbs" else _lib.QA_PROPOSAL_METROPOLIS)
            kernel = ctx.last_kernel
            t2 = time.perf_counter_ns()
            self.last_stats = st.as_dict()
            energies = energies[:done]
            extra = {}
            if device_states:
                # rank on the device, export k rows: (all energies, k best samples, their global read indices, occurrences)
                energies_all, samples, index, occ = self._best_k(ctx, dev_buf, energies, done, lo, num_best, aggregate, world)
                info["energies"] = energies_all + model.offset
                info["best_read_index"] = index
                energies = energies_all[index] if len(index) else energies_all[:0]
                local_states = samples
                extra["num_occurrences"] = occ
                aggregate = False               # done on the device
                sort_result = False             # already in ascending energy order
            else:
                local_states = local_states[:done]
                if world > 1:
                    local_states, energies = _gather_reads(local_states, energies, world)
        finally:
            if dev_buf is not None:
                dev_buf.close()
            if not on_device:
                gm.close()
        energies = energies + model.offset
        samples = local_states if vartype is SPIN else ((local_states + 1) // 2).astype(np.int8)
        info["timing"] = {"preprocessing_ns": t1 - t0, "sampling_ns": t2 - t1, "postprocessing_ns": 0}
        info["b200"] = {"mode": mode, "seed_mode": seed_mode, "world_size": world, "return_samples": return_samples,
                        "randomize_order": randomize_order, "proposal_acceptance_criteria": criteria, "kernel": kernel,
                        **{k: self.last_stats[k] for k in
                           ("attempts", "accepted", "draws", "candidates", "nbr_updates", "near_ties", "ms_anneal")}}
        ss = SampleSet.from_samples((samples, labels), energy=energies, vartype=vartype, info=info, **extra)
        if aggregate:
            ss = ss.aggregate()
        if sort_result:
            ss = ss.sorted()
        ss.info["timing"]["postprocessing_ns"] = time.perf_counter_ns() - t2
        return ss

    @staticmethod
    def _best_k(ctx, dev_buf, energies, done, lo, k, aggregate, world):
        """Device-side post-processing of one rank's reads (qa_aggregate_reads / qa_sort_reads / qa_gather_samples), then the
        SURVEY 8(e) exchange: per-rank candidates (k energies, k rows) and the energy vectors -- never the state matrices."""
        n = dev_buf.shape[1]
        view = _Rows(dev_buf, done)
        if aggregate and done:
            first, count = ctx.aggregate_reads(view)
        else:
            first, count = np.arange(done, dtype=np.int32), np.ones(done, dtype=np.int32)
        if done:
            order = ctx.sort_reads(energies)                      # stable: ties keep read order
            rank_of = np.empty(done, dtype=np.int64)
            rank_of[order] = np.arange(done)
            cand = first[np.argsort(rank_of[first], kind="stable")][:k]      # distinct samples by ascending energy
            occ = count[np.argsort(rank_of[first], kind="stable")][:k]
            rows = ctx.gather_samples(view, cand.astype(np.int32)) if len(cand) else np.empty((0, n), dtype=np.int8)
        else:
            cand, occ, rows = np.empty(0, dtype=np.int32), np.empty(0, dtype=np.int32), np.empty((0, n), dtype=np.int8)
        cand_e = energies[cand] if len(cand) else np.empty(0)
        if world == 1:
            return energies, rows, cand.astype(np.int64), occ.astype(np.int64)
        return _gather_best(energies, rows, cand.astype(np.int64) + lo, cand_e, occ.astype(np.int64), k, world, aggregate)


def _try_dense(gm: IsingModel, model) -> bool:
    """``mode='throughput'`` on a dense model (BASELINE config 5; materialised all-pairs models): ask the library for the dense
    k-way form -- it verifies the structure on the device -- so that the fp64 tensor-core kernel runs.  Sparse models are left
    alone: their exact replay kernel is faster than any recompute."""
    K = int(model.meta.get("num_cases", 1)) if isinstance(getattr(model, "meta", None), dict) else 1
    n = gm.num_variables
    if K not in (1, 2, 4, 8) or n % K:
        K = 1
    cells = n // K
    if cells < 64 or gm.num_couplers < 0.25 * K * cells * (cells - 1) / 2:
        return False
    return gm.enable_dense(K)


class _Rows:
    """The first ``rows`` rows of a device state matrix (what an interrupted run completed)."""

    def __init__(self, buf, rows):
        self._buf = buf
        self.shape = (int(rows), buf.shape[1])

    def data_ptr(self):
        return self._buf.data_ptr()


# ------------------------------------------------------------------------------------------------
def _coerce_bqm(obj) -> BinaryQuadraticModel:
    """Accept a real dimod BQM (anything with to_numpy_vectors / vartype / variables)."""
    if hasattr(obj, "to_numpy_vectors") and hasattr(obj, "vartype"):
        labels = list(obj.variables)
        vec = obj.to_numpy_vectors(variable_order=labels)
        ldata, (irow, icol, qdata), offset = vec[0], vec[1], vec[2]
        return BinaryQuadraticModel.from_numpy_vectors(ldata, (irow, icol, qdata), offset, as_vartype(obj.vartype), labels)
    raise TypeError(f"cannot sample an object of type {type(obj)!r}")


def _dist_rank_world():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except Exception:
        pass
    return 0, 1


def _shard(num_reads: int, rank: int, world: int):
    """Contiguous block of reads for ``rank`` (first ``num_reads % world`` ranks take one more)."""
    base, rem = divmod(num_reads, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _dist_device():
    import torch
    import torch.distributed as dist
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")


def _broadcast_int(value: int) -> int:
    import torch
    import torch.distributed as dist
    t = torch.tensor([int(value)], dtype=torch.int64, device=_dist_device())
    dist.broadcast(t, 0)
    return int(t.item())


def _all_gather_var(arr: np.ndarray, world: int):
    """all_gather of per-rank arrays whose first dimension differs (an interrupted rank completed fewer reads): the lengths are
    exchanged first, the payload is padded to the longest -- no row that was never annealed is ever returned."""
    import torch
    import torch.distributed as dist
    dev = _dist_device()
    cnt = torch.tensor([arr.shape[0]], dtype=torch.int64, device=dev)
    cnts = [torch.zeros_like(cnt) for _ in range(world)]
    dist.all_gather(cnts, cnt)
    lens = [int(c.item()) for c in cnts]
    per = max(max(lens), 1)
    pad = torch.zeros((per,) + tuple(arr.shape[1:]), dtype=torch.from_numpy(arr[:0]).dtype, device=dev)
    if arr.shape[0]:
        pad[: arr.shape[0]] = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
    out = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(out, pad)
    return [o[:ln].cpu().numpy() for o, ln in zip(out, lens)]


def _gather_reads(states: np.ndarray, energies: np.ndarray, world: int):
    """``return_samples='all'``: every rank ends with every completed read, in global read order."""
    return np.concatenate(_all_gather_var(states, world)), np.concatenate(_all_gather_var(energies, world))


def _gather_best(energies, rows, index, cand_e, occ, k, world, merge_duplicates):
    """SURVEY 8(e): what crosses NVLink is the energy vectors (8 bytes per read) and k candidate rows per rank.  The winners
    are the k lowest-energy candidates over all ranks, ties to the lower global read index."""
    e_all = np.concatenate(_all_gather_var(energies, world))
    c_rows = np.concatenate(_all_gather_var(rows, world))
    c_idx = np.concatenate(_all_gather_var(index, world))
    c_e = np.concatenate(_all_gather_var(cand_e, world))
    c_occ = np.concatenate(_all_gather_var(occ, world))
    if merge_duplicates and len(c_idx):          # the same sample may have been found on several ranks
        keep, seen = [], {}
        for p in np.lexsort((c_idx, c_e)):
            key = c_rows[p].tobytes()
            if key in seen:
                c_occ[seen[key]] += c_occ[p]
            else:
                seen[key] = p
                keep.append(p)
        sel = np.array(keep[:k], dtype=np.int64)
    else:
        sel = np.lexsort((c_idx, c_e))[:k]
    # index into the concatenated energy vector == global read index only when no rank was interrupted; report both
    return e_all, c_rows[sel], c_idx[sel], c_occ[sel]


def _decode_discrete(ss: SampleSet, model: LoweredModel, dqm=None) -> SampleSet:
    K = model.meta["num_cases"]
    cells = model.meta["cells"]
    n = len(cells)
    case, ok = decode_onehot(ss.record.sample, n, K)
    feasible = ok.all(axis=1)
    # energy of the decoded (repaired) assignment under the lowered model
    bits = np.zeros((len(ss), model.num_variables), dtype=np.int8)
    rows = np.repeat(np.arange(len(ss)), n)
    bits[rows, (np.tile(np.arange(n) * K, len(ss)) + case.ravel())] = 1
    if isinstance(model, DeviceModel):     # energies of the repaired assignments from the library (neal's summation order)
        energy = model.gm.energies((2 * bits - 1).astype(np.int8))[0] + model.offset
    else:
        energy = model.energies(2 * bits.astype(np.int16) - 1)
    out = SampleSet.from_samples((case.astype(np.int8) if K < 128 else case, cells), energy=energy, vartype=BINARY,
                                 info=dict(ss.info), is_feasible=feasible)
    out.vartype_name = "DISCRETE"
    out.info["onehot_penalty"] = model.meta.get("penalty")
    return out


def _annotate_cqm(ss: SampleSet, model: LoweredModel) -> SampleSet:
    if model.meta.get("kind") == "cqm_generic":
        cqm = model.meta["cqm"]
        feasible = cqm.check_feasible(np.asarray(ss.record.sample), ss.variables)
        out = SampleSet.from_samples((ss.record.sample, ss.variables), energy=ss.record.energy, vartype=BINARY,
                                     info=dict(ss.info), is_feasible=feasible)
        out.info["onehot_penalty"] = model.meta.get("onehot_penalty")
        out.info["size_penalty"] = model.meta.get("size_penalty")
        return out
    K = model.meta["num_cases"]
    n = len(model.meta["cells"])
    case, ok = decode_onehot(ss.record.sample, n, K)
    x = np.asarray(ss.record.sample)[:, : n * K].reshape(-1, n, K)
    sizes = x.sum(axis=1)
    feasible = ok.all(axis=1) & (sizes >= model.meta["min_size"]).all(axis=1)
    out = SampleSet.from_samples((ss.record.sample, ss.variables), energy=ss.record.energy, vartype=BINARY, info=dict(ss.info),
                                 is_feasible=feasible, cluster_sizes=sizes.astype(np.int32))
    out.info["onehot_penalty"] = model.meta.get("onehot_penalty")
    out.info["size_penalty"] = model.meta.get("size_penalty")
    return out
