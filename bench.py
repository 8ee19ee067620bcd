#!/usr/bin/env python
"""bench.py -- spin-flip attempts/sec of the annealing hot path on BASELINE.json's config 3.

Workload ("config.workload"): 8-way CQM-style clustering lowered to penalties on a 16 384-cell synthetic SNN graph
(131 072 cell variables + 112 slack bits), neal-order Metropolis, 1000 sweeps, geometric beta schedule.  A "step" is
one pass of the hot path over one batch of reads (``--reads`` per GPU): annealing kernel + energy kernel (+ the
per-rank best gather at N > 1).  Reads shard over ranks with no data-path collective -> weak scaling.

    value  whole-job attempts/s with model, states, seeds and schedule already resident in HBM
    e2e    the same through the neal-shaped C-ABI call qa_sa_sample_ising with HOST (pinned) buffers: model vectors
           and initial states copied in, adjacency built on the device, final states and energies copied out
    roofline  algorithmic bytes of the annealing kernel / its CUDA-event duration / measured HBM copy bandwidth
    cpu_baseline  the CPU oracle (restatement of neal's loop, oracle/) on a bounded sample of the same workload
    full_job / strong  the config AS STATED: 100 000 reads x 1000 sweeps, split over the N ranks (strong scaling), once;
           with the feasibility fraction of the reads and the time to the CPU arm's best energy
    config5  BASELINE config 5 (dense Gaussian-affinity 4-way model, 4096 cells x 4) on the fp64 tensor-core kernel, with its own
           roofline block (achieved TFLOP/s against the measured DMMA peak)

``--impl reference`` times the oracle alone, with all host threads, on bounded samples of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "spin_flip_attempts_per_sec"
UNIT = "attempts/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cells", type=int, default=16384)
    ap.add_argument("--clusters", type=int, default=8)
    ap.add_argument("--reads", type=int, default=75776, help="reads per GPU per step (148 SMs x 16 warps x 32 reads: one full wave)")
    ap.add_argument("--sweeps", type=int, default=50,
                    help="points of the geometric beta schedule per step (the full config-3 job is 1000; the per-attempt "
                         "phase mix, hence attempts/s, is the same for any length over the same beta range)")
    ap.add_argument("--size-penalty", type=float, default=None,
                    help="CQM size penalty B (default: onehot_penalty / cells, the library's default; 1.0 reproduces the round-1 "
                         "workload, whose binary slack freezes and leaves no read feasible)")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--cpu-reads", type=int, default=0, help="reads of the CPU sample (0: 2 x host threads)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-full-job", action="store_true", help="skip the 100 000 reads x 1000 sweeps job (full_job / strong blocks)")
    ap.add_argument("--job-reads", type=int, default=100000, help="reads of the stated job (split over the ranks)")
    ap.add_argument("--job-sweeps", type=int, default=1000)
    ap.add_argument("--job-share", default="", help="development, N = 1 only: 'r/w' anneals the share of rank r of w ranks")
    ap.add_argument("--no-config5", action="store_true", help="skip the dense tensor-core block (BASELINE config 5)")
    ap.add_argument("--c5-reads", type=int, default=37888, help="reads per GPU of the config-5 block (148 SMs x 8 warps x 32 reads)")
    ap.add_argument("--c5-sweeps", type=int, default=20)
    ap.add_argument("--budget-s", type=float, default=840.0,
                    help="wall-clock budget of the whole run: the stated job is shortened (fewer sweeps, said so) when it would not fit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0's reads) as DIR/*.npy, at most 60 MB, so that two builds "
                         "can be compared output for output; see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def build_workload(args):
    from scrna_seq_qannealing_clustering_b200 import models, schedule, snn
    graph, _ = snn.synthetic_snn(args.cells, k=5, dim=15, centres=args.clusters, seed=0)
    model = models.cqm_model(graph, args.clusters, min_size=20, size_penalty=getattr(args, "size_penalty", None))
    # beta range from the explicit couplers (one-hot + objective), not from the rank-1 size penalty: neal's default on
    # the penalty would start at beta ~ 1e-8 and spend most sweeps at ~100 % acceptance (SURVEY.md hard part 4)
    beta_range = schedule.default_ising_beta_range(model.h, model.starts, model.ends, model.weights, None)
    betas, spb = schedule.make_beta_schedule(beta_range, args.sweeps, 1, "geometric")
    return model, beta_range, betas, spb


def workload_config(args, model, beta_range):
    return {
        "workload": f"config3: {args.clusters}-way CQM lowered to penalties, {args.cells}-cell synthetic SNN (k=5, trim 15), "
                    f"{model.num_variables} vars, {model.num_couplers} couplers + {args.clusters} rank-1 size groups",
        "reads_per_gpu_per_step": args.reads,
        "num_sweeps": args.sweeps,
        "beta_range": [float(beta_range[0]), float(beta_range[1])],
        "beta_schedule_type": "geometric",
        "onehot_penalty": model.meta["onehot_penalty"],
        "size_penalty": model.meta["size_penalty"],
        "mode": "reference-order (bit-exact vs oracle), per-read seeds",
        "full_job": "100000 reads x 1000 sweeps = 1.31e13 attempts; a step anneals one read wave over the same beta range; the "
                    "job as stated is run once and reported in the full_job (N=1) / strong (N>1) block",
        "l2_policy": "per-step state (reads x n x 8 B of local fields) exceeds the 126 MB L2",
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows if len(r) > 3 + i)]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


KERNEL_NAMES = {1: "k_anneal_ref<groups> (one warp per read)", 2: "k_anneal_lockstep<push,groups> (32 reads per warp, eager updates)",
                5: "k_anneal_dense<K> (dense k-way model, fields by mma.sync f64)",
                4: "k_anneal_replay<groups> (32 reads per warp, deferred exact updates, TMA-staged coupling slabs; auto-selected)"}


def algorithmic_bytes(stats: dict, entries_per_read_sweep: float, reads_per_cta: int) -> float:
    """SURVEY.md 8(d): bytes = 8*N_att + 9*N_acc + 17*D_acc + 12*D_row for the reference layout (fp64 field per attempt,
    spin + field written per accepted flip, spin read + field read-modify-write per neighbour update, 12-byte CSR entries).
    D_row -- the coupling rows -- is fetched once per CTA and visit for all the reads the CTA holds, so it is amortised over
    them: 12 * (directed entries per sweep) * sweeps * reads / reads_per_cta."""
    sweeps_x_reads = stats["attempts"] / stats["num_variables"]
    return (8.0 * stats["attempts"] + 9.0 * stats["accepted"] + 17.0 * stats["nbr_updates"]
            + 12.0 * entries_per_read_sweep * sweeps_x_reads / reads_per_cta)


def field_layout_bytes(stats: dict) -> float:
    """The same unit in THIS kernel's layout (DESIGN.md section 4): 8 B local field + 2 bits per attempt, and an 8 B read +
    8 B write of one local field per neighbour update.  Reported next to the SURVEY figure, not used for `frac`."""
    return 8.25 * stats["attempts"] + 16.0 * stats["nbr_updates"]


DUMP_ENERGY_BYTES = 16 << 20     # energies.npy + energy_reads.npy
DUMP_STATE_BYTES = 44 << 20      # states.npy + state_reads.npy


def dump_outputs(out_dir, states, energies, seed: int) -> None:
    """Write what one step of the timed path hands its caller -- final states int8 [R][n] and energies fp64 [R], both on the
    device -- as .npy files in float32 / float64, at most 60 MB in all:

        energies.npy      fp64, every read's energy (a seeded sample of 1 M reads when R is larger)
        energy_reads.npy  fp64, the read index of each entry of energies.npy
        states.npy        fp32 (+-1), whole final states of a seeded sample of reads, as many as fit 44 MB with their indices
        state_reads.npy   fp64, the read index of each row of states.npy

    The sample depends on (R, n, seed) only, so two runs with the same arguments dump the same reads."""
    import torch
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    R, n = states.shape
    rng = np.random.default_rng(seed)

    def sample(k):
        return np.arange(R) if k >= R else np.sort(rng.choice(R, size=k, replace=False))

    e_idx = sample(DUMP_ENERGY_BYTES // 16)
    s_idx = sample(max(1, DUMP_STATE_BYTES // (4 * n + 8)))
    e = energies[torch.from_numpy(e_idx).to(energies.device)].cpu().numpy()
    s = states[torch.from_numpy(s_idx).to(states.device)].cpu().numpy()
    np.save(out / "energies.npy", e.astype(np.float64))
    np.save(out / "energy_reads.npy", e_idx.astype(np.float64))
    np.save(out / "states.npy", s.astype(np.float32))
    np.save(out / "state_reads.npy", s_idx.astype(np.float64))


def run_cpu_sample(model, betas, spb, seed, reads, threads, states=None, seeds=None):
    """The CPU restatement on `reads` reads (its own seeded inputs, or the given initial states / per-read seeds)."""
    from oracle import oracle
    from scrna_seq_qannealing_clustering_b200 import schedule
    if states is None:
        states = schedule.random_spin_states(reads, model.num_variables, seed)
    if seeds is None:
        seeds = schedule.per_read_seeds(seed, reads)
    t0 = time.perf_counter()
    e, st = oracle.sample_ising(model.h, model.starts, model.ends, model.weights, states, betas, spb, seeds,
                                groups=model.groups.astuple() if model.groups is not None else None, nthreads=threads)
    dt = time.perf_counter() - t0
    return st["attempts"] / dt, dt, e + model.offset, states


DMMA_PEAK_TFLOPS = 37.1   # measured on this pool's B200: tools/ubench_dmma.cu, profiles/r2_ubench_dmma_peak.log (DFMA: 24.7)


def config5_block(args, ctx, dev, rank, world, allmax, cpu_threads):
    """BASELINE.json config 5 (dense Gaussian-affinity QUBO, 4096 cells x 4 clusters, batched local fields on fp64 tensor cores):
    `c5_reads` reads per GPU x `c5_sweeps` sweeps on k_anneal_dense (QA_MODE_THROUGHPUT), inputs resident.  Roofline: the kernel
    is bound by the fp64 tensor pipe -- 2 * n_cells flops per attempt against the measured DMMA peak."""
    import torch
    from scrna_seq_qannealing_clustering_b200 import _lib, models, schedule, snn
    from scrna_seq_qannealing_clustering_b200.engine import IsingModel
    cells, K = 4096, 4
    X, _ = snn.gaussian_mixture_embedding(cells, dim=15, centres=K, sep=4.0, seed=2)
    m = models.dense_kway_model(snn.gaussian_affinity(X, k=10), K, 0.05)
    n = m.num_variables
    hot = schedule.default_ising_beta_range(m.h, m.starts, m.ends, m.weights, None)[0]
    beta_range = (hot, 1000.0 * hot)     # the default cold end follows the smallest non-zero coupling: ~1e7 on a Gaussian affinity
    betas, spb = schedule.make_beta_schedule(beta_range, args.c5_sweeps, 1, "geometric")
    R = args.c5_reads
    gm = IsingModel(ctx, m.h, m.starts, m.ends, m.weights)
    try:
        if not gm.enable_dense(K):
            raise RuntimeError("config 5 model lost its dense k-way form")
        g = torch.Generator(device=dev)
        g.manual_seed(args.seed + 5 + rank)
        states = torch.randint(0, 2, (R, n), dtype=torch.int8, device=dev, generator=g)
        states.mul_(2).sub_(1)
        head = states[:4].cpu().numpy() if cpu_threads else None
        seeds = schedule.per_read_seeds(args.seed + 5, R, first_read=rank * R)
        seeds_dev = torch.from_numpy(seeds.view(np.int64)).to(dev)
        energies = torch.empty(R, dtype=torch.float64, device=dev)
        betas_dev = torch.from_numpy(betas).to(dev)
        torch.cuda.synchronize()
        keep = states.clone()
        gm.sample(states, betas_dev, spb, seeds_dev, mode=_lib.QA_MODE_THROUGHPUT, energies=energies)      # warm-up
        states.copy_(keep)
        torch.cuda.synchronize()
        _, st, done = gm.sample(states, betas_dev, spb, seeds_dev, mode=_lib.QA_MODE_THROUGHPUT, energies=energies)
        assert done == R and ctx.last_kernel == _lib.QA_KERNEL_DENSE
        t = allmax(st.ms_anneal * 1e-3)
        attempts = float(n) * len(betas) * spb * R * world
        tflops = 2.0 * cells * attempts / t / 1e12
        out = {"workload": f"config5: dense Gaussian-affinity {K}-way model, {cells} cells x {K} = {n} vars, {m.num_couplers} couplers",
               "reads_per_gpu": R, "num_sweeps": len(betas) * spb, "beta_range": [float(beta_range[0]), float(beta_range[1])],
               "mode": "QA_MODE_THROUGHPUT (neal's sweep order and RNG, fields by mma.sync f64; tolerance parity)",
               "value": attempts / t, "unit": UNIT, "seconds": t, "acceptance": st.accepted / st.attempts,
               "best_energy": float(energies.min().item() + m.offset),
               "roofline": {"bound": "tensor", "achieved": tflops / world, "peak": DMMA_PEAK_TFLOPS, "unit": "TFLOP/s",
                            "frac": tflops / world / DMMA_PEAK_TFLOPS, "traffic": None, "kernel": "k_anneal_dense<4> (DMMA.8x8x4)",
                            "flops_per_attempt": 2.0 * cells,
                            "peak_source": "measured fp64 mma.sync m8n8k4 rate of this pool's B200 (profiles/r2_ubench_dmma_peak.log); "
                                           "MEASURED_PEAKS.json carries no fp64 figure"}}
        if cpu_threads:
            # the CPU arm anneals the first reads: same trajectories (generic real weights), energies to 1e-9 of neal's order
            hs = head.copy()
            t0 = time.perf_counter()
            from oracle import oracle
            ce, cst = oracle.sample_ising(m.h, m.starts, m.ends, m.weights, hs, betas, spb, seeds[:4], nthreads=cpu_threads)
            dt = time.perf_counter() - t0
            ge = energies[:4].cpu().numpy()
            out["cpu_arm"] = {"reads": 4, "seconds": dt, "value": cst["attempts"] / dt, "cores": min(cpu_threads, 4),
                              "final_states_identical_to_gpu": bool(np.array_equal(hs, states[:4].cpu().numpy())),
                              "max_rel_energy_diff": float(np.max(np.abs(ge - ce) / np.maximum(np.abs(ce), 1.0)))}
        return out
    finally:
        gm.close()


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model, beta_range, betas, spb = build_workload(args)
    threads = len(os.sched_getaffinity(0))  # torchrun exports OMP_NUM_THREADS=1: ask for every host core explicitly
    reads = args.cpu_reads or 8 * threads
    for _ in range(max(0, min(args.warmup, 1))):
        run_cpu_sample(model, betas[: max(1, len(betas) // 50)], spb, args.seed, threads, threads)
    rates, times = [], []
    for s in range(args.steps):
        r, dt, _, _ = run_cpu_sample(model, betas, spb, args.seed + s, reads, threads)
        rates.append(r)
        times.append(dt)
    total_attempts = model.num_variables * len(betas) * spb * reads * args.steps
    value = total_attempts / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, model, beta_range),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{reads} reads x {len(betas) * spb} sweeps x {model.num_variables} vars per step, OpenMP over reads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "`config` names the workload of the GPU arm; a CPU step anneals the bounded sample in cpu_baseline.sample of that "
                "workload (same model, schedule, seeding rule) -- a rate, so the read count does not enter the metric",
    }
    emit(line)


def emit(line: dict):
    """Rank 0 prints ONE JSON line on the real stdout (libraries such as NCCL may write banners to fd 1: it is pointed at
    stderr for the duration of the run, see main())."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    t_start = time.perf_counter()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse_args()
    if args.impl == "reference":
        return main_reference(args)

    import torch
    import torch.distributed as dist
    from scrna_seq_qannealing_clustering_b200 import schedule
    from scrna_seq_qannealing_clustering_b200.engine import Context, IsingModel

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # The path's only exchange is 16 bytes per rank and step.  With NCCL's peer-to-peer transport enabled (peer mappings of
        # the other ranks' memory), the annealing kernel of rank 0 ran 45 % longer in the part-filled strong leg (117 s against
        # 83 s for the same 50 000-read share; measured four ways: torchrun default, NVLS off, P2P off, two independent
        # processes -- profiles/r2_strong_leg_n2_investigation.md).  Default to NCCL's shared-memory transport; an explicit
        # NCCL_P2P_DISABLE in the environment wins.
        os.environ.setdefault("NCCL_P2P_DISABLE", "1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    def allmax(x: float) -> float:
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def allsum(x: float) -> float:
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return float(tt.item())

    model, beta_range, betas, spb = build_workload(args)
    n = model.num_variables
    R = args.reads
    groups = model.groups.astuple()
    first_read = rank * R
    seeds = schedule.per_read_seeds(args.seed, R, first_read=first_read)
    rng = np.random.default_rng(args.seed + 7919 * rank)
    # one pinned host buffer of initial states per rank (filled in chunks: no pageable 10 GB temporaries), reused by the e2e leg
    init_host = torch.empty((R, n), dtype=torch.int8, pin_memory=True)
    ih = init_host.numpy()
    for r0 in range(0, R, 4096):
        r1 = min(R, r0 + 4096)
        ih[r0:r1] = rng.integers(0, 2, size=(r1 - r0, n), dtype=np.int8) * 2 - 1
    # the reads the CPU leg anneals, too (full-size parity check): the head of the wave, a tile in its middle (another CTA,
    # other SMs) and the last reads of the wave
    threads = len(os.sched_getaffinity(0))
    ncpu = min(R, args.cpu_reads or 8 * threads)
    part = max(1, ncpu // 3)
    mid0 = min(max(0, (R // 2) // 32 * 32), max(0, R - part))
    sel = np.unique(np.concatenate([np.arange(0, min(R, ncpu - 2 * part)), np.arange(mid0, min(R, mid0 + part)),
                                    np.arange(max(0, R - part), R)]))
    init_sel = ih[sel].copy()

    ctx = Context(local_rank)
    gm = IsingModel(ctx, model.h, model.starts, model.ends, model.weights)
    gm.set_groups(*groups)

    # device-resident inputs (torch tensors used purely as HBM buffers)
    init_dev = init_host.to(dev, non_blocking=False)
    states_dev = torch.empty_like(init_dev)
    energies_dev = torch.empty(R, dtype=torch.float64, device=dev)
    seeds_dev = torch.from_numpy(seeds.view(np.int64)).to(dev)
    betas_dev = torch.from_numpy(betas).to(dev)
    best_buf = torch.zeros(2, dtype=torch.float64, device=dev)
    gathered = [torch.zeros(2, dtype=torch.float64, device=dev) for _ in range(world)] if world > 1 else None

    stats_acc = {}
    kernel_used = 0

    def step_resident(record: bool):
        states_dev.copy_(init_dev)
        torch.cuda.synchronize()
        e, st, done = gm.sample(states_dev, betas_dev, spb, seeds_dev, energies=energies_dev)
        assert done == R
        if world > 1:  # the path's only exchange: per-rank best (energy, global read index) from the library's argmin kernel
            ctx.argmin_into(energies_dev, first_read, best_buf)      # device -> device: the all_gather's send buffer
            dist.all_gather(gathered, best_buf)
        if record:
            for k, v in st.as_dict().items():
                stats_acc[k] = stats_acc.get(k, 0) + v
        return st

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_resident(False)
    kernel_used = ctx.last_kernel
    barrier()
    with ClockSampler(local_rank) as clocks:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_resident(True)
        barrier()
        elapsed = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, states_dev, energies_dev, args.seed)
    wall_s = allmax(elapsed)
    attempts_per_step_per_gpu = n * len(betas) * spb * R
    # device time: the library brackets every call with CUDA events on the stream it launches on (qa_stats.ms_total);
    # max over ranks.  The host wall clock around the same region is reported next to it.
    elapsed = allmax(stats_acc["ms_total"] * 1e-3)
    value = attempts_per_step_per_gpu * world * args.steps / elapsed
    stats_acc["num_variables"] = n

    # ---- e2e: HOST buffers through the neal-shaped C-ABI entry point, copies inside the timed region -----------------
    e2e = None
    if not args.no_e2e:
        host_states = init_host                # the same pinned buffer: refilled from the device copy before every step
        host_energies = torch.empty(R, dtype=torch.float64, pin_memory=True)
        hs, he = host_states.numpy(), host_energies.numpy()

        def step_e2e_groups():
            host_states.copy_(init_dev)        # harness: a fresh copy of the initial states (the call works in place)
            barrier()
            t0 = time.perf_counter()           # timed: model upload + adjacency/slab build + H2D + anneal + energies + D2H
            m2 = IsingModel(ctx, model.h, model.starts, model.ends, model.weights)
            m2.set_groups(*groups)
            _, st, done = m2.sample(hs, betas, spb, seeds, energies=he)
            dt = time.perf_counter() - t0      # the call is blocking: results are in the host buffers here
            m2.close()
            assert done == R
            return dt

        e2e_steps = max(1, min(args.steps, 2))
        step_e2e_groups()
        el = 0.0
        for _ in range(e2e_steps):
            el += step_e2e_groups()
        barrier()
        el = allmax(el)
        h2d = (model.h.nbytes + model.starts.nbytes + model.ends.nbytes + model.weights.nbytes + R * n + seeds.nbytes + betas.nbytes
               + sum(np.asarray(g).nbytes for g in groups))
        d2h = R * n + R * 8
        e2e = {"value": attempts_per_step_per_gpu * world * e2e_steps / el, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": 1e3 * el / e2e_steps,
               "api": "IsingModel(h, starts, ends, weights) + set_groups + sample(host states) [qa_model_from_ising + "
                      "qa_model_set_groups + qa_sa_sample_model]"}

    # ---- e2e through the dimod-shaped sampler with return_samples='best_k': the state matrix is created (counter-based
    # generator), annealed, ranked and reduced to k rows on the device -- what crosses PCIe is the model, the seeds, R energies
    # and k samples.  Reported NEXT TO `e2e` (whose inputs and outputs are full host state matrices), not instead of it.
    e2e_k = None
    if not args.no_e2e:
        from scrna_seq_qannealing_clustering_b200.sampler import B200SimulatedAnnealingSampler
        smp = B200SimulatedAnnealingSampler(context=ctx)
        kbest = 16

        def step_best_k():
            barrier()
            t0 = time.perf_counter()
            ss = smp.sample(model, num_reads=R * world, beta_schedule_type="custom", beta_schedule=betas, seed=args.seed,
                            initial_states_generator="counter", return_samples="best_k", num_best=kbest)
            dt = time.perf_counter() - t0
            assert len(ss.info["energies"]) == R * world
            return dt, ss

        step_best_k()
        elk = 0.0
        k_steps = max(1, min(args.steps, 2))
        for _ in range(k_steps):
            dt, ss_k = step_best_k()
            elk += dt
        elk = allmax(elk)
        h2d_k = (model.h.nbytes + model.starts.nbytes + model.ends.nbytes + model.weights.nbytes + seeds.nbytes + betas.nbytes
                 + sum(np.asarray(g).nbytes for g in groups))
        d2h_k = R * 8 + R * 4 + kbest * n
        e2e_k = {"value": attempts_per_step_per_gpu * world * k_steps / elk, "unit": UNIT, "h2d_bytes_per_step": int(h2d_k),
                 "d2h_bytes_per_step": int(d2h_k), "steps": k_steps, "ms_per_step": 1e3 * elk / k_steps, "num_best": kbest,
                 "best_energy": float(ss_k.first.energy),
                 "api": "B200SimulatedAnnealingSampler.sample(model, num_reads, beta_schedule, seed, initial_states_generator='counter', "
                        "return_samples='best_k') -> SampleSet of the k best samples + info['energies']"}

    # ---- roofline of the dominant kernel (annealing), from the library's own CUDA events on its stream --------------
    peak, peak_src = peaks()
    launches = max(int(stats_acc.get("anneal_launches", 1)), 1)
    ms_kernel = stats_acc["ms_anneal"] / launches
    reads_per_cta = 256                      # replay kernel: 8 warps x 32 reads share every coupling-slab fetch
    alg = algorithmic_bytes(stats_acc, 2.0 * model.num_couplers, reads_per_cta) / launches
    achieved = alg / (ms_kernel * 1e-3) / 1e9
    # measured DRAM bytes of the same launch shape, from the committed ncu launch list (a bench value is never taken under ncu)
    traffic = None
    tfile = ROOT / "profiles" / "traffic_replay_config3.json"
    if tfile.exists():
        t = json.loads(tfile.read_text())
        if (t["kernel"], t["reads"], t["num_sweeps"], t["num_variables"]) == (kernel_used, R, len(betas) * spb, n) and \
                t.get("library_round", 1) >= 2:
            traffic = t["dram_bytes_per_launch"]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "kernel": KERNEL_NAMES.get(kernel_used, str(kernel_used)), "ms_per_launch": ms_kernel,
                "algorithmic_bytes_per_launch": alg,
                "formula": "SURVEY 8(d): 8*N_att + 9*N_acc + 17*D_acc + 12*D_row, D_row amortised over the 256 reads of a CTA",
                "bytes_per_attempt": alg * launches / stats_acc["attempts"],
                "field_layout_bytes_per_attempt": field_layout_bytes(stats_acc) / stats_acc["attempts"],
                "field_layout_GBps": field_layout_bytes(stats_acc) / launches / (ms_kernel * 1e-3) / 1e9,
                "acceptance": stats_acc["accepted"] / stats_acc["attempts"],
                "candidates": stats_acc["candidates"] / stats_acc["attempts"],
                "kernel_share_of_step": stats_acc["ms_anneal"] / (elapsed * 1e3)}
    if traffic is not None:
        # what the kernel really moves (ncu, same launch shape): the replay form does not perform the per-(flip, neighbour)
        # read-modify-writes the reference formulation's byte count charges for, so `frac` can approach (or pass) 1 while
        # DRAM is far from busy -- the measured figure is the honest bandwidth statement
        roofline["traffic_bytes_per_attempt"] = traffic * launches / stats_acc["attempts"]
        roofline["traffic_GBps"] = traffic / (ms_kernel * 1e-3) / 1e9
        roofline["traffic_frac_of_peak"] = roofline["traffic_GBps"] / peak
        roofline["note"] = ("achieved = algorithmic bytes of the REFERENCE formulation (SURVEY 8(d)) / kernel time; the kernel's own DRAM "
                            "traffic (ncu) is traffic_GBps")

    # ---- CPU baseline on rank 0, N = 1 only ---------------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the CPU sample anneals reads of the GPU step (same initial states, same per-read seeds) from the head, the middle and
        # the tail of the wave, so it is also a full-size parity check: final states bytewise AND energies bitwise
        v, dt, cpu_energies, cpu_states = run_cpu_sample(model, betas, spb, args.seed, len(sel), threads, states=init_sel.copy(),
                                                         seeds=seeds[sel])
        isel = torch.from_numpy(sel).to(dev)
        gpu_states = states_dev[isel].cpu().numpy()
        gpu_e = energies_dev[isel].cpu().numpy()
        e_bad = np.flatnonzero(cpu_energies.view(np.uint64) != (gpu_e + model.offset).view(np.uint64))
        if len(e_bad):   # say where and by how much (stderr; the JSON line carries the verdict)
            print("[bench] energy mismatches at reads", sel[e_bad][:16].tolist(), "cpu", cpu_energies[e_bad][:4].tolist(),
                  "gpu", (gpu_e + model.offset)[e_bad][:4].tolist(), file=sys.stderr)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "seconds": dt,
               "sample": f"{len(sel)} reads x {len(betas) * spb} sweeps x {n} vars of the same workload (head, middle and tail of the "
                         "wave), OpenMP over reads",
               "parity_check": {"reads": int(len(sel)), "read_indices": [int(sel[0]), int(sel[len(sel) // 2]), int(sel[-1])],
                                "final_states_identical_to_gpu": bool(np.array_equal(cpu_states, gpu_states)),
                                "energies_bitwise_identical_to_gpu": bool(np.array_equal(cpu_energies.view(np.uint64),
                                                                                         (gpu_e + model.offset).view(np.uint64)))}}
    best_weak = float(energies_dev.min().item() + model.offset)

    # ---- BASELINE config 5: dense Gaussian-affinity 4-way model on the fp64 tensor-core kernel (every rank its own reads) ---
    c5 = None
    if not args.no_config5:
        c5 = config5_block(args, ctx, dev, rank, world, allmax, threads if (rank == 0 and world == 1 and not args.no_cpu_baseline) else 0)

    # ---- the config AS STATED: job_reads x job_sweeps, reads split over the ranks (strong scaling), once ---------------
    job = None
    if not args.no_full_job:
        del init_dev, states_dev, init_host, ih
        if not args.no_e2e:
            del host_states, hs
        torch.cuda.empty_cache()
        srank, sworld = rank, world
        if args.job_share and world == 1:      # development: anneal the share rank r of w would get (same reads, seeds, initial states)
            srank, sworld = (int(x) for x in args.job_share.split("/"))
        lo = srank * args.job_reads // sworld
        hi = (srank + 1) * args.job_reads // sworld
        Rj = hi - lo
        # shorten the job when it would not fit the wall-clock budget (the rate does not depend on the schedule length: same
        # beta range, same phase mix -- measured, see `full_job.value` against `value`)
        rate = value / world
        waves = max(1.0, np.ceil(Rj / 32 / (148 * 16)))
        est = lambda sw: n * sw * max(Rj, 1) / rate * (waves * 148 * 16 * 32 / max(Rj, 1))  # noqa: E731  (tail waves run the SMs part-full)
        left = args.budget_s - (time.perf_counter() - t_start) - 45.0
        job_sweeps = args.job_sweeps
        while job_sweeps > 50 and est(job_sweeps) > left:
            job_sweeps //= 2
        job_sweeps = int(allmax(float(-job_sweeps)) * -1) if world > 1 else job_sweeps      # the same on every rank: the minimum
        jbetas, jspb = schedule.make_beta_schedule(beta_range, job_sweeps, 1, "geometric")
        jseeds = schedule.per_read_seeds(args.seed + 1, Rj, first_read=lo)
        g = torch.Generator(device=dev)
        g.manual_seed(args.seed + 17 + srank)
        jstates = torch.randint(0, 2, (Rj, n), dtype=torch.int8, device=dev, generator=g)
        jstates.mul_(2).sub_(1)
        ncj = min(Rj, 2 * threads) if (rank == 0 and not args.no_cpu_baseline) else 0
        jinit_head = jstates[:ncj].cpu().numpy() if ncj else None
        jenergies = torch.empty(Rj, dtype=torch.float64, device=dev)
        jseeds_dev = torch.from_numpy(jseeds.view(np.int64)).to(dev)
        barrier()
        with ClockSampler(local_rank) as jclocks:      # a two-minute launch: clocks and throttle reasons of THIS leg, per rank
            _, jst, jdone = gm.sample(jstates, torch.from_numpy(jbetas).to(dev), jspb, jseeds_dev, energies=jenergies)
        assert jdone == Rj
        jck = jclocks.summary()
        jck["sm_mhz_min_over_ranks"] = -allmax(-(jck["sm_mhz"] or 0.0))
        jck["slowest_rank_seconds"] = allmax(jst.ms_total * 1e-3)
        jck["fastest_rank_seconds"] = -allmax(-jst.ms_total * 1e-3)
        jck["throttled_ranks"] = allsum(1.0 if jck["reasons"] else 0.0)
        if world > 1:      # who was slow: kernel seconds of every rank, in rank order
            mine = torch.tensor([jst.ms_anneal * 1e-3], dtype=torch.float64, device=dev)
            every = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            jck["kernel_seconds_by_rank"] = [float(x.item()) for x in every]
        t_job = allmax(jst.ms_total * 1e-3)
        job_attempts = float(n) * job_sweeps * args.job_reads
        cells = len(model.meta["cells"])
        _, viol = ctx.decode_onehot(jstates, cells, args.clusters, on_value=1, min_size=model.meta["min_size"], want_labels=False)
        feasible = allsum(float(((viol[:, 0] == 0) & (viol[:, 1] == 0)).sum()))
        onehot_ok = allsum(float((viol[:, 0] == 0).sum()))
        bad_cells = allsum(float(viol[:, 0].sum()))
        small_clusters = allsum(float(viol[:, 1].sum()))
        ej = jenergies.cpu().numpy() + model.offset
        best_job = -allmax(-float(ej.min()))
        job = {"reads": args.job_reads, "num_sweeps": job_sweeps, "num_sweeps_stated": args.job_sweeps, "reads_per_rank": int(Rj),
               "seconds": t_job, "value": job_attempts / t_job, "unit": UNIT, "scaling": "strong",
               "read_waves_per_gpu": float(Rj / 32 / (148 * 16)),
               "feasible_fraction": feasible / args.job_reads, "onehot_satisfied_fraction": onehot_ok / args.job_reads,
               "mean_cells_not_onehot_per_read": bad_cells / args.job_reads, "cells": cells,
               "mean_clusters_below_min_size_per_read": small_clusters / args.job_reads,
               "best_energy": best_job, "kernel_ms": allmax(jst.ms_anneal), "vs_weak_value_per_gpu": (job_attempts / t_job / world) / rate,
               "clocks": jck}
        if ncj:
            # the CPU arm on the first reads of the job: the converged target of the time-to-best-energy figure, and one more
            # parity check at the full schedule length
            vj, dtj, cej, csj = run_cpu_sample(model, jbetas, jspb, args.seed + 1, ncj, threads, states=jinit_head.copy(), seeds=jseeds[:ncj])
            target = float(cej.min())
            job["cpu_arm"] = {"reads": int(ncj), "seconds": dtj, "value": vj, "best_energy": target,
                              "final_states_identical_to_gpu": bool(np.array_equal(csj, jstates[:ncj].cpu().numpy())),
                              "energies_bitwise_identical_to_gpu": bool(np.array_equal(cej.view(np.uint64), ej[:ncj].view(np.uint64)))}
        else:
            target = None
        if world > 1:   # every rank needs the target to count its hits
            tt = torch.tensor([target if target is not None else 0.0], dtype=torch.float64, device=dev)
            dist.broadcast(tt, 0)
            target = float(tt.item()) if not args.no_cpu_baseline else None
        if target is not None:
            hits = allsum(float((ej <= target + 1e-9 * abs(target)).sum()))
            p_hit = hits / args.job_reads
            ttb = {"target_energy": target, "target": "best energy the CPU arm reached on its reads of the same job",
                   "p_hit_per_read": p_hit, "p_hit_estimated_on_reads": args.job_reads}
            if 0.0 < p_hit < 1.0:
                need = float(np.log(0.01) / np.log1p(-p_hit))
                ttb.update({"reads_for_99pct": need, "gpu_tts99_s": need / args.job_reads * t_job})
                if "cpu_arm" in job:
                    ttb["cpu_tts99_s"] = need * job["cpu_arm"]["seconds"] / job["cpu_arm"]["reads"]
                    ttb["cpu_cores"] = threads
            job["time_to_best_energy"] = ttb

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / args.steps, "wall_ms_per_step": 1e3 * wall_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, model, beta_range),
            "clocks": clocks.summary(), "e2e": e2e, "e2e_best_k": e2e_k, "gpu_launches": int(stats_acc.get("total_launches", 0)),
            "roofline": roofline, "cpu_baseline": cpu, "best_energy": best_weak,
            "full_job" if world == 1 else "strong": job, "config5": c5,
        }
        emit(line)
    gm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
