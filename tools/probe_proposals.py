"""dwave-samplers' sample options on the bench's config-3 model (16 384 cells x 8 clusters, CQM lowered to penalties, beta range
and schedule of bench.build_workload).  One JSON line per case, with the card's name, power limit and SM clock read in this
process:

  seq_metropolis / seq_gibbs   sequential order on the replay kernel at the bench's read count (75 776) and 50 sweeps,
                               alternated --runs times
  random_metropolis / random_gibbs
                               random order on the warp-per-read kernel at its resident read count (one read per resident
                               warp) and --random-sweeps sweeps (16: a window of about 5 s on a B200), after a one-sweep
                               warm-up run

Rates are attempts / qa_stats.ms_anneal (the annealing kernel's own CUDA-event time); acceptance = accepted / attempts;
draws counts every xorshift128+ output consumed (random order: one order draw per attempt included).

    python tools/probe_proposals.py [--reads 75776] [--sweeps 50] [--runs 2] [--random-sweeps 16] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import types
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (the config-3 workload, unchanged)
from scrna_seq_qannealing_clustering_b200 import _lib, schedule  # noqa: E402
from scrna_seq_qannealing_clustering_b200.engine import Context, IsingModel  # noqa: E402

KERNEL_NAMES = {1: "WARP_PER_READ", 2: "LOCKSTEP_PUSH", 4: "REPLAY", 5: "DENSE"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit": power, "sm_clock": clock}


def run(ctx, gm, nv, R, betas, spb, seed, var_order, proposal):
    import torch
    states = torch.empty((R, nv), dtype=torch.int8, device="cuda")
    ctx.random_states(seed, 0, R, nv, out=states)
    seeds = torch.from_numpy(schedule.per_read_seeds(seed, R).view(np.int64)).cuda()
    energies = torch.empty(R, dtype=torch.float64, device="cuda")
    _, st, done = gm.sample(states, torch.from_numpy(np.ascontiguousarray(betas)).cuda(), spb, seeds, energies=energies,
                            var_order=var_order, proposal=proposal)
    torch.cuda.synchronize()
    assert done == R
    return {"kernel": KERNEL_NAMES.get(ctx.last_kernel, ctx.last_kernel), "reads": R, "sweeps": len(betas) * spb,
            "attempts": st.attempts, "ms_anneal": round(st.ms_anneal, 3),
            "attempts_per_s": float(f"{st.attempts / (st.ms_anneal / 1e3):.4g}"),
            "acceptance": float(f"{st.accepted / st.attempts:.5g}"), "draws": st.draws,
            "draws_per_attempt": float(f"{st.draws / st.attempts:.5g}"), "candidates": st.candidates,
            "near_ties": st.near_ties, "best_energy": float(energies.min().item())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=75776)
    ap.add_argument("--sweeps", type=int, default=50)
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--random-sweeps", type=int, default=16)
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    a = ap.parse_args()
    lines = []

    def emit(case, r):
        line = json.dumps({"case": case, **card(), **r})
        print(line, flush=True)
        lines.append(line)

    args = types.SimpleNamespace(cells=16384, clusters=8, sweeps=a.sweeps, size_penalty=None)
    model, beta_range, betas, spb = bench.build_workload(args)
    nv = model.num_variables
    M, G = _lib.QA_PROPOSAL_METROPOLIS, _lib.QA_PROPOSAL_GIBBS
    with Context(0) as ctx:
        gm = IsingModel(ctx, model.h, model.starts, model.ends, model.weights)
        gm.set_groups(*model.groups.astuple())
        ctx.set_kernel(_lib.QA_KERNEL_REPLAY)
        run(ctx, gm, nv, a.reads, betas[:2], spb, 99, _lib.QA_ORDER_SEQUENTIAL, G)   # warm-up: module load, slabs
        for k in range(a.runs):
            for case, prop in (("seq_metropolis", M), ("seq_gibbs", G)):
                emit(case, run(ctx, gm, nv, a.reads, betas, spb, 1234 + k, _lib.QA_ORDER_SEQUENTIAL, prop))
        ctx.set_kernel(_lib.QA_KERNEL_AUTO)
        R = ctx.resident_reads
        for case, prop in (("random_metropolis", M), ("random_gibbs", G)):
            run(ctx, gm, nv, R, betas[:1], 1, 7, _lib.QA_ORDER_RANDOM, prop)   # warm-up
            rb, rspb = schedule.make_beta_schedule(beta_range, a.random_sweeps, 1, "geometric")   # the bench's range
            emit(case, run(ctx, gm, nv, R, rb, rspb, 1234, _lib.QA_ORDER_RANDOM, prop))
        gm.close()
    if a.out:
        out = Path(a.out)
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
