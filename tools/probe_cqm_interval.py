"""Config 3 (16 384 cells x 8 clusters, 75 776 reads x 50 sweeps) with the CQM size constraint lowered two ways: slack bits
(models.cqm_model default, B = A/n) and interval groups (size_lowering="interval", B = A).  Alternating runs, 3 each, then a
binding variant (min_size = 1900 of 2048 cells per cluster on average).  Per run: attempts/s from the kernel's own timing
(qa_stats.ms_anneal), the kernel that ran, the feasible fraction and reads with clusters below min_size (qa_decode_onehot),
and the best CQM objective among the feasible reads (exact, over the 64 lowest-energy feasible reads).

    python tools/probe_cqm_interval.py [--reads 75776] [--sweeps 50] [--out LOGFILE]   (the lines also go to stdout)
"""
from __future__ import annotations

import argparse
import subprocess
import sys
import types
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (the config-3 workload, unchanged)
from scrna_seq_qannealing_clustering_b200 import _lib, models, schedule, snn  # noqa: E402
from scrna_seq_qannealing_clustering_b200.engine import Context, IsingModel  # noqa: E402

KERNEL_NAMES = {1: "WARP_PER_READ", 2: "LOCKSTEP_PUSH", 3: "LOCKSTEP_PULL", 4: "REPLAY", 5: "DENSE"}


def run_one(ctx, model, graph_arrays, betas, spb, R, seed, min_size):
    import torch
    n_cells, K = len(model.meta["cells"]), model.meta["num_cases"]
    nv = model.num_variables
    gm = IsingModel(ctx, model.h, model.starts, model.ends, model.weights)
    gm.set_groups(*model.groups.astuple())
    states = torch.empty((R, nv), dtype=torch.int8, device="cuda")
    ctx.random_states(seed, 0, R, nv, out=states)
    seeds = torch.from_numpy(schedule.per_read_seeds(seed, R).view(np.int64)).cuda()
    energies = torch.empty(R, dtype=torch.float64, device="cuda")
    e, st, done = gm.sample(states, torch.from_numpy(betas).cuda(), spb, seeds, energies=energies)
    torch.cuda.synchronize()
    kernel = ctx.last_kernel
    _, viol = ctx.decode_onehot(states, n_cells, K, on_value=1, min_size=min_size, want_labels=False)
    feasible = (viol[:, 0] == 0) & (viol[:, 1] == 0)
    e_host = energies.cpu().numpy() + model.offset
    best = None
    if feasible.any():
        idx = np.nonzero(feasible)[0]
        idx = idx[np.argsort(e_host[idx], kind="stable")[:64]]
        rows = states[torch.from_numpy(idx).cuda()].cpu().numpy()[:, : n_cells * K]
        _, eu, ev, w = graph_arrays
        lab = rows.reshape(len(idx), n_cells, K).argmax(axis=2)
        same = lab[:, eu] == lab[:, ev]
        best = float(np.min(2.0 * len(w) - 2.0 * (same * w).sum(axis=1)))
    gm.close()
    return {"attempts_per_s": st.attempts / (st.ms_anneal / 1e3), "ms_anneal": st.ms_anneal, "kernel": KERNEL_NAMES.get(kernel, kernel),
            "feasible": float(feasible.mean()), "reads_with_small_clusters": int((viol[:, 1] > 0).sum()),
            "reads_not_onehot": int((viol[:, 0] > 0).sum()), "best_feasible_objective": best, "done": int(done)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=75776)
    ap.add_argument("--sweeps", type=int, default=50)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    a = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout
    log("card: " + " | ".join(gpu.strip().splitlines()))
    args = types.SimpleNamespace(cells=16384, clusters=8, sweeps=a.sweeps, size_penalty=None)
    slack_model, beta_range, betas, spb = bench.build_workload(args)
    graph, _ = snn.synthetic_snn(args.cells, k=5, dim=15, centres=args.clusters, seed=0)   # bench.build_workload's graph
    ga = models.graph_arrays(graph)
    log(f"config 3: {args.cells} cells x {args.clusters} clusters, {a.reads} reads x {a.sweeps} sweeps, beta range {beta_range}")
    with Context(0) as ctx:
        for min_size, label in ((20, "stated job (min_size 20)"), (1900, "binding (min_size 1900 of 2048 per cluster)")):
            slack = bench.build_workload(args)[0] if min_size == 20 else models.cqm_model(graph, 8, min_size=min_size)
            ivl = models.cqm_model(graph, 8, min_size=min_size, size_lowering="interval")
            log(f"--- {label}: slack n={slack.num_variables} B={slack.meta['size_penalty']:.6g} | interval n={ivl.num_variables} "
                f"B={ivl.meta['size_penalty']:.6g} (A={ivl.meta['onehot_penalty']:.6g})")
            runs = a.runs if min_size == 20 else 1
            for k in range(runs):
                for name, m in (("slack", slack), ("interval", ivl)):
                    r = run_one(ctx, m, ga, betas, spb, a.reads, 1234 + k, min_size)
                    log(f"{name:8s} run {k}: " + " ".join(f"{key}={val:.4g}" if isinstance(val, float) else f"{key}={val}"
                                                      for key, val in r.items()))
    if a.out:
        out = Path(a.out)
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
