"""Same-signature stand-ins for the reference's clustering functions, with the sampler injected.

    clustering_bqm / _2 / _3     Python_Functions/BQM_clustering.py:25, :206, :353
    clustering_dqm               Python_Functions/DQM_clustering.py:24
    clustering_cqm / _2          Python_Functions/CQM_clustering.py:25, :57
    graph_subsampling            Python_Functions/QA_subsampling.py:24

Each builds the reference's model (models.py), hands it to ``sampler`` (default: B200SimulatedAnnealingSampler) through
the dimod call the reference makes, and consumes the SampleSet the way the reference does (labels on the graph,
recursion rules).  ``solver`` / ``dirs`` / ``chain_strength`` are accepted for signature compatibility; QPU-only
kwargs are forwarded and dropped by the sampler with a warning, as neal would.
The recursion rules are restated literally in ``bqm_rule`` / ``bqm2_rule`` (ratio test, |e3| <= 0.1 early return with
one colour, ``min(len) > 5``, labels overwritten after a ``conf`` recursion, ``100 - color`` labels of ``clustering_bqm_2``).
Deviations, all deliberate: the reference's recursive calls omit ``chain_strength`` (TypeError on first recursion,
SURVEY.md 3.1) -- here the argument is passed; its ``conf`` rule reads ``record.energy[0]/[3]`` assuming an
energy-sorted record -- here the SampleSet is requested sorted; the functions return the level's SampleSet on every path
(the reference returns None on most).
"""
from __future__ import annotations

import random
import warnings
from typing import Optional

import numpy as np

from . import models
from .sampler import B200SimulatedAnnealingSampler

_default_sampler = None


def _sampler(sampler):
    global _default_sampler
    if sampler is not None:
        return sampler
    if _default_sampler is None:
        _default_sampler = B200SimulatedAnnealingSampler()
    return _default_sampler


def _on_device(sampler, device_build) -> bool:
    """Models are built by the qa_build_* kernels when the sampler can (ours); ``device_build=False`` forces the host builders."""
    return hasattr(sampler, "build_on_device") if device_build is None else bool(device_build)


def _close(model):
    if hasattr(model, "gm"):      # a DeviceModel owns a device handle
        model.close()


def _sample(sampler, model, quiet_kwargs: dict, sa_kwargs: dict):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)  # label / chain_strength / return_embedding are QPU-only
        return sampler.sample(model, sorted=True, **quiet_kwargs, **sa_kwargs)


def _split(G, response):
    lut = response.first.sample
    S0 = [node for node in G.nodes if not lut[node]]
    S1 = [node for node in G.nodes if lut[node]]
    return S0, S1


def _label(G, nodes, label, value):
    for i in nodes:
        G.nodes[i][label] = value


def bqm_rule(terminate_on, n0, n1, energies, iteration, size_limit, iter_limit):
    """The reference's termination rules for ``clustering_bqm``, restated literally (BQM_clustering.py:113-203).

    ``energies`` is the energy-sorted record (``response.record.energy``).  Returns ``(recurse, labels)`` where ``labels``
    says what the reference writes into ``G.nodes[.]['label<iteration>']`` at this level: ``'split'`` (one random colour
    per half), ``'single'`` (one random colour for every node) or ``None`` (nothing written).  In the ``conf`` branch the
    reference labels the halves, recurses, and then overwrites the level's label with a single colour: the net effect on
    this level's label is ``'single'``.
    """
    if terminate_on == "min_size":                                   # :113-131
        go = n0 > size_limit and n1 > size_limit and iteration < iter_limit
        return go, ("split" if go else None)
    if terminate_on == "conf":                                       # :133-178
        if len(energies) > 3:
            e0, e3 = float(energies[0]), float(energies[3])
            if not (e3 > 0.1 or e3 < -0.1):                          # "3rd lowest energy too close to zero"
                return False, "single"
            ratio = e0 / e3
            go = ratio > 1.5 and min(n0, n1) > 5 and iteration < iter_limit
            return go, "single"
        if min(n0, n1) > 5 and iteration < iter_limit:
            return True, "split"
        return False, "single"
    if terminate_on == "once":                                       # :180-187
        return False, "split"
    if terminate_on == "iter_limit":                                 # :189-201
        go = iteration < iter_limit
        return go, ("split" if go else None)
    return False, None


def bqm2_rule(terminate_on, n0, n1, energies, size_limit):
    """``clustering_bqm_2``'s rules (BQM_clustering.py:302-350): ``'color'`` = the deterministic ``100 - color`` /
    ``color - 100`` labels of its ``min_size`` branch.  (The reference indexes ``energy[3]`` unconditionally in the ``conf``
    branch; fewer than four reads end the recursion here instead of raising IndexError.)"""
    if terminate_on == "min_size":
        return (n0 > size_limit and n1 > size_limit), "color"
    if terminate_on == "conf":
        if len(energies) < 4:
            return False, None
        go = abs(float(energies[0]) - float(energies[3])) > 10 and min(n0, n1) > 5
        return go, ("split" if go else None)
    if terminate_on == "once":
        return False, "split"
    return False, None


def _write_labels(G, S0, S1, label, how, color=0):
    if how == "split":
        _label(G, S0, label, random.randint(0, 100))
        _label(G, S1, label, random.randint(120, 220))
    elif how == "single":
        _label(G, list(G.nodes), label, random.randint(0, 100))
    elif how == "color":
        _label(G, S0, label, 100 - color)
        _label(G, S1, label, color - 100)


def clustering_bqm(G, iteration, dirs, solver, gamma_factor, color=0, terminate_on="once", size_limit=40, iter_limit=2,
                   chain_strength=None, sampler=None, structured=True, device_build=None, **sa_kwargs):
    """2-way cut+balance partition (BQM_clustering.py:25-203); returns the SampleSet of this level."""
    smp = _sampler(sampler)
    if structured and _on_device(smp, device_build):
        model = smp.build_on_device("cut_balance", G, gamma_factor=gamma_factor, k=8.0)
    else:
        model = models.cut_balance_model(G, gamma_factor, k=8, structured=structured)
    sa_kwargs.setdefault("num_reads", 500)  # BQM_clustering.py:52
    try:
        response = _sample(smp, model, {"label": str(dirs.get("name", "")) + "_" + str(solver),
                                        "chain_strength": chain_strength}, sa_kwargs)
    finally:
        _close(model)
    S0, S1 = _split(G, response)
    go, how = bqm_rule(terminate_on, len(S0), len(S1), response.record.energy, iteration, size_limit, iter_limit)
    label = "label" + str(iteration)
    if go:
        _write_labels(G, S0, S1, label, "split")     # the reference labels the halves before it recurses
        for part in (S0, S1):
            clustering_bqm(G.subgraph(part), iteration + 1, dirs, solver, gamma_factor, color=color + 20, terminate_on=terminate_on,
                           size_limit=size_limit, iter_limit=iter_limit, chain_strength=chain_strength, sampler=sampler,
                           structured=structured, device_build=device_build, **sa_kwargs)
    if how is not None and not (go and how == "split"):
        _write_labels(G, S0, S1, label, how)
    return response


def clustering_bqm_2(G, iteration, dirs, solver, gamma_factor, color=0, terminate_on="once", size_limit=40, k=1,
                     chain_strength=None, sampler=None, device_build=None, **sa_kwargs):
    """2-way cut + linear gamma with the reference's recursion (BQM_clustering.py:206-350)."""
    if terminate_on not in ("min_size", "conf", "once"):
        raise NotImplementedError(f"clustering_bqm_2 has no terminate_on={terminate_on!r} branch (BQM_clustering.py:302-350)")
    smp = _sampler(sampler)
    if _on_device(smp, device_build):
        model = smp.build_on_device("cut_linear", G, gamma_factor=gamma_factor, k=k)
    else:
        model = models.cut_linear_model(G, gamma_factor, k)
    sa_kwargs.setdefault("num_reads", 5000)  # BQM_clustering.py:240
    try:
        response = _sample(smp, model, {"label": str(dirs.get("name", "")) + "_" + str(solver)}, sa_kwargs)
    finally:
        _close(model)
    S0, S1 = _split(G, response)
    go, how = bqm2_rule(terminate_on, len(S0), len(S1), response.record.energy, size_limit)
    _write_labels(G, S0, S1, "label" + str(iteration), how, color)
    if go:
        for part in (S0, S1):
            clustering_bqm_2(G.subgraph(part), iteration + 1, dirs, solver, gamma_factor, color=color + 20, terminate_on=terminate_on,
                             size_limit=size_limit, k=k, chain_strength=chain_strength, sampler=sampler, device_build=device_build,
                             **sa_kwargs)
    return response


def clustering_bqm_3(G, iteration, dirs, solver, gamma_factor, color=0, terminate_on="once", size_limit=40, sampler=None,
                     **sa_kwargs):
    """2-way cut + size window as a slack penalty, sampled with ``sampler.sample(bqm)`` (BQM_clustering.py:353-426)."""
    bqm = models.cut_inequality_bqm(G, gamma_factor, size_limit, k=8)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        response = _sampler(sampler).sample(bqm, sorted=True, max_iter=1, qpu_reads=100, tabu_timeout=200, **sa_kwargs)
    S0, S1 = _split(G, response)
    label = "label" + str(iteration)
    _label(G, S0, label, random.randint(0, 100))
    _label(G, S1, label, random.randint(120, 220))
    return response


def clustering_dqm(G, num_of_clusters, gamma, sampler=None, penalty=None, semantics="as_written", structured=True,
                   device_build=None, **sa_kwargs):
    """k-way DQM clustering (DQM_clustering.py:24-47): returns a SampleSet of case indices per cell."""
    smp = _sampler(sampler)
    if structured and _on_device(smp, device_build):
        model = smp.build_on_device("dqm", G, num_of_clusters=num_of_clusters, gamma=gamma, penalty=penalty, semantics=semantics)
    else:
        model = models.dqm_model(G, num_of_clusters, gamma, penalty=penalty, semantics=semantics, structured=structured)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)
            return smp.sample_dqm(model, label="DQM - scRAN-seq", **sa_kwargs)
    finally:
        _close(model)


def _cqm(G, num_of_clusters, sampler, onehot_penalty, size_penalty, min_size, subindex, device_build, sa_kwargs,
         size_lowering="slack"):
    smp = _sampler(sampler)
    if _on_device(smp, device_build):
        model = smp.build_on_device("cqm", G, num_of_clusters=num_of_clusters, min_size=min_size, onehot_penalty=onehot_penalty,
                                    size_penalty=size_penalty, subindex=subindex, size_lowering=size_lowering)
    else:
        model = models.cqm_model(G, num_of_clusters, min_size, onehot_penalty, size_penalty, subindex=subindex,
                                 size_lowering=size_lowering)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)
            return smp.sample_cqm(model, label="CQM - scRAN-seq", **sa_kwargs)
    finally:
        _close(model)


def clustering_cqm(G, num_of_clusters, sampler=None, onehot_penalty=None, size_penalty=None, min_size=20, device_build=None,
                   size_lowering="slack", **sa_kwargs):
    """k-way CQM clustering with one-hot and minimum-size constraints (CQM_clustering.py:25-55).  ``size_lowering``:
    'slack' (slack-bit equality penalty) or 'interval' (B * max(0, min_size - N_j)^2, no slack bits; models.cqm_model)."""
    return _cqm(G, num_of_clusters, sampler, onehot_penalty, size_penalty, min_size, None, device_build, sa_kwargs,
                size_lowering)


def clustering_cqm_2(G, num_of_clusters, sampler=None, onehot_penalty=None, size_penalty=None, min_size=20, device_build=None,
                     size_lowering="slack", **sa_kwargs):
    """As ``clustering_cqm`` but variables are named by the node attribute ``subindex`` (CQM_clustering.py:57-91)."""
    sub = [G.nodes[i]["subindex"] for i in G.nodes]
    return _cqm(G, num_of_clusters, sampler, onehot_penalty, size_penalty, min_size, sub, device_build, sa_kwargs,
                size_lowering)


def graph_subsampling(G, gamma, solver="hybrid", sampler=None, device_build=None, **sa_kwargs):
    """Pruning QUBO (QA_subsampling.py:24-97): labels nodes ``label1`` in {0, 1} and returns the SampleSet."""
    smp = _sampler(sampler)
    model = smp.build_on_device("subsampling", G, gamma=gamma) if _on_device(smp, device_build) else models.subsampling_model(G, gamma)
    sa_kwargs.setdefault("num_reads", 100)  # QA_subsampling.py:37
    try:
        response = _sample(smp, model, {"label": "prun_data", "chain_strength": 4}, sa_kwargs)
    finally:
        _close(model)
    S0, S1 = _split(G, response)
    _label(G, S0, "label1", 0)
    _label(G, S1, "label1", 1)
    return response


def disconnected_components(G):
    """``other_tools.disconnected_components`` (other_tools.py:71-86): ``subindex`` / ``valid`` node attributes."""
    import networkx as nx

    comps = list(nx.connected_components(G))
    lengths = [len(c) for c in sorted(comps, key=len, reverse=True)]
    S = [G.subgraph(c).copy() for c in comps]
    for s in S:
        if len(s.nodes()) > 15:
            for subindex, n in enumerate(s.nodes()):
                G.nodes[n]["subindex"] = subindex
                G.nodes[n]["valid"] = 1
        else:
            for n in s.nodes():
                G.nodes[n]["valid"] = 0
    return G, S, lengths


def recursive_bipartition_batched(G, gamma_factor, k=8.0, size_limit=40, iter_limit=2, num_reads=64, num_sweeps=200,
                                  beta_range=None, seed=None, context=None, model="cut_balance", terminate_on="min_size",
                                  write_labels=False):
    """Level-synchronous form of the recursion in ``clustering_bqm`` / ``clustering_bqm_2`` (BQM_clustering.py:113-203,
    302-350): instead of one sampler call per sub-graph, ALL sub-graphs of a recursion level are extracted, built and annealed
    on the device as one batch of independent problems in a single launch (the launch behind QA_subsampling's config 4).

    Per level: ``qa_graph_split`` cuts the root graph into the level's sub-graphs on the device (``G.subgraph`` semantics: the
    parent's node and edge order), ``qa_build_cut_balance`` builds each one's structured model (k * cut + gamma * s(s - n) with
    the balance term as a rank-1 group -- ``model="cut_balance"``; ``qa_build_cut_linear``: the sparse ``clustering_bqm_2`` model --
    ``model="cut_linear"``), ``qa_model_concat`` joins them and ``qa_sa_sample_model_batch`` anneals ``num_reads`` reads of
    every problem, each with the beta schedule of ITS OWN default range unless ``beta_range`` is given.  Initial states and
    per-read seeds are those a separate ``sampler.sample(model, seed=seed, num_reads=...)`` call per sub-graph would use, so
    the tree equals the one ``clustering_bqm(..., sampler=B200SimulatedAnnealingSampler(), seed=seed)`` builds call by call
    (tests/test_gpu_recursion.py).  Every termination rule of the reference is applied through ``bqm_rule`` / ``bqm2_rule``:
    ``terminate_on`` in 'min_size', 'conf', 'once', 'iter_limit'.

    Returns ``({node: leaf index}, levels, level_energies)``: ``levels[i]`` lists the node lists annealed at level i,
    ``level_energies[i]`` their best energies.  ``write_labels=True`` also writes the reference's ``label<level>`` node
    attributes (random colours) into ``G``."""
    from . import schedule
    from .engine import Context

    if model not in ("cut_balance", "cut_linear"):
        raise ValueError("model must be 'cut_balance' or 'cut_linear'")
    own_ctx = context is None
    ctx = Context(0) if own_ctx else context
    try:
        labels, eu, ev, w = models.graph_arrays(G)
        n_root = len(labels)
        root = (n_root, eu.astype(np.int32), ev.astype(np.int32), w)
        base_seed = schedule.resolve_seed(seed)
        frontier = [np.arange(n_root, dtype=np.int64)]
        leaves, levels, level_energies = [], [], []
        iteration = 0
        while frontier:
            levels.append([[labels[i] for i in part] for part in frontier])
            P = len(frontier)
            part_of = np.full(n_root, -1, dtype=np.int32)
            for p, part in enumerate(frontier):
                part_of[part] = p
            dg = ctx.split_graph(root, part_of, P)
            gms, offsets = [], []
            try:
                for p in range(P):
                    if model == "cut_balance":
                        gm, off, _ = ctx.build_cut_balance(dg.device_graph(p), gamma_factor, k)
                    else:
                        gm, off, _ = ctx.build_cut_linear(dg.device_graph(p), gamma_factor, k)
                    gms.append(gm)
                    offsets.append(off)
                if beta_range is None:   # every problem the default range of its own vectors, as separate sampler calls would
                    sched = [schedule.make_beta_schedule(schedule.default_ising_beta_range(*gm.get_ising(), None), num_sweeps, 1,
                                                         "geometric") for gm in gms]
                    betas, spb = np.stack([b for b, _ in sched]), sched[0][1]
                else:
                    betas, spb = schedule.make_beta_schedule(beta_range, num_sweeps, 1, "geometric")
                sizes = [gm.num_variables for gm in gms]
                states = np.concatenate([schedule.random_spin_states(num_reads, nv, base_seed).ravel() for nv in sizes])
                seeds = np.tile(schedule.per_read_seeds(base_seed, num_reads), P)
                bm = ctx.concat_models(gms)
                try:
                    e, _, done = ctx.sample_model_batch(bm, num_reads, states, betas, spb, seeds)
                finally:
                    bm.close()
                assert done == num_reads
            finally:
                for gm in gms:
                    gm.close()
                dg.close()
            nxt, best = [], []
            off = 0
            for p, part in enumerate(frontier):
                nv = sizes[p]
                rows = states[off:off + num_reads * nv].reshape(num_reads, nv)
                off += num_reads * nv
                ep = e[p * num_reads:(p + 1) * num_reads] + offsets[p]
                b = int(np.argmin(ep))          # first minimum == SampleSet.first of an energy-sorted, stable record
                best.append(float(ep[b]))
                S0, S1 = part[rows[b] < 0], part[rows[b] > 0]          # x = 0 / x = 1
                if model == "cut_balance":
                    go, how = bqm_rule(terminate_on, len(S0), len(S1), np.sort(ep, kind="stable"), iteration, size_limit, iter_limit)
                    # the reference's conf branch labels the halves, recurses, then overwrites the level with one colour
                    shown = "split" if (go and terminate_on != "conf") else how
                else:
                    go, how = bqm2_rule(terminate_on, len(S0), len(S1), np.sort(ep, kind="stable"), size_limit)
                    shown = how
                if write_labels and shown is not None:
                    sub = G.subgraph([labels[i] for i in part])
                    _write_labels(sub, [labels[i] for i in S0], [labels[i] for i in S1], "label" + str(iteration), shown, 20 * iteration)
                if go:
                    nxt.extend(x for x in (S0, S1) if len(x))
                elif how in ("split", "color"):
                    leaves.extend(x for x in (S0, S1) if len(x))
                else:
                    leaves.append(part)
            level_energies.append(best)
            frontier = nxt
            iteration += 1
        out = {labels[i]: idx for idx, part in enumerate(leaves) for i in part}
        return out, levels, level_energies
    finally:
        if own_ctx:
            ctx.close()
