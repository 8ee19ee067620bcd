"""Close the loop for dwave-samplers' sample options wherever the real library is importable (not in this project's test
environments): tests/native/proposals_sa_ref.cpp restates `randomize_order` and `proposal_acceptance_criteria` from
SURVEY.md Appendix C.8, and every GPU parity claim for them is GPU == that reference.

    python tests/check_proposals_against_dwave_samplers.py   # 0: every case matches bit for bit, 1: a mismatch, 2: absent

For each case of tests/check_against_neal.py and each of {sequential, random order} x {Metropolis, Gibbs} it runs

    dwave.samplers.SimulatedAnnealingSampler().sample(bqm, num_reads=R, num_sweeps=S, beta_range=..., seed=seed,
        beta_schedule_type='geometric', initial_states=..., initial_states_generator='none',
        randomize_order=..., proposal_acceptance_criteria=...)

and the reference in stream-seeding mode (one xorshift128+ stream over all reads, as dwave-samplers seeds), and compares
final states bytewise and energies to the last bit.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
sys.path.insert(0, str(HERE))


def main() -> int:
    try:
        import dimod
        from dwave.samplers import SimulatedAnnealingSampler
    except Exception as e:  # pragma: no cover - depends on the machine
        print(f"SKIP: dimod / dwave.samplers not importable: {e}")
        return 2
    import proposals_reference as pref
    from check_against_neal import cases
    from scrna_seq_qannealing_clustering_b200 import schedule
    sampler = SimulatedAnnealingSampler()
    R, sweeps, seed = 24, 200, 1234
    bad = 0
    for name, model, beta_range in cases():
        n = model.num_variables
        h = {i: float(model.h[i]) for i in range(n)}
        J = {(int(a), int(b)): float(w) for a, b, w in zip(model.starts, model.ends, model.weights)}
        bqm = dimod.BinaryQuadraticModel.from_ising(h, J)
        order = list(range(n))
        ldata, (irow, icol, qdata), _ = bqm.to_numpy_vectors(variable_order=order)
        init = schedule.random_spin_states(R, n, seed)
        betas, spb = schedule.make_beta_schedule(beta_range, sweeps, 1, "geometric")
        for var_order in (pref.SEQUENTIAL, pref.RANDOM):
            for criterion, proposal in (("Metropolis", pref.METROPOLIS), ("Gibbs", pref.GIBBS)):
                ss = sampler.sample(bqm, num_reads=R, num_sweeps=sweeps, beta_range=beta_range, beta_schedule_type="geometric",
                                    seed=seed, initial_states=(init.copy(), order), initial_states_generator="none",
                                    randomize_order=bool(var_order), proposal_acceptance_criteria=criterion)
                cols = [list(ss.variables).index(v) for v in order]
                ref_states = np.asarray(ss.record.sample)[:, cols].astype(np.int8)
                ref_e = np.asarray(ss.record.energy, dtype=np.float64)
                states = init.copy()
                e, _ = pref.sample_ising(np.asarray(ldata, dtype=np.float64), np.asarray(irow, dtype=np.int32),
                                         np.asarray(icol, dtype=np.int32), np.asarray(qdata, dtype=np.float64), states, betas,
                                         spb, np.array([seed], dtype=np.uint64), seed_mode=1, var_order=var_order,
                                         proposal=proposal)
                same_states = np.array_equal(states, ref_states)
                same_e = np.array_equal((e + bqm.offset).view(np.uint64), ref_e.view(np.uint64))
                close_e = np.allclose(e + bqm.offset, ref_e, rtol=1e-12, atol=1e-9)
                ok = same_states and (same_e or close_e)
                bad += not ok
                print(f"{'PASS' if ok else 'FAIL'}  {name} [{'random' if var_order else 'sequential'}, {criterion}]: states "
                      f"{'identical' if same_states else 'DIFFER'}, energies "
                      f"{'bit-identical' if same_e else ('equal to 1e-12' if close_e else 'DIFFER')}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
