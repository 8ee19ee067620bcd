"""The bench line's contract (driver-facing keys) checked on the committed final lines of the round, and the byte accounting
of SURVEY.md 8(d) on a hand-computed case."""
import json
from pathlib import Path

import pytest

import bench

PROFILES = Path(__file__).resolve().parents[1] / "profiles"


@pytest.mark.parametrize("name,n_gpus", [("r2_bench_final_n1.json", 1), ("r2_bench_final_n2.json", 2)])
def test_committed_bench_lines_carry_the_contract_keys(name, n_gpus):
    line = json.loads((PROFILES / name).read_text().strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["metric"] == "spin_flip_attempts_per_sec" and line["unit"] == "attempts/s" and line["higher_is_better"] is True
    assert line["n_gpus"] == n_gpus and line["scaling"] == "weak" and line["vs_baseline"] is None and line["dtype"] == "f64"
    assert "workload" in line["config"] and "config3" in line["config"]["workload"]
    assert line["gpu_launches"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert line["e2e"]["h2d_bytes_per_step"] > 9e9 and line["e2e"]["d2h_bytes_per_step"] > 9e9      # the state matrices cross PCIe
    assert line["e2e"]["value"] < line["value"]
    r = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"])
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"]) and line["clocks"]["reasons"] == []
    if n_gpus == 1:
        c = line["cpu_baseline"]
        assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] == "port"
        assert c["parity_check"]["final_states_identical_to_gpu"] and c["parity_check"]["energies_bitwise_identical_to_gpu"]
        job = line["full_job"]
        assert job["reads"] == 100000 and job["num_sweeps"] == 1000 and job["feasible_fraction"] == 1.0
        assert job["cpu_arm"]["final_states_identical_to_gpu"] and job["cpu_arm"]["energies_bitwise_identical_to_gpu"]
        c5 = line["config5"]
        assert c5["roofline"]["bound"] == "tensor" and 0.5 < c5["roofline"]["frac"] < 1.0
        assert c5["cpu_arm"]["final_states_identical_to_gpu"] and c5["cpu_arm"]["max_rel_energy_diff"] < 1e-9
    else:
        assert line["strong"]["reads"] == 100000 and line["strong"]["reads_per_rank"] == 50000


def test_steps_must_be_positive(monkeypatch):
    monkeypatch.setattr("sys.argv", ["bench.py", "--steps", "2", "--warmup", "0"])
    assert bench.parse_args().steps == 2
    monkeypatch.setattr("sys.argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args()


@pytest.mark.parametrize("state_budget", [None, 3 * (4 * 50 + 8)])
def test_dump_outputs_writes_float_arrays_of_a_fixed_sample(tmp_path, monkeypatch, state_budget):
    import numpy as np
    import torch
    if state_budget is not None:      # force the sampled form: 3 rows of states, 7 energies
        monkeypatch.setattr(bench, "DUMP_STATE_BYTES", state_budget)
        monkeypatch.setattr(bench, "DUMP_ENERGY_BYTES", 7 * 16)
    R, n = 20, 50
    g = torch.Generator().manual_seed(0)
    states = (torch.randint(0, 2, (R, n), dtype=torch.int8, generator=g) * 2 - 1)
    energies = torch.randn(R, dtype=torch.float64, generator=g)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, states, energies, seed=1234)
    files = {p.name: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert set(files) == {"energies.npy", "energy_reads.npy", "states.npy", "state_reads.npy"}
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    e_idx, s_idx = files["energy_reads.npy"], files["state_reads.npy"]
    assert len(e_idx) == (R if state_budget is None else 7) and len(s_idx) == (R if state_budget is None else 3)
    assert np.array_equal(files["energies.npy"], energies.numpy()[e_idx.astype(int)])
    assert np.array_equal(files["states.npy"], states.numpy()[s_idx.astype(int)].astype(np.float32))
    for name, a in files.items():      # same arguments, same sample and bytes
        assert np.array_equal(a, np.load(tmp_path / "b" / name))
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 << 20


def test_algorithmic_bytes_follow_survey_8d():
    # 10 attempts, 3 accepted flips with 7 neighbour updates in total, 40 directed entries per read and sweep, 1 sweep of 2 reads,
    # rows shared by 2 reads: 8*10 + 9*3 + 17*7 + 12*40*(10/5)/2 with num_variables = 5
    stats = {"attempts": 10, "accepted": 3, "nbr_updates": 7, "num_variables": 5}
    assert bench.algorithmic_bytes(stats, 40.0, 2) == 8 * 10 + 9 * 3 + 17 * 7 + 12 * 40 * 2 / 2
    assert bench.field_layout_bytes(stats) == 8.25 * 10 + 16 * 7
