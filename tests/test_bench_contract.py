"""CPU: the shape of bench.py's one JSON line -- the reference arm run for real on a small workload, and the last
committed device line under profiles/ (the device arm itself needs a GPU) -- and its --dump-outputs files."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def _check_common(line):
    assert BASE_KEYS <= set(line), BASE_KEYS - set(line)
    assert line["metric"] == "leapfrog_grad_evals_per_sec" and line["unit"] == "grad-evals/s"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["data"] == "synthetic"
    assert isinstance(line["config"], dict) and "workload" in line["config"] and "model" not in line["config"]
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])


def test_reference_arm_prints_exactly_one_json_line():
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c3",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    _check_common(line)
    assert line["impl"] == "reference"
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "NUTS transition" in cb["sample"]
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0 == line["e2e"]["d2h_bytes_per_step"]


def test_reference_arm_other_ranks_exit_without_work():
    env = dict(os.environ, PYTHONPATH=ROOT, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_committed_device_line_has_the_contract_keys():
    with open(os.path.join(ROOT, "profiles", "r01_bench_default_v9_skip.json")) as f:
        line = json.loads(f.read())
    _check_common(line)
    assert line["n_gpus"] == 1 and line["warmup"] >= 3 and line["gpu_launches"] > 0 and line["scaling"] == "weak"
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"])
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(line["clocks"]["reasons"])
    r = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] in ("hbm", "tensor")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
    cb = line["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] in ("port", "reference")
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["e2e"]["value"] != line["value"]          # measured separately, not a copy of the device-timed value


def test_committed_round2_lines_have_the_contract_keys():
    """the one-GPU line and the 8-GPU strong-scaling line of round 2 (profiles/), as the driver would parse them"""
    with open(os.path.join(ROOT, "profiles", "r02_bench_default_v6.json")) as f:
        one = json.loads(f.read())
    with open(os.path.join(ROOT, "profiles", "r02_bench_c4_n8_strong_v2.json")) as f:
        eight = json.loads(f.read())
    for line in (one, eight):
        _check_common(line)
        assert line["scaling"] == "strong" and line["gpu_launches"] > 0 and "workload" in line["config"] and "run" in line
        assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(line["clocks"]["reasons"])
        r = line["roofline"]
        assert r["bound"] == "tensor" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
        assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert one["config"] == eight["config"]                       # the same workload at every N (strong scaling)
    assert one["n_gpus"] == 1 and eight["n_gpus"] == 8
    assert eight["value"] / one["value"] >= 6.0                   # BASELINE.json north_star: >= 6x at 8 GPUs
    par = eight["parity"]
    assert par["obs_sharded_logp_rel_err"] < 1e-6 and par["obs_sharded_grad_normwise_err"] < 1e-6
    assert par["merged_draws_bit_equal_across_ranks"] is True
    assert par["peer_vs_allreduce_first_draw"]["chains_agreeing_within_1e-2_sd"] > 0.98
    assert par["peer_vs_allreduce_grad_evals"][0] == par["peer_vs_allreduce_grad_evals"][1]
    # pointwise workloads report the FP32-issue bound, with the HBM figure alongside; C1 carries the single-chain drop-in
    for name in ("c2", "c1", "c5"):
        ro = one["other_workloads"][name]["roofline"]
        assert ro["bound"] == "fp32" and 0 < ro["frac"] < 1 and ro["hbm"]["frac"] < 0.1
    assert one["other_workloads"]["c1"]["single_chain_drop_in"]["grad_evals_per_s"] > 0
    assert len(one["other_workloads"]["c1"]["chain_sweep"]) >= 5
    full = one["cpu_baseline"]["full_length"]
    assert set(full) == {"c1", "c2", "c5"} and all("min_ess_per_s" in v for v in full.values())
    assert one["ess"]["draws"] >= 500 and one["ess"]["warmup"] > 0 and one["ess"]["wall_s"] > 0


def test_strong_scaling_is_refused_for_pointwise_workloads():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--scaling", "strong", "--impl", "reference"],
                         capture_output=True, text=True, timeout=120, env=dict(os.environ, PYTHONPATH=ROOT), cwd=ROOT)
    assert out.returncode != 0 and "observation sharding" in (out.stderr + out.stdout)


def test_dump_outputs_keeps_a_fixed_sample_of_chains_within_the_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    draws = torch.arange(4 * 4096 * 32, dtype=torch.float32).reshape(4, 4096, 32)         # 2 MB: twice the budget
    depths = torch.randint(0, 10, (4, 4096), dtype=torch.int32, generator=torch.Generator().manual_seed(0))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), draws, depths)
    a = {f: np.load(tmp_path / "a" / f"{f}.npy") for f in ("draws", "tree_depth")}
    assert sum(os.path.getsize(tmp_path / "a" / f"{f}.npy") for f in a) <= 1 << 20
    assert a["draws"].dtype == a["tree_depth"].dtype == np.float32
    assert np.array_equal(a["tree_depth"], depths.numpy())
    kept = a["draws"][0, :, 0].astype(np.int64) // 32                                      # chain index of each kept row
    assert 1000 < len(kept) < 4096 and np.all(np.diff(kept) > 0)
    assert np.array_equal(a["draws"], draws.numpy()[:, kept])
    for f, v in a.items():
        assert np.array_equal(np.load(tmp_path / "b" / f"{f}.npy"), v)


@pytest.mark.gpu
def test_dump_outputs_are_identical_for_identical_arguments(cuda, tmp_path):
    """--dump-outputs on a small regression run, twice: the timed path starts from the same inputs every time, so the
    draws and tree depths of the last timed step agree bit for bit; --steps is the number of timed steps."""
    import numpy as np
    dumps = []
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c3", "--chains", "256",
                              "--steps", "2", "--warmup", "0", "--no-others", "--no-cpu-baseline", "--no-ess",
                              "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        assert json.loads(out.stdout)["steps"] == 2
        dumps.append({f: np.load(tmp_path / d / f"{f}.npy") for f in ("draws", "tree_depth")})
    a, b = dumps
    assert a["draws"].shape == (16, 256, 100) and a["tree_depth"].shape == (16, 256)
    assert np.isfinite(a["draws"]).all()
    for f in a:
        assert np.array_equal(a[f], b[f]), f
