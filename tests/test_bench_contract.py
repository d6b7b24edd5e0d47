"""bench.py's output contract: the committed GPU line carries every key the driver reads, and the reference arm
(`--impl reference`, CPU only: the oracle port on the host cores) runs here and prints the same shape."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "gpu_launches"}


def validate_gpu_line(d, steps=None):
    assert BASE_KEYS <= set(d) and {"roofline", "cpu_baseline", "clocks"} <= set(d)
    assert d["metric"] == "env_steps_per_sec" and d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True
    assert "workload" in d["config"] and d["config"]["games_per_gpu"] == 65536 and "model" not in d["config"]
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(d["value"] - 65536 * 256 * d["steps"] / (d["ms_per_step"] * d["steps"] / 1e3)) / d["value"] < 1e-6
    c = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] in ("port", "reference") and c["cores"] == 1
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    assert d["gpu_launches"] == d["steps"] and (steps is None or d["steps"] == steps)
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_committed_gpu_line_has_the_contract_keys():
    d = json.loads(open(os.path.join(ROOT, "profiles", "r02j_bench.json")).read().strip().splitlines()[-1])
    validate_gpu_line(d)
    assert d["clocks"]["samples"] >= 10                     # NVML sampler: tens of samples inside a 70 ms timed region
    assert d["cpu_baseline"]["kind"] == "reference"         # the unmodified Python reference ran on the GPU box's host


@pytest.mark.gpu
def test_fresh_gpu_line_has_the_contract_keys():
    """the line bench.py prints NOW, on this GPU (not a committed one)"""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "4", "--warmup", "3", "--no-extra"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    validate_gpu_line(d, steps=4)
    assert d["value"] > 1e9                                 # the north_star's bar, with a wide margin below the measured 4.9e9
    assert d["config"] == __import__("bench").workload_config(65536)


def load_dump(d):
    import numpy as np
    s = np.load(os.path.join(d, "state.npy"))
    assert s.dtype == np.float64 and s.shape[0] == 8 and s.shape[2] == 2
    words = s[..., 0].astype(np.uint64) | (s[..., 1].astype(np.uint64) << np.uint64(32))
    return words, np.load(os.path.join(d, "wins.npy")), np.load(os.path.join(d, "game_index.npy")).astype(np.int64)


def test_dump_outputs_is_exact_and_samples_under_the_byte_cap(tmp_path, monkeypatch):
    import numpy as np
    import oracle as orc
    sys.path.insert(0, ROOT)
    import bench
    st, wins, _ = orc.step_random(orc.start_states(3000), bench.SEED, 0, 64, nthreads=4)
    bench.dump_outputs(str(tmp_path / "all"), st, wins)
    words, w, idx = load_dump(str(tmp_path / "all"))
    assert np.array_equal(words, st) and np.array_equal(idx, np.arange(3000)) and np.array_equal(w, wins.astype(np.float64))
    monkeypatch.setattr(bench, "DUMP_BYTES", 200 * 1024)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), st, wins)
        assert sum(os.path.getsize(str(tmp_path / d / f)) for f in os.listdir(str(tmp_path / d))) <= 200 * 1024
    words, _, idx = load_dump(str(tmp_path / "a"))
    assert 1000 < len(idx) < 3000 and np.array_equal(words, st[:, idx])
    assert np.array_equal(idx, load_dump(str(tmp_path / "b"))[2])      # the sample is fixed


@pytest.mark.gpu
def test_dumped_outputs_are_the_state_after_the_timed_steps(tmp_path):
    """--dump-outputs: the env state after warm-up + timed steps, the oracle replays it bit for bit (first 2,048 games; the
    words the env step maintains, 0-4)"""
    import numpy as np
    import oracle as orc
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-extra", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["gpu_launches"] == 2
    words, wins, idx = load_dump(str(tmp_path))
    assert words.shape == (8, 65536) and np.array_equal(idx, np.arange(65536))
    sys.path.insert(0, ROOT)
    import bench
    k = 2048
    ost, owins, _ = orc.step_random(orc.start_states(k), bench.SEED, 0, (d["warmup"] + d["steps"]) * bench.PLIES_PER_STEP, nthreads=8)
    assert np.array_equal(words[:5, :k], ost[:5])
    assert wins.shape == (2,) and (wins >= owins).all()


def run_reference(env_extra):
    env = dict(os.environ, **env_extra)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                        "--no-extra"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=300)
    assert p.returncode == 0, p.stderr
    return p.stdout.strip()


def test_reference_arm_runs_on_cpu_and_only_rank0_prints():
    out = run_reference({"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"})
    d = json.loads(out.splitlines()[-1])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d) and d["metric"] == "env_steps_per_sec" and d["value"] > 0
    import refrun
    # the unmodified reference when its staged copy exists (build container, GPU box), else the C port of the same loop
    assert d["cpu_baseline"]["kind"] == ("reference" if refrun.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(bench.GAMES_PER_GPU)          # the same dict the GPU arm prints (same_config)
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
    assert run_reference({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == ""
