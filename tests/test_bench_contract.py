"""bench.py --impl reference runs without a GPU: check the JSON-line contract of the reference arm (same metric / unit / config
keys as the GPU arm prints, real slice time, CPU baseline bookkeeping)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=300,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    import bench
    d = _run(["--impl", "reference", "--steps", "3", "--warmup", "3", "--cpu-seconds", "1.5"])
    assert d["impl"] == "reference"
    assert d["metric"] == bench.WORKLOADS["quadrotor"]["metric"] and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None
    # the same `config` object the GPU arm prints for this workload at N = 1 (VERDICT round 1: same_config)
    assert d["config"] == bench.base_config("quadrotor", 1)
    # each step is one bounded slice of CPU work; ms_per_step is its real duration, not a derived number
    assert 0.2e3 <= d["ms_per_step"] <= 1.5e3, d["ms_per_step"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert set(cb["per_process_steps_per_s"]) == {"min", "median", "max"}
    assert cb["cores"] <= cb["cores_how"]["affinity"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


def test_reference_arm_other_workload_has_its_own_metric():
    import bench
    d = _run(["--impl", "reference", "--workload", "maze3d", "--steps", "3", "--warmup", "3", "--cpu-seconds", "1.5"])
    assert d["metric"] == bench.WORKLOADS["maze3d"]["metric"]
    assert d["config"] == bench.base_config("maze3d", 1)
    assert d["cpu_baseline"]["value"] == d["value"] > 0


def test_dump_outputs_keeps_a_fixed_sample_under_the_budget(tmp_path):
    """--dump-outputs: float32 (float64 kept), and above 64 MB the same seeded env sample on every run."""
    import numpy as np
    import bench
    obs = np.random.RandomState(1).randint(0, 256, (1024, 128, 128, 3)).astype(np.uint8)
    arrays = {"obs": obs, "reward": np.arange(1024, dtype=np.float64), "done": np.arange(1024) % 3 == 0}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(k + s for k in arrays for s in (".npy", "_env_index.npy"))
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 * 10 ** 6
    for n in names:
        assert np.array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n))
    idx = np.load(tmp_path / "a" / "obs_env_index.npy").astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "obs.npy"), obs[idx].astype(np.float32))
    assert np.load(tmp_path / "a" / "reward.npy").dtype == np.float64
    assert np.load(tmp_path / "a" / "done.npy").dtype == np.float32
    small = {"obs": np.ones((64, 19), np.float32), "done": np.zeros(64, np.uint8)}
    bench.dump_outputs(str(tmp_path / "c"), small)
    assert sorted(p.name for p in (tmp_path / "c").iterdir()) == ["done.npy", "obs.npy"]
