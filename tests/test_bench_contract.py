"""bench.py contract checks: the reference arm (CPU oracle port) prints exactly one JSON line with the
contract keys, the GPU arm refuses to run without CUDA, the roofline assembly, and --dump-outputs (its
host logic on the CPU, its repeatability on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUTPUT_NAMES = {"obs", "reward", "done", "collision", "reached_goal", "goal_distance", "progress", "terminal_observation"}


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["metric"].startswith("env-steps/sec")


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_cuda():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode != 0 and "no CPU fallback" in (res.stderr + res.stdout)


def test_roofline_block_names_the_longest_single_launch():
    """bench.roofline_block: three step kernels, each with its own CUDA-event interval; the headline roofline is that of
    the single launch with the longest duration (k_lidar -> FP32 roof, a navigation kernel -> HBM roof); a timer that
    brackets the navigation pair as one interval keeps the pair whole.  Pure host logic: no GPU, no oracle."""
    import numpy as np

    import bench

    kms = np.array([[0.052, 0.037, 0.075], [0.054, 0.039, 0.077]], dtype=np.float32)
    t = bench.kernel_times(kms)
    assert abs(t["k_vessel_nav"] - 0.053) < 1e-6 and abs(t["k_nav_cull"] - 0.038) < 1e-6 and abs(t["nav_pair"] - 0.091) < 1e-6
    assert t["k_lidar_min_med_max"][0] <= t["k_lidar"] <= t["k_lidar_min_med_max"][2]
    kw = dict(N=65536, R=180, obs_dim=186, step_ms=0.164, records_per_step=1.4 * 65536, seg_tests_per_step=1200.0 * 65536,
              k_moving=16, k_static=16, refresh_interval=25, table_tracks=False, fp32_peak_tflops=64.0, workload="moving")
    r = bench.roofline_block(kernel_ms=t, **kw)
    assert r["kernel"] == "k_lidar" and r["bound"] == "fp32" and r["unit"] == "TFLOP/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0.2 < r["frac"] < 0.6
    assert set(r["kernels"]) == {"k_vessel_nav", "k_nav_cull", "k_lidar"}
    assert all(k["hbm_frac"] > 0 and k["algo_bytes_per_launch"] > 0 for k in r["kernels"].values())
    assert r["traffic"] is None or r["traffic"] > 0  # profiles/ncu_traffic.json: per launch, like `achieved`
    # the navigation kernel as the longest launch -> HBM roof
    slow = dict(t, k_vessel_nav=0.2, nav_pair=0.238)
    r = bench.roofline_block(kernel_ms=slow, **kw)
    assert r["kernel"] == "k_vessel_nav" and r["bound"] == "hbm" and r["unit"] == "GB/s" and 0 < r["frac"] < 1
    # an older timer: interval 0 ~ 0, interval 1 = the pair
    t2 = bench.kernel_times(np.array([[0.0004, 0.091, 0.075]], dtype=np.float32))
    assert t2["k_nav_cull"] is None and abs(t2["k_vessel_nav"] - 0.0914) < 1e-5
    r = bench.roofline_block(kernel_ms=t2, **kw)
    assert r["kernel"] == "k_vessel_nav + k_nav_cull" and set(r["kernels"]) == {"k_vessel_nav", "k_lidar"}
    assert r["traffic"] is None or r["traffic"] > 5e7
    import json

    json.dumps(r)  # serialisable


def test_dump_outputs_writes_the_step_tuple_as_float32_and_samples_the_same_rows(tmp_path, monkeypatch):
    """bench.dump_outputs: one float32 .npy per array of AUVVecEnv.step's (obs, reward, done, info); above the byte
    budget every array keeps the same seeded sample of env rows.  CPU tensors stand in for the device buffers."""
    torch = pytest.importorskip("torch")
    import bench

    n, d = 1000, 186
    g = torch.Generator().manual_seed(3)
    obs = torch.rand((n, d), generator=g)
    flag = lambda: (torch.rand(n, generator=g) < 0.3).to(torch.uint8)
    info = dict(collision=flag(), reached_goal=flag(), goal_distance=torch.rand(n, generator=g),
                progress=torch.rand(n, generator=g), terminal_observation=torch.rand((n, d), generator=g))
    step = (obs, torch.rand(n, generator=g), flag(), info)

    assert bench.dump_outputs(str(tmp_path / "all"), step) == n
    out = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in OUTPUT_NAMES}
    assert set(os.listdir(tmp_path / "all")) == {f"{k}.npy" for k in OUTPUT_NAMES}
    assert all(a.dtype == np.float32 and a.shape[0] == n for a in out.values())
    assert np.array_equal(out["obs"], obs.numpy()) and np.array_equal(out["done"], step[2].numpy().astype(np.float32))

    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 100 * (2 * d + 6))
    assert bench.dump_outputs(str(tmp_path / "a"), step) == 100
    assert bench.dump_outputs(str(tmp_path / "b"), step) == 100
    a = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in OUTPUT_NAMES}
    b = {k: np.load(tmp_path / "b" / f"{k}.npy") for k in OUTPUT_NAMES}
    assert all(np.array_equal(a[k], b[k]) and a[k].shape[0] == 100 for k in OUTPUT_NAMES)
    rows = np.flatnonzero(np.isin(obs.numpy()[:, 0], a["obs"][:, 0]))  # the sampled env rows, in order
    assert len(rows) == 100
    assert np.array_equal(a["obs"], obs.numpy()[rows]) and np.array_equal(a["progress"], info["progress"].numpy()[rows])
    assert np.array_equal(a["terminal_observation"], info["terminal_observation"].numpy()[rows])


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_with_the_same_arguments(tmp_path):
    """Two bench.py runs with the same arguments time --steps steps and write the same outputs of the last one."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "7", "--warmup", "3", "--envs", "512",
           "--n-paths", "64", "--preroll-steps", "60", "--no-cpu-baseline", "--no-e2e"]
    for run in ("a", "b"):
        res = subprocess.run(cmd + ["--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600,
                             cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        d = json.loads(res.stdout.strip())
        assert d["steps"] == 7 and d["outputs_dumped"] == {"dir": str(tmp_path / run), "envs": 512, "of": 512}
    a = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in OUTPUT_NAMES}
    b = {k: np.load(tmp_path / "b" / f"{k}.npy") for k in OUTPUT_NAMES}
    assert a["obs"].shape == (512, 186) and all(v.dtype == np.float32 for v in a.values())
    assert np.abs(a["obs"]).max() > 0
    for k in OUTPUT_NAMES:
        assert np.array_equal(a[k], b[k]), k
