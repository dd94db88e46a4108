#!/usr/bin/env python
"""bench.py -- env-steps/s of the gym-auv step path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this framework
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port)

Workload (BASELINE.json configs[2]): MovingObstacles, 65536 envs per GPU x 180 rays x
32 obstacles (16 moving vessel pentagons + 16 static polygonised circles), paths shared
from a bank of 1024 random curves, random actions, auto-reset on (non-test mode).
One "step" = one full env.step() for every env of the batch (obstacle update, RKF45
vessel step, path projection / navigation, 180-ray LiDAR with reference culling,
reward, done, auto-reset).

Prints ONE JSON line (rank 0).  `value` = whole-job env-steps/s with actions resident
in HBM; `e2e` = the same through auv_step_host with host buffers (H2D actions, D2H
obs/reward/done inside the timed region).  `--dump-outputs DIR` also writes what the last
timed step returned as DIR/<name>.npy (see dump_outputs): the inputs depend only on the
arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (180-ray LiDAR, whole box)"
UNIT = "env-steps/s"
WORKLOAD = "MovingObstacles 65536 envs/GPU x 180 rays x 32 obstacles (16 moving + 16 static), 1024-path bank"

# algorithmic bytes per env-step of the fused step, SURVEY.md section 8(d), FP64 state build:
#   read : state 48 + action 8 + aux 40 + path tables ~ 3 x 64 + moving 16 x 40 + static 16 x 24
#   write: state 48 + aux 40 + moving 16 x 40 + obs 186 x 4 + reward/done/info 14
ALGO_BYTES_PER_ENV_STEP = (48 + 8 + 40 + 192 + 16 * 40 + 16 * 24) + (48 + 40 + 16 * 40 + 186 * 4 + 14)
FLOP_PER_SEG_TEST = 16  # SURVEY.md section 8(d)
FLOP_PER_RAY = 60


DENSE_RANGE = 1500.0  # --dense: a sensor range that covers the whole 800 m scenario area


def workload_config(args, use_lidar=True):
    """`config` of the JSON line: what names the workload -- identical for this arm and for `--impl reference`."""
    R = args.rays if use_lidar else 0
    dense = bool(getattr(args, "dense", False))
    default = (args.workload == "moving" and args.envs == 65536 and args.rays == 180 and args.n_moving == 16
               and args.n_static == 16 and not dense)
    name = WORKLOAD if default else (
        f"{args.workload}: {args.envs} envs/GPU x {R} rays x {args.n_moving}+{args.n_static} obstacles"
        + (f" + {args.n_polygons} shared land polygons" if args.workload == "land" else "")
        + (f", DENSE: sensor range {DENSE_RANGE:.0f} m, every obstacle slot is a record at every step" if dense else ""))
    return {"workload": name, "envs_per_gpu": args.envs, "rays": R, "obstacles": args.n_moving + args.n_static,
            "paths": args.n_paths, "auto_reset": True,
            "scenarios": "a fresh scenario of the MovingObstacles distribution for every episode" if args.workload == "moving"
            else "fixed pool, replayed on reset",
            "l2": "the per-step working set (state, records, observations, path tables) exceeds the 126 MB L2; no explicit flush"}


def n_ranges(n, chunks):
    """env ranges auv_step_chunked cuts n envs into (range size = ceil(n/chunks) rounded up to 64)."""
    if chunks <= 1:
        return 1
    cs = -(-(-(-n // chunks)) // 256) * 256
    return -(-n // cs)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--n-moving", type=int, default=16)
    ap.add_argument("--n-static", type=int, default=16)
    ap.add_argument("--n-paths", type=int, default=1024)
    ap.add_argument("--rays", type=int, default=180)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--workload", default="moving", choices=["moving", "land", "pathfollow"],
                    help="moving = BASELINE config 3 (headline); land = config 4 shape (shared world of "
                         "--n-polygons static land polygons); pathfollow = config 2 (no LiDAR, PathFollowRewarder)")
    ap.add_argument("--n-polygons", type=int, default=512)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="do not pin the process to the CPU cores local to its GPU (NVML affinity)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-sample-envs", type=int, default=8)
    ap.add_argument("--cpu-sample-steps", type=int, default=400)
    ap.add_argument("--chunks", type=int, default=2,
                    help="env ranges per step on the pipeline's own streams (auv_step_chunked); 1 = single stream")
    ap.add_argument("--chunk-streams", type=int, default=None)
    ap.add_argument("--host-transfer", default="auto", choices=["auto", "delta", "compact", "dense"],
                    help="how the e2e leg delivers observations to host memory (auto: measures delta and compact, "
                         "the faster one is e2e.value, the other is listed under e2e.other)")
    ap.add_argument("--dense", action="store_true",
                    help="stress line: sensor range 1500 m, so all obstacle slots are nearby and cast against at every step")
    ap.add_argument("--e2e-groups", type=int, nargs="+", default=[4],
                    help="env groups of the e2e leg (each value is measured; the fastest run is e2e.value)")
    ap.add_argument("--delta-gran", type=int, default=16, help="floats per chunk of the delta transfer (8, 16, 32)")
    ap.add_argument("--host-threads", type=int, default=None, help="host threads of auv_compact_expand (default: min(16, cores))")
    ap.add_argument("--host-chunks", type=int, default=4,
                    help="env ranges of the host-buffer step (auv_step_host_chunked): D2H of a range overlaps the next")
    ap.add_argument("--gpu-scenarios", action="store_true", help="(default; kept for old command lines)")
    ap.add_argument("--host-scenarios", action="store_true",
                    help="sample vessel starts and obstacles with the host generator once (pool of N scenarios, replayed "
                         "on reset) instead of the default: GPU generator, pool of 2N, a fresh scenario per episode")
    ap.add_argument("--host-paths", action="store_true",
                    help="build the path bank with SciPy on the host (~14 s for 1024 paths) instead of auv_pathbank_build")
    ap.add_argument("--refresh-every", type=int, default=8,
                    help="steps between auv_refresh_finished calls (fresh scenarios for the envs that finished)")
    ap.add_argument("--preroll-steps", type=int, default=2000,
                    help="untimed steps before the timed region (steady state: vessels spread along their paths, "
                         "episodes desynchronised); also gives the clock sampler its samples under load")
    ap.add_argument("--scenario-cache", default=None,
                    help="pickle the generated scenario set here / reuse it (tuning sweeps; same seeds => same set)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what AUVVecEnv.step returned in the last timed step as DIR/<name>.npy (rank 0, float32), "
                         "to compare two builds output for output; see dump_outputs")
    return ap.parse_args()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": float(max(mx)) if mx else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def build_workload(args, rank):
    import pickle

    cache = getattr(args, "scenario_cache", None)
    if cache:
        cache = (f"{cache}.{args.workload}.{args.envs}.{args.rays}.{args.n_moving}.{args.n_static}.{args.n_paths}."
                 f"{args.seed}.{rank}.{int(bool(getattr(args, 'host_scenarios', False)))}{int(bool(getattr(args, 'host_paths', False)))}"
                 f"{int(bool(getattr(args, 'dense', False)))}")
        if os.path.exists(cache):
            with open(cache, "rb") as f:
                return pickle.load(f)
    out = _build_workload(args, rank)
    if cache:
        with open(cache, "wb") as f:
            pickle.dump(out, f, protocol=4)
    return out


def _build_workload(args, rank):
    from gym_auv_b200 import scenarios as S
    from gym_auv_b200.config import Config

    cfg = Config()
    if getattr(args, "workload", "moving") == "pathfollow":
        return cfg, S.path_follow_no_obstacles(args.envs, seed=args.seed + 1000 * rank, n_paths=args.n_paths)
    cfg.vessel.use_lidar = True
    per_sector = args.rays // cfg.vessel.n_sectors
    if per_sector * cfg.vessel.n_sectors != args.rays:
        cfg.vessel.n_sectors = 8
        per_sector = args.rays // 8
    cfg.vessel.n_sensors_per_sector = per_sector
    if getattr(args, "dense", False):
        cfg.vessel.sensor_range = DENSE_RANGE
    if getattr(args, "workload", "moving") == "land":
        scn = S.land_scenarios(args.envs, n_polygons=args.n_polygons, n_moving=args.n_moving, n_static=args.n_static,
                               seed=args.seed + 1000 * rank, n_paths=args.n_paths)
    elif not getattr(args, "host_scenarios", False):
        # pool of 2N slots, path-major within N: env e alternates between slots e and e + N
        # the path bank is built on the GPU as well (auv_pathbank_build) unless --host-paths asks for SciPy
        scn = S.moving_obstacles_template(2 * args.envs, args.n_moving, args.n_static, seed=args.seed + 1000 * rank,
                                          n_paths=args.n_paths, path_period=args.envs,
                                          device_paths=not getattr(args, "host_paths", False))
    else:
        scn = S.moving_obstacles(args.envs, args.n_moving, args.n_static, seed=args.seed + 1000 * rank,
                                 n_paths=args.n_paths)
    return cfg, scn


# --------------------------------------------------------------------------------------
# CPU arm: the oracle port (restated reference; Shapely/GEOS not installable)
# --------------------------------------------------------------------------------------
def _cpu_worker(job):
    descs, cfgd, actions, warmup = job
    from oracle.sim import OracleEnv

    envs = [OracleEnv(d, cfgd, test_mode=False) for d in descs]
    T = actions.shape[0]
    t0 = None
    n = 0
    for t in range(T):
        if t == warmup:
            t0 = time.perf_counter()
        for i, env in enumerate(envs):
            _, _, done, _ = env.step(actions[t, i])
            if done:
                env.reset()
            if t >= warmup:
                n += 1
    return n, time.perf_counter() - t0


def cpu_baseline(args, cfg, scn, n_envs, steps, warmup, procs):
    """env-steps/s of the oracle port on `procs` host processes (each its own envs)."""
    import multiprocessing as mp
    from tests._parity import oracle_cfg

    cfgd = oracle_cfg(cfg)
    rng = np.random.RandomState(123)
    per = max(1, n_envs // procs)
    jobs = []
    for p in range(procs):
        ids = [(p * per + i) % scn.n_scenarios for i in range(per)]
        acts = rng.uniform([-1, -0.15], [1, 0.15], size=(steps + warmup, per, 2))
        jobs.append(([scn.describe(i) for i in ids], cfgd, acts, warmup))
    if procs == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    total = sum(r[0] for r in res)
    tmax = max(r[1] for r in res)
    return total / tmax, total, tmax


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    small = argparse.Namespace(**vars(args))
    small.envs = max(cores * 16, 64)  # seconds of work per process per step, not milliseconds
    small.n_paths = min(args.n_paths, 64)  # (SciPy builds each path in ~14 ms: untimed set-up)
    small.host_scenarios = True
    cfg, scn = build_workload(small, 0)
    per_step_envs = small.envs
    val, total, tmax = cpu_baseline(args, cfg, scn, per_step_envs, args.steps, args.warmup, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tmax / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "sample": f"{per_step_envs} envs per step on {cores} processes (a bounded sample of the workload's scenario distribution)",
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{total} env-steps ({per_step_envs} envs x {args.steps} steps on {cores} processes), "
                                   "oracle/sim.py FP64 restatement (Shapely/GEOS not installable)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def kernel_times(kms):
    """kms[K][3] = the three intervals of auv_step_timed per step (ms): k_vessel_nav, k_nav_cull, k_lidar.  (A library
    whose timer still brackets the navigation pair as one interval reports ~0 in the first: the pair is then kept whole.)"""
    kms = np.asarray(kms, dtype=np.float64)
    mmm = lambda v: [float(v.min()), float(np.median(v)), float(v.max())]
    pair = kms[:, 0] + kms[:, 1]
    out = {"k_lidar": float(kms[:, 2].mean()), "nav_pair": float(pair.mean()),
           "k_lidar_min_med_max": mmm(kms[:, 2]), "nav_pair_min_med_max": mmm(pair)}
    if kms[:, 0].mean() > 0.02 * pair.mean():
        out.update({"k_vessel_nav": float(kms[:, 0].mean()), "k_nav_cull": float(kms[:, 1].mean())})
    else:
        out.update({"k_vessel_nav": float(pair.mean()), "k_nav_cull": None})
    return out


def roofline_block(N, R, obs_dim, step_ms, kernel_ms, records_per_step, seg_tests_per_step, k_moving, k_static,
                   refresh_interval, table_tracks, fp32_peak_tflops, workload):
    """The `roofline` object of the JSON line: every step kernel with its algorithmic bytes (DESIGN.md section 5) against
    the measured HBM peak, k_lidar also with the SURVEY 8(d) FLOP count against the FP32 FMA probe; the headline fields
    are those of the DOMINANT kernel = the single launch with the longest duration in the steady state."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    flops_per_launch = FLOP_PER_SEG_TEST * seg_tests_per_step + FLOP_PER_RAY * R * N
    lidar_tflops = flops_per_launch / (kernel_ms["k_lidar"] * 1e-3) / 1e12
    # Algorithmic bytes per launch, steady state, per env:
    #   k_vessel_nav: reads state 48 + action 8 + counters / ids 44 + the path's header line 64 + the winning polyline
    #     segment 48, writes state 48 + counters 16 + the arclength 8.
    #   k_nav_cull: reads state 48 + ids 20 + header 64 + 2 PCHIP piece records 2 x 96 + its obstacle records' sources
    #     (64 B per nearby moving slot, 32 B per nearby static slot; all slots once per refresh interval), writes the
    #     navigation record 192 + obs[0..5] 24 + its obstacle records (80 B each).
    #   k_lidar: reads the hand-over line 128 and its obstacle records (80 B each), writes the closeness part of obs
    #     4 * (obs_dim - 6), reward / done / info 15, counters 20.
    rec_per_env = records_per_step / N
    slot_bytes = (k_moving * 64 + k_static * 32) / max(refresh_interval, 1) + rec_per_env * 48
    if table_tracks:
        slot_bytes += k_moving * (80 + 40)  # table-driven tracks: per-env obstacle state read + written every step
    split = kernel_ms.get("k_nav_cull") is not None
    nav_bytes = N * (48 + 8 + 44 + 64 + 48 + 48 + 16 + 8)
    cull_bytes = N * (48 + 20 + 64 + 192 + slot_bytes + 192 + 24) + 80.0 * records_per_step
    kbytes = {"k_vessel_nav": nav_bytes if split else nav_bytes + cull_bytes,
              "k_lidar": N * (128 + 4 * (obs_dim - 6) + 15 + 20) + 80.0 * records_per_step}
    if split:
        kbytes["k_nav_cull"] = cull_bytes
    traffic = {}
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture (profiles/)
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        if workload == "moving" and N == tr["envs"] and R == tr["rays"]:
            traffic = {k: tr[k]["dram_bytes_per_launch"] for k in kbytes if k in tr}
            if not split and "k_nav_cull" in tr:
                traffic["k_vessel_nav"] = tr["k_vessel_nav"]["dram_bytes_per_launch"] + tr["k_nav_cull"]["dram_bytes_per_launch"]
    except Exception:
        pass
    kernels = {}
    for k, nbytes in kbytes.items():
        gbs = nbytes / (kernel_ms[k] * 1e-3) / 1e9
        kernels[k] = {"ms_per_launch": kernel_ms[k], "algo_bytes_per_launch": nbytes, "hbm_gbs": gbs,
                      "hbm_frac": gbs / hbm_peak, "traffic": traffic.get(k)}
    kernels["k_lidar"].update({"fp32_tflops": lidar_tflops, "fp32_peak_tflops": fp32_peak_tflops,
                               "fp32_frac": lidar_tflops / fp32_peak_tflops if fp32_peak_tflops else None,
                               "seg_tests_per_env_step": seg_tests_per_step / N})
    dominant = max(kernels, key=lambda k: kernels[k]["ms_per_launch"])
    step_gbs = ALGO_BYTES_PER_ENV_STEP * N / (step_ms * 1e-3) / 1e9
    if dominant != "k_lidar":
        roof = {"kernel": dominant if split else "k_vessel_nav + k_nav_cull", "bound": "hbm",
                "achieved": kernels[dominant]["hbm_gbs"], "peak": hbm_peak,
                "unit": "GB/s", "frac": kernels[dominant]["hbm_frac"], "traffic": kernels[dominant]["traffic"],
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"}
    else:  # SURVEY 8(d): lidar_cast is bound by the FP32 pipe / instruction issue, not by tensor cores or HBM
        roof = {"kernel": dominant, "bound": "fp32", "achieved": lidar_tflops, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                "frac": kernels[dominant]["fp32_frac"], "traffic": kernels[dominant]["traffic"],
                "peak_source": "FP32 FMA probe measured in this run (no FP32 peak in MEASURED_PEAKS.json)"}
    roof.update({
        "ms_per_launch": kernels[dominant]["ms_per_launch"],
        "algo_bytes_per_launch": kernels[dominant]["algo_bytes_per_launch"],
        "records_per_env_step": rec_per_env,
        "kernels": kernels,
        "kernel_ms": kernel_ms,
        "note": "dominant kernel = the single launch with the longest duration in the STEADY STATE (CUDA events around "
                "every kernel of a single-stream run of K steps, auv_step_timed).  k_vessel_nav / k_nav_cull: algorithmic "
                "bytes against the measured HBM peak; k_lidar: SURVEY 8(d) FLOPs (16 x reference-semantics ray/segment "
                "tests + 60 x rays) against an FP32 FMA probe; ncu pipe / issue numbers of all three: profiles/.",
        "step_hbm_view": {"achieved": step_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": step_gbs / hbm_peak,
                          "algo_bytes_per_env_step": ALGO_BYTES_PER_ENV_STEP,
                          "note": "whole step (all kernels), SURVEY 8(d) bytes per env-step / timed-region time per step"},
    })
    return roof


DUMP_BYTES = 60 << 20  # array data of --dump-outputs; with the .npy headers the directory stays under 64 MB


def dump_outputs(out_dir, step_result):
    """Write the (obs, reward, done, info) tuple of AUVVecEnv.step as out_dir/<name>.npy, every array as float32
    (done / collision / reached_goal as 0.0 / 1.0), one row per env.  When all rows exceed DUMP_BYTES, every array
    keeps the same rows: a sorted sample drawn with a fixed seed, so that two runs with the same arguments write the
    same envs."""
    import torch

    obs, reward, done, info = step_result
    arrays = {"obs": obs, "reward": reward, "done": done, **info}
    n = obs.shape[0]
    row_bytes = 4 * sum(a[0].numel() for a in arrays.values())
    keep = min(n, DUMP_BYTES // row_bytes)
    rows = None
    if keep < n:
        rows = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, keep, replace=False))).to(obs.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if rows is not None:
            a = a.index_select(0, rows)
        np.save(os.path.join(out_dir, f"{name}.npy"), a.to(torch.float32).cpu().numpy())
    return keep


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes as C

    import torch
    import torch.distributed as dist
    from gym_auv_b200 import _lib
    from gym_auv_b200.vec_env import AUVVecEnv

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback on the product path)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    from gym_auv_b200.sharding import bind_to_gpu_numa

    numa_cores = bind_to_gpu_numa(local_rank) if not args.no_numa_bind else ()
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _lib.load()

    t_setup = time.perf_counter()
    cfg, scn = build_workload(args, rank)
    N, K, Wm = args.envs, args.steps, max(args.warmup, 3)
    R = cfg.vessel.n_sensors
    fresh = args.workload == "moving" and not args.host_scenarios  # a fresh GPU-generated scenario per episode
    # host threads of the compact-transfer expansion: the cores this rank may use, shared by the ranks of the box
    cores_here = len(os.sched_getaffinity(0))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    host_threads = args.host_threads or max(1, min(16, cores_here // max(local_world, 1)))
    env = AUVVecEnv(scn, N, cfg, device=device, test_mode=False, auto_reset=True, env_offset=0,
                    chunks=args.chunks, chunk_streams=args.chunk_streams, host_chunks=args.host_chunks,
                    host_threads=host_threads, delta_gran=args.delta_gran,
                    host_transfer=None if args.host_transfer == "auto" else args.host_transfer)
    seed = args.seed + 1000 * rank
    scenario_gen = {"where": "host", "scenarios": scn.n_scenarios}
    if fresh:
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        env.regenerate_scenarios(seed=seed, epoch=1)
        g1.record()
        torch.cuda.synchronize()
        scenario_gen = {"where": "gpu", "scenarios": scn.n_scenarios, "ms_incl_reset_cache": g0.elapsed_time(g1),
                        "per_episode": "every finished env gets a freshly generated scenario "
                                       "(auv_refresh_finished every %d steps, inside the timed region)" % args.refresh_every}
    gen = torch.Generator(device=device)
    gen.manual_seed(1234 + rank)
    lo = torch.tensor([-1.0, -0.15], device=device)
    hi = torch.tensor([1.0, 0.15], device=device)
    n_act = 16
    actions = [lo + (hi - lo) * torch.rand((N, 2), device=device, generator=gen) for _ in range(n_act)]
    env.reset()
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_no = [0]
    last_step = [None]  # what the latest AUVVecEnv.step returned (views of the env's output buffers)

    def run_steps(k):
        """k steps through the public API (AUVVecEnv.step), scenario refresh included"""
        for _ in range(k):
            i = step_no[0]
            last_step[0] = env.step(actions[i % n_act])
            if fresh and i % args.refresh_every == args.refresh_every - 1:
                env.refresh_finished_device(seed=seed)
            step_no[0] = i + 1

    stream = torch.cuda.current_stream(device)

    def timed(k):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record(stream)
        run_steps(k)
        b.record(stream)
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up, then the phase right after reset() as a side note (every vessel still at its path
    #      start, nearby lists refreshed in lock-step: the favourable phase)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    run_steps(Wm)
    after_reset_ms = timed(K) / K
    # ---- pre-roll into the steady state: vessels spread along their paths, episodes desynchronised,
    #      auto-reset and scenario refresh running.  The clock sampler (nvidia-smi every 100 ms) gets its
    #      samples under exactly this load.
    run_steps(max(0, args.preroll_steps - step_no[0]))
    barrier()
    env._out["stats"].zero_()
    env.total_steps = 0
    # ---- timed region: K steps of the steady state through AUVVecEnv.step
    ms_max = timed(K)
    value = world * N * K / (ms_max * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    stats_timed = env.episode_stats(reduce=True)  # the only collective on the path (NCCL all-reduce)
    dones_per_step = stats_timed["episodes"] / max(K, 1) / world
    steady_records = float(env._scratch["rec_cnt"].sum().item()) / N
    cross_track = float(env._st["nav"][:, 2].abs().mean().item())
    dumped_rows = None
    if args.dump_outputs and rank == 0:  # before the legs below step the env again
        dumped_rows = dump_outputs(args.dump_outputs, last_step[0])

    # ---- per-kernel attribution: K more steps of the same steady state on ONE stream with CUDA events
    #      around each kernel (auv_step_timed); these are the launch durations the roofline uses
    cfgp, rays, paths, pool, batch = env._refs()
    sp = C.c_void_p(stream.cuda_stream)
    timer = env.lib.auv_timer_create(K)
    assert timer, "auv_timer_create failed"
    torch.cuda.synchronize()
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0.record(stream)
    for i in range(K):
        a = actions[(step_no[0] + i) % n_act]
        _lib.check(env.lib.auv_step_timed(cfgp, rays, paths, pool, batch, C.c_void_p(a.data_ptr()), C.byref(env.out),
                                          sp, timer, i), "auv_step_timed")
    es1.record(stream)
    torch.cuda.synchronize()
    step_no[0] += K
    serial_ms_per_step = es0.elapsed_time(es1) / K
    kms = np.zeros((K, 3), dtype=np.float32)
    for i in range(K):
        _lib.check(env.lib.auv_timer_read(timer, i, kms[i].ctypes.data_as(C.POINTER(C.c_float))), "auv_timer_read")
    env.lib.auv_timer_destroy(timer)
    kernel_ms = kernel_times(kms)
    kernel_ms["single_stream_ms_per_step"] = serial_ms_per_step

    # ---- counting pass (untimed): K more steps with the seg-test counter on
    seg = torch.zeros(1, dtype=torch.int64, device=device)
    env.out.seg_tests = seg.data_ptr()
    recs = torch.zeros(1, dtype=torch.int64, device=device)
    for i in range(K):
        env.step(actions[(step_no[0] + i) % n_act])
        recs += env._scratch["rec_cnt"].sum()
    torch.cuda.synchronize()
    step_no[0] += K
    env.out.seg_tests = None
    seg_tests_per_step = float(seg.item()) / K
    records_per_step = float(recs.item()) / K  # obstacle records k_vessel_nav hands to k_lidar

    # ---- FP32 FMA peak probe (roofline denominator for the LiDAR kernel), measured live
    sink = torch.zeros(1, device=device)
    fl = C.c_double(0)
    blocks = 148 * 8
    for _ in range(2):
        env.lib.auv_fma_probe(C.c_void_p(sink.data_ptr()), blocks, 256, 1 << 15, C.c_void_p(stream.cuda_stream), C.byref(fl))
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    env.lib.auv_fma_probe(C.c_void_p(sink.data_ptr()), blocks, 256, 1 << 15, C.c_void_p(stream.cuda_stream), C.byref(fl))
    p1.record(stream)
    torch.cuda.synchronize()
    fp32_peak_tflops = fl.value / (p0.elapsed_time(p1) * 1e-3) / 1e12

    # ---- e2e through the host-buffer C ABI call
    e2e = None
    if not args.no_e2e:
        acts_np = [a.cpu().numpy() for a in actions[:4]]
        for i in range(2):
            env.step_host(acts_np[i % 4])
        barrier()
        ke = max(3, min(K, 20))
        t0 = time.perf_counter()
        for i in range(ke):
            env.step_host(acts_np[i % 4])
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t_e = torch.tensor([dt], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        # what the link alone would need for the DENSE rows: a D2H copy of obs, reward, done with no kernels
        probe = torch.empty(env._out["obs"].shape, dtype=torch.float32).pin_memory()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        c0.record(stream)
        for _ in range(10):
            probe.copy_(env._out["obs"], non_blocking=True)
        c1.record(stream)
        torch.cuda.synchronize()
        d2h_ms = c0.elapsed_time(c1) / 10
        dense_bytes = N * (env.obs_dim * 4 + 4 + 1)
        del probe
        e2e_ms = 1e3 * float(t_e.item()) / ke
        e2e = {"value": world * N * ke / float(t_e.item()), "unit": UNIT,
               "h2d_bytes_per_step": env.h2d_bytes_per_step * world,
               "d2h_bytes_per_step": env.d2h_bytes_per_step * world, "steps": ke, "ms_per_step": e2e_ms,
               "host_chunks": env.host_chunks, "host_transfer": env.host_transfer, "host_threads": env.host_threads,
               "dense_d2h_bytes_per_step": dense_bytes * world,
               "pcie": {"dense_d2h_only_ms_per_step": d2h_ms, "d2h_gbs": dense_bytes / (d2h_ms * 1e-3) / 1e9,
                        "note": "rank-0 link: time of a plain D2H copy of the dense [N, obs_dim] rows alone (what bounded "
                                "the host-buffer step before the compact transfer)"}}

    # ---- e2e, asynchronous interface: two env groups of N/2 stepped alternately with
    #      step_async / step_wait (stable-baselines' VecEnv interface) so that one group's
    #      observations travel while the other group is computed.  Same env count, same host
    #      buffers, every step's actions come from host memory and every observation lands there.
    def async_e2e(mode, n_groups):
        ring = env.ring(n_groups, host_transfer=mode, delta_gran=args.delta_gran, host_chunks=1)
        G, part = len(ring), ring.envs_per_group  # G envs of N/G sharing this env's device tables
        ring.reset()
        ah = [[a[g * part:(g + 1) * part].copy() for a in acts_np] for g in range(G)]
        count = [0] * G

        def turn_around(g):  # what the consumer does with a finished group: (refresh its vacated scenarios,) next step
            count[g] += 1
            if fresh and count[g] % args.refresh_every == 0:
                with torch.cuda.stream(ring.groups[g]._async_stream):  # ordered after the group's step on its own stream
                    ring.groups[g].refresh_finished_device(seed=seed + 17)
            ring.send(g, ah[g][count[g] % 4])

        for g in range(G):
            ring.send(g, ah[g][0])
        for _ in range(3 * G):  # warm-up (graph capture happens here)
            turn_around(ring.recv()[0])
        ring.drain()
        for g in range(G):  # warm-up of the refresh path (creates its worker batch)
            with torch.cuda.stream(ring.groups[g]._async_stream):
                ring.groups[g].refresh_finished_device(seed=seed + 17)
            ring.groups[g].d2h_bytes_per_step  # (delta transfer: start the byte count at the timed region)
        torch.cuda.synchronize()
        barrier()
        w0 = sum(g.wait_seconds for g in ring.groups)
        x0 = sum(g.expand_seconds for g in ring.groups)
        t0 = time.perf_counter()
        for g in range(G):
            ring.send(g, ah[g][0])
        for _ in range(ke * G):
            turn_around(ring.recv()[0])
        ring.drain()
        dt = time.perf_counter() - t0
        t_a = torch.tensor([dt], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_a, op=dist.ReduceOp.MAX)
        a_ms = 1e3 * float(t_a.item()) / (ke + 1)
        res = {"value": world * G * part * (ke + 1) / float(t_a.item()), "ms_per_step": a_ms, "steps": ke + 1,
               "host_transfer": mode + (f"/{args.delta_gran * 4}B" if mode == "delta" else ""), "groups": G,
               "d2h_bytes_per_step": sum(g.d2h_bytes_per_step for g in ring.groups) * world,
               "host_expand_ms_per_step": 1e3 * (sum(g.expand_seconds for g in ring.groups) - x0) / (ke + 1),
               "host_threads": ring.groups[0].host_threads if mode == "compact" else 0,
               "host_blocked_ms_per_step": 1e3 * (sum(g.wait_seconds for g in ring.groups) - w0) / (ke + 1)}
        torch.cuda.synchronize()
        ring.close()
        return res

    if e2e is not None and N >= 128:
        modes = ["delta", "compact"] if args.host_transfer == "auto" else [args.host_transfer]
        if "compact" in modes and args.host_transfer == "auto" and (
                not cfg.vessel.use_lidar or cfg.vessel.sensor_use_velocity_observations):
            modes.remove("compact")
        runs = [async_e2e(m, g) for m in modes for g in args.e2e_groups]
        runs.sort(key=lambda r: -r["value"])
        sync_part = {"value": e2e["value"], "ms_per_step": e2e["ms_per_step"], "host_chunks": e2e["host_chunks"],
                     "host_transfer": env.host_transfer, "call": "AUVVecEnv.step_host (one synchronous call per step)"}
        e2e.update(runs[0])
        e2e.update({"mode": "EnvGroupRing.recv / send over G groups of N/G envs (AUVVecEnv.step_async / step_wait per group)"
                            + (", fresh scenario per episode" if fresh else ""),
                    "sync": sync_part, "other": runs[1:]})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    print(f"[bench] value={value:.4g} ms/step={ms_max / K:.4f} after_reset_ms={after_reset_ms:.4f} kernel_ms={kernel_ms} "
          f"setup_s={setup_s:.1f} e2e={e2e}", file=sys.stderr)
    roof = roofline_block(N=N, R=R if cfg.vessel.use_lidar else 0, obs_dim=env.obs_dim, step_ms=ms_max / K, kernel_ms=kernel_ms,
                          records_per_step=records_per_step, seg_tests_per_step=seg_tests_per_step, k_moving=env.k_moving,
                          k_static=env.k_static, refresh_interval=cfg.vessel.sensor_interval_load_obstacles,
                          table_tracks=env.linear is None, fp32_peak_tflops=fp32_peak_tflops, workload=args.workload)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 ray casting on f64 state/culling", "data": "synthetic",
        "config": workload_config(args, bool(cfg.vessel.use_lidar)),
        "run": {"phase": "steady state: %d steps after reset(), auto-reset running, timed through AUVVecEnv.step" % (step_no[0] - 3 * K),
                "dones_per_step": dones_per_step, "records_per_env_step": steady_records,
                "mean_abs_cross_track_m": cross_track, "chunks": env.chunks, "chunk_streams": getattr(env, "chunk_streams", 1),
                "scenario_generation": scenario_gen, "setup_s": setup_s, "host_cores_bound": len(numa_cores),
                "working_set_mb": {"per_step_state_and_outputs": N * ALGO_BYTES_PER_ENV_STEP / 1e6,
                                   "path_bank": sum(v.numel() * v.element_size() for v in env._bank.values()) / 1e6}},
        "clocks": clocks,
        "after_reset": {"value": world * N / (after_reset_ms * 1e-3), "ms_per_step": after_reset_ms,
                        "note": "side note: the same K steps right after reset() (vessels at their path starts, nearby "
                                "lists refreshed in lock-step) -- NOT the headline"},
        "e2e": e2e,
        # k_vessel_nav + k_nav_cull + k_lidar per env range, 6 kernels + 1 memset per scenario refresh
        "gpu_launches": 3 * K * n_ranges(N, env.chunks) + (7 * (K // args.refresh_every) if fresh else 0),
        "roofline": roof,
        "episode_stats": stats_timed,
    }
    if dumped_rows is not None:
        line["outputs_dumped"] = {"dir": args.dump_outputs, "envs": dumped_rows, "of": N}
    if not args.no_cpu_baseline and world == 1:  # reported on rank 0 at N=1 only
        small = argparse.Namespace(**vars(args))
        small.envs = args.cpu_sample_envs
        small.n_paths = min(args.n_paths, small.envs)
        small.host_scenarios = True
        ccfg, cscn = build_workload(small, 0)
        v, total, tmax = cpu_baseline(args, ccfg, cscn, small.envs, args.cpu_sample_steps, 4, 1)
        line["cpu_baseline"] = {
            "value": v, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{total} env-steps ({small.envs} envs x {args.cpu_sample_steps} steps) of the same workload "
                      "distribution, oracle/sim.py FP64 restatement (Shapely/GEOS not installable), %.1f s" % tmax,
        }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (NCCL's version
    # banner, torchrun children) are diverted to stderr for the whole run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
