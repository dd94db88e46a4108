#!/usr/bin/env python
"""Cost of recording episode tracks (AUVVecEnv(record_tracks=...), AuvStepOut.tracks) on the BASELINE
config 3 shape: N = 65536 envs, a moving_obstacles_template pool of 2N with 16 + 16 obstacle slots,
refresh_finished_device every 8 steps.

Usage: python tools/track_overhead.py [--envs N] [--tracks K] [--capacity T] [--out FILE]

Two envs are built in one process, one with record_tracks = 0 and one with K tracked envs x T steps, on
identical pools.  Each gets 2000 warm-up steps; then 7 windows of 400 steps are timed for each, the two
envs alternating window by window (host clock around work that ends in a device synchronise), and the
median window gives env-steps/s.  Then 100 steps of each are timed per kernel with CUDA events
(auv_step_timed) for the median k_lidar time.  Prints one JSON line with both rates, their ratio, the
k_lidar times and the card's name, power limit and clocks read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gym_auv_b200 import _lib, lidar_config, scenarios as S  # noqa: E402
from gym_auv_b200.vec_env import AUVVecEnv  # noqa: E402
from tools.gen_throughput import card  # noqa: E402


def build(N, tracks, capacity):
    cfg = lidar_config()
    scn = S.moving_obstacles_template(2 * N, 16, 16, seed=0, n_paths=1024, path_period=N)
    env = AUVVecEnv(scn, N, cfg, auto_reset=True, record_tracks=tracks, track_capacity=capacity)
    env.regenerate_scenarios(seed=1, epoch=1)
    env.reset()
    return env


def run(env, acts, steps, t0):
    for i in range(steps):
        env.step(acts[(t0 + i) % len(acts)])
        if (t0 + i) % 8 == 7:
            env.refresh_finished_device(seed=3)
    return t0 + steps


def lidar_ms(env, acts, steps, t0):
    timer = env.lib.auv_timer_create(steps)
    cfg, rays, paths, pool, batch = env._refs()
    stream = env._stream()
    for i in range(steps):
        a = acts[(t0 + i) % len(acts)]
        _lib.check(env.lib.auv_step_timed(cfg, rays, paths, pool, batch, C.c_void_p(a.data_ptr()), C.byref(env.out), stream,
                                          timer, i), "auv_step_timed")
        if (t0 + i) % 8 == 7:
            env.refresh_finished_device(seed=3)
    torch.cuda.synchronize()
    ms, got = (C.c_float * 3)(), []
    for i in range(steps):
        _lib.check(env.lib.auv_timer_read(timer, i, ms), "auv_timer_read")
        got.append(float(ms[2]))
    env.lib.auv_timer_destroy(timer)
    return statistics.median(got), t0 + steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--tracks", type=int, default=256)
    ap.add_argument("--capacity", type=int, default=2048)
    ap.add_argument("--warmup", type=int, default=2000)
    ap.add_argument("--window", type=int, default=400)
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("track_overhead.py measures on a CUDA device; none is visible")
    N = a.envs
    envs = {"off": build(N, 0, a.capacity), "on": build(N, a.tracks, a.capacity)}
    g = torch.Generator(device="cuda").manual_seed(0)
    lo, hi = torch.tensor([-1.0, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    acts = [lo + (hi - lo) * torch.rand((N, 2), device="cuda", generator=g) for _ in range(16)]
    pos = {k: run(e, acts, a.warmup, 0) for k, e in envs.items()}
    torch.cuda.synchronize()
    rates = {k: [] for k in envs}
    for _ in range(a.windows):
        for k, e in envs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pos[k] = run(e, acts, a.window, pos[k])
            torch.cuda.synchronize()
            rates[k].append(N * a.window / (time.perf_counter() - t0))
    lidar = {}
    for k, e in envs.items():
        lidar[k], pos[k] = lidar_ms(e, acts, 100, pos[k])
    on = envs["on"]
    finished = int((on._tracks["head"][:, :, 2] != 0).sum().item())
    res = dict(
        workload="config3_tracks", envs=N, pool=2 * N, k_moving=16, k_static=16, refresh_every=8,
        tracked_envs=a.tracks, track_capacity=a.capacity, warmup_steps=a.warmup, window_steps=a.window, windows=a.windows,
        env_steps_per_s_off=statistics.median(rates["off"]), env_steps_per_s_on=statistics.median(rates["on"]),
        ratio_on_off=statistics.median(rates["on"]) / statistics.median(rates["off"]),
        windows_off=rates["off"], windows_on=rates["on"], k_lidar_ms_off=lidar["off"], k_lidar_ms_on=lidar["on"],
        track_rows_finished=finished,
        track_bytes=int(sum(t.numel() * t.element_size() for t in (on._tracks["points"], on._tracks["head"], on._tracks["snap"]))),
        card=card(),
    )
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
