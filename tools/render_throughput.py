#!/usr/bin/env python
"""Cost of rendering frames (AUVVecEnv.render, kernel k_render) on the BASELINE config 3 shape: N = 65536 envs, a
moving_obstacles_template pool of 2N with 16 + 16 obstacle slots, refresh_finished_device every 8 steps.

Usage: python tools/render_throughput.py [--envs N] [--out FILE]

After 2000 warm-up steps:
  * the time of one render call (CUDA events around it, median of 20 calls after 3 warm-up calls) for K = 1, 16 and
    256 frames at 400 x 400 and for 16 frames at 1024 x 1024, of envs spread evenly over the batch;
  * the step rate with one 16-frame 400 x 400 render every 100 steps against none: 7 windows of 400 steps each,
    the two regimes alternating window by window (host clock around work that ends in a device synchronise),
    median window.
Prints one JSON line with both, and the card's name, power limit and clocks read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gym_auv_b200 import lidar_config, scenarios as S  # noqa: E402
from gym_auv_b200.vec_env import AUVVecEnv  # noqa: E402
from tools.gen_throughput import card  # noqa: E402


def run(env, acts, steps, t0, render_every=0, ids=None):
    for i in range(steps):
        env.step(acts[(t0 + i) % len(acts)])
        if (t0 + i) % 8 == 7:
            env.refresh_finished_device(seed=3)
        if render_every and (t0 + i) % render_every == render_every - 1:
            env.render(ids, width=400, height=400)
    return t0 + steps


def render_ms(env, ids, width, height, reps=20):
    for _ in range(3):
        env.render(ids, width=width, height=height)
    got = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        env.render(ids, width=width, height=height)
        b.record()
        b.synchronize()
        got.append(a.elapsed_time(b))
    return statistics.median(got)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--warmup", type=int, default=2000)
    ap.add_argument("--window", type=int, default=400)
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("render_throughput.py measures on a CUDA device; none is visible")
    N = a.envs
    cfg = lidar_config()
    scn = S.moving_obstacles_template(2 * N, 16, 16, seed=0, n_paths=1024, path_period=N)
    env = AUVVecEnv(scn, N, cfg, auto_reset=True)
    env.regenerate_scenarios(seed=1, epoch=1)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    lo, hi = torch.tensor([-1.0, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    acts = [lo + (hi - lo) * torch.rand((N, 2), device="cuda", generator=g) for _ in range(16)]
    pos = run(env, acts, a.warmup, 0)
    torch.cuda.synchronize()
    spread = lambda k: [int(i) * (N // k) for i in range(k)]
    calls = {}
    for k, w, h in ((1, 400, 400), (16, 400, 400), (256, 400, 400), (16, 1024, 1024)):
        calls[f"k{k}_{w}x{h}_ms"] = render_ms(env, spread(k), w, h)
    ids16 = spread(16)
    rates = {"off": [], "on": []}
    for _ in range(a.windows):
        for mode in ("off", "on"):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pos = run(env, acts, a.window, pos, render_every=100 if mode == "on" else 0, ids=ids16)
            torch.cuda.synchronize()
            rates[mode].append(N * a.window / (time.perf_counter() - t0))
    off, on = statistics.median(rates["off"]), statistics.median(rates["on"])
    res = dict(
        workload="config3_render", envs=N, pool=2 * N, k_moving=16, k_static=16, refresh_every=8, warmup_steps=a.warmup,
        render_ms=calls, render_every=100, render_frames=16, render_size=[400, 400], window_steps=a.window,
        windows=a.windows, env_steps_per_s_off=off, env_steps_per_s_on=on, ratio_on_off=on / off,
        windows_off=rates["off"], windows_on=rates["on"], card=card(),
    )
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
