#!/usr/bin/env python
"""GPU-side scenario generation throughput (auv_generate_moving_obstacles + reset-cache refill)
and the cost of the ping-pong refresh during stepping.

Usage: python tools/gen_throughput.py [N] [--workload moving|land]

moving (default): MovingObstacles template pool of 2N, host refresh every 10 steps.
land: the BASELINE config 4 shape with a fresh scenario per episode -- N envs, a land_template pool of 2N
      scenarios in one shared world of 512 land polygons, 16 + 16 obstacles.  Prints one JSON line with the
      generation of all 2N scenarios (generator alone and including the reset cache) with the world and for
      the same pool without it, the steady-state env-steps/s through AUVVecEnv.step after 2000 warm-up steps
      (median of 7 windows) with refresh_finished_device every 8 steps and with the fixed pool, and the card's
      name, power limit and clocks read in the same run."""
import argparse
import ctypes as C
import dataclasses
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gym_auv_b200 import _lib, lidar_config, scenarios as S  # noqa: E402
from gym_auv_b200.vec_env import AUVVecEnv  # noqa: E402


def moving(N):
    cfg = lidar_config()
    t0 = time.perf_counter()
    scn = S.moving_obstacles_template(2 * N, 16, 16, seed=0, n_paths=1024)
    t_host = time.perf_counter() - t0
    env = AUVVecEnv(scn, N, cfg, auto_reset=True, chunks=4)
    out = {"envs": N, "pool": 2 * N, "host_path_bank_s": t_host}
    for rep in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        env.regenerate_scenarios(seed=1, epoch=rep + 1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    out["regenerate_all_s"] = dt
    out["scenarios_per_s_incl_reset_cache"] = 2 * N / dt
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = [torch.rand((N, 2), device="cuda", generator=g) * 2 - 1 for _ in range(8)]
    for i in range(20):
        env.step(acts[i % 8])
    env.refresh_finished(seed=3)
    torch.cuda.synchronize()
    K, every = 200, 10
    t0 = time.perf_counter()
    for i in range(K):
        env.step(acts[i % 8])
    torch.cuda.synchronize()
    t_plain = time.perf_counter() - t0
    refreshed = 0
    t0 = time.perf_counter()
    for i in range(K):
        env.step(acts[i % 8])
        if i % every == every - 1:
            refreshed += env.refresh_finished(seed=3)
    torch.cuda.synchronize()
    t_ref = time.perf_counter() - t0
    out.update(steps=K, refresh_every=every, env_steps_per_s_plain=N * K / t_plain, env_steps_per_s_with_refresh=N * K / t_ref,
               scenarios_refreshed=refreshed, refreshed_per_s=refreshed / t_ref)
    return out


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        row = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return dict(name=row[0], power_limit_w=float(row[1]), sm_mhz=float(row[2]), sm_max_mhz=float(row[3]))
    except (OSError, IndexError, ValueError, subprocess.SubprocessError) as e:
        return dict(name=torch.cuda.get_device_name(0), error=f"nvidia-smi: {e}")


def time_generation(env, reps=5):
    """(ms of the generator launches alone, ms including the reset-cache refill) for all pool scenarios,
    medians over `reps` epochs (CUDA events)."""
    M = env.scenarios.n_scenarios
    gen_ms, all_ms = [], []
    for rep in range(reps):
        gp = env.gen_params(1, 100 + rep)
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        _lib.check(env.lib.auv_generate_moving_obstacles(C.byref(gp), C.byref(env.paths), C.byref(env.pool), None, M,
                                                        C.c_void_p(env._scratch["status"].data_ptr()), env._stream()),
                   "auv_generate_moving_obstacles")
        b.record()
        env._build_reset_cache()
        c.record()
        torch.cuda.synchronize()
        gen_ms.append(a.elapsed_time(b))
        all_ms.append(a.elapsed_time(c))
    env.check_status()
    return statistics.median(gen_ms), statistics.median(all_ms)


def steady(env, acts, refresh, warmup=2000, window=400, windows=7, every=8):
    """env-steps/s through AUVVecEnv.step, median over windows after `warmup` steps; with `refresh`
    refresh_finished_device every `every` steps (inside the timed windows)."""
    N = env.num_envs
    step = [0]

    def run(k):
        for _ in range(k):
            i = step[0]
            env.step(acts[i % len(acts)])
            if refresh and i % every == every - 1:
                env.refresh_finished_device(seed=5)
            step[0] = i + 1

    env.reset()
    run(warmup)
    torch.cuda.synchronize()
    rates, recs, dones = [], [], []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ep0 = env._out["stats"][0].item()
        a.record()
        run(window)
        b.record()
        torch.cuda.synchronize()
        rates.append(N * window / (a.elapsed_time(b) * 1e-3))
        dones.append((env._out["stats"][0].item() - ep0) / window)
        recs.append(float(env._scratch["rec_cnt"].float().mean()))
    env.check_status()
    return dict(env_steps_per_s=statistics.median(rates), window_rates=rates, records_per_env_step=statistics.mean(recs),
                dones_per_step=statistics.mean(dones))


def query_stats(env, g, sample=200000, seed=0):
    """What the land query of the generator (auv_generate.cuh: land_clear) does per call, counted on the host for a
    sample of the objects the world pool holds (accepted draws; rejected candidates are not in the pool): grid
    cells visited, polygons whose enclosing circle is tested, rings walked and vertices on those rings."""
    import numpy as np

    M = g.n_scenarios
    pts = np.concatenate([g.vessel_init[:, :2], g.mov_start.reshape(-1, 2), g.st_pos.reshape(-1, 2)])
    d = np.concatenate([np.full(M, S.LAND_CLEARANCE), g.mov_width.ravel(), g.st_radius.ravel()])
    pick = np.random.RandomState(seed).choice(len(pts), size=min(sample, len(pts)), replace=False)
    pts, d = pts[pick], d[pick]
    w = env.scenarios.world
    grid = env._pool["world_grid"]
    off, items, nx, ny, cell = grid["off"], grid["items"], grid["nx"], grid["ny"], grid["cell"]
    fx0, fx1 = np.floor((pts[:, 0] - d - grid["x0"]) / cell), np.floor((pts[:, 0] + d - grid["x0"]) / cell)
    fy0, fy1 = np.floor((pts[:, 1] - d - grid["y0"]) / cell), np.floor((pts[:, 1] + d - grid["y0"]) / cell)
    on = (fx1 >= 0) & (fy1 >= 0) & (fx0 <= nx - 1) & (fy0 <= ny - 1)
    ix0, ix1 = np.maximum(fx0, 0).astype(int), np.minimum(fx1, nx - 1).astype(int)
    iy0, iy1 = np.maximum(fy0, 0).astype(int), np.minimum(fy1, ny - 1).astype(int)
    cells = np.where(on, (ix1 - ix0 + 1) * (iy1 - iy0 + 1), 0)
    tested = np.zeros(len(pts), np.int64)
    walked = np.zeros(len(pts), np.int64)
    verts = np.zeros(len(pts), np.int64)
    nv = np.diff(w.voff)
    for dy in range(int((iy1 - iy0).max(initial=0)) + 1):
        for dx in range(int((ix1 - ix0).max(initial=0)) + 1):
            sel = np.nonzero(on & (ix0 + dx <= ix1) & (iy0 + dy <= iy1))[0]
            c = (iy0[sel] + dy) * nx + ix0[sel] + dx
            cnt = off[c + 1] - off[c]
            tested[sel] += cnt
            rep = np.repeat(sel, cnt)
            j = items[np.concatenate([np.arange(a, b) for a, b in zip(off[c], off[c + 1])]) if len(sel) else []]
            near = np.hypot(pts[rep, 0] - w.circle[j, 0], pts[rep, 1] - w.circle[j, 1]) <= w.circle[j, 2] + d[rep]
            np.add.at(walked, rep[near], 1)
            np.add.at(verts, rep[near], nv[j[near]] - 1)
    return dict(objects_sampled=len(pts), grid_cell_m=cell, grid_cells=nx * ny,
                polygons_per_nonempty_cell=float(np.diff(off)[np.diff(off) > 0].mean()),
                cells_visited_per_query=float(cells.mean()), circle_tests_per_query=float(tested.mean()),
                rings_walked_per_query=float(walked.mean()), ring_edges_per_query_at_most=float(verts.mean()),
                share_of_queries_walking_a_ring=float((walked > 0).mean()))


def land(N):
    cfg = lidar_config()
    t0 = time.perf_counter()
    scn = S.land_template(2 * N, n_polygons=512, n_moving=16, n_static=16, seed=0, n_paths=1024, path_period=N)
    t_host = time.perf_counter() - t0
    plain = dataclasses.replace(scn, world_polygons=[], _world=None)
    out = {"workload": "land: %d envs, pool of %d generated scenarios, 512 shared land polygons, 16 + 16 obstacles"
           % (N, 2 * N), "envs": N, "pool": 2 * N, "polygons": 512, "host_template_s": t_host}
    gen = {}
    for name, s in (("world", scn), ("no_world", plain)):
        env = AUVVecEnv(s, N, cfg, auto_reset=True)
        g_ms, all_ms = time_generation(env)
        gen[name] = dict(generator_ms=g_ms, ms_incl_reset_cache=all_ms, scenarios_per_s_incl_reset_cache=2 * N / (all_ms * 1e-3))
        pulled = env.pull_scenarios()  # both pools end on the same seed and epoch
        if name == "world":
            gen["land_query"] = query_stats(env, pulled)
            world_pool = pulled
        else:  # objects whose draw in the world differs from the world-less one: redrawn because of land
            for k in ("vessel_init", "mov_start", "st_pos"):
                a, b = getattr(world_pool, k), getattr(pulled, k)
                gen["land_query"][f"{k}_redrawn_share"] = float((a != b).any(axis=-1).mean())
        del env
        torch.cuda.empty_cache()
    gen["world_over_no_world_incl_reset_cache"] = gen["world"]["ms_incl_reset_cache"] / gen["no_world"]["ms_incl_reset_cache"]
    gen["world_over_no_world_generator"] = gen["world"]["generator_ms"] / gen["no_world"]["generator_ms"]
    out["generation"] = gen
    g = torch.Generator(device="cuda").manual_seed(0)
    lo, hi = torch.tensor([-1.0, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    acts = [lo + (hi - lo) * torch.rand((N, 2), device="cuda", generator=g) for _ in range(16)]
    runs = {}
    for name, refresh in (("device_refresh_every_8", True), ("fixed_pool", False)):
        env = AUVVecEnv(scn, N, cfg, auto_reset=True)
        env.regenerate_scenarios(seed=1, epoch=1)
        runs[name] = steady(env, acts, refresh)
        del env
        torch.cuda.empty_cache()
    out["steady_state"] = dict(warmup_steps=2000, window_steps=400, windows=7, statistic="median", **runs)
    out["records_per_env_step"] = runs["device_refresh_every_8"]["records_per_env_step"]
    out["dones_per_step"] = runs["device_refresh_every_8"]["dones_per_step"]
    out["card"] = card()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("N", nargs="?", type=int, default=65536, help="envs (the pool holds 2 N scenarios)")
    ap.add_argument("--workload", default="moving", choices=["moving", "land"])
    args = ap.parse_args()
    print(json.dumps(land(args.N) if args.workload == "land" else moving(args.N)))


if __name__ == "__main__":
    main()
