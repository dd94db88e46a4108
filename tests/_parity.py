"""Shared harness: run the same injected scenarios through the CPU oracle and the CUDA
path and compare.  Tolerances follow BASELINE.json north_star: collision / done /
reached_goal / culling windows / sector indices bit-exact (conditioned on the oracle's
margin to the threshold being above the FP32 error band), vessel state, LiDAR ranges
and rewards within a stated tolerance."""
from __future__ import annotations

import numpy as np

RANGE_RTOL = 1e-4  # LiDAR ranges: |d_gpu - d_ref| <= RANGE_ATOL + RANGE_RTOL * d_ref
RANGE_ATOL = 1e-4
STATE_TOL = 1e-9   # vessel state is integrated in FP64 on the GPU
REWARD_RTOL = 1e-4
REWARD_ATOL = 1e-4
OBS_ATOL = 2e-5    # closeness in [0,1] (FP32 log)
COLLISION_BAND = 2e-4  # |min d - vessel_width| below this: FP32 may legitimately differ


def oracle_cfg(config, **extra):
    v, e, s = config.vessel, config.episode, config.simulation
    d = dict(
        min_cumulative_reward=e.min_cumulative_reward, max_timesteps=e.max_timesteps,
        min_goal_distance=e.min_goal_distance, min_path_progress=e.min_path_progress,
        t_step_size=s.t_step_size, thrust_max_auv=v.thrust_max_auv, moment_max_auv=v.moment_max_auv,
        vessel_width=v.vessel_width, look_ahead_distance=v.look_ahead_distance, use_lidar=v.use_lidar,
        sensor_interval_load_obstacles=v.sensor_interval_load_obstacles,
        n_sensors_per_sector=v.n_sensors_per_sector, n_sectors=v.n_sectors, sensor_range=v.sensor_range,
        sensor_log_transform=v.sensor_log_transform,
        sensor_use_velocity_observations=v.sensor_use_velocity_observations,
    )
    d.update(extra)
    return d


def rollout_oracle(scn, config, actions, test_mode=True, on_step=None, **cfg_extra):
    """actions: [T, M, 2].  Returns dict of arrays [T(+1), M, ...] (stops an env at done).
    on_step(t, m, env), if given, is called after every step with the stepped OracleEnv."""
    from oracle.sim import OracleEnv

    T, M = actions.shape[0], scn.n_scenarios
    R = config.vessel.n_sensors if config.vessel.use_lidar else 0
    D = 6 + R + (2 * R if (R and config.vessel.sensor_use_velocity_observations) else 0)
    out = dict(
        obs0=[], obs=np.full((T, M, D), np.nan), reward=np.full((T, M), np.nan),
        done=np.zeros((T, M), bool), collision=np.zeros((T, M), bool), reached=np.zeros((T, M), bool),
        state=np.full((T, M, 6), np.nan), dists=np.full((T, M, max(R, 1)), np.nan),
        progress=np.full((T, M), np.nan), goal_distance=np.full((T, M), np.nan),
        min_dist=np.full((T, M), np.inf), alive=np.zeros((T, M), bool), s=np.full((T, M), np.nan),
        windows=[[None] * M for _ in range(T)], n_tests=np.zeros(M, np.int64), mov_pos=[[None] * M for _ in range(T)],
    )
    out["slot_of"] = [
        np.concatenate([np.nonzero(scn.mov_width[m] > 0)[0], scn.k_moving + np.nonzero(scn.st_radius[m] > 0)[0],
                        scn.k_moving + scn.k_static + np.arange(len(scn.world_polygons))]).astype(int)
        for m in range(M)
    ]
    for m in range(M):
        env = OracleEnv(scn.describe(m), oracle_cfg(config, **cfg_extra), test_mode=test_mode)
        out["obs0"].append(env.reset())
        for t in range(T):
            obs, rew, done, info = env.step(actions[t, m])
            out["alive"][t, m] = True
            out["obs"][t, m] = obs
            out["reward"][t, m] = rew
            out["done"][t, m] = done
            out["collision"][t, m] = info["collision"]
            out["reached"][t, m] = info["reached_goal"]
            out["state"][t, m] = env.vessel.state
            out["progress"][t, m] = info["progress"]
            out["goal_distance"][t, m] = info["goal_distance"]
            out["s"][t, m] = env.vessel.nav["vessel_arclength"]
            if R:
                out["dists"][t, m] = env.vessel.dists
                out["min_dist"][t, m] = env.vessel.dists.min()
            out["mov_pos"][t][m] = np.array([o.position for o in env.obstacles if not o.static])
            if R and env.vessel.nearby:
                slot = {id(o): j for j, o in enumerate(env.obstacles)}
                out["windows"][t][m] = {slot[id(o)]: w for o, w in zip(env.vessel.nearby, env.vessel.windows)}
            else:
                out["windows"][t][m] = {}
            if on_step is not None:
                on_step(t, m, env)
            if done:
                break
        out["n_tests"][m] = env.vessel.n_tests
    return out


def rollout_gpu(scn, config, actions, test_mode=True, device="cuda:0", cull_mode="reference", **env_kw):
    import torch
    from gym_auv_b200.vec_env import AUVVecEnv

    T, M = actions.shape[0], scn.n_scenarios
    env = AUVVecEnv(scn, M, config, device=device, test_mode=test_mode, auto_reset=False, debug=True,
                    cull_mode=cull_mode, **env_kw)
    obs0 = env.reset().cpu().numpy().copy()
    R = config.vessel.n_sensors if config.vessel.use_lidar else 0
    out = dict(obs0=obs0, obs=[], reward=[], done=[], collision=[], reached=[], state=[], dists=[], progress=[],
               goal_distance=[], s=[], windows=[], mov_pos=[])
    a = torch.as_tensor(actions, dtype=torch.float32, device=device)
    for t in range(T):
        obs, rew, done, info = env.step(a[t])
        out["obs"].append(obs.cpu().numpy().copy())
        out["reward"].append(rew.cpu().numpy().copy())
        out["done"].append(done.cpu().numpy().astype(bool))
        out["collision"].append(info["collision"].cpu().numpy().astype(bool))
        out["reached"].append(info["reached_goal"].cpu().numpy().astype(bool))
        out["state"].append(env.state.cpu().numpy().T.copy())
        out["progress"].append(info["progress"].cpu().numpy().copy())
        out["goal_distance"].append(info["goal_distance"].cpu().numpy().copy())
        out["s"].append(env.get_attr("nav")[:, 0].cpu().numpy().copy())
        if R:
            out["dists"].append(env.get_attr("lidar_dist").cpu().numpy().copy())
        out["windows"].append(env.get_attr("windows").cpu().numpy().copy())
        out["mov_pos"].append(env.get_attr("mov_pos").cpu().numpy().copy())
    for k in ("obs", "reward", "done", "collision", "reached", "state", "dists", "progress", "goal_distance", "s",
              "windows", "mov_pos"):
        if out[k]:
            out[k] = np.stack(out[k])
    out["seg_tests"] = int(env.get_attr("seg_tests").item())
    return out, env


def compare(ref, gpu, config, label=""):
    """Assert parity; returns a small report dict."""
    alive = ref["alive"]
    width = config.vessel.vessel_width
    rep = dict(label=label, env_steps=int(alive.sum()))
    # state (FP64 on both sides)
    ds = np.abs(gpu["state"] - ref["state"])[alive]
    rep["state_max_abs"] = float(ds.max())
    assert ds.max() <= STATE_TOL * max(1.0, float(np.abs(ref["state"][alive]).max())), (label, ds.max())
    # arclength / progress
    d_s = np.abs(gpu["s"] - ref["s"])[alive]
    rep["arclength_max_abs"] = float(d_s.max())
    assert d_s.max() <= 1e-7, (label, "arclength", d_s.max())
    if config.vessel.use_lidar:
        dr, dg = ref["dists"][alive], gpu["dists"][alive]
        err = np.abs(dg - dr)
        tol = RANGE_ATOL + RANGE_RTOL * dr
        rep["range_max_abs"] = float(err.max())
        rep["range_max_rel"] = float((err / np.maximum(dr, 1e-9))[dr > 1e-3].max()) if (dr > 1e-3).any() else 0.0
        bad = err > tol
        assert not bad.any(), (label, "ranges", int(bad.sum()), float(err.max()), np.argwhere(bad)[:5], dr[bad][:5], dg[bad][:5])
    # bit-exact flags, conditioned on margin
    margin = np.abs(ref["min_dist"] - width)
    decisive = alive & (margin > COLLISION_BAND)
    rep["collision_decisive"] = int(decisive.sum())
    rep["collision_skipped_in_band"] = int((alive & ~decisive).sum())
    assert np.array_equal(gpu["collision"][decisive], ref["collision"][decisive]), (label, "collision")
    assert np.array_equal(gpu["reached"][alive], ref["reached"][alive]), (label, "reached_goal")
    assert np.array_equal(gpu["done"][decisive], ref["done"][decisive]), (label, "done")
    # culling windows: bit-exact integers for every nearby obstacle (slots are packed in the
    # same order on both sides when every slot is used)
    if config.vessel.use_lidar and "windows" in gpu and len(gpu["windows"]):
        T, M = alive.shape
        nwin = 0
        for t in range(T):
            for m in range(M):
                if not alive[t, m] or ref["windows"][t][m] is None:
                    continue
                gw = gpu["windows"][t, m]
                for j, (a, b) in ref["windows"][t][m].items():
                    js = ref["slot_of"][m][j] if "slot_of" in ref else j
                    if a < -config.vessel.n_sensors:
                        continue  # IndexError corner: defined as all rays
                    assert (int(gw[js, 0]), int(gw[js, 1])) == (a, b), (label, "window", t, m, j, gw[js], (a, b))
                    nwin += 1
        rep["windows_checked"] = nwin
    # rewards
    rr, rg = ref["reward"][decisive], gpu["reward"][decisive]
    rerr = np.abs(rg - rr)
    rep["reward_max_abs"] = float(rerr.max()) if rerr.size else 0.0
    assert np.all(rerr <= REWARD_ATOL + REWARD_RTOL * np.abs(rr)), (label, "reward", rerr.max())
    # observations
    oerr = np.abs(gpu["obs"] - ref["obs"])[alive]
    rep["obs_max_abs"] = float(oerr.max())
    assert oerr.max() <= max(OBS_ATOL, RANGE_RTOL), (label, "obs", oerr.max())
    return rep


# ---------------------------------------------------------------------------------------
# Oracle replay of LIVE envs of a running batch (the regime bench.py measures)
# ---------------------------------------------------------------------------------------
def _oracle_from_live(scn_host, config, m, state, step_counter, max_progress, t_step, cum_reward, mask_words,
                      mov_pos, mov_disp, mov_counter, **cfg_extra):
    """OracleEnv of pool scenario m put into the given live state (vessel, counters, nearby list,
    moving-obstacle positions / last displacement / waypoint counter)."""
    import math

    from oracle.sim import OracleEnv

    o = OracleEnv(scn_host.describe(m), oracle_cfg(config, **cfg_extra), test_mode=False)
    o.vessel.state = np.array(state, dtype=np.float64)
    o.vessel.step_counter = int(step_counter)
    o.vessel.max_progress = float(max_progress)
    o.t_step = int(t_step)
    o.cumulative_reward = float(cum_reward)
    used_m = np.nonzero(scn_host.mov_width[m] > 0)[0]
    used_s = np.nonzero(scn_host.st_radius[m] > 0)[0]
    slots = list(used_m) + [scn_host.k_moving + j for j in used_s] + [
        scn_host.k_moving + scn_host.k_static + k for k in range(len(scn_host.world_polygons))]
    for ob, j in zip(o.obstacles, slots):
        if not ob.static:
            ob.position = np.array(mov_pos[j], dtype=np.float64)
            ob.dx, ob.dy = float(mov_disp[j][0]), float(mov_disp[j][1])
            ob.heading = math.atan2(ob.dy, ob.dx)
            ob.counter = float(mov_counter[j])
            ob._rebuild()
    bits = np.asarray(mask_words).astype(np.uint32)
    o.vessel.nearby = [ob for ob, j in zip(o.obstacles, slots) if (int(bits[j >> 5]) >> (j & 31)) & 1]
    return o


def live_sample_compare(env, config, acts, horizon, n_sample, start, prefer_records=False, **cfg_extra):
    """env: a running AUVVecEnv(auto_reset=True, debug=True).  Steps it `horizon` more steps with
    acts[(start + t) % len(acts)], then replays a sample of its envs through the oracle from their
    full live state at the start of the window -- through auto-resets onto the next pool scenario --
    and compares ranges, observations (terminal and first-of-next-episode), rewards and done flags."""
    import torch

    N, M = env.num_envs, env.scenarios.n_scenarios
    width = config.vessel.vessel_width
    R = config.vessel.n_sensors
    scn_host = env.pull_scenarios()
    snap = {k: v.clone().cpu().numpy() for k, v in env._st.items()}
    pos, disp, cnt = [x.clone().cpu().numpy() for x in env.obstacle_state()]
    rec_cnt = env._scratch["rec_cnt"].clone().cpu().numpy()
    outs = []
    for t in range(horizon):
        obs, rew, done, info = env.step(acts[(start + t) % len(acts)])
        outs.append(dict(obs=obs.clone(), reward=rew.clone(), done=done.clone(),
                         dists=env.get_attr("lidar_dist").clone(), term=info["terminal_observation"].clone()))
    env.check_status()
    done_any = torch.stack([o["done"] for o in outs]).any(0).cpu().numpy().astype(bool)
    rs = np.random.RandomState(0)
    with_done = rs.permutation(np.nonzero(done_any)[0])[: max(2, n_sample // 5)]
    with_rec = rs.permutation(np.nonzero((rec_cnt > 0) & ~done_any)[0])
    with_rec = with_rec[: (n_sample - len(with_done)) if prefer_records else (n_sample - len(with_done)) // 2]
    rest = rs.permutation(np.nonzero(~done_any)[0])[: max(0, n_sample - len(with_done) - len(with_rec))]
    sample = np.unique(np.concatenate([with_done, with_rec, rest])).astype(int)
    tid = torch.as_tensor(sample, device=env.device)
    G = [dict(obs=o["obs"][tid].cpu().numpy(), reward=o["reward"][tid].cpu().numpy(),
              done=o["done"][tid].cpu().numpy().astype(bool), dists=o["dists"][tid].cpu().numpy(),
              term=o["term"][tid].cpu().numpy()) for o in outs]
    A = [acts[(start + t) % len(acts)][tid].cpu().numpy().astype(np.float64) for t in range(horizon)]
    rep = dict(envs=len(sample), resets=0, refreshes=0, with_records=0, env_steps=0, skipped_in_band=0,
               range_max_abs=0.0, obs_max_abs=0.0, reward_max_abs=0.0)
    interval = config.vessel.sensor_interval_load_obstacles
    for k, e in enumerate(sample):
        m = int(snap["scn_id"][e])
        o = _oracle_from_live(scn_host, config, m, snap["state"][:, e], snap["step_counter"][e], snap["max_progress"][e],
                              snap["t_step"][e], snap["cum_reward"][e], snap["nearby_mask"][e], pos[e], disp[e], cnt[e],
                              **cfg_extra)
        saw_records = False
        for t in range(horizon):
            ob, rew, done, info = o.step(A[t][k])
            g = G[t]
            margin = abs(float(o.vessel.dists.min()) - width) if config.vessel.use_lidar else np.inf
            if margin <= COLLISION_BAND or abs(o.cumulative_reward - config.episode.min_cumulative_reward) < 0.05:
                rep["skipped_in_band"] += 1  # FP32 casting may legitimately decide the other way: stop this env here
                break
            rep["env_steps"] += 1
            rep["refreshes"] += int(o.vessel.step_counter % interval == 0)
            saw_records = saw_records or bool(o.vessel.nearby)
            assert bool(g["done"][k]) == bool(done), ("done", e, t)
            g_obs = g["term"][k] if done else g["obs"][k]
            derr = np.abs(g["dists"][k] - o.vessel.dists)
            assert (derr <= RANGE_ATOL + RANGE_RTOL * o.vessel.dists).all(), ("ranges", e, t, derr.max())
            oerr = np.abs(g_obs - ob).max()
            assert oerr <= max(OBS_ATOL, RANGE_RTOL), ("obs", e, t, oerr)
            rerr = abs(float(g["reward"][k]) - rew)
            assert rerr <= REWARD_ATOL + REWARD_RTOL * abs(rew), ("reward", e, t, rerr)
            rep["range_max_abs"] = max(rep["range_max_abs"], float(derr.max()))
            rep["obs_max_abs"] = max(rep["obs_max_abs"], float(oerr))
            rep["reward_max_abs"] = max(rep["reward_max_abs"], rerr)
            if done:  # VecEnv auto-reset: the env moves on to pool scenario (m + stride) mod M
                from oracle.sim import OracleEnv

                rep["resets"] += 1
                m = (m + (env.reset_stride or N)) % M  # a ring group strides by the whole ring, not its own size
                o = OracleEnv(scn_host.describe(m), oracle_cfg(config, **cfg_extra), test_mode=False)
                first = o.reset()  # (the constructor already reset once; the second reset is identical)
                ferr = np.abs(g["obs"][k] - first).max()
                assert ferr <= max(OBS_ATOL, RANGE_RTOL), ("first obs of the next episode", e, t, ferr)
        rep["with_records"] += int(saw_records)
    return rep
