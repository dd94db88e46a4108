"""AUVVecEnv -- the batched, VecEnv-shaped entry point added in front of the reference's
gym.Env contract (SURVEY.md section 8b).

``step(actions[N,2]) -> (obs[N,D], reward[N], done[N], info)`` runs one full
``BaseEnvironment.step`` (environment.py:292-366) for N envs on one B200 through the
C ABI in ``include/auv_b200.h``; finished envs are auto-reset inside the same call
(stable-baselines VecEnv semantics: the returned obs of a done env is the first obs of
its next episode, the last obs of the finished one is in ``info["terminal_observation"]``).

PyTorch is used for device memory and streams only; all arithmetic is in
``libauv_b200.so``.  There is no CPU fallback: constructing an env without CUDA raises.
"""
from __future__ import annotations

import ctypes as C
import time
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .config import Config
from .scenarios import LAND_CLEARANCE, ScenarioSet, linear_track_positions, table_track_positions
from .spaces import Box, Dict as DictSpace


def sector_partition(isensor: int, n_sensors: int, n_sectors: int, c: float = 0.1) -> int:
    """utils/sector_partitioning.py:4-9."""
    a, b = n_sensors, n_sectors

    def sigma(x):
        return b / (1 + np.exp((-x + a / 2) / (c * a)))

    return int(np.floor(sigma(isensor) - sigma(0)))


def ray_table(n_sensors: int, n_sectors: int):
    """Per-ray constants: body angles (vessel.py:63-68), reward weights
    (rewarder.py:203-205, gamma_theta = 10), sector ids."""
    d = 2 * np.pi / n_sensors
    ang = np.array([-np.pi + (i + 1) * d for i in range(n_sensors)], dtype=np.float64)
    cos_sin = np.stack([np.cos(ang), np.sin(ang)], axis=1)
    weight = 1.0 / (1.0 + np.abs(10.0 * ang))
    wsum = 0.0
    for w in weight:
        wsum += float(w)
    sector = np.array([sector_partition(i, n_sensors, n_sectors) for i in range(n_sensors)], dtype=np.uint8)
    return ang, cos_sin, weight.astype(np.float32), wsum, sector


def make_auv_config(cfg: Config, rewarder: str, test_mode: bool, auto_reset: bool, cull_mode: str,
                    velocity_mode: str = "zero") -> _lib.AuvConfig:
    v, e, s = cfg.vessel, cfg.episode, cfg.simulation
    if cfg.vessel.sensor_use_feasibility_pooling:
        raise NotImplementedError(
            "sensor_use_feasibility_pooling is broken in the reference at HEAD (SURVEY.md quirk #7)"
        )
    return _lib.AuvConfig(
        t_step_size=float(s.t_step_size),
        thrust_max_auv=float(v.thrust_max_auv),
        moment_max_auv=float(v.moment_max_auv),
        vessel_width=float(v.vessel_width),
        look_ahead_distance=float(v.look_ahead_distance),
        sensor_range=float(v.sensor_range),
        min_goal_distance=float(e.min_goal_distance),
        min_path_progress=float(e.min_path_progress),
        min_cumulative_reward=float(e.min_cumulative_reward),
        feasibility_width_multiplier=float(v.feasibility_width_multiplier),
        max_timesteps=int(e.max_timesteps),
        sensor_interval_load_obstacles=int(v.sensor_interval_load_obstacles),
        n_sensors=int(v.n_sensors),
        n_sectors=int(v.n_sectors),
        use_lidar=int(bool(v.use_lidar)),
        sensor_log_transform=int(bool(v.sensor_log_transform)),
        sensor_use_velocity_observations=int(bool(v.sensor_use_velocity_observations)),
        rewarder=_lib.REWARDER_IDS[rewarder],
        test_mode=int(bool(test_mode)),
        cull_mode=_lib.CULL_IDS[cull_mode],
        auto_reset=int(bool(auto_reset)),
        velocity_mode=_lib.VELOCITY_IDS[velocity_mode],
    )


def pick_finished_row(head) -> Optional[int]:
    """Row (0 / 1) of a track slot's ``head`` [2, 8] that holds the most recent finished episode: of the
    rows whose finished flag is set, the one with the greater episode number; None if neither is."""
    head = np.asarray(head)
    rows = [p for p in (0, 1) if head[p, 2]]
    if not rows:
        return None
    return max(rows, key=lambda p: int(head[p, 0]))


def track_rows(head_row, points_row, capacity: int):
    """The recorded points of one track row in step order: (points [n, 4], step_index [n] = steps taken
    after each point, truncated).  An episode longer than ``capacity`` keeps its last ``capacity`` points."""
    n, T = int(head_row[1]), int(capacity)
    pts = np.asarray(points_row)
    if n <= T:
        return pts[:n].copy(), np.arange(1, n + 1), False
    t = np.arange(n - T, n)
    return pts[t % T].copy(), t + 1, True


def assemble_episode(head_row, points_row, snap_row, capacity: int, k_moving: int, k_static: int, dt: float,
                     linear: Optional[dict], scenarios: Optional[ScenarioSet], path_table=None, polygons=()):
    """The ``save_latest_episode`` dict (environment.py:466-489) of one track row: ``head_row`` [8],
    ``points_row`` [T, 4] and the scenario snapshot ``snap_row`` [4 + 8 k_moving + 4 k_static] (layout of
    AuvTracks in include/auv_b200.h).  ``linear``: the pool's closed-form track constants (``AUVVecEnv.linear``)
    or None for table-driven pools, whose tracks are re-run from ``scenarios`` (slot = the row's scenario id).
    ``path_table(path_id)`` evaluates the path (None: no ``"path"``)."""
    snap = np.asarray(snap_row, np.float64)
    pts, step_index, truncated = track_rows(head_row, points_row, capacity)
    n = int(head_row[1])
    init = snap[1:4].copy()
    if truncated:
        xy, psi, steps = pts[:, 0:2].astype(np.float64), pts[:, 2].astype(np.float64), step_index
    else:
        xy = np.concatenate([init[None, 0:2], pts[:, 0:2].astype(np.float64)], axis=0)
        psi = np.concatenate([init[2:3], pts[:, 2].astype(np.float64)])
        steps = np.arange(n + 1)
    pid = int(snap[0])
    km, ks = int(k_moving), int(k_static)
    mov = None
    updates = int(head_row[6]) - (n - steps)  # obstacle updates since reset at each row
    moving_taken = np.zeros((len(steps), 0, 2))
    if km:
        rec = snap[4:4 + 8 * km].reshape(km, 8)
        if linear is not None:
            used = rec[:, 4] > 0
            moving_taken = linear_track_positions(rec[used], updates, linear["first_wrap"], linear["wrap_period"])
            d = rec[used, 2:4]
            mov = dict(width=rec[used, 4].copy(), start=rec[used, 5:7].copy(),
                       vel_tables=[np.repeat(v[None] / dt, linear["vel_len"], axis=0) for v in d])
        else:
            m = int(head_row[5])
            used = scenarios.mov_width[m] > 0
            moving_taken = table_track_positions(scenarios, m, updates, dt)[:, used]
            mov = scenarios.describe(m)["moving"]
    st = None
    if ks:
        sr = snap[4 + 8 * km:].reshape(ks, 4)
        used = sr[:, 2] > 0
        st = dict(pos=sr[used, 0:2].copy(), radius=sr[used, 2].copy())
    obstacles = dict(
        waypoints=scenarios.waypoints[pid] if scenarios is not None else None, vessel_init=init, moving=mov, static=st,
        rewarder=scenarios.rewarder if scenarios is not None else None,
        post_generate_update=scenarios.post_generate_update if scenarios is not None else None,
        polygons=list(polygons), moving_path_taken=moving_taken,
    )
    ep = dict(
        path=None, path_taken=xy, heading_taken=psi, rewards=pts[:, 3].astype(np.float64), obstacles=obstacles,
        episode=int(head_row[0]), timesteps=n, collision=bool(head_row[3]), reached_goal=bool(head_row[4]),
        truncated=bool(truncated), scenario=int(head_row[5]), path_id=pid,
    )
    if truncated:
        ep["step_index"] = steps
    if path_table is not None:
        tab = path_table(pid)
        ep["path"] = tab(np.linspace(0, tab.length, 1000))
    return ep


class AUVVecEnv:
    """N gym-auv environments stepped together on one GPU.

    Parameters
    ----------
    scenarios : ScenarioSet   pool of M scenarios (env i starts on scenario
                              (env_offset + i) % M and moves on by N at every reset)
    num_envs  : N
    config    : gym_auv_b200.Config (reference field names)
    device    : torch device (must be CUDA)
    test_mode : as BaseEnvironment(test_mode=...) (environment.py:32,380-382)
    auto_reset: VecEnv semantics (default) or manual ``reset_envs``
    debug     : also record per-ray distances, culling windows and FP64 navigation values
    count_ray_tests : count the reference-semantics ray/segment tests (get_attr("seg_tests")); default: ``debug``
    sector_outputs : also produce per-sector min-pooled and feasibility-pooled ranges
                     (get_attr("sector_min_dist") / get_attr("sector_feasible_dist"))
    chunks    : > 1 cuts the batch into that many env ranges which run their kernels on
                ``chunk_streams`` internal streams (auv_step_chunked); results are identical
    host_chunks : ranges of step_host (auv_step_host_chunked): each range's observations start
                their D2H copy while the next range is computed (default: ``chunks``)
    velocity_mode : "zero" (default) = the LiDAR speed measurements are (0, 0) as in the reference's live
                ``simulate_sensor`` (sensor.py:140-159); "nearest" = ``simulate_sensor_brute_force``
                (sensor.py:100-137): per ray the displacement of the nearest hit obstacle rotated into the
                ray frame -- it feeds ``max(0, v_y)`` of the Colav penalty (rewarder.py:199-206) and, with
                ``sensor_use_velocity_observations``, the 2 R velocity channels of the observation
    world_grid : nearby-list refreshes over a shared world of more than 32 land polygons go through a
                uniform grid over their enclosing circles instead of testing every polygon (same result)
    host_transfer : how step_host / step_async deliver the observations, all three bit-identical:
                "delta" (default) = the dense [N, obs_dim] array lives in pinned host memory and the device stores
                only the 64 B chunks of it that changed since the previous step (auv_step_host_delta_submit:
                no host-side work, every observation layout; ~85 % of a row stays exactly 0 step after step);
                "compact" = head + hit mask + non-zero closeness values written to pinned memory
                (auv_step_host_compact_submit) and scattered into the dense array by ``host_threads`` host
                threads (auv_compact_expand; LiDAR observations without velocity channels only);
                "dense" = plain D2H copy of all rows.
    compact_host : legacy switch (True = "compact", False = "dense") used when host_transfer is None
    delta_gran : floats per chunk of the delta transfer (8, 16 or 32; 16 = one host cache line)
    linear_tracks : "auto" (default) = pools whose moving obstacles all follow constant-velocity tracks
                (the MovingObstacles family) are stepped with the closed form of the update and keep no
                per-env obstacle state; False forces the general table-driven update
    record_tracks : record the episode tracks (path_taken, headings, rewards, the scenario) of this many envs,
                spread evenly (stride N // record_tracks; indices in ``tracked_envs``), in the step kernel:
                ``last_episode(i)`` / ``current_episode(i)``.  0 (default) = off.  The ray-test counting
                kernels do not record: with ``debug`` pass ``count_ray_tests=False`` (else ValueError); the env
                then has no ``seg_tests`` output
    track_capacity : steps kept per recorded episode; a longer episode keeps its last ``track_capacity``
    """

    def __init__(
        self,
        scenarios: ScenarioSet,
        num_envs: int,
        config: Optional[Config] = None,
        device="cuda:0",
        test_mode: bool = False,
        auto_reset: bool = True,
        cull_mode: str = "reference",
        debug: bool = False,
        env_offset: int = 0,
        sector_outputs: bool = False,
        max_nearby: Optional[int] = None,
        chunks: int = 1,
        chunk_streams: Optional[int] = None,
        host_chunks: Optional[int] = None,
        velocity_mode: str = "zero",
        linear_tracks="auto",
        reset_stride: int = 0,
        world_grid: bool = True,
        compact_host: Optional[bool] = None,
        host_threads: Optional[int] = None,
        host_transfer: Optional[str] = None,
        delta_gran: int = 16,
        record_tracks: int = 0,
        track_capacity: int = 2048,
        count_ray_tests: Optional[bool] = None,
        _shared: Optional[dict] = None,
    ):
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("AUVVecEnv needs a CUDA device: the step path has no CPU fallback")
        self.lib = _lib.load()
        self.config = config.copy() if config is not None else Config()
        self.scenarios = scenarios
        if _shared is None:
            scenarios.validate()
        self.num_envs = N = int(num_envs)
        self.test_mode = test_mode
        self.debug = debug
        self.env_offset = int(env_offset)
        self.cfg = make_auv_config(self.config, scenarios.rewarder, test_mode, auto_reset, cull_mode, velocity_mode)
        self._velocity_mode = velocity_mode
        self.obs_dim = self.lib.auv_obs_dim(C.byref(self.cfg))
        self.n_sensors = R = int(self.config.vessel.n_sensors)
        dev = self.device
        t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt).to(dev)

        # ---- ray table
        self.sensor_angles, cos_sin, weight, wsum, sector = ray_table(R, int(self.config.vessel.n_sectors))
        k64 = np.arange(64) * (2 * np.pi / 64)
        unit64 = np.stack([np.cos(k64), np.sin(k64)], axis=1)
        unit64[np.abs(unit64) < 1e-15] = 0.0
        if _shared is not None:
            self._ray = _shared["ray"]
        else:
            self._ray = dict(cos_sin=t(cos_sin, torch.float64), weight=t(weight, torch.float32),
                             sector=t(sector, torch.uint8), unit64=t(unit64, torch.float64))
        self.sector_index = sector
        self.rays = _lib.AuvRayTable(
            self._ray["cos_sin"].data_ptr(), self._ray["weight"].data_ptr(), self._ray["sector"].data_ptr(), self._ray["unit64"].data_ptr(), wsum
        )

        # ---- path bank
        bank = scenarios.bank
        self._bank = _shared["bank"] if _shared is not None else bank.device_arrays(dev)
        b = self._bank
        self.paths = _lib.AuvPathBank(
            bank.n_paths, getattr(bank, "n_knots", None) or bank.knots.shape[1], b["hdr"].data_ptr(), b["poly_xy"].data_ptr(), b["poly_cum"].data_ptr(),
            b["poly_f32"].data_ptr(), b["blk_chord"].data_ptr(), b["blk_dev"].data_ptr(), b["sb_chord"].data_ptr(), b["sb_dev"].data_ptr(),
            b["pp"].data_ptr(), b["sub_chord"].data_ptr(), b["sub_dev"].data_ptr(),
        )

        # ---- scenario pool
        M, Km, Ks = scenarios.n_scenarios, scenarios.k_moving, scenarios.k_static
        self.k_moving, self.k_static = Km, Ks
        mw = max(1, (Km + Ks + scenarios.world.n + 31) // 32)
        if mw > 32:
            raise ValueError("at most 1024 obstacle slots (moving + static + world polygons) per env")
        if _shared is None:
            pos0, disp0, counter0 = scenarios.initial_obstacle_state(float(self.config.simulation.t_step_size))
            vel = scenarios.vel_table if len(scenarios.vel_table) else np.zeros((1, 2))
        self._pool = _shared["pool"] if _shared is not None else dict(
            path_id=t(scenarios.path_id, torch.int32),
            vessel_init=t(scenarios.vessel_init, torch.float64),
            mov_start=t(scenarios.mov_start, torch.float64),
            mov_width=t(scenarios.mov_width, torch.float64),
            mov_track=t(scenarios.mov_track, torch.int32),
            mov_pos0=t(pos0, torch.float64),
            mov_disp0=t(disp0, torch.float64),
            mov_counter0=t(counter0, torch.float64),
            vel_table=t(vel, torch.float64),
            st_pos=t(scenarios.st_pos, torch.float64),
            st_radius=t(scenarios.st_radius, torch.float64),
            st_rec=torch.zeros((M, max(Ks, 1), 4), dtype=torch.float64, device=dev),
        )
        # closed-form obstacle update for pools of constant-velocity tracks (AuvScenarioPool.linear_tracks)
        if _shared is not None:
            self.linear = _shared["linear"]
        else:
            lin = scenarios.linear_track_info(float(self.config.simulation.t_step_size)) if linear_tracks else None
            self.linear = None
            if lin is not None and Km > 0:
                first, period = C.c_int32(0), C.c_int32(0)
                _lib.check(self.lib.auv_linear_wrap(float(self.config.simulation.t_step_size), lin["counter0"],
                                                    lin["vel_len"], C.byref(first), C.byref(period)), "auv_linear_wrap")
                self.linear = dict(first_wrap=int(first.value), wrap_period=int(period.value), **lin)
                self._pool["mov_lin"] = torch.zeros((M, Km, 8), dtype=torch.float64, device=dev)
        world = scenarios.world
        self.n_world = Pw = world.n
        if Pw and _shared is None:
            self._pool.update(
                world_circle=t(world.circle, torch.float64), world_voff=t(world.voff, torch.int32),
                world_verts=t(world.verts, torch.float64),
            )
            if world_grid and Pw > 32:  # broad phase of the nearby refresh: uniform grid over the enclosing circles
                g = world.grid(float(self.config.vessel.sensor_range) + 10.0)
                self._pool.update(world_cell_off=t(g["off"], torch.int32), world_cell_items=t(g["items"], torch.int32))
                self._pool["world_grid"] = g
        if _shared is None:
            # cached first observation of every scenario (filled by _build_reset_cache)
            self._pool.update(
                reset_obs=torch.zeros((M, self.obs_dim), dtype=torch.float32, device=dev),
                reset_max_progress=torch.zeros(M, dtype=torch.float64, device=dev),
                reset_mask=torch.zeros((M, mw), dtype=torch.int32, device=dev),
            )
        p = self._pool
        wptr = lambda k: p[k].data_ptr() if k in p else None
        lin = self.linear
        self.pool = _lib.AuvScenarioPool(
            M, Km, Ks, Pw, p["path_id"].data_ptr(), p["vessel_init"].data_ptr(), p["mov_start"].data_ptr(),
            p["mov_width"].data_ptr(), p["mov_track"].data_ptr(), p["mov_pos0"].data_ptr(), p["mov_disp0"].data_ptr(),
            p["mov_counter0"].data_ptr(), p["vel_table"].data_ptr(), p["st_pos"].data_ptr(), p["st_radius"].data_ptr(),
            p["st_rec"].data_ptr(), wptr("mov_lin"), int(lin is not None), lin["first_wrap"] if lin else 0,
            lin["wrap_period"] if lin else 0, 0,
            wptr("world_circle"), wptr("world_voff"), wptr("world_verts"),
            wptr("world_cell_off"), wptr("world_cell_items"),
            p["world_grid"]["x0"] if "world_grid" in p else 0.0, p["world_grid"]["y0"] if "world_grid" in p else 0.0,
            p["world_grid"]["cell"] if "world_grid" in p else 0.0,
            p["world_grid"]["nx"] if "world_grid" in p else 0, p["world_grid"]["ny"] if "world_grid" in p else 0,
            p["reset_obs"].data_ptr(), p["reset_max_progress"].data_ptr(), p["reset_mask"].data_ptr(),
        )
        if _shared is None:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.auv_pool_pack(C.byref(self.cfg), C.byref(self.pool), None, M, self._stream()),
                           "auv_pool_pack")

        # ---- mutable batch state
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        self._st = dict(
            scn_id=((torch.arange(N, device=dev, dtype=torch.int64) + self.env_offset) % M).to(torch.int32),
            episode=z(N, torch.int32),
            state=z((6, N), torch.float64),
            step_counter=z(N, torch.int32),
            t_step=z(N, torch.int32),
            cum_reward=z(N, torch.float64),
            max_progress=z(N, torch.float64),
            cte_sum=z(N, torch.float64),
            nearby_mask=z((N, mw), torch.int32),
            nav=z((N, _lib.NAV_W), torch.float64),
            obst_steps=z(N, torch.int32),
            prev_seg=torch.full((N,), -1, dtype=torch.int32, device=dev),
            env_pid=z(N, torch.int32),
        )
        if self.linear is None:  # table-driven tracks keep per-env obstacle state
            self._st.update(
                mov_pos=z((N, max(Km, 1), 2), torch.float64),
                mov_disp=z((N, max(Km, 1), 2), torch.float64),
                mov_counter=z((N, max(Km, 1)), torch.float64),
            )
        # scratch between the culling and the casting stage: one record slot per obstacle slot
        # can never overflow; worlds with many polygons cap it (overflow raises, never silent)
        slots = Km + Ks + Pw
        self.rec_cap = int(max_nearby) if max_nearby is not None else (slots if slots <= 64 else 64)
        self.rec_cap = max(1, min(self.rec_cap, max(slots, 1)))
        self._scratch = dict(
            rec=torch.zeros((N, self.rec_cap, _lib.REC_BYTES), dtype=torch.uint8, device=dev),
            rec_cnt=z(N, torch.int32), status=z(1, torch.int32),
        )
        s = self._st
        sptr = lambda k: s[k].data_ptr() if k in s else None
        self.reset_stride = int(reset_stride)
        self.batch = _lib.AuvBatch(
            N, mw, self.env_offset, self.reset_stride, s["scn_id"].data_ptr(), s["episode"].data_ptr(), s["state"].data_ptr(),
            s["step_counter"].data_ptr(), s["t_step"].data_ptr(), s["cum_reward"].data_ptr(),
            s["max_progress"].data_ptr(), s["cte_sum"].data_ptr(), s["nearby_mask"].data_ptr(),
            sptr("mov_pos"), sptr("mov_disp"), sptr("mov_counter"), s["nav"].data_ptr(),
            self._scratch["rec"].data_ptr(), self._scratch["rec_cnt"].data_ptr(),
            self._scratch["status"].data_ptr(), self.rec_cap, 0,
            s["obst_steps"].data_ptr(), s["prev_seg"].data_ptr(), s["env_pid"].data_ptr(),
        )

        # ---- outputs
        K = Km + Ks + Pw
        self._out = dict(
            obs=z((N, self.obs_dim), torch.float32),
            reward=z(N, torch.float32),
            done=z(N, torch.uint8),
            collision=z(N, torch.uint8),
            reached_goal=z(N, torch.uint8),
            goal_distance=z(N, torch.float32),
            progress=z(N, torch.float32),
            terminal_obs=z((N, self.obs_dim), torch.float32),
            stats=z(_lib.N_STATS, torch.float64),
            seg_tests=z(1, torch.int64),
            episode_out=z((N, 8), torch.float32),
        )
        if sector_outputs and self.config.vessel.use_lidar:
            ns = int(self.config.vessel.n_sectors)
            self._out["sector_min_dist"] = z((N, ns), torch.float32)
            self._out["sector_feasible_dist"] = z((N, ns), torch.float32)
        if debug:
            self._out["lidar_dist"] = z((N, max(R, 1)), torch.float32)
            self._out["windows"] = z((N, max(K, 1), 2), torch.int32)
        count_ray_tests = bool(debug) if count_ray_tests is None else bool(count_ray_tests)
        if count_ray_tests and int(record_tracks) > 0:
            raise ValueError("record_tracks cannot be combined with the ray-test counter of debug: "
                             "pass count_ray_tests=False")
        if int(record_tracks) > 0:
            del self._out["seg_tests"]  # not counted: get_attr("seg_tests") raises instead of reading 0
        o = self._out
        ptr = lambda k: o[k].data_ptr() if k in o else None
        # episode tracks of a sample of the envs (AuvTracks), recorded by the step kernel
        self.record_tracks = Kt = max(0, min(int(record_tracks), N))
        self.track_capacity = T = int(track_capacity)
        self.tracked_envs = np.zeros(0, dtype=np.int64)
        self._tracks, self.tracks = None, None
        if Kt:
            if T < 1:
                raise ValueError("track_capacity must be >= 1")
            stride = N // Kt
            self.tracked_envs = np.arange(Kt, dtype=np.int64) * stride
            W = _lib.track_snap_width(Km, Ks)
            self._tracks = dict(points=z((Kt, 2, T, 4), torch.float32), head=z((Kt, 2, _lib.TRACK_HEAD_W), torch.int32),
                                snap=z((Kt, 2, W), torch.float64), stride=stride)
            tk = self._tracks
            self.tracks = _lib.AuvTracks(Kt, stride, T, 0, tk["points"].data_ptr(), tk["head"].data_ptr(),
                                         tk["snap"].data_ptr())
        self.out = _lib.AuvStepOut(
            ptr("obs"), ptr("reward"), ptr("done"), ptr("collision"), ptr("reached_goal"), ptr("goal_distance"),
            ptr("progress"), ptr("lidar_dist"), ptr("windows"), ptr("terminal_obs"), ptr("sector_min_dist"),
            ptr("sector_feasible_dist"), ptr("stats"),
            ptr("seg_tests") if count_ray_tests else None, ptr("episode_out"),
            C.addressof(self.tracks) if Kt else None,
        )
        self.actions_dev = z((N, 2), torch.float32)
        self._pinned = None
        can_compact = bool(self.config.vessel.use_lidar) and not bool(self.config.vessel.sensor_use_velocity_observations)
        if host_transfer not in (None, "dense", "compact", "delta"):
            raise ValueError("host_transfer must be 'dense', 'compact' or 'delta'")
        if host_transfer == "compact" and not can_compact:
            raise ValueError("host_transfer='compact' needs LiDAR observations without velocity channels")
        if host_transfer is None:
            host_transfer = "delta" if compact_host is None else ("compact" if compact_host and can_compact else "dense")
        self.host_transfer = host_transfer
        self.compact_host = self.host_transfer == "compact"
        self.delta_gran = int(delta_gran)
        self._delta_seen = (0, 0)  # (chunks, steps) at the last d2h_bytes_per_step query
        import os as _os

        self.host_threads = int(host_threads) if host_threads else max(1, min(16, len(_os.sched_getaffinity(0))))
        self.expand_seconds = 0.0  # host time spent in auv_compact_expand (diagnostic)
        self.wait_seconds = 0.0  # host time spent blocked in step_wait (diagnostic)
        self.chunks = max(1, int(chunks))
        self.host_chunks = max(1, min(64, int(host_chunks))) if host_chunks else self.chunks
        self._pipe = None
        if self.chunks > 1 or self.host_chunks > 1:
            ns = int(chunk_streams) if chunk_streams else max(2, min(self.chunks, 4))
            with torch.cuda.device(self.device):
                self._pipe = self.lib.auv_pipeline_create(ns)
            if not self._pipe:
                raise _lib.AuvLibraryError("auv_pipeline_create failed: " + self.lib.auv_last_error().decode())
            self.chunk_streams = ns
        self.total_steps = 0

        self.action_space = Box(low=np.array([-1, -0.15]), high=np.array([1, 0.15]), dtype=np.float32)
        self.observation_space = Box(low=-np.ones(self.obs_dim), high=np.ones(self.obs_dim), dtype=np.float32)
        self.dict_observation = bool(self.config.vessel.use_dict_observation) and bool(self.config.vessel.use_lidar)
        if self.dict_observation:  # environment.py:116-137
            self.observation_space = DictSpace({
                "proprioceptive": Box(-1.0, 1.0, shape=(6,), dtype=np.float32),
                "lidar": Box(-1.0, 1.0, shape=((self.obs_dim - 6) // R, R), dtype=np.float32),
            })
        self._max_nearby = max_nearby
        self._cull_mode = cull_mode
        if auto_reset and _shared is None:
            self._build_reset_cache()

    def _worker(self, cap: int) -> "AUVVecEnv":
        """A batch of `cap` envs that shares this env's device tables: the scratch the reset cache is
        computed on (auv_reset_cache_fill / auv_refresh_finished)."""
        if not hasattr(self, "_workers"):
            self._workers = {}
        w = self._workers.get(cap)
        if w is None:
            w = self._workers[cap] = AUVVecEnv(
                self.scenarios, cap, self.config, device=self.device, test_mode=self.test_mode, auto_reset=False,
                cull_mode=self._cull_mode, max_nearby=self._max_nearby, velocity_mode=self._velocity_mode,
                _shared=self._shared_tables())
        return w

    def _build_reset_cache(self, ids: Optional[torch.Tensor] = None, chunk: int = 65536):
        """reset() of scenario m always returns the same observation (it depends on the
        scenario only), so it is computed once per pool scenario -- by the same kernels, over a
        worker batch that shares this env's device tables (auv_reset_cache_fill) -- and the in-step
        auto-reset of a finished env becomes a copy (pool.reset_obs / reset_max_progress /
        reset_mask).  ``ids``: int tensor of pool scenarios to (re)compute, default all."""
        M = self.scenarios.n_scenarios
        total = M if ids is None else int(ids.numel())
        if total == 0:
            return
        cap = 1024 if total <= 1024 else (8192 if total <= 8192 else min(chunk, 65536))
        w = self._worker(cap)
        idp = ids.to(self.device, torch.int32).contiguous() if ids is not None else None
        cfg, rays, paths, pool, _ = self._refs()
        with torch.cuda.device(self.device):
            for start in range(0, total, cap):
                n = min(cap, total - start)
                p = C.c_void_p(idp.data_ptr() + 4 * start) if idp is not None else None
                _lib.check(self.lib.auv_reset_cache_fill(cfg, rays, paths, pool, C.byref(w.batch), C.byref(w.out), p,
                                                         start if idp is None else 0, n, self._stream()),
                           "auv_reset_cache_fill")
        if cap > 8192:  # the big worker is only needed once
            torch.cuda.synchronize(self.device)
            self._workers.pop(cap, None)

    # ------------------------------------------------------------------ GPU-side scenario generation
    def gen_params(self, seed: int, epoch: int) -> "_lib.AuvGenParams":
        v = self.config.vessel
        return _lib.AuvGenParams(
            seed=int(seed) & 0xFFFFFFFFFFFFFFFF, epoch=int(epoch) & 0xFFFFFFFF,
            post_generate_update=int(bool(self.scenarios.post_generate_update)),
            t_step_size=float(self.config.simulation.t_step_size), vessel_width=float(v.vessel_width),
            init_pos_jitter=50.0, mov_disp_std=500.0, mov_width_mean=10.0, mov_speed_lo=1.0, mov_speed_hi=3.0,
            st_disp_std=250.0, st_radius_mean=30.0,
            path_group=int(self.scenarios.path_group), path_period=int(self.scenarios.path_period or self.scenarios.n_scenarios),
            land_clearance=LAND_CLEARANCE,
        )

    def regenerate_scenarios(self, ids: Optional[torch.Tensor] = None, seed: int = 0, epoch: int = 1):
        """Draw fresh MovingObstacles scenarios ON THE GPU (auv_generate_moving_obstacles:
        movingobstacles.py:28-95 + helpers.py:5-35 with Philox streams keyed by (seed; scenario,
        slot, epoch)) into the listed pool slots (default: all) and refill their cached first
        observation.  Slots that a live env is running must not be listed -- see
        ``refresh_finished``.  The host copy ``self.scenarios`` goes stale: ``pull_scenarios()``.

        In a pool with a shared world of land polygons every placed object is also clear of land
        (outside every polygon and farther than d from every ring): the vessel start by
        ``scenarios.LAND_CLEARANCE``, a static circle's centre by its radius, a moving obstacle's track
        start by its width; rejected draws are redrawn from the same stream.  Paths, goals and the later
        course of moving obstacles are not tested.  A start area that stays covered after 4096 draws raises
        in ``check_status()``."""
        M, Km = self.scenarios.n_scenarios, self.k_moving
        if Km and self._pool["vel_table"].shape[0] < M * Km:
            raise ValueError("pool.vel_table must hold n_scenarios * k_moving entries (constant-velocity tracks)")
        gp = self.gen_params(seed, epoch)
        self._pool["host_stale"] = True  # the host ScenarioSet no longer describes every pool slot
        idp, n = None, M
        if ids is not None:
            ids = ids.to(self.device, torch.int32).contiguous()
            idp, n = C.c_void_p(ids.data_ptr()), int(ids.numel())
            if n == 0:
                return 0
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_generate_moving_obstacles(
                C.byref(gp), C.byref(self.paths), C.byref(self.pool), idp, n,
                C.c_void_p(self._scratch["status"].data_ptr()), self._stream()), "auv_generate_moving_obstacles")
        self._build_reset_cache(ids)
        return n

    def regenerate_paths(self, ids: Optional[torch.Tensor] = None, seed: int = 0, epoch: int = 1, length: float = 800.0):
        """Draw fresh ``RandomCurveThroughOrigin`` paths ON THE GPU (path.py:96-120 waypoints with Philox
        streams, then ``Path.__init__``'s three PCHIP rounds, polyline and search tables:
        auv_random_curve_waypoints + auv_pathbank_build) into the listed slots of a device-built bank
        (default: all).  Scenarios that follow those paths are stale afterwards -- regenerate them
        (``regenerate_scenarios``) before the next ``reset()``; ``MovingObstacles._generate`` does the same
        pair of draws per episode (movingobstacles.py:28-95).  The ``"path"`` of a recorded episode
        (``last_episode``) is evaluated from the bank when it is read, so it is stale for an episode
        whose path slot was replaced here."""
        from .pathbank import DevicePathBank

        bank = self.scenarios.bank
        if not isinstance(bank, DevicePathBank):
            raise ValueError("regenerate_paths needs a device-built path bank (scenarios built with device_paths=True)")
        n = bank.n_paths
        idp = None
        if ids is not None:
            ids = ids.to(self.device, torch.int32).contiguous()
            idp, n = C.c_void_p(ids.data_ptr()), int(ids.numel())
            if n == 0:
                return 0
        wp = torch.zeros((n, 2, 8), dtype=torch.float64, device=self.device)
        nwp = torch.zeros(n, dtype=torch.int32, device=self.device)
        bs = bank.build_struct(self._bank)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_random_curve_waypoints(int(seed) & 0xFFFFFFFFFFFFFFFF, int(epoch) & 0xFFFFFFFF, float(length),
                                                           idp, n, C.c_void_p(wp.data_ptr()), C.c_void_p(nwp.data_ptr()),
                                                           self._stream()), "auv_random_curve_waypoints")
            _lib.check(self.lib.auv_pathbank_build(C.c_void_p(wp.data_ptr()), C.c_void_p(nwp.data_ptr()), idp, n, C.byref(bs),
                                                   C.c_void_p(self._scratch["status"].data_ptr()), self._stream()),
                       "auv_pathbank_build")
        # keep the host copy of the waypoints in step (oracle replay / pull_scenarios)
        hw, hn = wp.cpu().numpy(), nwp.cpu().numpy()
        slots = range(bank.n_paths) if ids is None else ids.cpu().numpy().tolist()
        for k, pth in enumerate(slots):
            bank.waypoints[int(pth)] = hw[k, :, : int(hn[k])].copy()
            self.scenarios.waypoints[int(pth)] = bank.waypoints[int(pth)]
        bank._tables = None
        self.check_status()
        return n

    def refresh_finished(self, seed: int = 0) -> int:
        """Ping-pong scenario refresh for sustained training: with a pool of M = 2 N scenarios env
        e alternates between slots e and e + N at every reset, so the slot it is NOT running is
        free.  Every env that finished an episode since the last call gets a freshly generated
        scenario in its free slot (the one its next reset moves to).  Returns how many."""
        N, M = self.reset_stride or self.num_envs, self.scenarios.n_scenarios
        if M != 2 * N:
            raise ValueError("refresh_finished needs a pool of exactly 2 * reset_stride (default num_envs) scenarios")
        ep = self._st["episode"]
        if getattr(self, "_seen_episode", None) is None:
            self._seen_episode = torch.zeros_like(ep)
            self._gen_epoch = 1
        changed = torch.nonzero(ep != self._seen_episode).flatten()
        self._seen_episode.copy_(ep)
        if changed.numel() == 0:
            return 0
        free = (self._st["scn_id"][changed].to(torch.int64) + N) % M
        self._gen_epoch += 1
        return self.regenerate_scenarios(free, seed=seed, epoch=self._gen_epoch)

    def refresh_finished_device(self, seed: int = 0, capacity: int = 4096):
        """``refresh_finished`` without a host round trip (auv_refresh_finished): collecting the envs
        that finished, generating fresh scenarios into the slots they vacated and recomputing those
        slots' cached first observation are all enqueued on the current stream -- nothing is read back,
        so it can sit inside a training loop (the reference draws a new scenario in every reset()).
        At most ``capacity`` slots per call; the rest are picked up by the next call."""
        N, M = self.num_envs, self.scenarios.n_scenarios
        if M != 2 * (self.reset_stride or N):
            raise ValueError("refresh_finished_device needs a pool of exactly 2 * reset_stride (default num_envs) scenarios")
        capacity = int(min(capacity, 65536))
        rs = getattr(self, "_refresh", None)
        if rs is None or rs["cap"] != capacity:
            dev = self.device
            # episode counters seen so far: envs that finished before the first call are not listed again
            rs = self._refresh = dict(
                cap=capacity, seen=self._st["episode"].clone(), ids=torch.zeros(capacity, dtype=torch.int32, device=dev),
                count=torch.zeros(1, dtype=torch.int32, device=dev), epoch=getattr(self, "_gen_epoch", 1))
            rs["struct"] = _lib.AuvRefreshScratch(rs["seen"].data_ptr(), rs["ids"].data_ptr(), rs["count"].data_ptr(),
                                                  capacity, 0)
        w = self._worker(1024 if capacity <= 1024 else (8192 if capacity <= 8192 else 65536))
        rs["epoch"] += 1
        self._gen_epoch = rs["epoch"]
        gp = self.gen_params(seed, rs["epoch"])
        self._pool["host_stale"] = True
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_refresh_finished(cfg, rays, paths, pool, batch, C.byref(w.batch), C.byref(w.out),
                                                     C.byref(rs["struct"]), C.byref(gp), self._stream()),
                       "auv_refresh_finished")

    def pull_scenarios(self) -> ScenarioSet:
        """Host copy of the device pool (after regenerate_scenarios), e.g. to replay generated
        scenarios through the CPU oracle."""
        import dataclasses

        p = self._pool
        h = lambda k: p[k].cpu().numpy().copy()
        return dataclasses.replace(
            self.scenarios, path_id=h("path_id"), vessel_init=h("vessel_init"), mov_start=h("mov_start"),
            mov_width=h("mov_width"), mov_track=h("mov_track"), vel_table=h("vel_table"), st_pos=h("st_pos"),
            st_radius=h("st_radius"), _bank=self.scenarios.bank, _world=self.scenarios._world,
        )

    # ------------------------------------------------------------------ helpers
    def _shared_tables(self):
        return dict(ray=self._ray, bank=self._bank, pool=self._pool, linear=self.linear)

    def obstacle_state(self):
        """(position [N, Km, 2], last displacement [N, Km, 2], waypoint counter [N, Km]) of the moving
        obstacles -- VesselObstacle.position / (dx, dy) / waypoint_counter (obstacles.py:195-215).  Pools
        of constant-velocity tracks keep no per-env obstacle state: the values are evaluated on demand."""
        if self.linear is None:
            return self._st["mov_pos"], self._st["mov_disp"], self._st["mov_counter"]
        N, Km = self.num_envs, max(self.k_moving, 1)
        pos = torch.zeros((N, Km, 2), dtype=torch.float64, device=self.device)
        disp = torch.zeros_like(pos)
        cnt = torch.zeros((N, Km), dtype=torch.float64, device=self.device)
        if self.k_moving:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.auv_obstacle_state(
                    C.byref(self.cfg), C.byref(self.pool), C.byref(self.batch), C.c_void_p(pos.data_ptr()),
                    C.c_void_p(disp.data_ptr()), C.c_void_p(cnt.data_ptr()), self._stream()), "auv_obstacle_state")
        return pos, disp, cnt

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _refs(self):
        return C.byref(self.cfg), C.byref(self.rays), C.byref(self.paths), C.byref(self.pool), C.byref(self.batch)

    def check_status(self):
        """Raise if a kernel flagged a problem (synchronises).  Called by reset() and
        episode_stats(); call it yourself after long unattended runs."""
        st = int(self._scratch["status"].item())
        if st & _lib.STATUS_GEN_GAVE_UP:
            raise RuntimeError("scenario generator: an obstacle slot was still rejected after 100000 draws")
        if st & _lib.STATUS_GEN_LAND_BLOCKED:
            raise RuntimeError("scenario generator: a scenario's start area is covered by land "
                               "(no vessel start clear of land after 4096 draws)")
        if st & _lib.STATUS_BOUNDS:
            raise RuntimeError("AUV_DEBUG_BOUNDS build: an index check inside a step kernel failed "
                               f"(source lines OR-ed together: {st >> 8})")
        if st & _lib.STATUS_PATH_TOO_LONG:
            raise RuntimeError("a generated path's polyline does not fit its slot: raise DevicePathBank(vcap=...)")
        if st & _lib.STATUS_POLY_TOO_LARGE:
            raise RuntimeError(f"a world polygon has more than {_lib.MAX_POLY_VERTS} vertices: split it")
        if st & _lib.STATUS_REC_OVERFLOW:
            raise RuntimeError(
                f"more than max_nearby={self.rec_cap} obstacles were within sensor range of one env: "
                "construct AUVVecEnv with a larger max_nearby"
            )

    def observation_dict(self, obs=None):
        """The Dict observation of environment.py:116-137,281-288 for the whole batch, as zero-copy views of
        the flat observation: ``proprioceptive`` [N, 6] and the LiDAR "image" ``lidar`` [N, C, R] -- channel 0
        closeness, with ``sensor_use_velocity_observations`` channels 1-2 the obstacle velocity in the ray
        frame (v_x, v_y).  (The reference always stacks the two velocity rows; without velocity observations
        they are all zero upstream and are simply not materialised here: C = 1.)"""
        o = self._out["obs"] if obs is None else obs
        R = self.n_sensors
        return {"proprioceptive": o[:, :6], "lidar": o[:, 6:].reshape(o.shape[0], -1, R)}

    def _fmt(self, obs):
        return self.observation_dict(obs) if self.dict_observation else obs

    # ------------------------------------------------------------------ gym/VecEnv API
    def reset(self, check: bool = True) -> torch.Tensor:
        """Reset every env (BaseEnvironment.reset, environment.py:176-245)."""
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_reset(cfg, pool, batch, None, self._stream()), "auv_reset")
            _lib.check(
                self.lib.auv_observe(cfg, rays, paths, pool, batch, C.byref(self.out), _lib.OBSERVE_RESET, self._stream()),
                "auv_observe",
            )
        if check:
            self.check_status()
        return self._fmt(self._out["obs"])

    def reset_envs(self, mask: torch.Tensor, scenario_ids: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Reset the envs where mask != 0 (optionally onto explicit scenario ids)."""
        mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        if scenario_ids is not None:
            sel = mask.bool()
            self._st["scn_id"][sel] = scenario_ids.to(self.device, torch.int32)[sel]
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_reset(cfg, pool, batch, C.c_void_p(mask.data_ptr()), self._stream()), "auv_reset")
            # observe everything in RESET mode would clobber live envs' max_progress only
            # with identical values; obs of untouched envs is simply recomputed
            _lib.check(
                self.lib.auv_observe(cfg, rays, paths, pool, batch, C.byref(self.out), _lib.OBSERVE_RESET, self._stream()),
                "auv_observe",
            )
        return self._out["obs"]

    def step(self, actions: torch.Tensor):
        """actions: [N, 2] float32 CUDA tensor (thrust, steer) -- environment.py:101-106."""
        if actions.shape != (self.num_envs, 2):
            raise ValueError(f"actions must have shape ({self.num_envs}, 2), got {tuple(actions.shape)}")
        a = actions.to(device=self.device, dtype=torch.float32).contiguous()
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            if self._pipe and self.chunks > 1:
                _lib.check(
                    self.lib.auv_step_chunked(cfg, rays, paths, pool, batch, C.c_void_p(a.data_ptr()), C.byref(self.out),
                                              self._stream(), self._pipe, self.chunks),
                    "auv_step_chunked",
                )
            else:
                _lib.check(
                    self.lib.auv_step(cfg, rays, paths, pool, batch, C.c_void_p(a.data_ptr()), C.byref(self.out), self._stream()),
                    "auv_step",
                )
        self.total_steps += 1
        return self._fmt(self._out["obs"]), self._out["reward"], self._out["done"], self.info()

    def step_host(self, actions: np.ndarray):
        """NumPy in / NumPy out: the call a CPU-side VecEnv consumer makes (the e2e
        path).  Copies actions H2D and obs/reward/done D2H through pinned buffers."""
        if self.host_transfer != "dense":
            self.step_async(actions)
            return self.step_wait()
        pin = self.step_host_buffers()
        pin["act"].numpy()[...] = actions
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            hargs = (cfg, rays, paths, pool, batch, C.c_void_p(pin["act"].data_ptr()),
                     C.c_void_p(self.actions_dev.data_ptr()), C.byref(self.out), C.c_void_p(pin["obs"].data_ptr()),
                     C.c_void_p(pin["reward"].data_ptr()), C.c_void_p(pin["done"].data_ptr()), self._stream())
            if self._pipe and self.host_chunks > 1:
                _lib.check(self.lib.auv_step_host_chunked(*hargs, self._pipe, self.host_chunks), "auv_step_host_chunked")
            else:
                _lib.check(self.lib.auv_step_host(*hargs), "auv_step_host")
        self.total_steps += 1
        return pin["obs"].numpy(), pin["reward"].numpy(), pin["done"].numpy()

    # stable-baselines' asynchronous VecEnv interface (vec_env/base_vec_env.py: step_async /
    # step_wait): the step is submitted on a stream owned by this env; step_wait blocks on it.
    # Two env groups stepped alternately (wait A, submit A, wait B, submit B, ...) keep the
    # D2H link busy: one group's observations travel while the other group is computed.
    def step_async(self, actions: np.ndarray):
        if getattr(self, "_async_pending", False):
            raise RuntimeError("step_async() called twice without step_wait()")
        if self._pinned is None:
            self.step_host_buffers()
        if self._pipe is None:
            with torch.cuda.device(self.device):
                self._pipe = self.lib.auv_pipeline_create(2)
            if not self._pipe:
                raise _lib.AuvLibraryError("auv_pipeline_create failed: " + self.lib.auv_last_error().decode())
            self.chunk_streams = 2
        if getattr(self, "_async_stream", None) is None:
            self._async_stream = torch.cuda.Stream(device=self.device)
            self._async_done = torch.cuda.Event()
        pin = self._pinned
        if getattr(self, "_async_call", None) is None:  # the argument list never changes: build it once
            cfg, rays, paths, pool, batch = self._refs()
            head = (cfg, rays, paths, pool, batch, C.c_void_p(pin["act"].data_ptr()), C.c_void_p(self.actions_dev.data_ptr()),
                    C.byref(self.out))
            tail = (C.c_void_p(pin["reward"].data_ptr()), C.c_void_p(pin["done"].data_ptr()),
                    C.c_void_p(self._async_stream.cuda_stream), self._pipe, max(1, self.host_chunks))
            if self.host_transfer == "delta":
                self._async_call = (self.lib.auv_step_host_delta_submit, head + (C.byref(pin["delta"]),) + tail,
                                    "auv_step_host_delta_submit")
            elif self.compact_host:
                self._async_call = (self.lib.auv_step_host_compact_submit, head + (C.byref(pin["compact"]),) + tail,
                                    "auv_step_host_compact_submit")
            else:
                self._async_call = (self.lib.auv_step_host_submit, head + (C.c_void_p(pin["obs"].data_ptr()),) + tail,
                                    "auv_step_host_submit")
            self._act_np = pin["act"].numpy()
        self._act_np[...] = actions
        cur = torch.cuda.current_stream(self.device)
        if cur != self._async_stream:
            self._async_stream.wait_stream(cur)  # earlier work of this env (reset, step) is ordered before
        fn, fargs, name = self._async_call
        with torch.cuda.device(self.device):
            rc = fn(*fargs)
        if rc:
            _lib.check(rc, name)
        self._async_done.record(self._async_stream)
        self._async_pending = True
        self.total_steps += 1

    def step_wait(self):
        if not getattr(self, "_async_pending", False):
            raise RuntimeError("step_wait() without a pending step_async()")
        t0 = time.perf_counter()
        self._async_done.synchronize()
        self.wait_seconds += time.perf_counter() - t0
        torch.cuda.current_stream(self.device).wait_event(self._async_done)
        self._async_pending = False
        pin = self._pinned
        if self.compact_host:  # scatter head / mask / packed values into the dense array (host threads)
            t0 = time.perf_counter()
            _lib.check(self.lib.auv_compact_expand(
                C.byref(self.cfg), self.num_envs, C.byref(pin["compact"]), C.c_void_p(pin["prev_mask"].ctypes.data),
                C.c_void_p(pin["obs_dense"].ctypes.data), self.host_threads), "auv_compact_expand")
            self.expand_seconds += time.perf_counter() - t0
            return pin["obs_dense"], pin["reward"].numpy(), pin["done"].numpy()
        return pin["obs"].numpy(), pin["reward"].numpy(), pin["done"].numpy()

    def groups(self, n_groups: int = 2, **kw):
        """``n_groups`` envs of num_envs / n_groups each that SHARE this env's device tables
        (ray table, path bank, scenario pool incl. the cached first observations): the
        asynchronous pattern ``wait(A); submit(A); wait(B); submit(B); ...`` with
        step_async / step_wait keeps the host link busy.  Group g starts on the scenarios
        g * n .. (g + 1) * n - 1; every group advances through the whole pool on resets."""
        n = self.num_envs // int(n_groups)
        if n <= 0:
            raise ValueError("more groups than envs")
        shared = self._shared_tables()
        kw.setdefault("host_chunks", max(1, self.host_chunks // int(n_groups)))
        kw.setdefault("host_transfer", self.host_transfer)
        kw.setdefault("delta_gran", self.delta_gran)
        kw.setdefault("record_tracks", self.record_tracks)
        kw.setdefault("track_capacity", self.track_capacity)
        return [AUVVecEnv(self.scenarios, n, self.config, device=self.device, test_mode=self.test_mode,
                          auto_reset=bool(self.cfg.auto_reset), cull_mode=self._cull_mode, env_offset=g * n,
                          max_nearby=self._max_nearby, velocity_mode=self._velocity_mode,
                          reset_stride=self.reset_stride or self.num_envs, host_threads=self.host_threads,
                          _shared=shared, **kw)
                for g in range(int(n_groups))]

    def ring(self, n_groups: int = 4, **kw) -> "EnvGroupRing":
        """The env groups of ``groups(n_groups)`` behind a send / recv interface (the asynchronous mode
        of batched env pools): ``recv()`` hands out whichever group's step has finished, ``send(g, actions)``
        submits that group's next step.  See EnvGroupRing."""
        return EnvGroupRing(self.groups(n_groups, **kw))

    def step_host_buffers(self):
        """Pinned host buffers of step_host / step_async (actions in; obs, reward, done out)."""
        N = self.num_envs
        if self._pinned is None:
            self._pinned = dict(
                act=torch.zeros((N, 2), dtype=torch.float32).pin_memory(),
                reward=torch.zeros(N, dtype=torch.float32).pin_memory(),
                done=torch.zeros(N, dtype=torch.uint8).pin_memory(),
            )
            if self.compact_host:
                W = (self.n_sensors + 31) // 32
                p = self._pinned
                p["head"] = torch.zeros((N, 8), dtype=torch.float32).pin_memory()
                p["mask"] = torch.zeros((N, W), dtype=torch.int32).pin_memory()
                p["vals"] = torch.zeros(N * W * 32, dtype=torch.float32).pin_memory()
                p["counter"] = torch.zeros(1, dtype=torch.int32, device=self.device)
                p["prev_mask"] = np.zeros((N, W), dtype=np.uint32)
                p["obs_dense"] = np.zeros((N, self.obs_dim), dtype=np.float32)
                p["compact"] = _lib.AuvCompact(p["head"].data_ptr(), p["mask"].data_ptr(), p["vals"].data_ptr(),
                                               p["counter"].data_ptr(), W, N * W * 32)
            else:
                self._pinned["obs"] = torch.zeros((N, self.obs_dim), dtype=torch.float32).pin_memory()
                if self.host_transfer == "delta":  # the device's copy of what the host array holds
                    p = self._pinned
                    p["shadow"] = torch.zeros((N, self.obs_dim), dtype=torch.float32, device=self.device)
                    p["shipped"] = torch.zeros(1, dtype=torch.int64, device=self.device)
                    p["delta"] = _lib.AuvDelta(p["obs"].data_ptr(), p["shadow"].data_ptr(), p["shipped"].data_ptr(),
                                               self.delta_gran)
        return self._pinned

    @property
    def h2d_bytes_per_step(self) -> int:
        return self.num_envs * 2 * 4

    @property
    def d2h_bytes_per_step(self) -> int:
        """bytes that cross the link per step: dense rows, or -- compact transfer -- heads, masks, reward,
        done plus the packed non-zero values of the LAST step (read from its head records)"""
        if self.compact_host and self._pinned is not None:
            p = self._pinned
            nz = int(p["head"].numpy().view(np.int32)[:, 6].sum())
            return self.num_envs * (32 + 4 * p["mask"].shape[1] + 4 + 1) + 4 * nz
        if self.host_transfer == "delta" and self._pinned is not None:  # average since the previous query
            chunks, steps = int(self._pinned["shipped"].item()), self.total_steps
            c0, s0 = self._delta_seen
            self._delta_seen = (chunks, steps)
            return self.num_envs * (4 + 1) + int((chunks - c0) * self.delta_gran * 4 / max(1, steps - s0))
        return self.num_envs * (self.obs_dim * 4 + 4 + 1)

    def info(self) -> Dict[str, torch.Tensor]:
        o = self._out
        return dict(
            collision=o["collision"],
            reached_goal=o["reached_goal"],
            goal_distance=o["goal_distance"],
            progress=o["progress"],
            terminal_observation=o["terminal_obs"],
        )

    # ------------------------------------------------------------------ staged entry points
    def obstacle_update(self):
        cfg, _, _, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_obstacle_update(cfg, pool, batch, self._stream()), "auv_obstacle_update")

    def vessel_step(self, actions: torch.Tensor):
        a = actions.to(device=self.device, dtype=torch.float32).contiguous()
        cfg, _, _, _, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_vessel_step(cfg, batch, C.c_void_p(a.data_ptr()), self._stream()), "auv_vessel_step")

    def navigate(self):
        """Vessel.navigate for every env -> nav record [N, 12] (s, chi, y_e, s_la, look-ahead
        heading error, heading error, goal distance, progress, cos psi, sin psi, reached, ...)."""
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_navigate(cfg, rays, paths, pool, batch, self._stream()), "auv_navigate")
        return self._st["nav"]

    def observe(self, mode=_lib.OBSERVE_STEP):
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(
                self.lib.auv_observe(cfg, rays, paths, pool, batch, C.byref(self.out), mode, self._stream()),
                "auv_observe",
            )
        return self._out["obs"]

    # ------------------------------------------------------------------ rendering
    def render(self, env_ids, width: int = 400, height: int = 400, half_width: Optional[float] = None) -> torch.Tensor:
        """Top-down RGB frames of envs ``env_ids`` as their last step or reset left them: a CUDA ``uint8`` tensor
        [K, height, width, 3], north up, centred on each vessel, ``2 half_width / width`` metres per pixel (the
        frame rule is stated at ``AuvRender`` in include/auv_b200.h).  A visual tap: no parity with the
        reference's pygame renderer is claimed.  Enqueued on the current stream (auv_render, kernel k_render)
        with no host synchronisation; it reads env state and the device observation rows only -- every step
        path (``step``, ``step_host``, ``step_async`` / ``step_wait`` with each host transfer) computes those
        rows on the device before any copy, so the rays are the last step's.

        ``env_ids``: at least one id; ints on the host (checked: ValueError when out of range) or an int CUDA
        tensor (not read back; a frame whose id is out of range comes out all zeros).  ``half_width`` defaults to
        ``config.vessel.render_distance`` when that is a number.  RuntimeError between ``step_async()`` and
        ``step_wait()``: the step in flight is writing what a frame would show."""
        if getattr(self, "_async_pending", False):
            raise RuntimeError("render() between step_async() and step_wait(): call step_wait() first")
        if half_width is None:
            rd = self.config.vessel.render_distance
            if isinstance(rd, bool) or not isinstance(rd, (int, float)):
                raise ValueError(f"config.vessel.render_distance is {rd!r}, not a number: pass half_width")
            half_width = float(rd)
        if isinstance(env_ids, torch.Tensor) and env_ids.is_cuda:
            # ids outside [0, N) become -1 before the narrowing to int32, so that none can wrap into the batch
            t = env_ids.to(device=self.device).reshape(-1)
            ids = torch.where((t >= 0) & (t < self.num_envs), t, torch.full_like(t, -1)).to(torch.int32).contiguous()
        else:
            host = np.asarray(env_ids.cpu() if isinstance(env_ids, torch.Tensor) else env_ids, dtype=np.int64).reshape(-1)
            if host.size and (host.min() < 0 or host.max() >= self.num_envs):
                raise ValueError(f"env ids must be in [0, {self.num_envs}), got {host.tolist()}")
            # pinned + non_blocking: the copy is ordered on the stream without waiting for it
            ids = torch.from_numpy(host.astype(np.int32)).pin_memory().to(self.device, non_blocking=True)
        K = int(ids.numel())
        if K == 0:
            raise ValueError("render() needs at least one env id")
        frames = torch.empty((K, int(height), int(width), 3), dtype=torch.uint8, device=self.device)
        desc = _lib.AuvRender(K, int(width), int(height), 0, ids.data_ptr(), float(half_width))
        cfg, rays, paths, pool, batch = self._refs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.auv_render(cfg, rays, paths, pool, batch, C.c_void_p(self._out["obs"].data_ptr()),
                                           C.byref(desc), C.c_void_p(frames.data_ptr()), self._stream()), "auv_render")
        return frames

    # ------------------------------------------------------------------ episode tracks (record_tracks)
    def _track_slot(self, i: int) -> Optional[int]:
        if self._tracks is None:
            return None
        i, stride = int(i), self._tracks["stride"]
        if i < 0 or i % stride or i // stride >= self.record_tracks:
            return None
        return i // stride

    def _track_sync(self):
        torch.cuda.current_stream(self.device).synchronize()
        if getattr(self, "_async_stream", None) is not None:
            self._async_stream.synchronize()

    def _path_table(self, pid: int):
        from .pathbank import DevicePathBank, build_path

        bank = self.scenarios.bank
        if isinstance(bank, DevicePathBank) and bank._tables is None:  # one path, not the whole bank
            return build_path(bank.waypoints[pid])
        return bank.tables[pid]

    def _assemble(self, head_row, points_row, snap_row):
        if self.linear is None and self.k_moving and self._pool.get("host_stale"):
            # table-driven histories are re-run from the host ScenarioSet (snapshots hold no velocity tables)
            raise RuntimeError("obstacle histories of a table-driven pool are rebuilt from the host scenarios, which "
                               "GPU scenario generation has made stale: record tracks with linear_tracks='auto' "
                               "on generated pools")
        return assemble_episode(head_row, points_row, snap_row, self.track_capacity, self.k_moving, self.k_static,
                                float(self.config.simulation.t_step_size), self.linear, self.scenarios,
                                self._path_table, self.scenarios.world_polygons)

    def last_episode(self, i: int) -> Optional[dict]:
        """The most recent FINISHED episode of env ``i`` as ``BaseEnvironment.save_latest_episode`` stores it
        (environment.py:466-489): ``path``, ``path_taken`` [n + 1, 2] (row 0 = the scenario's vessel_init, the
        other rows the recorded FP32 positions after each step), ``heading_taken`` [n + 1], ``rewards`` [n],
        ``obstacles`` (``ScenarioSet.describe``-shaped, from the scenario snapshot taken when the episode
        ended, plus ``moving_path_taken`` [n + 1, k_used, 2]), ``episode``, ``timesteps``, ``collision``,
        ``reached_goal``, ``truncated`` (episode longer than ``track_capacity``: the last ``track_capacity``
        rows are kept, numbered by ``step_index``).  None when env ``i`` is not tracked or has finished no
        episode.  Synchronises the env's stream; copies one track slot."""
        slot = self._track_slot(i)
        if slot is None:
            return None
        self._track_sync()
        tk = self._tracks
        head = tk["head"][slot].cpu().numpy()
        p = pick_finished_row(head)
        if p is None:
            return None
        return self._assemble(head[p], tk["points"][slot, p].cpu().numpy(), tk["snap"][slot, p].cpu().numpy())

    def current_episode(self, i: int) -> Optional[dict]:
        """``last_episode``'s dict for the episode env ``i`` is running now (finished or not: without
        auto-reset a finished env stays on its episode until reset), read from its live pool slot -- which a
        refresh never regenerates while the env runs it.  None when env ``i`` is not tracked."""
        slot = self._track_slot(i)
        if slot is None:
            return None
        self._track_sync()
        tk, i = self._tracks, int(i)
        ep, scn = int(self._st["episode"][i].item()), int(self._st["scn_id"][i].item())
        p = ep & 1
        head = tk["head"][slot, p].cpu().numpy()
        if int(head[0]) != ep or int(head[1]) == 0:  # no step of this episode yet: the row is stale
            head = np.array([ep, 0, 0, 0, 0, scn, 0, 0], dtype=np.int32)
        pool, km, ks = self._pool, self.k_moving, self.k_static
        parts = [pool["path_id"][scn:scn + 1].to(torch.float64), pool["vessel_init"][scn]]
        if km:
            parts.append(pool["mov_lin"][scn].reshape(-1) if "mov_lin" in pool
                         else torch.zeros(8 * km, dtype=torch.float64, device=self.device))
        if ks:
            parts.append(pool["st_rec"][scn, :ks].reshape(-1))
        snap = torch.cat(parts).cpu().numpy()
        return self._assemble(head, tk["points"][slot, p].cpu().numpy(), snap)

    # ------------------------------------------------------------------ attributes the reference driver reads
    @property
    def state(self) -> torch.Tensor:
        """[6, N] FP64 vessel state x, y, psi, u, v, r."""
        return self._st["state"]

    def get_attr(self, name: str):
        """SubprocVecEnv.get_attr-shaped access to per-env counters (scripts/run.py:415-426)."""
        table = dict(
            t_step=self._st["t_step"], cumulative_reward=self._st["cum_reward"], episode=self._st["episode"],
            step_counter=self._st["step_counter"], max_progress=self._st["max_progress"], scn_id=self._st["scn_id"],
            nearby_mask=self._st["nearby_mask"], nav=self._st["nav"], obst_steps=self._st["obst_steps"],
        )
        if name in table:
            return table[name]
        if name in ("mov_pos", "mov_disp", "mov_counter"):
            return dict(zip(("mov_pos", "mov_disp", "mov_counter"), self.obstacle_state()))[name]
        if name in self._out:
            return self._out[name]
        raise AttributeError(name)

    def episode_stats(self, reduce: bool = True) -> Dict[str, float]:
        """Per-episode means in the keys of ``env.history`` (environment.py:476-489).
        With ``torch.distributed`` initialised and reduce=True the accumulators are summed
        over ranks first -- the only collective on this path (SURVEY.md section 8e)."""
        from .sharding import reduce_stats, summarize_stats

        self.check_status()
        st = self._out["stats"].clone()
        st[9] = float(self.total_steps) * self.num_envs
        if reduce:
            st = reduce_stats(st)
        return summarize_stats(st.cpu().numpy(), float(self.config.simulation.t_step_size))

    def close(self):
        if self._pipe:
            torch.cuda.synchronize(self.device)
            self.lib.auv_pipeline_destroy(self._pipe)
            self._pipe = None
            self._async_call = None  # (its argument list holds the destroyed pipeline)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EnvGroupRing:
    """G env groups stepped out of order: ``send(g, actions)`` submits group g's step (step_async),
    ``recv()`` returns ``(g, obs, reward, done)`` of the first group whose step has finished and whose
    results are complete in host memory.  Unlike a fixed ``wait(A); submit(A); wait(B); submit(B)`` loop --
    which pulls the groups into lock-step (a group that finishes early is only resubmitted after the one
    before it, so all of them compute at the same time and then queue on the host link together) -- the
    groups keep whatever phase offset they have, and with G >= 3 the link and the SMs both stay busy
    while the host turns one group around."""

    def __init__(self, groups):
        self.groups = list(groups)
        self.pending = []  # group indices in submission order
        self.spins = 0

    def __len__(self):
        return len(self.groups)

    @property
    def envs_per_group(self) -> int:
        return self.groups[0].num_envs

    def reset(self):
        return [g.reset() for g in self.groups]

    def send(self, g: int, actions: np.ndarray):
        self.groups[g].step_async(actions)
        self.pending.append(g)

    def recv(self):
        if not self.pending:
            raise RuntimeError("recv() with no step in flight")
        t0 = time.perf_counter()
        while True:
            for k, g in enumerate(self.pending):
                if self.groups[g]._async_done.query():
                    del self.pending[k]
                    self.groups[g].wait_seconds += time.perf_counter() - t0
                    obs, rew, done = self.groups[g].step_wait()
                    return g, obs, rew, done
            self.spins += 1

    def drain(self):
        out = []
        while self.pending:
            out.append(self.recv())
        return out

    def close(self):
        for g in self.groups:
            g.close()
        self.groups = []
