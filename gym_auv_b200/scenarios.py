"""Batched scenario plug-ins: what the reference's ``_generate()`` hooks produce, as
struct-of-arrays for M scenarios at once.

Reference anchors: envs/movingobstacles.py:28-120 (MovingObstacles family),
envs/testscenario.py:20-360 (deterministic fixtures), utils/helpers.py:5-35
(obstacle rejection sampler), objects/obstacles.py:144-215 (VesselObstacle track /
velocity table / update), objects/path.py:96-120 (random curve).

A ``ScenarioSet`` is pure host data (NumPy).  ``describe(i)`` returns the neutral
single-scenario dict that the parity tests inject into the CPU oracle, so both sides
always run the same scenario (the reference's generation mixes a seeded and the global
unseeded RNG -- SURVEY.md quirk #9 -- so seeds alone cannot reproduce it).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from .pathbank import DevicePathBank, PathBank, PathTable, build_path, random_curve_waypoints

VESSEL_TRACK_LEN = 9999  # a 10000-point trajectory yields 9999 per-second velocities
# GPU scenario generation in a shared land-polygon world: a vessel start must be clear of land by this much
# (outside every polygon, farther from every ring) -- the margin random_land keeps around vessel starts
LAND_CLEARANCE = 30.0


def princip(a):
    return ((a + np.pi) % (2 * np.pi)) - np.pi


@dataclass
class ScenarioSet:
    waypoints: List[np.ndarray]  # P arrays [2, n_wp]
    path_id: np.ndarray  # [M] int32
    vessel_init: np.ndarray  # [M, 3]
    mov_start: np.ndarray  # [M, Km, 2]
    mov_width: np.ndarray  # [M, Km]   (<= 0: unused slot)
    mov_track: np.ndarray  # [M, Km, 4] int32: vel_off, vel_len, vel_stride, 0
    vel_table: np.ndarray  # [n_vel, 2]
    st_pos: np.ndarray  # [M, Ks, 2]
    st_radius: np.ndarray  # [M, Ks]   (<= 0: unused slot)
    rewarder: str = "colav"
    post_generate_update: bool = False  # scenario's _generate() ends with self._update()
    name: str = ""
    world_polygons: List[np.ndarray] = field(default_factory=list)  # static land shared by all scenarios
    # path-major layout: scenario m follows path ((m mod path_period) // path_group) mod n_paths, so that
    # consecutive envs share a path (0 = no such structure; the GPU generator then draws paths at random)
    path_group: int = 0
    path_period: int = 0
    _bank: Optional[PathBank] = field(default=None, repr=False)
    _world: Optional[object] = field(default=None, repr=False)

    @property
    def n_scenarios(self) -> int:
        return int(self.path_id.shape[0])

    @property
    def k_moving(self) -> int:
        return int(self.mov_width.shape[1])

    @property
    def k_static(self) -> int:
        return int(self.st_radius.shape[1])

    @property
    def bank(self) -> PathBank:
        if self._bank is None:
            self._bank = PathBank.from_waypoints(self.waypoints)
        return self._bank

    @property
    def world(self):
        if self._world is None:
            from .polygons import World

            self._world = World(self.world_polygons)
        return self._world

    def validate(self):
        if np.any(self.st_radius < 0):
            raise ValueError("negative obstacle radius")  # obstacles.py:95-96
        if self.path_id.min() < 0 or self.path_id.max() >= len(self.waypoints):
            raise ValueError("path_id out of range")

    # -- state right after reset(): VesselObstacle.__init__ does update(dt=0.1)
    #    (obstacles.py:192-193) and MovingObstacles/TestHeadOn/TestCrossing end their
    #    _generate() with one more self._update() (movingobstacles.py:95)
    def initial_obstacle_state(self, dt: float):
        pos = self.mov_start.astype(np.float64).copy()
        counter = np.zeros(self.mov_width.shape, dtype=np.float64)
        disp = np.zeros_like(pos)
        steps = [0.1] + ([dt] if self.post_generate_update else [])
        for h in steps:
            pos, disp, counter = advance_obstacles(self, pos, counter, h)
        return pos, disp, counter

    def linear_track_info(self, dt: float):
        """``dict(vel_len, counter0)`` when every used moving slot follows a constant-velocity track
        (stride 0) of one common length -- the MovingObstacles family, movingobstacles.py:51-75 --
        else None.  Such pools are stepped with the closed form of ``VesselObstacle._update``."""
        if self.k_moving == 0:
            return None
        used = self.mov_width > 0
        tr = self.mov_track[used] if used.any() else self.mov_track.reshape(-1, 4)
        if len(tr) == 0 or np.any(tr[:, 2] != 0) or np.any(tr[:, 1] != tr[0, 1]) or tr[0, 1] < 2:
            return None
        return dict(vel_len=int(tr[0, 1]), counter0=0.1 + (float(dt) if self.post_generate_update else 0.0))

    def describe(self, i: int) -> dict:
        """Neutral single-scenario description (input of oracle.sim.OracleEnv)."""
        mov = None
        if self.k_moving:
            used = self.mov_width[i] > 0
            tables = []
            for j in np.nonzero(used)[0]:
                off, ln, stride, _ = self.mov_track[i, j]
                tables.append(self.vel_table[off + np.arange(ln) * stride])
            mov = dict(width=self.mov_width[i][used], start=self.mov_start[i][used], vel_tables=tables)
        st = None
        if self.k_static:
            used = self.st_radius[i] > 0
            st = dict(pos=self.st_pos[i][used], radius=self.st_radius[i][used])
        return dict(
            waypoints=self.waypoints[int(self.path_id[i])],
            vessel_init=self.vessel_init[i].copy(),
            moving=mov,
            static=st,
            rewarder=self.rewarder,
            post_generate_update=self.post_generate_update,
            polygons=[np.asarray(p, dtype=np.float64) for p in self.world_polygons],
        )


def advance_obstacles(scn: ScenarioSet, pos, counter, dt):
    """Vectorised ``VesselObstacle._update`` (obstacles.py:195-215)."""
    counter = counter + dt
    index = np.floor(counter).astype(np.int64)
    vlen = scn.mov_track[..., 1].astype(np.int64)
    wrap = index >= vlen - 1
    counter = np.where(wrap, 0.0, counter)
    index = np.where(wrap, 0, index)
    pos = np.where(wrap[..., None], scn.mov_start, pos)
    if scn.vel_table.shape[0] == 0:
        v = np.zeros(pos.shape)
    else:
        v = scn.vel_table[scn.mov_track[..., 0].astype(np.int64) + index * scn.mov_track[..., 2]]
    disp = dt * v
    used = (scn.mov_width > 0)[..., None]
    return np.where(used, pos + disp, pos), np.where(used, disp, 0.0), np.where(used[..., 0], counter, 0.0)


def _two_sum(a, b):
    """s + e == a + b exactly, s = RN(a + b) (Knuth)."""
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _fma(a, b, c):
    """Correctly rounded a * b + c element-wise -- the device's fma -- vectorised: a * b is split exactly into
    uh + ul (Dekker's product), c + uh into th + tl (TwoSum), tl + ul is rounded to odd, and th plus that is
    rounded to nearest once (Boldo & Melquiond, "Emulation of FMA and correctly rounded sums: proved
    algorithms using rounding to odd", IEEE TC 57(4), 2008; exact barring overflow / underflow)."""
    a, b, c = np.broadcast_arrays(np.asarray(a, np.float64), np.asarray(b, np.float64), np.asarray(c, np.float64))
    split = 134217729.0  # 2^27 + 1
    t = split * a
    ah = t - (t - a)
    al = a - ah
    t = split * b
    bh = t - (t - b)
    bl = b - bh
    uh = a * b
    ul = ((ah * bh - uh) + ah * bl + al * bh) + al * bl
    th, tl = _two_sum(c, uh)
    v, ve = _two_sum(tl, ul)
    # round to odd: an inexact v with an even significand moves one ulp towards the exact sum
    fix = (ve != 0) & ((v.view(np.int64) & 1) == 0)
    v = np.where(fix, np.nextafter(v, np.where(ve > 0, np.inf, -np.inf)), v)
    return th + v


def linear_track_positions(rec, n, first_wrap: int, wrap_period: int):
    """Positions of constant-velocity obstacle tracks after ``n`` updates since reset -- the closed form
    of obstacles.py:195-215 that the step and ``auv_obstacle_state`` evaluate (AuvScenarioPool.linear_tracks):
        n <  first_wrap : pos0 + n d
        n >= first_wrap : start + ((n - first_wrap) mod wrap_period + 1) d
    ``rec`` [k, 8] packed pool.mov_lin records (pos0, d, width, start, 0), ``n`` int array [S].
    Returns [S, k, 2], FP64 with fused multiply-adds: bit-identical to the device."""
    rec = np.asarray(rec, np.float64).reshape(-1, 8)
    n = np.asarray(n, np.int64).reshape(-1, 1, 1)
    wrapped = n >= first_wrap
    m = np.where(wrapped, (n - first_wrap) % wrap_period + 1, n).astype(np.float64)
    base = np.where(wrapped, rec[None, :, 5:7], rec[None, :, 0:2])
    return _fma(m, rec[None, :, 2:4], base)


def table_track_positions(scn: ScenarioSet, m: int, n, dt: float):
    """Positions of the moving obstacles of pool scenario ``m`` after ``n`` updates since reset ([S] ints,
    non-decreasing not required): ``initial_obstacle_state`` followed by ``advance_obstacles`` step by step.
    Returns [S, Km, 2]."""
    from types import SimpleNamespace

    one = SimpleNamespace(mov_start=scn.mov_start[m], mov_width=scn.mov_width[m], mov_track=scn.mov_track[m],
                          vel_table=scn.vel_table, post_generate_update=scn.post_generate_update)
    pos, _, counter = ScenarioSet.initial_obstacle_state(one, dt)
    n = np.asarray(n, np.int64).reshape(-1)
    out = np.zeros((n.size, one.mov_width.shape[0], 2))
    order = np.argsort(n, kind="stable")
    u = 0
    for k in order:
        while u < n[k]:
            pos, _, counter = advance_obstacles(one, pos, counter, dt)
            u += 1
        out[k] = pos
    return out


def _empty_moving(M):
    return (
        np.zeros((M, 0, 2)),
        np.zeros((M, 0)),
        np.zeros((M, 0, 4), dtype=np.int32),
        np.zeros((0, 2)),
    )


# ---------------------------------------------------------------------------------
# MovingObstacles family  (movingobstacles.py:28-120, helpers.py:5-35)
# ---------------------------------------------------------------------------------


def _sample_obstacles(rng, grng, path: PathTable, vessel_xy, count, n, disp_std, radius_mean, width):
    """``helpers.generate_obstacle`` for `count` scenarios x `n` slots sharing one path.
    rng = the env's seeded stream, grng = stand-in for the reference's global np.random."""
    pos = np.zeros((count, n, 2))
    rad = np.zeros((count, n))
    todo = np.ones((count, n), dtype=bool)
    goal = path(path.length)
    while todo.any():
        k = int(todo.sum())
        disp = grng.normal(0, disp_std, size=k)
        s = (0.1 + 0.8 * rng.rand(k)) * path.length
        p = path(s).T  # [k, 2]
        ang = princip(path.direction(s) - np.pi / 2)
        p = p + disp[:, None] * np.stack([np.cos(ang), np.sin(ang)], axis=1)
        r = np.maximum(1, grng.poisson(radius_mean, size=k)).astype(np.float64)
        ci, _ = np.nonzero(todo)
        vdist = np.linalg.norm(p - vessel_xy[ci], axis=1) - width - r
        gdist = np.linalg.norm(p - goal[None, :], axis=1) - r
        ok = np.minimum(vdist, gdist) > 0
        idx = np.argwhere(todo)
        acc = idx[ok]
        pos[acc[:, 0], acc[:, 1]] = p[ok]
        rad[acc[:, 0], acc[:, 1]] = r[ok]
        todo[acc[:, 0], acc[:, 1]] = False
    return pos, rad


def moving_obstacles(
    n_scenarios: int,
    n_moving: int = 17,
    n_static: int = 11,
    seed: int = 0,
    n_paths: Optional[int] = None,
    rewarder: str = "colav",
    vessel_width: float = 1.255,
    path_length: float = 800.0,
    name: str = "MovingObstaclesNoRules-v0",
    path_period: Optional[int] = None,
) -> ScenarioSet:
    """M scenarios distributed like ``MovingObstacles._generate``.  ``n_paths`` distinct
    random curves are shared by index, path-major (None = one path per scenario): scenario m
    follows path ``((m mod path_period) // group) mod P`` with ``group = path_period // P`` and
    ``path_period`` = M by default -- consecutive scenarios (hence consecutive envs, hence whole
    CTAs of the step kernels) share a path."""
    M = int(n_scenarios)
    P = M if n_paths is None else int(min(n_paths, M))
    period, group = _path_layout(M, P, path_period)
    rng = np.random.RandomState(seed)
    grng = np.random.RandomState(seed + 0x5EED)
    wps = []
    for _ in range(P):
        nwp = int(np.floor(4 * rng.rand() + 2))
        wps.append(random_curve_waypoints(rng, nwp, length=path_length))
    tables = [build_path(w) for w in wps]
    path_id = _path_major_ids(M, P, period, group)
    vessel_init = np.zeros((M, 3))
    mov_start = np.zeros((M, n_moving, 2))
    mov_width = np.zeros((M, n_moving))
    mov_vel = np.zeros((M, n_moving, 2))
    st_pos = np.zeros((M, n_static, 2))
    st_radius = np.zeros((M, n_static))
    for p in range(P):
        members = np.nonzero(path_id == p)[0]
        c = len(members)
        tab = tables[p]
        init = np.tile(tab(0.0), (c, 1))
        init += 50 * (rng.rand(c, 2) - 0.5)
        ang = princip(tab.direction(0.0) + 2 * np.pi * (rng.rand(c) - 0.5))
        vessel_init[members, 0:2] = init
        vessel_init[members, 2] = ang
        if n_moving:
            pos, rad = _sample_obstacles(rng, grng, tab, init, c, n_moving, 500, 10, vessel_width)
            direction = rng.rand(c, n_moving) * 2 * np.pi
            speed = grng.uniform(1, 3, size=(c, n_moving))
            mov_start[members] = pos
            mov_width[members] = rad
            mov_vel[members] = speed[..., None] * np.stack([np.cos(direction), np.sin(direction)], axis=-1)
        if n_static:
            pos, rad = _sample_obstacles(rng, grng, tab, init, c, n_static, 250, 30, vessel_width)
            st_pos[members] = pos
            st_radius[members] = rad
    # constant-velocity tracks: one table entry per obstacle, stride 0
    vel_table = mov_vel.reshape(-1, 2).copy()
    mov_track = np.zeros((M, n_moving, 4), dtype=np.int32)
    mov_track[..., 0] = np.arange(M * n_moving).reshape(M, n_moving)
    mov_track[..., 1] = VESSEL_TRACK_LEN
    mov_track[..., 2] = 0
    scn = ScenarioSet(
        waypoints=wps, path_id=path_id, vessel_init=vessel_init, mov_start=mov_start, mov_width=mov_width,
        mov_track=mov_track, vel_table=vel_table, st_pos=st_pos, st_radius=st_radius, rewarder=rewarder,
        post_generate_update=True, name=name, path_group=group, path_period=period,
    )
    scn._bank = PathBank(tables)
    return scn


def _path_layout(M: int, P: int, path_period: Optional[int]):
    period = int(path_period) if path_period else M
    group = max(1, period // P)
    return period, group


def _path_major_ids(M: int, P: int, period: int, group: int) -> np.ndarray:
    return (((np.arange(M) % period) // group) % P).astype(np.int32)


def moving_obstacles_template(
    n_scenarios: int,
    n_moving: int = 17,
    n_static: int = 11,
    seed: int = 0,
    n_paths: int = 1024,
    rewarder: str = "colav",
    path_length: float = 800.0,
    name: str = "MovingObstaclesNoRules-v0",
    path_period: Optional[int] = None,
    device_paths: bool = False,
) -> ScenarioSet:
    """Path bank + EMPTY obstacle slots for M scenarios: the input of
    ``AUVVecEnv.regenerate_scenarios`` (GPU-side sampling of vessel starts and obstacles).  Only
    the random curves (path.py:96-120, three SciPy PCHIP fits each) are built on the host."""
    M, P = int(n_scenarios), int(min(n_paths, n_scenarios))
    rng = np.random.RandomState(seed)
    wps = []
    for _ in range(P):
        nwp = int(np.floor(4 * rng.rand() + 2))
        wps.append(random_curve_waypoints(rng, nwp, length=path_length))
    period, group = _path_layout(M, P, path_period)
    path_id = _path_major_ids(M, P, period, group)
    vessel_init = np.zeros((M, 3))
    if device_paths:  # the path tables are built on the GPU too (auv_pathbank_build); vessel starts are generated there
        tables = None
    else:
        tables = [build_path(w) for w in wps]
        for p in range(P):
            vessel_init[path_id == p, 0:2] = tables[p](0.0)
    mov_track = np.zeros((M, n_moving, 4), dtype=np.int32)
    mov_track[..., 0] = np.arange(M * n_moving).reshape(M, n_moving)
    mov_track[..., 1] = VESSEL_TRACK_LEN
    scn = ScenarioSet(
        waypoints=wps, path_id=path_id, vessel_init=vessel_init, mov_start=np.zeros((M, n_moving, 2)),
        mov_width=np.zeros((M, n_moving)), mov_track=mov_track, vel_table=np.zeros((M * n_moving, 2)),
        st_pos=np.zeros((M, n_static, 2)), st_radius=np.zeros((M, n_static)), rewarder=rewarder,
        post_generate_update=True, name=name, path_group=group, path_period=period,
    )
    scn._bank = DevicePathBank(wps) if device_paths else PathBank(tables)
    return scn


def path_follow_no_obstacles(n_scenarios: int, seed: int = 0, n_paths: Optional[int] = None) -> ScenarioSet:
    """``PathFollowNoObstacles`` (movingobstacles.py:114-120)."""
    return moving_obstacles(
        n_scenarios, 0, 0, seed=seed, n_paths=n_paths, rewarder="pathfollow", name="PathFollowNoObstacles-v0"
    )


# ---------------------------------------------------------------------------------
# Deterministic fixtures  (testscenario.py)
# ---------------------------------------------------------------------------------


def _single(waypoints, vessel_init=None, static=None, moving_traj=None, rewarder="colav", post_update=False,
            name="") -> ScenarioSet:
    """One scenario from explicit pieces.  static = list of (pos, radius);
    moving_traj = list of (width, trajectory[(t_int, (x, y)), ...])."""
    wp = np.array(waypoints, dtype=np.float64)
    tab = build_path(wp)
    if vessel_init is None:
        vessel_init = np.hstack([tab(0.0), tab.direction(0.0)])
    static = static or []
    moving_traj = moving_traj or []
    ks, km = len(static), len(moving_traj)
    st_pos = np.zeros((1, ks, 2))
    st_radius = np.zeros((1, ks))
    for j, (pos, r) in enumerate(static):
        if r < 0:
            raise ValueError("negative obstacle radius")
        st_pos[0, j] = np.asarray(pos, dtype=np.float64).flatten()
        st_radius[0, j] = r
    mov_start = np.zeros((1, km, 2))
    mov_width = np.zeros((1, km))
    mov_track = np.zeros((1, km, 4), dtype=np.int32)
    vels = []
    off = 0
    for j, (width, traj) in enumerate(moving_traj):
        t = np.array([p[0] for p in traj], dtype=np.int64)
        xy = np.array([p[1] for p in traj], dtype=np.float64)
        v = (xy[1:] - xy[:-1]) / (t[1:] - t[:-1])[:, None]  # obstacles.py:160-172
        v = np.repeat(v, (t[1:] - t[:-1]), axis=0)
        vels.append(v)
        mov_start[0, j] = xy[0]
        mov_width[0, j] = width
        mov_track[0, j] = (off, len(v), 1, 0)
        off += len(v)
    vel_table = np.concatenate(vels, axis=0) if vels else np.zeros((0, 2))
    scn = ScenarioSet(
        waypoints=[wp], path_id=np.zeros(1, dtype=np.int32), vessel_init=np.asarray(vessel_init)[None, :],
        mov_start=mov_start, mov_width=mov_width, mov_track=mov_track, vel_table=vel_table, st_pos=st_pos,
        st_radius=st_radius, rewarder=rewarder, post_generate_update=post_update, name=name,
    )
    scn._bank = PathBank([tab])
    return scn


def test_scenario1() -> ScenarioSet:  # testscenario.py:20-37
    wp = [[0, 1100], [0, 1100]]
    tab = build_path(wp)
    static = []
    arc = 30
    for o in range(20):
        r = 10 + 10 * o**1.5
        arc += r * 2 + 30
        static.append((tab(arc), r))
    return _single(wp, static=static, name="TestScenario1-v0")


def test_scenario2() -> ScenarioSet:  # testscenario.py:40-83
    wp = np.vstack([[t * np.cos(t / 100), 2 * t] for t in range(500)]).T
    tab = build_path(wp)
    static = []
    arc, r = 30, 5
    while True:
        arc += 2 * r
        if arc >= tab.length:
            break
        dist = 140 - 120 / (1 + np.exp(-0.005 * arc))
        pos = tab(arc)
        ang = tab.direction(arc) - np.pi / 2
        disp = dist * np.array([np.cos(ang), np.sin(ang)])
        static.append((pos + disp, r))
        static.append((pos - disp, r))
    return _single(wp, static=static, name="TestScenario2-v0")


def test_scenario3() -> ScenarioSet:  # testscenario.py:86-105
    wp = np.vstack([[0, 0], [0, 500]]).T
    static = []
    for n in range(21):
        ang = np.pi / 4 + n / 20 * np.pi / 2
        static.append((np.array([np.cos(ang) * 100, np.sin(ang) * 100]), 25))
    return _single(wp, static=static, name="TestScenario3-v0")


def test_scenario4() -> ScenarioSet:  # testscenario.py:108-128
    wp = np.vstack([[0, 0], [0, 500]]).T
    static = []
    for n in range(21):
        ang = n / 20 * 2 * np.pi
        if abs(ang < 3 / 2 * np.pi) < np.pi / 12:  # sic: reference compares a bool
            continue
        static.append((np.array([np.cos(ang) * 100, np.sin(ang) * 100]), 25))
    return _single(wp, static=static, name="TestScenario4-v0")


def _straight_vessel_track(start, step_xy, n=5000):
    return [(i, (start[0] + step_xy[0] * i, start[1] + step_xy[1] * i)) for i in range(n)]


def test_head_on(start_angle: float = 0.0) -> ScenarioSet:  # testscenario.py:131-170
    """The reference draws start_angle ~ U(-5deg, 5deg) from the global `random`;
    it is an explicit argument here."""
    wp = np.vstack([[0, 0], [0, 250]]).T
    tab = build_path(wp)
    v0 = tab(0.0)
    sx = v0[0] + 150 * np.sin(start_angle)
    sy = v0[1] + 150 * np.cos(start_angle)
    traj = _straight_vessel_track((sx, sy), (-0.5 * np.sin(start_angle), -0.5 * np.cos(start_angle)))
    return _single(wp, moving_traj=[(30, traj)], post_update=True, name="TestHeadOn-v0")


def _crossing(shift_deg, start_deg, name):
    wp = np.vstack([[0, 0], [0, 500]]).T
    tab = build_path(wp)
    v0 = tab(0.0)
    sh, sa = np.deg2rad(shift_deg), np.deg2rad(start_deg)
    sx = v0[0] + 200 * np.sin(sa)
    sy = v0[1] + 200 * np.cos(sa)
    traj = _straight_vessel_track((sx, sy), (0.5 * np.sin(sh), 0.5 * np.cos(sh)))
    return _single(wp, moving_traj=[(30, traj)], post_update=True, name=name)


def test_crossing() -> ScenarioSet:  # testscenario.py:173-213
    return _crossing(90, -45, "TestCrossing-v0")


def test_crossing1() -> ScenarioSet:  # testscenario.py:216-256
    return _crossing(-50, 70, "TestCrossing1-v0")


def empty_scenario() -> ScenarioSet:  # testscenario.py:259-278
    wp = np.vstack([[25, 10], [25, 200]]).T
    return _single(wp, name="EmptyScenario-v0")


def debug_scenario(seed: int = 0) -> ScenarioSet:  # testscenario.py:281-350
    rng = np.random.RandomState(seed)
    wp = np.vstack([[250, 100], [250, 200]]).T
    moving = []
    i = np.arange(10000)
    for k in range(5):
        shift = rng.rand() * 2 * np.pi
        radius = rng.rand() * 40 + 30
        speed = rng.rand() * 0.003 + 0.003
        xs = 250 + radius * np.cos(speed * i + shift)
        ys = 150 + 70 * k + radius * np.sin(speed * i + shift)
        moving.append((6, [(int(t), (xs[t], ys[t])) for t in i]))
    for k in range(5):
        start = rng.rand() * 200 + 150
        speed = rng.rand() * 0.03 + 0.03
        shift = 10 * rng.rand()
        moving.append((6, [(int(t), (245 + 2.5 * k + shift, start - 10 * speed * t)) for t in i]))
    return _single(wp, moving_traj=moving, name="DebugScenario-v0")


def concat(sets: List[ScenarioSet]) -> ScenarioSet:
    """Stack scenario sets (padding obstacle slots) into one pool."""
    km = max(s.k_moving for s in sets)
    ks = max(s.k_static for s in sets)
    wps, pid, vinit, mstart, mwidth, mtrack, vtab, spos, srad = [], [], [], [], [], [], [], [], []
    poff = voff = 0
    tables = []
    for s in sets:
        M = s.n_scenarios
        wps += s.waypoints
        tables += s.bank.tables
        pid.append(s.path_id + poff)
        poff += len(s.waypoints)
        vinit.append(s.vessel_init)

        def pad(a, k, axis=1):
            w = [(0, 0)] * a.ndim
            w[axis] = (0, k - a.shape[axis])
            return np.pad(a, w)

        mstart.append(pad(s.mov_start, km))
        mwidth.append(pad(s.mov_width, km))
        tr = s.mov_track.copy()
        tr[..., 0] += voff
        mtrack.append(pad(tr, km))
        vtab.append(s.vel_table)
        voff += len(s.vel_table)
        spos.append(pad(s.st_pos, ks))
        srad.append(pad(s.st_radius, ks))
        assert M == s.vessel_init.shape[0]
    out = ScenarioSet(
        waypoints=wps, path_id=np.concatenate(pid).astype(np.int32), vessel_init=np.concatenate(vinit),
        mov_start=np.concatenate(mstart), mov_width=np.concatenate(mwidth), mov_track=np.concatenate(mtrack),
        vel_table=np.concatenate(vtab) if vtab else np.zeros((0, 2)), st_pos=np.concatenate(spos),
        st_radius=np.concatenate(srad), rewarder=sets[0].rewarder,
        post_generate_update=sets[0].post_generate_update, name="+".join(s.name for s in sets),
    )
    if any(s.post_generate_update != sets[0].post_generate_update for s in sets):
        raise ValueError("cannot concat scenario sets with different post_generate_update")
    out._bank = PathBank(tables)
    return out


def land_scenarios(n_scenarios: int, n_polygons: int = 512, n_moving: int = 0, n_static: int = 0, seed: int = 0,
                   n_paths: Optional[int] = None, extent: float = 6000.0) -> ScenarioSet:
    """BASELINE config 4 shape: MovingObstacles-style scenarios inside one shared world of
    static land polygons (synthetic; envs/realworld.py's data files are not shipped)."""
    from .polygons import random_land

    scn = moving_obstacles(n_scenarios, n_moving, n_static, seed=seed, n_paths=n_paths, name="LandPolygons")
    scn.world_polygons = random_land(n_polygons, extent, seed=seed + 77, keep_clear=scn.vessel_init[:, :2])
    return scn


def land_template(n_scenarios: int, n_polygons: int = 512, n_moving: int = 16, n_static: int = 16, seed: int = 0,
                  n_paths: int = 1024, extent: float = 6000.0, path_period: Optional[int] = None,
                  device_paths: bool = False) -> ScenarioSet:
    """``moving_obstacles_template`` inside a shared world of ``random_land`` polygons: the input of
    ``AUVVecEnv.regenerate_scenarios`` for the BASELINE config 4 shape with a fresh scenario per episode.
    Land is kept clear of every bank path's first and last waypoint by ``25 sqrt(2) + LAND_CLEARANCE + 1`` m,
    so that every corner of a path's +-25 m start square is clear of land by LAND_CLEARANCE and the
    template's own bank never forces a vessel start to be redrawn."""
    from .polygons import random_land

    scn = moving_obstacles_template(n_scenarios, n_moving, n_static, seed=seed, n_paths=n_paths, name="LandPolygons",
                                    path_period=path_period, device_paths=device_paths)
    ends = np.array([[w[0, 0], w[1, 0]] for w in scn.waypoints] + [[w[0, -1], w[1, -1]] for w in scn.waypoints])
    scn.world_polygons = random_land(n_polygons, extent, seed=seed + 77, keep_clear=ends,
                                     clear_margin=25.0 * np.sqrt(2.0) + LAND_CLEARANCE + 1.0)
    return scn


# registry: scenario id -> (builder, rewarder default); mirrors gym_auv/__init__.py:43-121
SCENARIOS = {
    "TestScenario1-v0": test_scenario1,
    "TestScenario2-v0": test_scenario2,
    "TestScenario3-v0": test_scenario3,
    "TestScenario4-v0": test_scenario4,
    "TestHeadOn-v0": test_head_on,
    "TestCrossing-v0": test_crossing,
    "TestCrossing1-v0": test_crossing1,
    "DebugScenario-v0": debug_scenario,
    "EmptyScenario-v0": empty_scenario,
    "MovingObstaclesNoRules-v0": lambda seed=0, n=1: moving_obstacles(n, 17, 11, seed=seed),
    "PathFollowNoObstacles-v0": lambda seed=0, n=1: path_follow_no_obstacles(n, seed=seed),
}
