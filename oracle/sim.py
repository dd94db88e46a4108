"""FP64 single-env restatement of the reference's step path.  TEST INFRASTRUCTURE.

An ``OracleEnv`` is built from a *scenario description* (plain dict of NumPy
arrays -- the same dict the product's scenario generators emit, see
``gym_auv_b200/scenarios.py``) so that the oracle and the CUDA path always
run on identical injected scenarios (the reference's own generation mixes a
seeded and an unseeded RNG, SURVEY.md quirk #9).

Reference anchors (file:line under /root/reference/gym_auv):
  environment.py:176-245 reset, :247-290 observe, :292-366 step, :375-384 _isdone,
  :386-392 _update;  objects/vessel/vessel.py:189-224 reset, :226-247 step,
  :249-368 perceive, :370-428 sensor loop, :461-541 navigate;
  objects/vessel/sensor.py:22-97 culling, :140-159 simulate_sensor;
  objects/path.py:19-93;  objects/obstacles.py:90-113 circle, :144-233 vessel
  obstacle, :235-262 enclosing circle;  objects/rewarder.py:78-140, :167-241.
"""
from __future__ import annotations

import math

import numpy as np
from scipy import interpolate

from . import geos_lite as G
from . import model as M

# defaults of gym_auv/config.py (declared values, not the DEBUG_CONFIG-mutated ones)
DEFAULT_CFG = dict(
    min_cumulative_reward=-2000.0,
    max_timesteps=10000,
    min_goal_distance=5.0,
    min_path_progress=0.99,
    t_step_size=1.0,
    thrust_max_auv=2.0,
    moment_max_auv=0.15,
    vessel_width=1.255,
    look_ahead_distance=300.0,
    use_lidar=True,
    sensor_interval_load_obstacles=25,
    n_sensors_per_sector=20,
    n_sectors=9,
    sensor_range=150.0,
    sensor_log_transform=True,
    sensor_use_velocity_observations=False,
    # "zero": simulate_sensor at HEAD returns (0, 0) speeds (sensor.py:140-159);
    # "nearest": simulate_sensor_brute_force (sensor.py:100-137)
    velocity_mode="zero",
)


# ---------------------------------------------------------------------------------
# Path (path.py:19-93)
# ---------------------------------------------------------------------------------


def _arc_len(coords):
    diff = np.diff(coords, axis=1)
    return np.concatenate([[0.0], np.cumsum(np.sqrt(np.sum(diff**2, axis=0)))])


class OraclePath:
    def __init__(self, waypoints):
        wp = np.array(waypoints, dtype=np.float64)
        for _ in range(3):
            arc = _arc_len(wp)
            spline = interpolate.PchipInterpolator(arc, wp, axis=1)
            wp = spline(np.linspace(arc[0], arc[-1], 1000))
        self.arclengths = arc
        self.spline = spline
        self.dspline = spline.derivative()
        self.length = float(arc[-1])
        samples = np.linspace(0, self.length, int(10 * self.length))
        self.points = np.transpose(spline(samples))  # (n, 2) 0.1 m polyline

    def __call__(self, s):
        return self.spline(s)

    @property
    def end(self):
        return self.spline(self.length)

    def direction(self, s):
        d = self.dspline(s)
        return math.atan2(d[1], d[0])

    def closest_arclength(self, pos):
        return G.linestring_project(self.points, pos)


# ---------------------------------------------------------------------------------
# Obstacles (obstacles.py)
# ---------------------------------------------------------------------------------


class OracleCircle:
    """CircularObstacle: boundary is a RING (LineString), obstacles.py:90-113."""

    static = True
    filled = False

    def __init__(self, position, radius):
        if radius < 0:
            raise ValueError("negative radius")
        self.position = np.array(position, dtype=np.float64).flatten()
        self.radius = float(radius)
        self.ring = G.circle_boundary_ring(self.position[0], self.position[1], self.radius)

    def enclosing_circle(self):
        return self.position, self.radius


class OraclePolygon:
    """PolygonObstacle: static FILLED polygon, enclosing circle cached
    (obstacles.py:116-127)."""

    static = True
    filled = True

    def __init__(self, points):
        pts = np.array(points, dtype=np.float64)
        if not np.array_equal(pts[0], pts[-1]):
            pts = np.vstack([pts, pts[:1]])
        self.ring = pts
        self._circle = G.enclosing_circle_of_ring(self.ring)

    def enclosing_circle(self):
        return self._circle


class OracleVesselObstacle:
    """VesselObstacle (obstacles.py:144-233).  ``vel_table`` is the per-integer-second
    velocity list the reference derives from the trajectory (:160-172)."""

    static = False
    filled = True

    def __init__(self, width, start, vel_table, init_update=True):
        self.width = float(width)
        self.start = np.array(start, dtype=np.float64)
        self.vel = np.asarray(vel_table, dtype=np.float64)
        self.counter = 0.0
        w = self.width
        self.body = np.array(
            [(-w / 2, -w / 2), (-w / 2, w / 2), (w / 2, w / 2), (3 / 2 * w, 0.0), (w / 2, -w / 2), (-w / 2, -w / 2)]
        )
        self.position = self.start.copy()
        self.heading = math.pi / 2
        self.dx = 0.0
        self.dy = 0.0
        self._rebuild()
        if init_update:
            self.update(0.1)

    @classmethod
    def from_trajectory(cls, width, trajectory, init_update=True):
        """trajectory = [(t_int, (x, y)), ...] as in the reference scenarios."""
        vel = []
        for i in range(len(trajectory) - 1):
            t0, p0 = trajectory[i]
            t1, p1 = trajectory[i + 1]
            dx = (p1[0] - p0[0]) / (t1 - t0)
            dy = (p1[1] - p0[1]) / (t1 - t0)
            vel.extend([(dx, dy)] * (t1 - t0))
        return cls(width, trajectory[0][1], np.array(vel), init_update)

    def update(self, dt):
        self.counter += dt
        idx = int(np.floor(self.counter))
        if idx >= len(self.vel) - 1:
            self.counter = 0
            idx = 0
            self.position = self.start.copy()
        self.dx = dt * self.vel[idx][0]
        self.dy = dt * self.vel[idx][1]
        self.heading = math.atan2(self.dy, self.dx)
        self.position = self.position + np.array([self.dx, self.dy])
        self._rebuild()

    def _rebuild(self):
        ring = G.rotate_about(self.body, self.heading, G.polygon_centroid(self.body))
        self.ring = ring + self.position

    def enclosing_circle(self):
        # NOT cached in the reference: MRR of the current boundary every call
        return G.enclosing_circle_of_ring(self.ring)


# ---------------------------------------------------------------------------------
# LiDAR culling + casting (sensor.py)
# ---------------------------------------------------------------------------------


def limit_angle_rays(centre, radius, p0, heading, angle_per_ray):
    """sensor.py:22-71 -> (idx_min_ray, idx_max_ray) before the -1 / modulo."""
    dist = math.hypot(centre[0] - p0[0], centre[1] - p0[1])
    safe = max(1e-8, dist)
    ratio = radius / safe
    delta = math.asin(ratio) if ratio <= 1.0 else math.pi  # np.arcsin -> nan -> pi
    n, e = centre[0] - p0[0], centre[1] - p0[1]
    bearing = math.atan2(e, n) - heading
    idx_min = int(math.floor((math.pi + (bearing - delta)) / angle_per_ray))
    idx_max = int(math.ceil((math.pi + (bearing + delta)) / angle_per_ray))
    return idx_min, idx_max


def rays_for_obstacles(obstacles, p0, heading, angle_per_ray, n_rays):
    """sensor.py:74-97 including Python's negative-index wrap; an index below
    -n_rays (IndexError in the reference) is defined as 'all rays' (SURVEY B14)."""
    per_ray = [[] for _ in range(n_rays)]
    windows = []
    for ob in obstacles:
        c, r = ob.enclosing_circle()
        lo, hi = limit_angle_rays(c, r, p0, heading, angle_per_ray)
        a, b = lo - 1, hi % n_rays
        windows.append((a, b))
        if a < -n_rays:
            for i in range(n_rays):
                per_ray[i].append(ob)
            continue
        for i in range(a, b):
            per_ray[i].append(ob)
    return per_ray, windows


def cast_ray(angle, p0, sensor_range, obstacles, with_obstacle=False):
    """sensor.py:140-159: min distance to ray∩boundary over the candidate list.  With
    ``with_obstacle`` also the obstacle of the nearest intersection, first one on ties
    (``min((distance, i))`` of simulate_sensor_brute_force, sensor.py:113-117)."""
    p1 = (p0[0] + math.cos(angle) * sensor_range, p0[1] + math.sin(angle) * sensor_range)
    best = None
    who = None
    for ob in obstacles:
        if ob.filled and G.point_in_ring(p0, ob.ring):
            d = 0.0
        else:
            d = G.ray_ring_min_distance_np(p0, p1, ob.ring)
        if d is not None and (best is None or d < best):
            best = d
            who = ob
    d = sensor_range if best is None else best
    return (d, who) if with_obstacle else d


def cast_ray_runner_up(angle, p0, sensor_range, obstacles):
    """cast_ray(with_obstacle=True) plus the nearest intersection on any OTHER obstacle: the margin by which
    the nearest obstacle -- whose velocity the ray reports -- wins.  Returns (d, obstacle, d_other,
    other_obstacle); (sensor_range, None, inf, None) for a clear ray, (d, obstacle, inf, None) for one hit."""
    p1 = (p0[0] + math.cos(angle) * sensor_range, p0[1] + math.sin(angle) * sensor_range)
    hits = []
    for i, ob in enumerate(obstacles):
        d = 0.0 if ob.filled and G.point_in_ring(p0, ob.ring) else G.ray_ring_min_distance_np(p0, p1, ob.ring)
        if d is not None:
            hits.append((d, i, ob))
    if not hits:
        return sensor_range, None, math.inf, None
    hits.sort(key=lambda h: (h[0], h[1]))  # first obstacle on ties, as cast_ray
    d, _, who = hits[0]
    d2, _, who2 = next((h for h in hits[1:] if h[2] is not who), (math.inf, -1, None))
    return d, who, d2, who2


def relative_speed(angle, ob):
    """sensor.py:118-128: Rz(-sensor_angle - pi/2) applied to the obstacle's last displacement (dx, dy)."""
    if ob is None or ob.static:
        return 0.0, 0.0
    a = -angle - math.pi / 2
    return (math.cos(a) * ob.dx - math.sin(a) * ob.dy, math.sin(a) * ob.dx + math.cos(a) * ob.dy)


# ---------------------------------------------------------------------------------
# Vessel (vessel.py)
# ---------------------------------------------------------------------------------


class OracleVessel:
    def __init__(self, cfg, init_state):
        self.cfg = cfg
        self.n_sensors = cfg["n_sensors_per_sector"] * cfg["n_sectors"]
        self.d_angle = 2 * math.pi / self.n_sensors
        self.sensor_angles = np.array([-math.pi + (i + 1) * self.d_angle for i in range(self.n_sensors)])
        self.state = np.hstack([np.array(init_state, dtype=np.float64), np.zeros(3)])
        self.dists = np.ones(self.n_sensors) * cfg["sensor_range"]
        self.speeds = np.zeros((2, self.n_sensors))
        self.collision = False
        self.progress = 0.0
        self.max_progress = 0.0
        self.reached_goal = False
        self.step_counter = 0
        self.nearby = []
        self.nav = {}
        self.n_tests = 0  # ray/segment tests performed (SURVEY 8d "T")

    @property
    def position(self):
        return self.state[0:2]

    @property
    def heading(self):
        return self.state[2]

    @property
    def speed(self):
        return float(np.linalg.norm(self.state[3:5]))

    def step(self, action):
        self.state = M.vessel_step(
            self.state, action, self.cfg["t_step_size"], self.cfg["thrust_max_auv"], self.cfg["moment_max_auv"]
        )
        self.step_counter += 1

    def closeness(self, d):
        rng = self.cfg["sensor_range"]
        if self.cfg["sensor_log_transform"]:
            return 1 - np.clip(np.log(1 + d) / np.log(1 + rng), 0, 1)
        return 1 - np.clip(d / rng, 0, 1)

    def perceive(self, obstacles):
        rng = self.cfg["sensor_range"]
        p0 = (float(self.state[0]), float(self.state[1]))
        width = self.cfg["vessel_width"]
        if self.step_counter % self.cfg["sensor_interval_load_obstacles"] == 0:
            self.nearby = [
                ob
                for ob in obstacles
                if (G.point_polygon_distance(p0, ob.ring) if ob.filled else G.point_ring_distance(p0, ob.ring)) - width
                < rng
            ]
        if not self.nearby:
            self.dists = np.ones(self.n_sensors) * rng
            self.speeds = np.zeros((2, self.n_sensors))
            self.collision = False
            return np.zeros(self.n_sensors), np.zeros((2, self.n_sensors))
        angles = self.sensor_angles + self.heading
        per_ray, self.windows = rays_for_obstacles(self.nearby, p0, self.heading, self.d_angle, self.n_sensors)
        d = np.empty(self.n_sensors)
        v = np.zeros((2, self.n_sensors))
        nearest = self.cfg.get("velocity_mode", "zero") == "nearest"
        for i in range(self.n_sensors):
            d[i], who = cast_ray(angles[i], p0, rng, per_ray[i], with_obstacle=True)
            if nearest:
                v[:, i] = relative_speed(angles[i], who)
            self.n_tests += sum(len(ob.ring) - 1 for ob in per_ray[i])
        self.dists = d
        self.speeds = v
        self.collision = bool(np.any(d < width))
        return self.closeness(d), v

    def navigate(self, path):
        cfg = self.cfg
        pos = self.position
        s = path.closest_arclength(pos)
        chi = path.direction(s)
        delta = path(s) - pos
        cross_track = -math.sin(chi) * delta[0] + math.cos(chi) * delta[1]
        s_la = min(path.length, s + cfg["look_ahead_distance"])
        la_heading_err = float(M.princip(path.direction(s_la) - self.heading))
        rel = path(s_la) - pos
        heading_err = float(M.princip(math.atan2(rel[1], rel[0]) - self.heading))
        self.progress = s / path.length
        self.max_progress = max(self.progress, self.max_progress)
        goal_distance = float(np.linalg.norm(path.end - pos))
        self.reached_goal = bool(
            goal_distance <= cfg["min_goal_distance"] or self.progress >= cfg["min_path_progress"]
        )
        self.nav = dict(
            cross_track_error=cross_track / 100,
            heading_error=heading_err,
            look_ahead_heading_error=la_heading_err,
            goal_distance=goal_distance,
            vessel_arclength=s,
            target_arclength=s_la,
        )
        return np.array([self.state[3], self.state[4], self.state[5], la_heading_err, heading_err, cross_track / 100])


# ---------------------------------------------------------------------------------
# Rewards (rewarder.py:78-140, 167-241)
# ---------------------------------------------------------------------------------


def colav_reward(v: OracleVessel):
    if v.collision:
        return -10000.0 * (1 - 0.5)
    cte = v.nav["cross_track_error"]
    he = v.nav["heading_error"]
    path_reward = (1 + math.cos(he) * v.speed / 2) * (1 + math.exp(-5.0 * abs(cte))) - 1
    num = 0.0
    den = 0.0
    rng = v.cfg["sensor_range"]
    for i in range(v.n_sensors):
        weight = 1 / (1 + abs(10.0 * v.sensor_angles[i]))
        raw = rng * math.exp(-0.1 * v.dists[i] + 1.0 * max(0, v.speeds[1, i]))
        num += weight * raw
        den += weight
    closeness_reward = -num / den if v.n_sensors > 0 else 0.0
    if v.progress < v.max_progress:
        path_reward = min(path_reward, 0)
    slow = -2 if v.speed < 0.04 else 0
    living = 0.5 * (2 * 0.05 + 1) + 0 * 0.05
    r = 0.5 * path_reward + 0.5 * closeness_reward - living + 0 * v.speed / 2 - 10.0 * abs(v.state[5]) + slow
    if r < 0:
        r *= 2.0
    return float(r)


def pathfollow_reward(v: OracleVessel):
    if v.collision:
        return -10000.0 * (1 - 0.5)
    cte = v.nav["cross_track_error"]
    he = v.nav["heading_error"]
    path_reward = (1 + math.cos(he) * v.speed / 2) * (1 + math.exp(-5.0 * abs(cte))) - 1
    slow = -2 if v.speed < 0.1 else 0
    living = 0.5 * (2 * 0.05 + 1) + 0 * 0.05
    return float(path_reward - living + 0 * v.speed / 2 - 10.0 * abs(v.state[5]) + slow)


REWARDERS = {"colav": colav_reward, "pathfollow": pathfollow_reward}


# ---------------------------------------------------------------------------------
# Environment (environment.py)
# ---------------------------------------------------------------------------------


def build_obstacles(scn):
    """Obstacle order = moving first, then static circles, then polygons (matches
    MovingObstacles._generate's append order, movingobstacles.py:51-90)."""
    obs = []
    mov = scn.get("moving")
    if mov is not None:
        for j in range(len(mov["width"])):
            if "vel_tables" in mov:
                table = mov["vel_tables"][j]
            else:  # constant-velocity linear track of `vel_len` entries
                table = np.broadcast_to(mov["vel"][j], (int(mov["vel_len"][j]), 2))
            obs.append(OracleVesselObstacle(mov["width"][j], mov["start"][j], table, init_update=True))
    st = scn.get("static")
    if st is not None:
        for j in range(len(st["radius"])):
            obs.append(OracleCircle(st["pos"][j], st["radius"][j]))
    for poly in scn.get("polygons", []):
        obs.append(OraclePolygon(poly))
    return obs


class OracleEnv:
    def __init__(self, scn, cfg=None, test_mode=False):
        self.cfg = dict(DEFAULT_CFG)
        if cfg:
            self.cfg.update(cfg)
        self.test_mode = test_mode
        self.scn = scn
        self.reward_fn = REWARDERS[scn.get("rewarder", "colav")]
        self.reset()

    def reset(self):
        scn = self.scn
        self.t_step = 0
        self.cumulative_reward = 0.0
        self.path = OraclePath(scn["waypoints"])
        self.vessel = OracleVessel(self.cfg, scn["vessel_init"])
        self.obstacles = build_obstacles(scn)
        if scn.get("post_generate_update", False):
            self._update()
        self.cross_track_errors = []
        return self.observe()

    def _update(self):
        for ob in self.obstacles:
            if not ob.static:
                ob.update(self.cfg["t_step_size"])

    def observe(self):
        nav = self.vessel.navigate(self.path)
        parts = [nav]
        if self.cfg["use_lidar"]:
            closeness, vel = self.vessel.perceive(self.obstacles)
            parts.append(closeness.flatten())
            if self.cfg["sensor_use_velocity_observations"]:
                parts.append(vel.flatten())
        return np.clip(np.hstack(parts), -1.0, 1.0)

    def step(self, action):
        action = np.asarray(action, dtype=np.float64)
        if np.isnan(action).any():
            action = np.zeros(action.shape)
        self._update()
        self.vessel.step(action)
        obs = self.observe()
        v = self.vessel
        reward = self.reward_fn(v)
        self.cumulative_reward += reward
        info = dict(
            collision=v.collision,
            reached_goal=v.reached_goal,
            goal_distance=v.nav["goal_distance"],
            progress=v.progress,
        )
        done = bool(
            v.collision
            or v.reached_goal
            or (self.t_step >= self.cfg["max_timesteps"] - 1 and not self.test_mode)
            or (self.cumulative_reward < self.cfg["min_cumulative_reward"] and not self.test_mode)
        )
        self.cross_track_errors.append(abs(v.nav["cross_track_error"]) * 100)
        self.t_step += 1
        return obs, reward, done, info


# ---------------------------------------------------------------------------------
# Sector pooling (sensor.py:215-296; utils/sector_partitioning.py).  The wiring of
# LidarPreprocessor is broken in the reference at HEAD (SURVEY quirk #7); the static
# pooling method itself is self-contained and restated here literally.
# ---------------------------------------------------------------------------------


def feasibility_pooling(measurements, width, theta):
    """LidarPreprocessor._feasibility_pooling (sensor.py:251-296)."""
    measurements = np.asarray(measurements, dtype=np.float64)
    n = measurements.shape[0]
    for idx in np.argsort(measurements):
        surviving = measurements > measurements[idx] + width
        d = measurements[idx] * theta
        opening_width = 0
        opening_span = 0
        opening_start = -theta * (n - 1) / 2
        found = False
        for isensor, ok in enumerate(surviving):
            if ok:
                opening_width += d
                opening_span += theta
                if opening_width > width:
                    if abs(opening_start + opening_span / 2) < theta * (n - 1) / 4:
                        found = True
            else:
                opening_width += 0.5 * d
                opening_span += 0.5 * theta
                if opening_width > width:
                    if abs(opening_start + opening_span / 2) < theta * (n - 1) / 4:
                        found = True
                opening_width = 0
                opening_span = 0
                opening_start = -theta * (n - 1) / 2 + isensor * theta
        if not found:
            return max(0, measurements[idx])
    return max(0, np.max(measurements))


def sector_pool(dists, n_sectors=9, vessel_width=1.255, width_multiplier=5.0):
    """(min-pooled, feasibility-pooled) ranges per sector for one ray vector."""
    dists = np.asarray(dists, dtype=np.float64)
    n = len(dists)
    table = M.sector_table(n, n_sectors)
    theta = 2 * math.pi / n
    mins, feas = [], []
    for s in range(n_sectors):
        m = dists[table == s]
        mins.append(m.min())
        feas.append(feasibility_pooling(m, vessel_width * width_multiplier, theta))
    return np.array(mins), np.array(feas)
