"""FP64 NumPy restatement of the frame rule stated at ``AuvRender`` (include/auv_b200.h), independent of the
kernel: what ``k_render`` must draw.  TEST INFRASTRUCTURE.

Shapes come from the oracle (``geos_lite.circle_boundary_ring``, the ``OracleVesselObstacle`` body rotated about
its centroid); the pixel predicates are vectorised restatements of ``geos_lite.point_in_ring`` and
``geos_lite.point_segment_distance`` (pinned against them by tests/test_render.py).  Besides the colour, every
pixel gets a margin: the distance in pixels from its centre to the nearest boundary of a layer that could decide
it (the deciding layer and every layer above it; inside a union of shapes, the depth in the deepest one), capped
at ``MARGIN_CAP``.  A pixel whose margin is at most ``NONDECISIVE_PX`` may legitimately differ from the kernel's
FP32 test.  That band is ~10x the FP32 rounding of camera-relative coordinates of a few hundred pixels, and narrow
enough that the 180 half-pixel rays of a LiDAR frame (whose capsule edges run ~40 000 px through a 256 x 192
frame) leave well under 0.1 % of the pixels in it: a band of 2e-3 px would hold ~0.2 %.
"""
from __future__ import annotations

import math

import numpy as np

from gym_auv_b200 import _lib
from oracle import geos_lite as G
from oracle.sim import OracleVesselObstacle

PALETTE = np.array([_lib.RGB_OWNSHIP, _lib.RGB_RAY_HIT, _lib.RGB_RAY_CLEAR, _lib.RGB_MOVING, _lib.RGB_STATIC,
                    _lib.RGB_GOAL, _lib.RGB_PATH, _lib.RGB_LAND, _lib.RGB_SEA], dtype=np.int64)
SHIP, RAY_HIT, RAY_CLEAR, MOVING, STATIC, GOAL, PATH, LAND, SEA = range(9)
NONDECISIVE_PX = 5e-4
MARGIN_CAP = 1.0


def rgb_of(layer):
    c = PALETTE[np.asarray(layer)]
    return np.stack([(c >> 16) & 255, (c >> 8) & 255, c & 255], axis=-1).astype(np.uint8)


def seg_dist(px, py, ax, ay, bx, by):
    """geos_lite.point_segment_distance, vectorised (same arithmetic)."""
    ex, ey = bx - ax, by - ay
    len2 = ex * ex + ey * ey
    with np.errstate(divide="ignore", invalid="ignore"):
        r = ((px - ax) * ex + (py - ay) * ey) / len2
        s = ((ay - py) * ex - (ax - px) * ey) / len2
    d = np.where(r <= 0.0, np.hypot(px - ax, py - ay),
                 np.where(r >= 1.0, np.hypot(px - bx, py - by), np.abs(s) * np.sqrt(len2)))
    return np.where(len2 == 0.0, np.hypot(px - ax, py - ay), d)


def in_ring(px, py, ring):
    """geos_lite.point_in_ring, vectorised: crossing number, a point met exactly by an edge counts as inside."""
    inside = np.zeros(np.shape(px), dtype=bool)
    on = np.zeros(np.shape(px), dtype=bool)
    for k in range(len(ring) - 1):
        x1, y1 = ring[k]
        x2, y2 = ring[k + 1]
        m = (y1 > py) != (y2 > py)
        with np.errstate(divide="ignore", invalid="ignore"):
            xint = x1 + (py - y1) * (x2 - x1) / (y2 - y1)
        on |= m & (xint == px)
        inside ^= m & (xint > px)
    return inside | on


def ring_dist(px, py, ring):
    d = np.full(np.shape(px), np.inf)
    for k in range(len(ring) - 1):
        d = np.minimum(d, seg_dist(px, py, ring[k, 0], ring[k, 1], ring[k + 1, 0], ring[k + 1, 1]))
    return d


def ray_length(c, sensor_range, log_transform):
    """Range d_i of a ray from its closeness c_i (the inverse of k_lidar's closeness; range when c_i = 0)."""
    c = np.asarray(c, dtype=np.float64)
    d = (1.0 + sensor_range) ** (1.0 - c) - 1.0 if log_transform else (1.0 - c) * sensor_range
    return np.where(c == 0.0, sensor_range, d)


def vessel_ring(width, position, heading):
    """The VesselObstacle pentagon of ``width`` (oracle body rotated about its centroid), placed at ``position``."""
    ob = OracleVesselObstacle(width, position, np.zeros((2, 2)), init_update=False)
    ob.heading = heading
    ob.position = np.asarray(position, dtype=np.float64)
    ob._rebuild()
    return ob.ring


class Canvas:
    def __init__(self, width, height, half_width):
        self.W, self.H, self.s = int(width), int(height), 2.0 * float(half_width) / int(width)
        self.px = (self.H / 2 - np.arange(self.H) - 0.5) * self.s  # [H] metres north of the vessel
        self.py = (np.arange(self.W) + 0.5 - self.W / 2) * self.s  # [W] metres east
        # signed depth of each pixel in each layer (pixels; > 0 inside): the max over the layer's shapes of
        # +distance to the shape's boundary inside it, -distance outside.  Outside every shape that is minus the
        # distance to the layer; inside, a lower bound of the distance to the boundary of the layer's union
        self.depth = np.full((9, self.H, self.W), -np.inf)

    def window(self, lo, hi):
        """row / column slices of the pixels within MARGIN_CAP px of the box lo..hi (camera metres), or None"""
        g = (MARGIN_CAP + 1.0) * self.s
        rows = np.nonzero((self.px >= lo[0] - g) & (self.px <= hi[0] + g))[0]
        cols = np.nonzero((self.py >= lo[1] - g) & (self.py <= hi[1] + g))[0]
        if len(rows) == 0 or len(cols) == 0:
            return None
        return slice(rows[0], rows[-1] + 1), slice(cols[0], cols[-1] + 1)

    def add(self, layer, win, inside, bdist):
        rs, cs = win
        d = np.where(inside, bdist, -bdist) / self.s
        self.depth[layer, rs, cs] = np.maximum(self.depth[layer, rs, cs], d)

    def grid(self, win):
        rs, cs = win
        return np.meshgrid(self.px[rs], self.py[cs], indexing="ij")

    def polygon(self, layer, ring):
        ring = np.asarray(ring, dtype=np.float64)
        win = self.window(ring.min(axis=0), ring.max(axis=0))
        if win is None:
            return
        X, Y = self.grid(win)
        self.add(layer, win, in_ring(X, Y, ring), ring_dist(X, Y, ring))

    def polyline(self, layer, pts, h):
        """capsule of half-width h around the polyline pts [n, 2], by blocks of 32 segments"""
        pts = np.asarray(pts, dtype=np.float64)
        for b in range(0, len(pts) - 1, 32):
            blk = pts[b:b + 33]
            win = self.window(blk.min(axis=0) - h, blk.max(axis=0) + h)
            if win is None:
                continue
            X, Y = self.grid(win)
            d = seg_dist(X[..., None], Y[..., None], blk[:-1, 0], blk[:-1, 1], blk[1:, 0], blk[1:, 1]).min(axis=-1)
            self.add(layer, win, d <= h, np.abs(d - h))

    def disc(self, layer, c, radius):
        win = self.window(np.asarray(c) - radius, np.asarray(c) + radius)
        if win is None:
            return
        X, Y = self.grid(win)
        d = np.hypot(X - c[0], Y - c[1])
        self.add(layer, win, d <= radius, np.abs(d - radius))

    def result(self):
        """(rgb [H, W, 3] uint8, layer [H, W], margin [H, W] px)"""
        inside = self.depth >= 0.0
        first = np.where(inside.any(axis=0), inside.argmax(axis=0), SEA)
        upto = np.arange(9)[:, None, None] <= first[None]
        margin = np.minimum(np.where(upto, np.abs(self.depth), np.inf).min(axis=0), MARGIN_CAP)
        return rgb_of(first), first, margin


def rasterise(scene: dict, width: int, height: int, half_width: float):
    """The frame of ``scene`` (world coordinates, x north, y east):
      pos (2,), psi, vessel_width,
      rays: None or dict(angles [R] body angles, closeness [R] channel 0, range, log_transform),
      moving: [(width, position (2,), displacement (2,))], static: [(centre (2,), radius)],
      goal (2,), path [n, 2], world: [closed rings].
    Returns (rgb, layer, margin)."""
    cv = Canvas(width, height, half_width)
    s = cv.s
    p0 = np.asarray(scene["pos"], dtype=np.float64)
    psi = float(scene["psi"])
    ship = vessel_ring(max(float(scene["vessel_width"]), _lib.RENDER_SHIP_MIN_PX * s), (0.0, 0.0), psi)
    cv.polygon(SHIP, ship - G.polygon_centroid(ship))
    rays = scene.get("rays")
    if rays is not None:
        d = ray_length(rays["closeness"], float(rays["range"]), bool(rays["log_transform"]))
        h = _lib.RENDER_RAY_HALF_PX * s
        for i, a in enumerate(np.asarray(rays["angles"], dtype=np.float64)):
            e = d[i] * np.array([math.cos(psi + a), math.sin(psi + a)])
            cv.polyline(RAY_HIT if rays["closeness"][i] > 0 else RAY_CLEAR, np.array([[0.0, 0.0], e]), h)
    for w, pos, disp in scene.get("moving", []):
        if w > 0:
            cv.polygon(MOVING, vessel_ring(w, pos, math.atan2(disp[1], disp[0])) - p0)
    for c, r in scene.get("static", []):
        if r > 0:
            cv.polygon(STATIC, G.circle_boundary_ring(c[0], c[1], r) - p0)
    cv.disc(GOAL, np.asarray(scene["goal"], dtype=np.float64) - p0, _lib.RENDER_GOAL_PX * s)
    if scene.get("path") is not None:
        cv.polyline(PATH, np.asarray(scene["path"], dtype=np.float64) - p0, _lib.RENDER_PATH_HALF_PX * s)
    for ring in scene.get("world", []):
        if 4 <= len(ring) <= _lib.MAX_POLY_VERTS:
            cv.polygon(LAND, np.asarray(ring, dtype=np.float64) - p0)
    return cv.result()


def env_scenes(env, ids):
    """Scenes (``rasterise`` input) of envs ``ids`` of an AUVVecEnv, read back through its public state:
    ``obstacle_state()``, ``pull_scenarios()`` (the device pool may have been regenerated), the path polyline
    read from the device bank by header, the world rings, the state and the observation row."""
    from gym_auv_b200.pathbank import HDR_DTYPE

    import torch

    torch.cuda.synchronize(env.device)
    scn = env.pull_scenarios()
    pos, disp, _ = (t.cpu().numpy() for t in env.obstacle_state())
    state = env.state.cpu().numpy()
    obs = env._out["obs"].cpu().numpy()
    sid = env.get_attr("scn_id").cpu().numpy()
    pid = env._st["env_pid"].cpu().numpy()
    hdr = env._bank["hdr"].cpu().numpy().view(HDR_DTYPE)
    poly = env._bank["poly_xy"].cpu().numpy().reshape(-1, 2)
    v = env.config.vessel
    out = []
    for e in ids:
        m, h = int(sid[e]), hdr[int(pid[e])]
        rays = None
        if v.use_lidar:
            rays = dict(angles=env.sensor_angles, closeness=obs[e, 6:6 + env.n_sensors].astype(np.float64),
                        range=float(v.sensor_range), log_transform=bool(v.sensor_log_transform))
        out.append(dict(
            pos=state[0:2, e], psi=state[2, e], vessel_width=float(v.vessel_width), rays=rays,
            moving=[(scn.mov_width[m, j], pos[e, j], disp[e, j]) for j in range(env.k_moving)],
            static=[(scn.st_pos[m, j], scn.st_radius[m, j]) for j in range(env.k_static)],
            goal=(h["end_x"], h["end_y"]), path=poly[h["v0"]:h["v0"] + h["nseg"] + 1],
            world=env.scenarios.world.rings if env.n_world else [],
        ))
    return out
