"""Host-side construction of the path bank (reset-time work, SURVEY.md section 8 a18).

A path is what ``gym_auv.objects.path.Path.__init__`` builds (path.py:19-40): three
rounds of chord-length re-parametrisation through SciPy PCHIP resampled at 1000
points, plus the 0.1 m polyline that ``LineString.project`` runs on.  The bank stores,
per distinct path, exactly the tables the device needs:

  * PPoly knots [1000] and coefficients [999][2][4] (FP64)      -> Path.__call__, get_direction
  * polyline vertices [n][2] and chord-length prefix sums [n]     -> LineString.project
  * one (chord, deviation) capsule per 8, 32 and 512 consecutive segments -> exact hierarchical search
  * length, end point, origin

Construction stays on the host with SciPy (the reference does the same); only
evaluation and projection are on the per-step path.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence

import numpy as np
from scipy import interpolate

from ._lib import PP_W

PATH_BLOCK = 32  # segments per projection block, AUV_PATH_BLOCK in include/auv_b200.h
PATH_SUPER = 16  # blocks per superblock, AUV_PATH_SUPER
PATH_SUB = 8  # segments per sub-block, AUV_PATH_SUB
N_KNOTS = 1000
HDR_DTYPE = np.dtype([("v0", "<i4"), ("nseg", "<i4"), ("b0", "<i4"), ("s0", "<i4"), ("ox", "<f8"), ("oy", "<f8"),
                      ("length", "<f8"), ("end_x", "<f8"), ("end_y", "<f8"), ("extent", "<f8")])  # AuvPathHdr


@dataclass
class PathTable:
    """One path, host arrays (FP64 unless noted)."""

    knots: np.ndarray  # [1000]
    coef: np.ndarray  # [999, 2, 4]
    poly: np.ndarray  # [n, 2]
    cum: np.ndarray  # [n]
    blk_chord: np.ndarray  # [nblk, 4] float32 (ax, ay, ex, ey), relative to origin
    blk_dev: np.ndarray  # [nblk, 2] float32 (1/|e|^2, deviation)
    sb_chord: np.ndarray  # [nsb, 4] float32
    sb_dev: np.ndarray  # [nsb, 2] float32
    sub_chord: np.ndarray  # [ceil(nseg / 8), 4] float32
    sub_dev: np.ndarray  # [ceil(nseg / 8), 2] float32
    origin: np.ndarray  # [2]
    length: float
    end: np.ndarray  # [2]
    spline: object  # scipy PPoly (host-side evaluation for scenario generation)

    def __call__(self, s):
        return self.spline(s)

    def direction(self, s):
        d = self.spline.derivative()(s)
        return np.arctan2(d[1], d[0])


def _chord_lengths(pts: np.ndarray) -> np.ndarray:
    seg = np.sqrt(np.sum(np.diff(pts, axis=1) ** 2, axis=0))
    return np.concatenate([[0.0], np.cumsum(seg)])


def _capsules(rel: np.ndarray, nseg: int, span: int):
    """One capsule per `span` consecutive segments.  Returns
      chord [n, 4] float32 = (ax, ay, ex, ey): first vertex and chord vector (last - first),
      aux   [n, 2] float32 = (1/|e|^2 or 0, deviation): the deviation is the max distance of
    the covered vertices from the ROUNDED chord (evaluated in FP64) plus a float32 rounding
    allowance, rounded up -- so dist(P, polyline part) is within [dc - dev, dc + dev] of the
    distance dc from P to the rounded chord."""
    n = (nseg + span - 1) // span
    first = np.arange(n) * span
    last = np.minimum(first + span, nseg)
    chord = np.concatenate([rel[first], rel[last] - rel[first]], axis=1).astype(np.float32)
    a = chord[:, 0:2].astype(np.float64)
    e = chord[:, 2:4].astype(np.float64)
    len2 = np.sum(e * e, axis=1)
    with np.errstate(divide="ignore"):
        inv = np.where(len2 > 0, 1.0 / len2, 0.0).astype(np.float32)
    dev = np.zeros(n)
    for k in range(span + 1):  # loop over the offset inside the node keeps memory O(n)
        v = rel[np.minimum(first + k, last)]
        w = v - a
        t = np.clip(np.sum(w * e, axis=1) * inv.astype(np.float64), 0.0, 1.0)
        dev = np.maximum(dev, np.sqrt(np.sum((w - t[:, None] * e) ** 2, axis=1)))
    extent = float(np.abs(rel).max()) + 1.0
    dev = dev + 8.0 * np.finfo(np.float32).eps * extent
    dev = np.nextafter(dev.astype(np.float32), np.float32(np.inf))
    return chord, np.stack([inv, dev], axis=1).astype(np.float32)


def build_path(waypoints) -> PathTable:
    """waypoints: array [2, n_wp] (x row, y row) as passed to the reference's Path()."""
    pts = np.array(waypoints, dtype=np.float64)
    if pts.ndim != 2 or pts.shape[0] != 2 or pts.shape[1] < 2:
        raise ValueError(f"waypoints must have shape [2, n>=2], got {pts.shape}")
    spline = None
    arc = None
    for _ in range(3):
        arc = _chord_lengths(pts)
        spline = interpolate.PchipInterpolator(arc, pts, axis=1)
        pts = spline(np.linspace(arc[0], arc[-1], N_KNOTS))
    length = float(arc[-1])
    n_poly = int(10 * length)
    if n_poly < 2:
        raise ValueError("path shorter than 0.2 m")
    poly = np.ascontiguousarray(spline(np.linspace(0, length, n_poly)).T)  # [n, 2]
    seglen = np.sqrt(np.sum(np.diff(poly, axis=0) ** 2, axis=1))
    cum = np.concatenate([[0.0], np.cumsum(seglen)])
    # PPoly.c has shape [4, 999, 2] (power, interval, axis) -> [999, 2, 4]
    coef = np.ascontiguousarray(np.transpose(spline.c, (1, 2, 0)))
    origin = poly[0].copy()

    nseg = n_poly - 1
    rel = poly - origin
    blk_chord, blk_dev = _capsules(rel, nseg, PATH_BLOCK)
    sb_chord, sb_dev = _capsules(rel, nseg, PATH_BLOCK * PATH_SUPER)
    sub_chord, sub_dev = _capsules(rel, nseg, PATH_SUB)
    return PathTable(
        knots=np.ascontiguousarray(spline.x),
        coef=coef,
        poly=poly,
        cum=cum,
        blk_chord=blk_chord,
        blk_dev=blk_dev,
        sb_chord=sb_chord,
        sb_dev=sb_dev,
        sub_chord=sub_chord,
        sub_dev=sub_dev,
        origin=origin,
        length=length,
        end=np.array(spline(length), dtype=np.float64),
        spline=spline,
    )


class PathBank:
    """A list of PathTable concatenated into the flat arrays of ``AuvPathBank``: one 64 B header
    per path, capsule tables whose per-path offsets are even (so a CTA can bulk-copy a path's
    tables into shared memory in 16 B units), one 96 B record per PCHIP piece.  A path's sub-block
    table is padded to PATH_BLOCK // PATH_SUB entries per (padded) block, so it starts at that multiple
    of the path's first block."""

    def __init__(self, tables: Sequence[PathTable]):
        if len(tables) == 0:
            raise ValueError("empty path bank")
        self.tables: List[PathTable] = list(tables)
        self.n_paths = len(tables)
        self.poly_off = np.zeros(self.n_paths + 1, dtype=np.int32)
        self.blk_off = np.zeros(self.n_paths + 1, dtype=np.int32)
        self.sb_off = np.zeros(self.n_paths + 1, dtype=np.int32)
        even = lambda k: (int(k) + 1) & ~1
        for i, t in enumerate(tables):
            self.poly_off[i + 1] = self.poly_off[i] + len(t.poly)
            self.blk_off[i + 1] = self.blk_off[i] + even(len(t.blk_dev))
            self.sb_off[i + 1] = self.sb_off[i] + even(len(t.sb_dev))

        def padded(parts, width, slot=lambda p: even(len(p))):
            out = np.zeros((int(sum(slot(p) for p in parts)), width), dtype=np.float32)
            o = 0
            for p in parts:
                out[o:o + len(p)] = p
                o += slot(p)
            return out

        per_blk = PATH_BLOCK // PATH_SUB

        self.sb_chord = padded([t.sb_chord for t in tables], 4)
        self.sb_dev = padded([t.sb_dev for t in tables], 2)
        self.blk_chord = padded([t.blk_chord for t in tables], 4)
        self.blk_dev = padded([t.blk_dev for t in tables], 2)
        self.sub_chord = padded([t.sub_chord for t in tables], 4, slot=lambda p: per_blk * even((len(p) + per_blk - 1) // per_blk))
        self.sub_dev = padded([t.sub_dev for t in tables], 2, slot=lambda p: per_blk * even((len(p) + per_blk - 1) // per_blk))
        self.poly_xy = np.concatenate([t.poly for t in tables], axis=0)
        self.poly_cum = np.concatenate([t.cum for t in tables])
        self.origin = np.stack([t.origin for t in tables])
        self.knots = np.stack([t.knots for t in tables])
        self.coef = np.stack([t.coef for t in tables])
        self.length = np.array([t.length for t in tables], dtype=np.float64)
        self.end_xy = np.stack([t.end for t in tables])

    @classmethod
    def from_waypoints(cls, waypoint_list) -> "PathBank":
        return cls([build_path(w) for w in waypoint_list])

    def header_array(self) -> np.ndarray:
        """[n_paths] records with the layout of ``AuvPathHdr`` (64 B)."""
        hdr = np.zeros(self.n_paths, dtype=HDR_DTYPE)
        hdr["v0"] = self.poly_off[:-1]
        hdr["nseg"] = np.diff(self.poly_off) - 1
        hdr["b0"] = self.blk_off[:-1]
        hdr["s0"] = self.sb_off[:-1]
        hdr["ox"], hdr["oy"] = self.origin[:, 0], self.origin[:, 1]
        hdr["length"] = self.length
        hdr["end_x"], hdr["end_y"] = self.end_xy[:, 0], self.end_xy[:, 1]
        hdr["extent"] = [float(np.abs(t.poly - t.origin).sum(axis=1).max()) for t in self.tables]
        return hdr

    def poly_f32_array(self) -> np.ndarray:
        """[total_vertices, 2] float32: polyline vertices relative to their path's origin."""
        return np.concatenate([(t.poly - t.origin).astype(np.float32) for t in self.tables], axis=0)

    def piece_array(self) -> np.ndarray:
        """[n_paths, n_knots - 1, 12]: knot j, knot j + 1, x c0..c3, y c0..c3, 2 unused (``AuvPathBank.pp``)."""
        nk = self.knots.shape[1]
        pp = np.zeros((self.n_paths, nk - 1, PP_W), dtype=np.float64)
        pp[:, :, 0] = self.knots[:, :-1]
        pp[:, :, 1] = self.knots[:, 1:]
        pp[:, :, 2:6] = self.coef[:, :, 0, :]
        pp[:, :, 6:10] = self.coef[:, :, 1, :]
        return pp

    def device_arrays(self, device):
        import torch

        def dev(a, dtype):
            return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(device)

        return dict(
            hdr=torch.from_numpy(self.header_array().view(np.uint8).copy()).to(device),
            poly_xy=dev(self.poly_xy, torch.float64),
            poly_cum=dev(self.poly_cum, torch.float64),
            poly_f32=dev(self.poly_f32_array(), torch.float32),
            blk_chord=dev(self.blk_chord, torch.float32),
            blk_dev=dev(self.blk_dev, torch.float32),
            sb_chord=dev(self.sb_chord, torch.float32),
            sb_dev=dev(self.sb_dev, torch.float32),
            pp=dev(self.piece_array(), torch.float64),
            sub_chord=dev(self.sub_chord, torch.float32),
            sub_dev=dev(self.sub_dev, torch.float32),
        )


class DevicePathBank:
    """A path bank whose tables are built ON THE GPU (auv_pathbank_build: the three PCHIP rounds of
    path.py:19-40, polyline, prefix sums, capsules) from host waypoints -- milliseconds for 1024 random
    curves instead of ~14 s of SciPy -- in fixed-size slots (``vcap`` polyline vertices per path), so that
    single slots can be rebuilt later (fresh random curves, ``AUVVecEnv.regenerate_paths``).  The host
    builder ``PathBank`` stays the reference implementation the device tables are tested against.

    ``vcap``: a PCHIP curve is monotone per coordinate between its knots, so its length is at most the L1
    length of the waypoint polygon; for ``RandomCurveThroughOrigin(length=800)`` with up to 5 waypoints
    (movingobstacles.py:30-31) that is < 4.08 x 800 m = 3264 m -> 32642 vertices: the default never overflows
    for that family (paths of ~1.7 km do occur among a few thousand samples).  It is rounded up to a multiple of
    2 x PATH_BLOCK x PATH_SUPER, so that every slot's first block and superblock are even (the step bulk-copies
    these tables in 16 B units)."""

    n_knots = N_KNOTS

    def __init__(self, waypoints: Sequence[np.ndarray], vcap: int = 32768):
        if len(waypoints) == 0:
            raise ValueError("empty path bank")
        self.waypoints = [np.asarray(w, dtype=np.float64) for w in waypoints]
        for w in self.waypoints:
            if w.ndim != 2 or w.shape[0] != 2 or not (2 <= w.shape[1] <= 8):
                raise ValueError(f"device-built paths take 2..8 waypoints of shape [2, n], got {w.shape}")
        self.n_paths = len(self.waypoints)
        span = 2 * PATH_BLOCK * PATH_SUPER
        self.vcap = (int(vcap) + span - 1) // span * span
        self._tables = None
        self._dev = None

    @property
    def tables(self) -> List[PathTable]:
        """Host tables (SciPy), built lazily: only scenario generation on the host and the tests need them."""
        if self._tables is None:
            self._tables = [build_path(w) for w in self.waypoints]
        return self._tables

    def waypoint_arrays(self):
        wp = np.zeros((self.n_paths, 2, 8))
        nwp = np.zeros(self.n_paths, dtype=np.int32)
        for i, w in enumerate(self.waypoints):
            wp[i, :, : w.shape[1]] = w
            nwp[i] = w.shape[1]
        return wp, nwp

    def allocate(self, device):
        import torch

        P, V = self.n_paths, self.vcap
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=device)
        return dict(
            hdr=z(P * HDR_DTYPE.itemsize, torch.uint8), poly_xy=z((P * V, 2), torch.float64), poly_cum=z(P * V, torch.float64),
            poly_f32=z((P * V, 2), torch.float32), blk_chord=z((P * V // PATH_BLOCK, 4), torch.float32),
            blk_dev=z((P * V // PATH_BLOCK, 2), torch.float32),
            sb_chord=z((P * V // (PATH_BLOCK * PATH_SUPER), 4), torch.float32),
            sb_dev=z((P * V // (PATH_BLOCK * PATH_SUPER), 2), torch.float32), pp=z((P, N_KNOTS - 1, PP_W), torch.float64),
            sub_chord=z((P * V // PATH_SUB, 4), torch.float32), sub_dev=z((P * V // PATH_SUB, 2), torch.float32),
        )

    def build_struct(self, arrays):
        from . import _lib

        a = arrays
        return _lib.AuvPathBuild(a["hdr"].data_ptr(), a["poly_xy"].data_ptr(), a["poly_cum"].data_ptr(), a["poly_f32"].data_ptr(),
                                 a["blk_chord"].data_ptr(), a["blk_dev"].data_ptr(), a["sb_chord"].data_ptr(),
                                 a["sb_dev"].data_ptr(), a["pp"].data_ptr(), N_KNOTS, self.vcap, a["sub_chord"].data_ptr(),
                                 a["sub_dev"].data_ptr())

    def device_arrays(self, device):
        """Allocate the slots and build every path on the device."""
        import ctypes as C

        import torch

        from . import _lib

        lib = _lib.load()
        arrays = self.allocate(device)
        wp, nwp = self.waypoint_arrays()
        d_wp = torch.as_tensor(wp).to(device)
        d_n = torch.as_tensor(nwp).to(device)
        status = torch.zeros(1, dtype=torch.int32, device=device)
        bs = self.build_struct(arrays)
        with torch.cuda.device(device):
            stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
            _lib.check(lib.auv_pathbank_build(C.c_void_p(d_wp.data_ptr()), C.c_void_p(d_n.data_ptr()), None, self.n_paths,
                                              C.byref(bs), C.c_void_p(status.data_ptr()), stream), "auv_pathbank_build")
        if int(status.item()) & _lib.STATUS_PATH_TOO_LONG:
            raise ValueError(f"a path's 0.1 m polyline has more than vcap={self.vcap} vertices: raise vcap")
        return arrays


def random_curve_waypoints(rng, nwaypoints: int, length: float = 400.0) -> np.ndarray:
    """Waypoints of ``RandomCurveThroughOrigin`` (path.py:96-120): start on a circle of
    radius length/2, end = -start, nwaypoints//2 rounds each inserting two jittered points
    (the jitter is a scalar added to BOTH coordinates) around the origin.  Returns [2, n]."""
    angle_init = 2 * np.pi * (rng.rand() - 0.5)
    start = np.array([0.5 * length * np.cos(angle_init), 0.5 * length * np.sin(angle_init)])
    end = -start
    wps = np.vstack([start, end])
    half = nwaypoints // 2
    for k in range(half):
        p1 = (half - k) * start / (half + 1) + length / (half + 1) * (rng.rand() - 0.5)
        p2 = (half - k) * end / (half + 1) + length / (half + 1) * (rng.rand() - 0.5)
        wps = np.vstack([wps[: k + 1, :], p1, np.array([0.0, 0.0]), p2, wps[-1 * k - 1 :, :]])
    return np.transpose(wps)
