"""The path projection of the step (``project_group``: FP32 capsule pruning over superblocks, blocks and
8-segment sub-blocks, then an FP64 refine with a cross-multiplied, shuffle arg-min) against an exact
reference of the operation it restates: GEOS ``LengthIndexOfPoint`` -- the FIRST segment at the minimum
distance wins, the measure is ``cum[k] + r |seg k|``.

The reference runs on the kernel's own polyline (read back from the device tables), screens every segment in
FP64 and decides the survivors with ``fractions.Fraction``.  Each query point is then one of

* decisive: the exact runner-up is farther than 1e-12 (relative, squared distance) -- the segment must be the
  exact one and the arclength its measure to 1e-9 m;
* an exact tie with a common nearest point (a vertex both segments reduce to): the kernel computes both sides
  with the same operations, so the lower index must win;
* a near tie: the segment must lie in the exact near-tie set and the arclength must be that segment's measure.

The point families are the inputs where a capsule search goes wrong: the medial line of a hairpin (two distant
branches nearly equidistant, displaced by less than the FP32 pads), the centre of a circular arc (every
sub-block survives the pruning), the far field, points past both ends, points on vertices and segment
interiors, and points outside convex corners.  Every family runs cold and warm from segments that are wrong on
purpose, on a host-built bank, a device-built bank, a bank without sub-block tables, and with envs of two
paths mixed in every CTA (global-table fallback).  The navigation features are compared with
``OracleVessel.navigate`` where the point is decisive, and with ``navigate``'s formulas at the kernel's
arclength elsewhere."""
import dataclasses
import math
from fractions import Fraction as F

import numpy as np
import pytest

from gym_auv_b200 import scenarios as S
from gym_auv_b200.pathbank import PathBank, build_path
from oracle import geos_lite as G
from tests.test_oracle_exact import exact_pt_seg_d2

TIE_REL = 1e-12  # exact gap (relative, squared distance) below which two segments are a near tie
SCREEN_REL, SCREEN_ABS = 1e-9, 1e-10  # FP64 screen: distance within this of the minimum -> decided exactly
S_TOL = 1e-9  # arclength, m


# ---------------------------------------------------------------------------------------------------------
# exact reference
# ---------------------------------------------------------------------------------------------------------
def _measure(poly, cum, p, k):
    """segmentNearestMeasure of segment k (geos_lite.linestring_project, FP64)."""
    a, b = poly[k], poly[k + 1]
    e = b - a
    len2 = e[0] * e[0] + e[1] * e[1]
    if len2 == 0.0:
        return float(cum[k])
    r = ((p[0] - a[0]) * e[0] + (p[1] - a[1]) * e[1]) / len2
    if r <= 0.0:
        return float(cum[k])
    seglen = math.sqrt(len2)
    return float(cum[k] + r * seglen) if r <= 1.0 else float(cum[k] + seglen)


def _fp64_d2(poly, pts):
    """[n_pts, nseg] squared point-segment distances, FP64."""
    a, e = poly[:-1], np.diff(poly, axis=0)
    len2 = (e * e).sum(1)
    w = pts[:, None, :] - a[None]
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(len2 > 0, (w * e[None]).sum(2) / len2, 0.0)
    r = np.clip(r, 0.0, 1.0)
    d = w - r[..., None] * e[None]
    return (d * d).sum(2)


def _exact_foot(p, a, b):
    px, py, ax, ay, bx, by = map(F, (*p, *a, *b))
    ex, ey = bx - ax, by - ay
    l2 = ex * ex + ey * ey
    r = F(0) if l2 == 0 else min(max(((px - ax) * ex + (py - ay) * ey) / l2, F(0)), F(1))
    return ax + r * ex, ay + r * ey


@dataclasses.dataclass
class Ref:
    kind: str  # "decisive" | "tie" | "near"
    best: int  # first exact minimum
    near: tuple  # exact near-tie set (segments within TIE_REL of the minimum)
    other: int  # nearest segment more than 300 segments away from `best` (a warm start on the wrong branch)


def reference(poly, pts, chunk=128):
    """Exact first-minimum projection of every point onto the polyline `poly` [n, 2]."""
    poly = np.asarray(poly, dtype=np.float64)
    out = []
    for c0 in range(0, len(pts), chunk):
        P = pts[c0:c0 + chunk]
        d2 = _fp64_d2(poly, P)
        d = np.sqrt(d2)
        for i, p in enumerate(P):
            dmin = d[i].min()
            cand = np.nonzero(d[i] <= dmin * (1 + SCREEN_REL) + SCREEN_ABS)[0]
            ex = {int(k): exact_pt_seg_d2(p, poly[k], poly[k + 1]) for k in cand}
            m = min(ex.values())
            mins = sorted(k for k, v in ex.items() if v == m)
            near = tuple(sorted(k for k, v in ex.items() if v - m <= TIE_REL * m))
            if len(near) == 1:
                kind = "decisive"
            elif len(mins) > 1 and len({_exact_foot(p, poly[k], poly[k + 1]) for k in mins}) == 1:
                kind = "tie"
            else:
                kind = "near"
            far = np.abs(np.arange(len(poly) - 1) - mins[0]) > 300
            other = int(np.argmin(np.where(far, d2[i], np.inf))) if far.any() else 0
            out.append(Ref(kind, mins[0], near, other))
    return out


def check_projection(poly, cum, p, ref, seg, s):
    """None if (seg, s) is a correct projection of p by the reference `ref`, else why not."""
    nseg = len(poly) - 1
    if not 0 <= seg < nseg:
        return f"segment {seg} out of [0, {nseg})"
    if ref.kind in ("decisive", "tie") and seg != ref.best:
        return f"{ref.kind}: segment {seg}, the first exact minimum is {ref.best}"
    if ref.kind == "near" and seg not in ref.near:
        return f"near tie: segment {seg} not in {ref.near}"
    want = _measure(poly, cum, p, seg)
    if not abs(s - want) <= S_TOL:
        return f"arclength {s!r} != measure {want!r} of segment {seg}"
    return None


# ---------------------------------------------------------------------------------------------------------
# paths and point families (at most 8 waypoints each, so that the device builder takes them too)
# ---------------------------------------------------------------------------------------------------------
def _rot(th):
    return np.array([[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]])


# a tapered hairpin, turned by 35 degrees: out along the x axis, a 20 m turn, back 3 m .. 40 m away
HAIRPIN = (_rot(0.61) @ np.array([[0.0, 350.0, 700.0, 720.0, 700.0, 350.0, 100.0],
                                   [0.0, 0.0, 0.0, 20.0, 40.0, 21.5, 3.0]])) + np.array([[250.0], [-180.0]])
# circular arcs (315 degrees): radius 150 m (staged tables) and 340 m (> 16384 segments: global tables, two
# windows of 32 superblocks).  Through 8 waypoints the PCHIP radius varies by metres; through 2000 / 4000 it
# varies by 0.8 / 1.7 mm, so that seen from the centre every (150 m) or most (340 m) sub-blocks lie within the
# capsule bounds of the nearest one and have to be refined in FP64.  The device builder takes 8 waypoints at
# most: its variant runs on the coarse arcs.
CENTRE = np.array([-420.0, 615.0])


def _arc(radius, n=8):
    th = np.linspace(0.0, 1.75 * np.pi, n)
    return np.stack([CENTRE[0] + radius * np.cos(th), CENTRE[1] + radius * np.sin(th)])


SCURVE = np.array([[0.0, 300.0, 600.0, 900.0], [0.0, 80.0, -50.0, 30.0]]) + np.array([[-60.0], [35.0]])
PATHS = dict(hairpin=HAIRPIN, arc150=_arc(150.0), arc340=_arc(340.0), circle150=_arc(150.0, 2000),
             circle340=_arc(340.0, 4000), scurve=SCURVE)
DEVICE_KEY = dict(circle150="arc150", circle340="arc340")  # waypoint sets the device builder takes instead


def _hairpin_medial(t):
    """Points on the medial line of the hairpin's straight part, displaced by delta towards the return branch."""
    poly = t.poly
    nseg = len(poly) - 1
    u = np.array([math.cos(0.61), math.sin(0.61)])
    along = (poly - poly[0]) @ u
    kturn = int(np.argmax(along))
    ks = np.linspace(0.12 * kturn, 0.93 * kturn, 56).astype(int)
    A = poly[ks]
    e = poly[ks + 1] - poly[ks]
    n = np.stack([-e[:, 1], e[:, 0]], 1) / np.linalg.norm(e, axis=1)[:, None]  # left normal: towards the return branch
    idx = np.arange(nseg)

    def gap(q):  # distance to the return branch - distance to the out branch
        d2 = _fp64_d2(poly, q)
        return np.sqrt(np.where(idx[None] > kturn, d2, np.inf).min(1)) - np.sqrt(np.where(idx[None] <= kturn, d2, np.inf).min(1))

    lo, hi = np.zeros(len(ks)), np.full(len(ks), 60.0)
    assert (gap(A + hi[:, None] * n) < 0).all()
    for _ in range(64):  # bisection to FP64 resolution
        mid = 0.5 * (lo + hi)
        pos = gap(A + mid[:, None] * n) > 0
        lo, hi = np.where(pos, mid, lo), np.where(pos, hi, mid)
    med = A + lo[:, None] * n
    deltas = (0.0, 1e-9, -1e-9, 1e-7, -1e-7, 1e-5, -1e-5, 1e-3, -1e-3)
    return np.concatenate([med + dl * n for dl in deltas])


def _circle_centre(_t):
    ang = np.linspace(0, 2 * np.pi, 40, endpoint=False)
    pts = [CENTRE[None]]
    for r in (1e-9, 1e-6, 1e-3, 0.1, 1.0, 10.0):
        pts.append(CENTRE + r * np.stack([np.cos(ang + r), np.sin(ang + r)], 1))
    return np.concatenate(pts)


def _far_field(t):
    c = t.poly.mean(0)
    ang = np.linspace(0, 2 * np.pi, 100, endpoint=False)
    return np.concatenate([c + r * np.stack([np.cos(ang + r), np.sin(ang + r)], 1) for r in (500.0, 1200.0, 2500.0, 5000.0)])


def _past_ends(t):
    poly = t.poly
    pts = []
    for end, nxt in ((poly[0], poly[1]), (poly[-1], poly[-2])):
        out = (end - nxt) / np.linalg.norm(end - nxt)
        nrm = np.array([-out[1], out[0]])
        for a in (0.05, 0.5, 3.0, 10.0, 40.0, 100.0, 400.0, 1000.0):
            for b in np.linspace(-0.6, 0.6, 13):
                pts.append(end + a * out + a * b * nrm)
    return np.array(pts)


def _on_path(t):
    rng = np.random.RandomState(11)
    poly = t.poly
    nseg = len(poly) - 1
    kv = np.concatenate([[0, nseg], rng.randint(1, nseg, 200)])
    ki = rng.randint(0, nseg, 200)
    u = rng.uniform(0.01, 0.99, 200)[:, None]
    return np.concatenate([poly[kv], poly[ki] + u * (poly[ki + 1] - poly[ki])])


def _corners(t):
    """Outside the convex corners of the arc: the foot on both segments of a vertex is the vertex itself."""
    rng = np.random.RandomState(12)
    poly = t.poly
    ks = rng.randint(1, len(poly) - 1, 150)
    pts = []
    for k, rho in zip(ks, np.tile([0.5, 5.0, 40.0], 50)):
        e0, e1 = poly[k] - poly[k - 1], poly[k + 1] - poly[k]
        b = np.array([e0[1], -e0[0]]) / np.linalg.norm(e0) + np.array([e1[1], -e1[0]]) / np.linalg.norm(e1)
        b *= np.sign(b @ (poly[k] - CENTRE))  # the bisector of the two outer normals
        pts.append(poly[k] + rho * b / np.linalg.norm(b))
    return np.array(pts)


FAMILIES = dict(
    hairpin=("hairpin", _hairpin_medial),
    circle_centre=("circle150", _circle_centre),
    circle_centre_long=("circle340", _circle_centre),
    far_field=("hairpin", _far_field),
    past_ends=("scurve", _past_ends),
    on_path=("hairpin", _on_path),
    corners=("arc150", _corners),
)


# ---------------------------------------------------------------------------------------------------------
# CPU tests of the checker
# ---------------------------------------------------------------------------------------------------------
def test_reference_agrees_with_linestring_project_on_decisive_points_and_vertex_ties():
    from gym_auv_b200.pathbank import random_curve_waypoints

    rng = np.random.RandomState(21)
    t = build_path(random_curve_waypoints(rng, 5, 120.0))
    pts = t.poly[rng.randint(0, len(t.poly), 150)] + rng.normal(0, 8.0, (150, 2))
    refs = reference(t.poly, pts)
    n = 0
    for p, r in zip(pts, refs):
        if r.kind == "near":
            continue
        n += 1
        assert abs(G.linestring_project(t.poly, p) - _measure(t.poly, t.cum, p, r.best)) <= S_TOL
        assert check_projection(t.poly, t.cum, p, r, r.best, G.linestring_project(t.poly, p)) is None
    assert n >= 140


def test_checker_rejects_subtly_wrong_projections():
    """Negative controls: the runner-up on a decisive point, an arclength 1e-7 m off, the higher index of an
    exact vertex tie and an out-of-range segment all fail; the right answers pass."""
    t = build_path(PATHS["arc150"])
    poly, cum = t.poly, t.cum
    dec = poly[[400, 2000]] + np.array([[0.0, 0.0]])
    dec = dec + 0.3 * (dec - CENTRE) / np.linalg.norm(dec - CENTRE, axis=1)[:, None]
    dec[:, 0] += 0.02  # off the vertex normal
    ties = _corners(t)[:6]
    pts = np.concatenate([dec, ties])
    refs = reference(poly, pts)
    assert [r.kind for r in refs[:2]] == ["decisive"] * 2 and all(r.kind == "tie" and len(r.near) == 2 for r in refs[2:])
    for p, r in zip(pts, refs):
        s = _measure(poly, cum, p, r.best)
        assert check_projection(poly, cum, p, r, r.best, s) is None
        assert check_projection(poly, cum, p, r, r.best, s + 1e-7) is not None
        assert check_projection(poly, cum, p, r, len(poly) - 1, s) is not None
        assert check_projection(poly, cum, p, r, -1, s) is not None
        if r.kind == "decisive":
            d2 = _fp64_d2(poly, p[None])[0]
            d2[r.best] = np.inf
            runner = int(np.argmin(d2))
            assert check_projection(poly, cum, p, r, runner, _measure(poly, cum, p, runner)) is not None
        else:
            hi = r.near[-1]
            assert hi > r.best and check_projection(poly, cum, p, r, hi, _measure(poly, cum, p, hi)) is not None


def test_point_families_cover_their_cases():
    """The families produce what they are meant to: decisive points and near ties on the hairpin's medial line,
    exact vertex ties on the path's vertices and outside corners, feet at both ends past the ends."""
    kinds = {}
    for fam in ("hairpin", "on_path", "corners", "past_ends"):
        key, gen = FAMILIES[fam]
        t = build_path(PATHS[key])
        pts = gen(t)
        refs = reference(t.poly, pts)
        kinds[fam] = {k: sum(r.kind == k for r in refs) for k in ("decisive", "tie", "near")}
        if fam == "past_ends":
            nseg = len(t.poly) - 1
            assert sum(r.best == 0 for r in refs) >= 90 and sum(r.best == nseg - 1 for r in refs) >= 90
    assert kinds["hairpin"]["decisive"] >= 300 and kinds["hairpin"]["near"] + kinds["hairpin"]["tie"] >= 20, kinds
    assert kinds["on_path"]["tie"] >= 190 and kinds["on_path"]["decisive"] >= 200, kinds
    assert kinds["corners"]["tie"] >= 140, kinds


def unprunable_sub_blocks(t, p):
    """Fraction of the path's sub-blocks that no exact capsule search can prune for the point p: their capsule
    lower bound (distance to the chord minus the deviation, FP64 on the stored tables) does not exceed the
    minimum distance itself, so every valid upper bound keeps them."""
    ch, dv = t.sub_chord.astype(np.float64), t.sub_dev.astype(np.float64)
    w = (np.asarray(p) - t.origin) - ch[:, :2]
    r = np.clip((w * ch[:, 2:]).sum(1) * dv[:, 0], 0.0, 1.0)
    lower = np.linalg.norm(w - r[:, None] * ch[:, 2:], axis=1) - dv[:, 1]
    return float((lower <= np.sqrt(_fp64_d2(t.poly, np.asarray(p)[None]).min())).mean())


def test_circle_centre_leaves_most_sub_blocks_to_the_fp64_refine():
    """Seen from the arc's centre the dense arcs are equidistant within the capsule bounds: at least 95 % (150 m)
    and 60 % (340 m) of the sub-blocks cannot be pruned by any valid bound, so the kernel refines them in FP64;
    the 8-waypoint arcs of the device variant prune nearly everything (their radius varies by metres)."""
    f150 = unprunable_sub_blocks(build_path(PATHS["circle150"]), CENTRE)
    f340 = unprunable_sub_blocks(build_path(PATHS["circle340"]), CENTRE)
    assert f150 >= 0.95 and f340 >= 0.6, (f150, f340)
    assert unprunable_sub_blocks(build_path(PATHS["arc150"]), CENTRE) < 0.05


# ---------------------------------------------------------------------------------------------------------
# the kernel
# ---------------------------------------------------------------------------------------------------------
VARIANTS = ("host", "device", "no_sub_tables", "mixed_paths")
_cache = {}


def _scenarios(key, variant):
    """One scenario per path (no obstacles); 'mixed_paths' adds the reversed path as a second one."""
    wp = PATHS[key]
    wps = [wp, wp[:, ::-1].copy()] if variant == "mixed_paths" else [wp]
    one = S._single(wp)
    M = len(wps)
    z = lambda *s: np.zeros((M, 0) + s)
    scn = S.ScenarioSet(waypoints=wps, path_id=np.arange(M, dtype=np.int32), vessel_init=np.repeat(one.vessel_init, M, 0),
                        mov_start=z(2), mov_width=z(), mov_track=np.zeros((M, 0, 4), np.int32), vel_table=np.zeros((0, 2)),
                        st_pos=z(2), st_radius=z(), name="projection-edges")
    if variant == "device":
        from gym_auv_b200.pathbank import DevicePathBank

        scn._bank = DevicePathBank(wps)
    else:
        scn._bank = PathBank([build_path(w) for w in wps])
    return scn


def _device_path(env, pid):
    """The polyline, prefix sums, header and PCHIP pieces the kernel reads for path pid."""
    from gym_auv_b200.pathbank import HDR_DTYPE

    h = env._bank["hdr"].cpu().numpy().view(HDR_DTYPE)[pid]
    v0, n = int(h["v0"]), int(h["nseg"]) + 1
    poly = env._bank["poly_xy"][v0:v0 + n].cpu().numpy().astype(np.float64)
    cum = env._bank["poly_cum"][v0:v0 + n].cpu().numpy().astype(np.float64)
    pp = env._bank["pp"][pid].cpu().numpy()
    from scipy.interpolate import PPoly

    spline = PPoly(np.stack([pp[:, 2:6].T, pp[:, 6:10].T], axis=-1), np.concatenate([pp[:, 0], pp[-1:, 1]]))
    return poly, cum, h, spline


def _wrap(a):
    return (a + np.pi) % (2 * np.pi) - np.pi


def _navigate_at(spline, h, cfg, p, psi, s):
    """Vessel.navigate's formulas (oracle/sim.py) at the arclength s, on the kernel's own PCHIP tables."""
    L = float(h["length"])
    pos = spline(s)
    d = spline.derivative()(s)
    chi = math.atan2(d[1], d[0])
    y_e = -math.sin(chi) * (pos[0] - p[0]) + math.cos(chi) * (pos[1] - p[1])
    s_la = min(L, s + cfg.vessel.look_ahead_distance)
    dl = spline.derivative()(s_la)
    la_err = _wrap(math.atan2(dl[1], dl[0]) - psi)
    rel = spline(s_la) - p
    head_err = _wrap(math.atan2(rel[1], rel[0]) - psi)
    goal = math.hypot(float(h["end_x"]) - p[0], float(h["end_y"]) - p[1])
    prog = s / L
    reached = goal <= cfg.episode.min_goal_distance or prog >= cfg.episode.min_path_progress
    return np.array([s, chi, y_e, s_la, la_err, head_err, goal, prog]), reached, math.hypot(*rel)


# nav[0..7] = s, chi, y_e, s_la, look-ahead heading error, heading error, goal distance, progress.  chi and the
# heading errors come from FP32 atan2 in the kernel (they feed float32 observations); the rest is FP64
NAV_ATOL = np.array([S_TOL, 1e-6, 1e-9, S_TOL, 1e-6, 1e-6, 1e-9, 1e-12])
NAV_RTOL = np.array([0.0, 0.0, 1e-12, 0.0, 0.0, 0.0, 1e-12, 0.0])
ANGLES = np.array([False, True, False, False, True, True, False, False])


def _nav_err(got, want, la_dist):
    d = np.abs(got - want)
    d[ANGLES] = np.abs(_wrap(got[ANGLES] - want[ANGLES]))
    if la_dist < 1e-3:  # the vessel sits on the look-ahead point (the path's end): its bearing is rounding noise
        d[5] = 0.0
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("family", list(FAMILIES))
def test_projection_matches_the_exact_first_minimum(family, variant, built_lib):
    import torch

    from gym_auv_b200 import lidar_config
    from gym_auv_b200.vec_env import AUVVecEnv
    from oracle.sim import OraclePath, OracleVessel
    from tests._parity import oracle_cfg

    key, gen = FAMILIES[family]
    if variant == "device":
        key = DEVICE_KEY.get(key, key)
    cfg = lidar_config()
    scn = _scenarios(key, variant)
    pts = gen(build_path(PATHS[key]))
    P = len(scn.waypoints)
    N = len(pts) * P  # mixed_paths: every point once on each path, envs shuffled across the CTAs
    env = AUVVecEnv(scn, N, cfg, test_mode=True, auto_reset=False, debug=True)
    if variant == "no_sub_tables":
        env.paths.sub_chord = None
        env.paths.sub_dev = None
    env.reset()
    perm = np.random.RandomState(1).permutation(N) if P > 1 else np.arange(N)
    pid = perm % P  # env e queries point perm[e] // P on path perm[e] % P
    pt = pts[perm // P]
    if P > 1:
        env.reset_envs(torch.ones(N, dtype=torch.uint8), torch.as_tensor(pid, dtype=torch.int32))
    assert np.array_equal(env._st["env_pid"].cpu().numpy(), pid)
    paths = [_device_path(env, q) for q in range(P)]
    refs = np.empty(N, dtype=object)
    for q in range(P):
        sel = np.nonzero(pid == q)[0]
        ck = (family, variant == "device", q)
        if ck not in _cache:
            _cache[ck] = reference(paths[q][0], pts)
        r = _cache[ck]
        refs[sel] = [r[i] for i in perm[sel] // P]
    nseg = np.array([len(paths[q][0]) - 1 for q in range(P)])[pid]
    best = np.array([r.best for r in refs])
    psi = 0.3 + 0.001 * np.arange(N)
    warms = dict(cold=np.full(N, -1), first=np.zeros(N, int), last=nseg - 1, other_branch=np.array([r.other for r in refs]),
                 far=(best + nseg // 2) % nseg)
    assert (np.abs(warms["far"] - best) >= 30 * 8).all()
    state0 = torch.zeros((6, N), dtype=torch.float64, device="cuda")
    state0[0] = torch.as_tensor(pt[:, 0], device="cuda")
    state0[1] = torch.as_tensor(pt[:, 1], device="cuda")
    state0[2] = torch.as_tensor(psi, device="cuda")
    zero = torch.zeros((N, 2), dtype=torch.float32, device="cuda")
    ocfg = oracle_cfg(cfg)
    opaths = [OraclePath(w) for w in scn.waypoints]
    counts = dict(decisive=0, tie=0, near=0)
    for r in refs:
        counts[r.kind] += 1
    worst = np.zeros(8)
    results = {}
    for name, w in warms.items():
        env.state.copy_(state0)
        env._st["prev_seg"].copy_(torch.as_tensor(w, dtype=torch.int32))
        env.step(zero)
        torch.cuda.synchronize()
        # with nu = 0 and tau = 0 the RKF45 step leaves the position as it is, bit for bit (the heading is
        # re-wrapped into [-pi, pi), which may round its last bit)
        assert torch.equal(env.state[:2], state0[:2]) and torch.equal(env.state[3:], state0[3:]), (name, "vessel moved")
        assert float((env.state[2] - state0[2]).abs().max()) <= 1e-15, name
        seg = env._st["prev_seg"].cpu().numpy()
        nav = env.get_attr("nav")[:, :11].cpu().numpy()
        results[name] = (seg, nav)
        bad = []
        for e in range(N):
            poly, cum, h, spline = paths[pid[e]]
            why = check_projection(poly, cum, pt[e], refs[e], int(seg[e]), float(nav[e, 0]))
            if why is not None:
                bad.append((e, refs[e].kind, why))
        assert not bad, (family, variant, name, len(bad), bad[:5])
    # navigation features (the same for every warm start: the projection is an exact arg-min)
    seg, nav = results["cold"]
    s_exact = sum(float(nav[e, 0]) == _measure(paths[pid[e]][0], paths[pid[e]][1], pt[e], int(seg[e])) for e in range(N))
    for name, (s2, n2) in results.items():
        assert np.array_equal(s2, seg) and np.array_equal(n2, nav), (family, variant, name)
    # Against navigate's formulas on the PCHIP pieces the kernel read (which isolates the projection), and at
    # decisive points against OracleVessel.navigate on the oracle's own SciPy path end to end.  The device-built
    # pieces and polyline differ from SciPy's in the last bits (1e-9 relative / 1e-10 m, pinned by
    # test_device_path_builder_matches_scipy_tables), so that comparison allows ten times the tolerance there.
    oracle_tol = 10.0 if variant == "device" else 1.0
    worst_oracle = np.zeros(8)
    for e in range(N):
        poly, cum, h, spline = paths[pid[e]]
        want, reached, la_dist = _navigate_at(spline, h, cfg, pt[e], psi[e], float(nav[e, 0]))
        err = _nav_err(nav[e, :8], want, la_dist)
        worst = np.maximum(worst, err)
        assert (err <= NAV_ATOL + NAV_RTOL * np.abs(want)).all(), (family, variant, e, err, nav[e, :8], want)
        assert bool(nav[e, 10]) == reached, (family, variant, e, "reached_goal")
        if refs[e].kind == "decisive":  # the oracle end to end: its own path and projection
            v = OracleVessel(ocfg, [pt[e][0], pt[e][1], psi[e]])
            v.navigate(opaths[pid[e]])
            o = v.nav
            want = np.array([o["vessel_arclength"], opaths[pid[e]].direction(o["vessel_arclength"]),
                             100 * o["cross_track_error"], o["target_arclength"], o["look_ahead_heading_error"],
                             o["heading_error"], o["goal_distance"], v.progress])
            err = _nav_err(nav[e, :8], want, la_dist)
            worst_oracle = np.maximum(worst_oracle, err)
            assert (err <= oracle_tol * (NAV_ATOL + NAV_RTOL * np.abs(want))).all(), (family, variant, e, "oracle", err)
            assert bool(nav[e, 10]) == v.reached_goal, (family, variant, e, "oracle reached_goal")
    if family == "past_ends":
        L = np.array([float(paths[q][2]["length"]) for q in range(P)])[pid]
        at_end = np.array([r.best in (0, n - 1) for r, n in zip(refs, nseg)])
        assert at_end.sum() >= 0.9 * N
        end_s = np.array([0.0 if r.best == 0 else float(paths[q][1][-1]) for r, q in zip(refs, pid)])
        assert np.abs(nav[at_end, 0] - end_s[at_end]).max() <= S_TOL
        assert np.array_equal(nav[at_end, 3], np.minimum(L[at_end], nav[at_end, 0] + cfg.vessel.look_ahead_distance))
        assert nav[at_end, 10].any() and not nav[at_end, 10].all()  # reached_goal at the far end only
    env.check_status()
    print(f"\n{family}/{variant}: {N} envs, {counts}, arclength bit-equal to the FP64 measure {s_exact}/{N}, nav max err "
          f"{np.array2string(worst, precision=2)}, vs oracle {np.array2string(worst_oracle, precision=2)}")
