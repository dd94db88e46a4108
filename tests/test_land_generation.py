"""Scenario generation on the GPU inside a shared world of land polygons (DESIGN.md section 6b).

Every object the generator places must be CLEAR OF LAND BY d: outside every world polygon (even-odd rule on
the closed ring) and at an FP64 distance > d from every ring -- the vessel start by LAND_CLEARANCE, a static
circle's centre by its radius, a moving obstacle's track start by its width.  The reference below restates
``oracle.geos_lite.point_in_ring`` / ``point_ring_distance`` vectorised over a polygon's ring (and is checked
against them); kernel decisions are compared where the reference is more than 1e-9 m from the threshold."""
import dataclasses

import numpy as np
import pytest
from scipy.spatial import cKDTree

from gym_auv_b200 import lidar_config, scenarios as S
from gym_auv_b200.polygons import World, star_polygon
from gym_auv_b200.scenarios import LAND_CLEARANCE
from oracle.geos_lite import point_in_ring, point_ring_distance

BAND = 1e-9  # m: decisions closer than this to the threshold are not compared


def signed_distance(points, rings, reach):
    """FP64 signed distance of each point to the union of the filled rings: + outside, - inside, 0 on a
    boundary (boundary points count as inside, as in point_in_ring).  Rings whose every vertex is farther
    than reach[i] + 1 m from point i are skipped (the result is then > reach[i] there).  Returns +inf
    where no ring is within reach."""
    points = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    reach = np.broadcast_to(np.asarray(reach, dtype=np.float64), (len(points),))
    out = np.full(len(points), np.inf)
    if not len(points) or not len(rings):
        return out
    tree = cKDTree(points)
    rmax = float(reach.max())
    for ring in rings:
        ring = np.asarray(ring, dtype=np.float64)
        c = 0.5 * (ring.min(axis=0) + ring.max(axis=0))
        rho = float(np.hypot(*(ring - c).T).max())
        cand = np.array(tree.query_ball_point(c, rho + rmax + 1.0), dtype=np.int64)
        if not len(cand):
            continue
        cand = cand[np.hypot(*(points[cand] - c).T) <= rho + reach[cand] + 1.0]
        if not len(cand):
            continue
        x, y = points[cand, 0:1], points[cand, 1:2]
        x1, y1, x2, y2 = ring[:-1, 0], ring[:-1, 1], ring[1:, 0], ring[1:, 1]
        # point_in_ring: crossing number, a crossing AT the point is "inside"
        cross = (y1 > y) != (y2 > y)
        with np.errstate(divide="ignore", invalid="ignore"):
            xint = x1 + (y - y1) * (x2 - x1) / np.where(cross, y2 - y1, 1.0)
        on = (cross & (xint == x)).any(axis=1)
        inside = on | ((cross & (xint > x)).sum(axis=1) % 2 == 1)
        # point_segment_distance, minimised over the ring
        ex, ey = x2 - x1, y2 - y1
        len2 = ex * ex + ey * ey
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.where(len2 > 0, ((x - x1) * ex + (y - y1) * ey) / np.where(len2 > 0, len2, 1.0), 0.0)
            s = ((y1 - y) * ex - (x1 - x) * ey) / np.where(len2 > 0, len2, 1.0)
        d_a, d_b = np.hypot(x - x1, y - y1), np.hypot(x - x2, y - y2)
        d = np.where(r <= 0.0, d_a, np.where(r >= 1.0, d_b, np.abs(s) * np.sqrt(len2)))
        dist = d.min(axis=1)
        sd = np.where(inside, -dist, dist)
        out[cand] = np.minimum(out[cand], sd)
    return out


def land_rule(points, d, rings):
    """(clear, decisive) of "clear of land by d" for each point."""
    d = np.broadcast_to(np.asarray(d, dtype=np.float64), (len(points),))
    sd = signed_distance(points, rings, d)
    return sd > d, np.abs(sd - d) > BAND


def objects(g):
    """(kind, scenario, points, d) of everything the generator places, scenario-major."""
    M, Km, Ks = g.n_scenarios, g.k_moving, g.k_static
    return [("start", np.arange(M), g.vessel_init[:, :2], np.full(M, LAND_CLEARANCE)),
            ("track", np.repeat(np.arange(M), Km), g.mov_start.reshape(-1, 2), g.mov_width.ravel()),
            ("circle", np.repeat(np.arange(M), Ks), g.st_pos.reshape(-1, 2), g.st_radius.ravel())]


def rule_per_object(g, rings):
    return {k: (m, *land_rule(p, d, rings)) for k, m, p, d in objects(g)}


def assert_rule_holds(g, rings, skip=None):
    """Every decisive object obeys the rule (scenarios in `skip` excluded for the vessel start).  Returns the
    number of non-decisive objects."""
    nd = 0
    for k, (m, clear, dec) in rule_per_object(g, rings).items():
        keep = np.ones(len(m), bool) if skip is None or k != "start" else ~np.isin(m, skip)
        bad = keep & dec & ~clear
        assert not bad.any(), (k, np.nonzero(bad)[0][:5])
        nd += int((keep & ~dec).sum())
    return nd


def square(cx, cy, h):
    return np.array([[cx - h, cy - h], [cx + h, cy - h], [cx + h, cy + h], [cx - h, cy + h]])


# ---------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------
def test_land_reference_rejects_its_negative_controls():
    rng = np.random.RandomState(4)
    star = star_polygon(rng, np.array([100.0, -50.0]), 80.0, 24)
    ring = np.vstack([star, star[:1]])
    d = 30.0
    # inside the non-convex star: its centre
    clear, dec = land_rule(np.array([[100.0, -50.0]]), d, [ring])
    assert dec[0] and not clear[0]
    # d -/+ 1e-6 below / above the bottom edge of a square
    sq = np.vstack([square(0.0, 0.0, 50.0), [[-50.0, -50.0]]])
    pts = np.array([[10.0, -50.0 - (d - 1e-6)], [10.0, -50.0 - (d + 1e-6)]])
    clear, dec = land_rule(pts, d, [sq])
    assert dec.all() and not clear[0] and clear[1]
    # a concave notch of the star: 0.5 m radially out of a vertex that lies closer to the centre than both
    # neighbours -- outside the polygon but within d of two edges; it must not be called inside
    rad = np.hypot(*(star - [100.0, -50.0]).T)
    k = next(i for i in range(len(star)) if rad[i] < rad[i - 1] and rad[i] < rad[(i + 1) % len(star)])
    u = (star[k] - [100.0, -50.0]) / rad[k]
    notch = star[k] + 0.5 * u
    sd = signed_distance(notch[None], [ring], d)[0]
    assert not point_in_ring(notch, ring) and 0.0 < sd < d
    clear, dec = land_rule(notch[None], d, [ring])
    assert dec[0] and not clear[0]
    # the vectorised restatement decides as geos_lite does, point by point
    pts = np.array([100.0, -50.0]) + rng.uniform(-150, 150, size=(600, 2))
    sd = signed_distance(pts, [ring], 400.0)
    for p, s in zip(pts, sd):
        inside = point_in_ring(p, ring)
        dist = point_ring_distance(p, ring)
        assert (s <= 0.0) == inside and abs(abs(s) - dist) <= 1e-9, (p, s, inside, dist)


def test_land_template_keeps_every_start_square_clear():
    scn = S.land_template(64, n_polygons=512, n_moving=4, n_static=4, seed=1, n_paths=32, extent=1600.0)
    rings = World(scn.world_polygons).rings
    assert len(rings) == 512
    p0 = np.array([t(0.0) for t in scn.bank.tables])
    corners = (p0[:, None, :] + np.array([[-25, -25], [25, -25], [25, 25], [-25, 25]])[None]).reshape(-1, 2)
    clear, dec = land_rule(corners, LAND_CLEARANCE, rings)
    assert clear.all() and dec.all()
    # the margin binds: land comes within 100 m of some start square
    assert (signed_distance(corners, rings, 100.0) < 100.0).any()


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib(built_lib):
    torch = pytest.importorskip("torch")
    from gym_auv_b200 import _lib

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return _lib.load()


def _without_world(scn):
    return dataclasses.replace(scn, world_polygons=[], _world=None)


def _scenario_equal(a, b):
    """[M] bool: every array the generator writes is bit-identical for the scenario."""
    M, Km = a.n_scenarios, a.k_moving
    eq = (a.path_id == b.path_id) & (a.vessel_init == b.vessel_init).all(1)
    eq &= (a.mov_start == b.mov_start).all((1, 2)) & (a.mov_width == b.mov_width).all(1)
    eq &= (a.vel_table.reshape(M, Km, 2) == b.vel_table.reshape(M, Km, 2)).all((1, 2))
    eq &= (a.st_pos == b.st_pos).all((1, 2)) & (a.st_radius == b.st_radius).all(1)
    return eq


@gpu
def test_generation_in_a_world_obeys_the_rule_and_changes_only_rejected_draws(lib):
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    M, Km, Ks = 4096, 16, 16
    scn = S.land_template(M, n_polygons=512, n_moving=Km, n_static=Ks, seed=5, n_paths=16, extent=4000.0)
    bank = scn.bank
    starts = np.array([t(0.0) for t in bank.tables])
    gap = np.array([np.delete(np.hypot(*(starts - c).T), p).min() for p, c in enumerate(starts)])
    extra = []
    for p in np.nonzero(gap > 150.0)[0]:  # over one corner of an isolated start square (no other path's is near)
        c0 = starts[p]
        extra.append(square(c0[0] + 25.0, c0[1] + 25.0, 15.0))
    assert len(extra) >= 2
    for p, t in enumerate(bank.tables):  # on the obstacles' sampling area, away from every start square
        mid, ang = t(0.5 * t.length), t.direction(0.5 * t.length) - np.pi / 2
        for side in (-1.0, 1.0):
            c = mid + side * 120.0 * np.array([np.cos(ang), np.sin(ang)])
            if np.hypot(*(starts - c).T).min() > 250.0:
                extra.append(star_polygon(np.random.RandomState(p), c, 50.0, 16))
    scn.world_polygons = list(scn.world_polygons) + extra
    rings = World(scn.world_polygons).rings
    ew = AUVVecEnv(scn, 1024, cfg, auto_reset=True)
    e0 = AUVVecEnv(_without_world(scn), 1024, cfg, auto_reset=True)
    assert ew.n_world == len(rings) and e0.n_world == 0
    ew.regenerate_scenarios(seed=7, epoch=3)
    e0.regenerate_scenarios(seed=7, epoch=3)
    ew.check_status(), e0.check_status()
    gw, g0 = ew.pull_scenarios(), e0.pull_scenarios()
    # the rule, and the existing vessel / goal acceptance and +-25 m jitter
    nondecisive = assert_rule_holds(gw, rings)
    assert nondecisive <= 5, nondecisive
    p0 = np.array([bank.tables[p](0.0) for p in gw.path_id])
    assert np.abs(gw.vessel_init[:, :2] - p0).max() <= 25.0 + 1e-9
    goal = np.array([bank.tables[p](bank.tables[p].length) for p in gw.path_id])
    for pos, rad in ((gw.mov_start, gw.mov_width), (gw.st_pos, gw.st_radius)):
        dv = np.linalg.norm(pos - gw.vessel_init[:, None, :2], axis=2) - cfg.vessel.vessel_width - rad
        dg = np.linalg.norm(pos - goal[:, None, :], axis=2) - rad
        assert np.minimum(dv, dg).min() > 0 and rad.min() >= 1.0
    # exact effect: the world-less draw, judged by the world's rule
    rule0 = rule_per_object(g0, rings)
    clear0 = np.ones(M, bool)
    decisive0 = np.ones(M, bool)
    for m, clear, dec in rule0.values():
        np.logical_and.at(clear0, m, clear)
        np.logical_and.at(decisive0, m, dec)
    same = _scenario_equal(gw, g0)
    assert same[clear0 & decisive0].all(), np.nonzero(clear0 & decisive0 & ~same)[0][:5]
    assert not (~same & clear0 & decisive0).any()
    assert (~clear0[~same]).all()
    assert (~same).sum() >= 50, int((~same).sum())
    # per object: a slot whose world-less draw was clear (and whose vessel start did not move) is unchanged
    vsame = (gw.vessel_init == g0.vessel_init).all(1)
    assert (~vsame).sum() >= 10, "the start-square polygons should force vessel redraws"
    for k, a_w, a_0 in (("track", gw.mov_start, g0.mov_start), ("circle", gw.st_pos, g0.st_pos)):
        m, clear, dec = rule0[k]
        slot_same = (a_w.reshape(-1, 2) == a_0.reshape(-1, 2)).all(1)
        keep = clear & dec & vsame[m]
        assert slot_same[keep].all(), k
        assert (~clear[~slot_same & vsame[m]]).all(), k


@gpu
def test_a_world_out_of_reach_changes_nothing(lib):
    import torch
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    scn = S.moving_obstacles_template(1024, 16, 16, seed=3, n_paths=64)
    rs = np.random.RandomState(1)
    far = [star_polygon(rs, np.array([60000.0, -40000.0]) + rs.uniform(-3000, 3000, 2), 80.0, 20) for _ in range(40)]
    envs = [AUVVecEnv(scn, 512, cfg, auto_reset=True)]
    for grid in (True, False):
        envs.append(AUVVecEnv(dataclasses.replace(scn, world_polygons=far, _world=None), 512, cfg, auto_reset=True,
                              world_grid=grid))
    assert "world_cell_off" in envs[1]._pool and "world_cell_off" not in envs[2]._pool
    for e in envs:
        e.regenerate_scenarios(seed=12, epoch=2)
        e.check_status()
    torch.cuda.synchronize()
    keys = [k for k, v in envs[0]._pool.items() if torch.is_tensor(v) and k != "reset_mask"]
    for e in envs[1:]:
        for k in keys:
            assert torch.equal(envs[0]._pool[k], e._pool[k]), k
        assert torch.equal(envs[0].reset(), e.reset())


@gpu
def test_a_start_square_under_land_raises_the_blocked_bit(lib):
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    scn = S.land_template(256, n_polygons=128, n_moving=6, n_static=6, seed=11, n_paths=4, extent=3000.0)
    starts = np.array([t(0.0) for t in scn.bank.tables])
    p = 3
    c = starts[p]
    assert np.delete(np.hypot(*(starts - c).T), p).min() > 300.0  # the square covers no other start square
    scn.world_polygons = list(scn.world_polygons) + [square(c[0], c[1], 200.0)]
    rings = World(scn.world_polygons).rings
    env = AUVVecEnv(scn, 256, cfg, auto_reset=True)
    env.regenerate_scenarios(seed=2, epoch=1)
    with pytest.raises(RuntimeError, match="start area is covered by land"):
        env.check_status()
    g = env.pull_scenarios()
    blocked = np.nonzero(g.path_id == p)[0]
    assert len(blocked) > 0
    assert_rule_holds(g, rings, skip=blocked)
    clear, _ = land_rule(g.vessel_init[blocked, :2], LAND_CLEARANCE, rings)
    assert not clear.any()
    assert np.abs(g.vessel_init[blocked, :2] - c).max() <= 25.0 + 1e-9  # the last draw is kept
    # a status bit, not a device fault: the env keeps stepping
    import torch

    env._scratch["status"].zero_()
    env.reset()
    for _ in range(5):
        env.step(torch.zeros((256, 2), device="cuda"))
    torch.cuda.synchronize()


@gpu
def test_fresh_device_paths_in_a_world(lib):
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    scn = S.land_template(512, n_polygons=256, n_moving=6, n_static=6, seed=3, n_paths=16, device_paths=True)
    rings = World(scn.world_polygons).rings
    env = AUVVecEnv(scn, 512, cfg, auto_reset=True)
    before = [w.copy() for w in scn.bank.waypoints]
    env.regenerate_paths(seed=41, epoch=2)
    env.regenerate_scenarios(seed=41, epoch=2)
    env.check_status()  # no blocked start, no give-up
    assert any(not np.array_equal(a, b) for a, b in zip(scn.bank.waypoints, before))
    g = env.pull_scenarios()
    assert assert_rule_holds(g, rings) <= 2


@gpu
def test_world_scenarios_generated_on_the_gpu_replay_through_the_oracle(lib):
    from gym_auv_b200.vec_env import AUVVecEnv
    from tests._parity import compare, rollout_gpu, rollout_oracle

    cfg = lidar_config()
    scn = S.land_template(8, n_polygons=48, n_moving=16, n_static=16, seed=9, n_paths=3, extent=1500.0)
    env = AUVVecEnv(scn, 8, cfg, auto_reset=True)
    env.regenerate_scenarios(seed=21, epoch=4)
    env.check_status()
    g = env.pull_scenarios()
    assert len(g.world_polygons) == 48 and (g.st_radius > 0).all() and (g.mov_width > 0).all()
    actions = np.asarray(np.random.RandomState(91).uniform([-1, -0.15], [1, 0.15], size=(40, 8, 2)),
                         dtype=np.float32).astype(np.float64)
    ref = rollout_oracle(g, cfg, actions)
    gpu_out, _ = rollout_gpu(g, cfg, actions)
    rep = compare(ref, gpu_out, cfg, "gpu-generated-world")
    assert rep["windows_checked"] > 0
    assert np.allclose(env._pool["reset_obs"].cpu().numpy(), np.array(ref["obs0"]), atol=2e-5)


@gpu
def test_steady_state_with_device_refresh_in_a_world_matches_the_oracle(lib):
    import torch
    from gym_auv_b200.vec_env import AUVVecEnv
    from tests._parity import live_sample_compare

    cfg = lidar_config()
    N = 16384
    scn = S.land_template(2 * N, n_polygons=512, n_moving=16, n_static=16, seed=2, n_paths=256, extent=4000.0,
                          path_period=N)
    rings = World(scn.world_polygons).rings
    env = AUVVecEnv(scn, N, cfg, test_mode=False, auto_reset=True, debug=True)
    env.regenerate_scenarios(seed=5, epoch=1)
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    lo, hi = torch.tensor([-1.0, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    acts = [lo + (hi - lo) * torch.rand((N, 2), device="cuda", generator=gen) for _ in range(16)]
    refreshed = 0
    for t in range(400):
        env.step(acts[t % 16])
        if t % 8 == 7:
            env.refresh_finished_device(seed=5)
            refreshed += int(env._refresh["count"].item())
    env.check_status()
    assert refreshed > 0
    rep = live_sample_compare(env, cfg, acts, horizon=30, n_sample=32, start=400, prefer_records=True)
    print(rep)
    assert rep["with_records"] >= 20, rep
    assert assert_rule_holds(env.pull_scenarios(), rings) <= 10


@gpu
def test_ring_with_delta_transfer_and_group_refresh_in_a_world_is_bit_identical(lib):
    import torch
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    cfg.episode.max_timesteps = 24  # episodes end inside the rollout: the refreshes have work
    N, G = 2048, 4
    n = N // G
    scn = S.land_template(2 * N, n_polygons=128, n_moving=6, n_static=6, seed=4, n_paths=32, extent=2500.0,
                          path_period=N)
    a, b = AUVVecEnv(scn, N, cfg, auto_reset=True), AUVVecEnv(scn, N, cfg, auto_reset=True)
    for e in (a, b):
        e.regenerate_scenarios(seed=3, epoch=1)
    ring = a.ring(G)
    twin = b.groups(G)
    assert ring.groups[0].host_transfer == "delta"
    ring.reset()
    for g in twin:
        g.reset()
    acts = np.random.RandomState(5).uniform([-1, -0.15], [1, 0.15], size=(80, G, n, 2)).astype(np.float32)
    dones = 0
    for t in range(80):
        for g in range(G):
            ring.send(g, acts[t, g])
        got = {}
        for _ in range(G):
            g, obs, rew, done = ring.recv()
            got[g] = (obs.copy(), rew.copy(), done.copy())
        for g in range(G):
            o, r, d, _ = twin[g].step(torch.as_tensor(acts[t, g], device="cuda"))
            assert np.array_equal(got[g][0], o.cpu().numpy()), (t, g)
            assert np.array_equal(got[g][1], r.cpu().numpy()) and np.array_equal(got[g][2], d.cpu().numpy()), (t, g)
            dones += int(got[g][2].sum())
        if t % 8 == 7:
            for g in range(G):
                ring.groups[g].refresh_finished_device(seed=9)
                twin[g].refresh_finished_device(seed=9)
    torch.cuda.synchronize()
    assert dones > N
    for k in ("path_id", "vessel_init", "mov_start", "st_pos", "reset_obs"):
        assert torch.equal(a._pool[k], b._pool[k]), k
    for g in ring.groups + twin:
        g.check_status()
    ring.close()


@gpu
def test_adapter_with_fresh_scenarios_runs_in_a_world(lib):
    import torch
    from gym_auv_b200.adapters import B200VecEnv

    cfg = lidar_config()
    cfg.episode.max_timesteps = 20
    n = 256
    scn = S.land_template(2 * n, n_polygons=128, n_moving=6, n_static=6, seed=8, n_paths=16, extent=2500.0,
                          path_period=n)
    env = B200VecEnv(scn, n, cfg, fresh_scenarios=True, refresh_every=8, seed=4)
    first = env.impl._pool["st_pos"].clone()
    obs = env.reset()
    assert obs.shape == (n, env.impl.obs_dim)
    rs = np.random.RandomState(2)
    dones = 0
    for _ in range(64):
        obs, rew, done, infos = env.step(rs.uniform([-1, -0.15], [1, 0.15], size=(n, 2)))
        dones += int(done.sum())
    torch.cuda.synchronize()
    env.impl.check_status()
    assert dones > n and np.isfinite(obs).all()
    assert not torch.equal(first, env.impl._pool["st_pos"]), "finished envs' slots were regenerated"
    assert_rule_holds(env.impl.pull_scenarios(), World(scn.world_polygons).rings)
    env.close()
