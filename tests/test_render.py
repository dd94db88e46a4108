"""Top-down RGB frames (auv_render / k_render, AUVVecEnv.render and the gym / VecEnv facades) against the FP64
reference rasteriser of tests/_render_ref.py, plus the C-ABI argument checks and the read-only guarantee."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from gym_auv_b200 import _lib
from oracle import geos_lite as G
from tests import _render_ref as RR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _scene(**kw):
    base = dict(pos=(1000.0, -500.0), psi=0.0, vessel_width=1.255, rays=None, moving=[], static=[],
                goal=(1e6, 1e6), path=None, world=[])
    base.update(kw)
    return base


# ---------------------------------------------------------------- reference rasteriser on hand-made scenes (CPU)
def test_ref_square_pixel_count():
    p0 = np.array([1000.0, -500.0])
    sq = np.array([[40.2, 40.2], [60.2, 40.2], [60.2, 60.2], [40.2, 60.2], [40.2, 40.2]]) + p0
    rgb, layer, margin = RR.rasterise(_scene(world=[sq]), 200, 200, 100.0)  # s = 1 m: centres at k + 0.5
    assert (layer == RR.LAND).sum() == 400
    assert (margin[layer == RR.LAND] > 0.2).all()


def test_ref_pentagon_points_north_at_heading_zero():
    rgb, layer, _ = RR.rasterise(_scene(vessel_width=20.0), 100, 100, 50.0)  # s = 1 m
    rows, cols = np.nonzero(layer == RR.SHIP)
    dx = 50 - rows - 0.5  # metres north of the vessel
    dy = cols + 0.5 - 50
    assert dx.max() > 20.0 and dx.min() > -16.0  # tip 11/9 w north, tail 7/9 w south of the centroid
    tip = dx == dx.max()
    assert np.abs(dy[tip]).max() <= 1.0  # the tip pixels are on the centre line
    assert (rgb[layer == RR.SHIP] == RR.rgb_of(RR.SHIP)).all()


def test_ref_pixel_origin_is_north_west_corner():
    W, H, hw = 64, 48, 32.0
    s = 2 * hw / W
    p0 = np.array([1000.0, -500.0])
    goal = p0 + np.array([(H / 2 - 0.5) * s, (0.5 - W / 2) * s])  # centre of pixel (0, 0)
    _, layer, _ = RR.rasterise(_scene(goal=tuple(goal)), W, H, hw)
    assert layer[0, 0] == RR.GOAL and layer[0, W - 1] != RR.GOAL and layer[H - 1, 0] != RR.GOAL


@pytest.mark.parametrize("radius", [3.0, 30.0])
def test_ref_ngon_area(radius):
    p0 = np.array([1000.0, -500.0])
    W, hw = 400, 50.0
    s = 2 * hw / W
    c = p0 + np.array([10.3, -7.1])
    _, layer, _ = RR.rasterise(_scene(static=[(c, radius)]), W, W, hw)
    n = G.circle_ngon_sides(radius)
    area = 0.5 * n * radius**2 * math.sin(2 * math.pi / n)
    perimeter = 2 * n * radius * math.sin(math.pi / n)
    assert abs((layer == RR.STATIC).sum() * s * s - area) <= perimeter * s


@pytest.mark.parametrize("log_transform", [True, False])
def test_ref_ray_length_inverts_k_lidar_closeness(log_transform):
    rng = 150.0
    d = np.concatenate([np.linspace(0.0, 149.9, 97), [1e-3, 1.255]])
    if log_transform:  # k_lidar: 1 - clip(log(1 + d) / log(1 + range), 0, 1)
        c = 1.0 - np.clip(np.log1p(d) / np.log1p(rng), 0.0, 1.0)
    else:
        c = 1.0 - np.clip(d / rng, 0.0, 1.0)
    back = RR.ray_length(c.astype(np.float32).astype(np.float64), rng, log_transform)
    np.testing.assert_allclose(back[c > 0], d[c > 0], rtol=1e-5, atol=1e-4)
    assert RR.ray_length(np.zeros(1), rng, log_transform)[0] == rng


def test_ref_predicates_match_oracle():
    rs = np.random.RandomState(3)
    ring = G.circle_boundary_ring(0.3, -0.2, 5.0)
    pts = rs.uniform(-7, 7, size=(400, 2))
    inside = RR.in_ring(pts[:, 0], pts[:, 1], ring)
    assert list(inside) == [G.point_in_ring(p, ring) for p in pts]
    a, b = rs.uniform(-3, 3, size=(2, 2))
    d = RR.seg_dist(pts[:, 0], pts[:, 1], a[0], a[1], b[0], b[1])
    ref = [G.point_segment_distance(p[0], p[1], a[0], a[1], b[0], b[1]) for p in pts]
    np.testing.assert_allclose(d, ref, rtol=1e-15, atol=0)  # np.hypot and math.hypot may differ in the last bit


# ---------------------------------------------------------------- binding (CPU)
def test_palette_and_layer_constants_match_header():
    hdr = open(os.path.join(ROOT, "include", "auv_b200.h")).read()
    found = 0
    for name, val in re.findall(r"#define AUV_(RGB_\w+|RENDER_\w+)\s+(0x[0-9A-Fa-f]+u?|[0-9.]+)", hdr):
        v = int(val.rstrip("u"), 16) if val.startswith("0x") else float(val)
        assert getattr(_lib, name) == v, name
        found += 1
    assert found == 14


def test_render_struct_size(built_lib):
    lib = _lib.load()
    assert C.sizeof(_lib.AuvRender) == lib.auv_sizeof(13)


def _bad_render_args():
    """host structs that every validation step accepts except the one each case breaks.  n_envs is 0 in every
    case, so even a check that did not fire could never reach a launch."""
    from gym_auv_b200 import Config
    from gym_auv_b200.vec_env import make_auv_config

    cfg = make_auv_config(Config(), "colav", False, True, "reference")
    cfg.use_lidar, cfg.n_sensors, cfg.n_sectors = 1, 180, 9
    dummy = 4096
    rays = _lib.AuvRayTable(dummy, dummy, dummy, dummy, 1.0)
    paths = _lib.AuvPathBank()
    pool = _lib.AuvScenarioPool()
    batch = _lib.AuvBatch()
    r = _lib.AuvRender(4, 64, 64, 0, dummy, 50.0)
    return cfg, rays, paths, pool, batch, r, dummy


@pytest.mark.parametrize("case", ["cfg", "rays", "paths", "pool", "batch", "desc", "frames", "env_ids", "obs",
                                  "count", "width0", "width_big", "height0", "height_big", "hw_zero", "hw_neg",
                                  "hw_nan", "hw_inf"])
def test_render_rejects_bad_arguments(built_lib, case):
    lib = _lib.load()
    cfg, rays, paths, pool, batch, r, dummy = _bad_render_args()
    obs, frames = dummy, dummy
    args = dict(cfg=C.byref(cfg), rays=C.byref(rays), paths=C.byref(paths), pool=C.byref(pool), batch=C.byref(batch),
                desc=C.byref(r))
    if case in args:
        args[case] = None
    elif case == "frames":
        frames = None
    elif case == "env_ids":
        r.env_ids = None
    elif case == "obs":
        obs = None
    elif case == "count":
        r.count = 0
    elif case.startswith("width") or case.startswith("height"):
        setattr(r, case.split("_")[0].rstrip("0"), 0 if case.endswith("0") else 4097)
    else:
        r.half_width = {"hw_zero": 0.0, "hw_neg": -1.0, "hw_nan": float("nan"), "hw_inf": float("inf")}[case]
    rc = lib.auv_render(args["cfg"], args["rays"], args["paths"], args["pool"], args["batch"], obs, args["desc"],
                        frames, None)
    assert rc == -1  # AUV_EINVAL
    msg = lib.auv_last_error().decode()
    expect = {"obs": "obs", "count": "count", "hw": "half_width", "width": "width and height",
              "height": "width and height"}
    key = next((k for k in expect if case.startswith(k)), None)
    assert (expect[key] if key else "NULL") in msg, msg


# ---------------------------------------------------------------- GPU: kernel against the reference
torch = pytest.importorskip("torch")


def _compare(env, ids, width, height, half_width, frames=None):
    if frames is None:
        frames = env.render(ids, width=width, height=height, half_width=half_width)
    got = frames.cpu().numpy()
    scenes = RR.env_scenes(env, ids)
    total_nd = 0
    for k, sc in enumerate(scenes):
        rgb, layer, margin = RR.rasterise(sc, width, height, half_width)
        decisive = margin > RR.NONDECISIVE_PX
        bad = decisive & (got[k] != rgb).any(axis=-1)
        assert not bad.any(), (ids[k], half_width, np.argwhere(bad)[:5], layer[bad][:5], got[k][bad][:5])
        total_nd += int((~decisive).sum())
    n_px = len(ids) * width * height
    print(f"non-decisive pixels: {total_nd} of {n_px} (half_width {half_width})")
    assert total_nd <= 1e-3 * n_px
    return got


def _random_steps(env, steps, seed):
    g = torch.Generator(device=env.device).manual_seed(seed)
    lo = torch.tensor([-1.0, -0.15], device=env.device)
    for _ in range(steps):
        a = torch.rand((env.num_envs, 2), generator=g, device=env.device) * (-2 * lo) + lo
        _, _, done, _ = env.step(a)
    return done


def _with_last_reset(env, done, picks):
    d = torch.nonzero(done).flatten().cpu().numpy()
    ids = list(picks)
    if len(d):
        ids[-1] = int(d[0])
    return ids, len(d) > 0


@pytest.mark.gpu
def test_render_config3_shape():
    from gym_auv_b200 import lidar_config, scenarios as S
    from gym_auv_b200.vec_env import AUVVecEnv

    N = 4096
    scn = S.moving_obstacles_template(2 * N, 17, 11, seed=3, n_paths=64, path_period=N, device_paths=True)
    env = AUVVecEnv(scn, N, lidar_config(), auto_reset=True)
    env.regenerate_scenarios(seed=5, epoch=1)
    env.reset()
    done = _random_steps(env, 300, 7)
    for extra in range(200):
        if bool(done.any()):
            break
        done = _random_steps(env, 1, 100 + extra)
    ids, has_reset = _with_last_reset(env, done, np.arange(16) * 251)
    assert has_reset
    for hw in (150.0, 300.0):
        _compare(env, ids, 256, 192, hw)


@pytest.mark.gpu
def test_render_land_grid_and_no_grid():
    from gym_auv_b200 import lidar_config, scenarios as S
    from gym_auv_b200.vec_env import AUVVecEnv

    N = 1024
    envs = []
    for grid in (True, False):
        scn = S.land_template(2 * N, 512, 16, 16, seed=2, n_paths=64, path_period=N, device_paths=True)
        env = AUVVecEnv(scn, N, lidar_config(), auto_reset=True, world_grid=grid, max_nearby=96)
        env.regenerate_scenarios(seed=9, epoch=1)
        env.reset()
        done = _random_steps(env, 120, 11)
        envs.append(env)
    assert "world_cell_off" in envs[0]._pool and "world_cell_off" not in envs[1]._pool
    ids = [int(i) for i in np.arange(16) * 61]
    a = _compare(envs[0], ids, 256, 192, 300.0)
    b = envs[1].render(ids, width=256, height=192, half_width=300.0).cpu().numpy()
    np.testing.assert_array_equal(a, b)  # same states, same frames with and without the grid
    land = (a == RR.rgb_of(RR.LAND)).all(axis=-1).mean()
    assert land > 0.0
    # zoomed out over the whole world: tile (1, 1) of a 96 x 96 frame spans 8 km around the vessel, so its display
    # list takes more than one chunk of polygons (every polygon without the grid, some listed once per cell with it)
    ids4, W, hw = ids[:4], 96, 12000.0
    s = 2 * hw / W
    st = envs[1].state.cpu().numpy()
    circ = envs[1].scenarios.world.circle
    for e in ids4:
        half = (W / 2 - 32 - 0.5) * s  # tile (1, 1)'s pixel centres span [-half, half] in both axes
        gap = np.maximum(np.abs(circ[:, :2] - st[0:2, e]) - half, 0.0)
        assert int((np.hypot(gap[:, 0], gap[:, 1]) <= circ[:, 2]).sum()) > 256  # polygons the tile lists
    a = _compare(envs[0], ids4, W, W, hw)
    b = _compare(envs[1], ids4, W, W, hw)
    np.testing.assert_array_equal(a, b)


@pytest.mark.gpu
def test_render_mostly_land_without_grid():
    """A ring with a slit into a hole around the vessel start: land everywhere in the frame but the hole."""
    from gym_auv_b200 import lidar_config, scenarios as S
    from gym_auv_b200.vec_env import AUVVecEnv

    scn = S.moving_obstacles(2, 0, 3, seed=4)
    x, y = scn.vessel_init[0, :2]
    ring = np.array([[-1000, -1000], [1000, -1000], [1000, 1000], [-1000, 1000], [-1000, 0.5], [-15, 0.5], [-15, 15],
                     [15, 15], [15, -15], [-15, -15], [-15, -0.5], [-1000, -0.5], [-1000, -1000]], dtype=np.float64)
    scn.world_polygons = [ring + np.array([x, y])]
    env = AUVVecEnv(scn, 2, lidar_config(), auto_reset=True)
    env.reset()
    _random_steps(env, 3, 1)
    got = _compare(env, [0], 320, 240, 150.0)
    assert (got[0] == RR.rgb_of(RR.LAND)).all(axis=-1).mean() > 0.5  # rays, obstacles and the path draw over the rest


@pytest.mark.gpu
def test_render_table_tracks_velocity_channels():
    from gym_auv_b200 import lidar_config, scenarios as S
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config(sensor_use_velocity_observations=True)
    cfg.simulation.t_step_size = 0.5
    env = AUVVecEnv(S.debug_scenario(), 8, cfg, auto_reset=True, linear_tracks=False, velocity_mode="nearest")
    assert env.linear is None and env.obs_dim == 6 + 3 * env.n_sensors
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(2)
    for _ in range(60):
        a = torch.stack([torch.full((8,), 0.8, device=env.device),
                         (torch.rand(8, generator=g, device=env.device) - 0.5) * 0.1], dim=1)
        env.step(a)
    got = _compare(env, list(range(8)), 256, 256, 150.0)
    assert (got == RR.rgb_of(RR.MOVING)).all(axis=-1).any()


@pytest.mark.gpu
def test_render_without_lidar_has_no_rays():
    from gym_auv_b200 import Config, scenarios as S
    from gym_auv_b200.vec_env import AUVVecEnv

    env = AUVVecEnv(S.path_follow_no_obstacles(8, seed=1), 8, Config(), auto_reset=True)
    assert not env.config.vessel.use_lidar
    env.reset()
    _random_steps(env, 20, 3)
    got = _compare(env, list(range(8)), 200, 200, 100.0)
    for layer in (RR.RAY_HIT, RR.RAY_CLEAR):
        assert not (got == RR.rgb_of(layer)).all(axis=-1).any()
    assert (got == RR.rgb_of(RR.PATH)).all(axis=-1).any()


def _twins(n=256, **kw):
    from gym_auv_b200 import lidar_config, scenarios as S
    from gym_auv_b200.vec_env import AUVVecEnv

    out = []
    for _ in range(2):
        env = AUVVecEnv(S.moving_obstacles(64, 17, 11, seed=6), n, lidar_config(), auto_reset=True, **kw)
        env.reset()
        out.append(env)
    return out


@pytest.mark.gpu
def test_render_is_read_only():
    a, b = _twins()
    g = torch.Generator(device=a.device).manual_seed(4)
    ids = list(range(0, 256, 17))
    for _ in range(200):
        act = torch.rand((256, 2), generator=g, device=a.device) * torch.tensor([2.0, 0.3], device=a.device) - torch.tensor(
            [1.0, 0.15], device=a.device)
        ra = a.step(act)
        a.render(ids, width=96, height=64, half_width=150.0)
        rb = b.step(act)
        for x, y in zip(ra[:3], rb[:3]):
            assert torch.equal(x, y)
        for k in ra[3]:
            assert torch.equal(ra[3][k], rb[3][k]), k
    assert torch.equal(a.state, b.state)
    for k in ("t_step", "cumulative_reward", "episode", "max_progress", "nearby_mask", "nav"):
        assert torch.equal(a.get_attr(k), b.get_attr(k)), k


@pytest.mark.gpu
def test_render_is_read_only_async_delta():
    a, b = _twins(host_transfer="delta")
    rs = np.random.RandomState(8)
    ids = list(range(0, 256, 17))
    for _ in range(200):
        act = rs.uniform([-1, -0.15], [1, 0.15], size=(256, 2)).astype(np.float32)
        a.step_async(act)
        with pytest.raises(RuntimeError):
            a.render(ids)
        oa, ra, da = (x.copy() for x in a.step_wait())
        a.render(ids, width=96, height=64, half_width=150.0)
        b.step_async(act)
        ob, rb, db = b.step_wait()
        np.testing.assert_array_equal(oa, ob)
        np.testing.assert_array_equal(ra, rb)
        np.testing.assert_array_equal(da, db)
    torch.cuda.synchronize()
    assert torch.equal(a.state, b.state)
    assert torch.equal(a._out["obs"], b._out["obs"])


@pytest.mark.gpu
def test_render_deterministic_and_out_of_range_ids():
    a, _ = _twins(n=64)
    _random_steps(a, 30, 5)
    f1 = a.render([3, 9, 40], width=200, height=150, half_width=120.0)
    f2 = a.render([3, 9, 40], width=200, height=150, half_width=120.0)
    assert torch.equal(f1, f2)
    ids = torch.tensor([3, 64, 9, -1, 40], dtype=torch.int32, device=a.device)
    f3 = a.render(ids, width=200, height=150, half_width=120.0)
    assert int(f3[1].abs().sum()) == 0 and int(f3[3].abs().sum()) == 0
    assert torch.equal(f3[[0, 2, 4]], f1)
    with pytest.raises(ValueError):
        a.render([0, 64])
    with pytest.raises(ValueError):
        a.render([-1])
    with pytest.raises(ValueError):
        a.render([])
    wide = torch.tensor([3, 2**32 + 3, 9, -(2**32) + 9, 40], dtype=torch.int64, device=a.device)  # no wrap into the batch
    f4 = a.render(wide, width=200, height=150, half_width=120.0)
    assert int(f4[1].abs().sum()) == 0 and int(f4[3].abs().sum()) == 0
    assert torch.equal(f4[[0, 2, 4]], f1)


@pytest.mark.gpu
def test_render_facades():
    from gym_auv_b200 import lidar_config, make, scenarios as S
    from gym_auv_b200.adapters import B200VecEnv

    env = make("MovingObstaclesNoRules-v0", lidar_config())
    assert env.metadata["render.modes"] == ["rgb_array"]
    env.step([0.5, 0.0])
    img = env.render()
    assert img.dtype == np.uint8 and img.shape == (400, 400, 3)
    assert (img[199:201, 199:201] == RR.rgb_of(RR.SHIP)).all()
    with pytest.raises(NotImplementedError):
        env.render(mode="human")
    cfg = lidar_config()
    cfg.vessel.render_distance = "auto"
    with pytest.raises(ValueError):
        make("MovingObstaclesNoRules-v0", cfg).render()
    assert env.render(width=64, height=32, half_width=50.0).shape == (32, 64, 3)

    venv = B200VecEnv(S.moving_obstacles(40, 17, 11, seed=2), 20, lidar_config())
    venv.reset()
    venv.step(np.zeros((20, 2), dtype=np.float32))
    imgs = venv.get_images()
    assert len(imgs) == 16 and all(i.shape == (400, 400, 3) and i.dtype == np.uint8 for i in imgs)
    tiled = venv.render()
    assert tiled.shape == (1600, 1600, 3)
    np.testing.assert_array_equal(tiled[400:800, 1200:1600], imgs[7])
    five = venv.render(indices=[0, 1, 2, 3, 19])
    assert five.shape == (800, 1200, 3)
    assert (five[400:800, 800:1200] == 0).all()  # padding
    np.testing.assert_array_equal(five[400:800, 400:800], venv.get_images([19])[0])
    with pytest.raises(NotImplementedError):
        venv.render(mode="human")
    with pytest.raises(ValueError):
        venv.get_images([20])
    with pytest.raises(ValueError):
        venv.render(indices=[])
    venv.config.vessel.render_distance = "auto"
    with pytest.raises(ValueError):
        venv.get_images()
    assert venv.render(indices=[0, 1], half_width=80.0).shape == (400, 800, 3)
    assert venv.get_images([2], half_width=80.0)[0].shape == (400, 400, 3)
    venv.step_async(np.zeros((20, 2), dtype=np.float32))
    with pytest.raises(RuntimeError):
        venv.render()
    venv.step_wait()
