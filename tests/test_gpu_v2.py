"""GPU parity tests for the round-2 kernel structure: closed-form constant-velocity obstacle
tracks (incl. the wrap of obstacles.py:195-215), shared-memory staged capsule tables vs the
global fallback, the warm-started projection, the LiDAR velocity channel of
simulate_sensor_brute_force (sensor.py:100-137), and oracle samples of the regime that is
benchmarked (steady state after >= 1000 steps with auto-reset and fresh scenarios)."""
import dataclasses
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from gym_auv_b200 import lidar_config, scenarios as S  # noqa: E402
from tests._parity import (compare, live_sample_compare, rollout_gpu, rollout_oracle)  # noqa: E402

pytestmark = pytest.mark.gpu


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def random_actions(T, M, seed):
    return f32(np.random.RandomState(seed).uniform([-1, -0.15], [1, 0.15], size=(T, M, 2)))


@pytest.fixture(scope="module", autouse=True)
def _lib_loaded(built_lib):
    from gym_auv_b200 import _lib

    _lib.load()
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"


def test_closed_form_tracks_equal_the_table_driven_update():
    """Pools of constant-velocity tracks are stepped with the closed form pos0 + n d (no per-env
    obstacle state); the general path accumulates pos += d like the reference.  Same scenarios, both
    ways: obstacle positions agree to 1e-9, everything downstream within the usual tolerances."""
    cfg = lidar_config()
    scn = S.moving_obstacles(12, 9, 7, seed=21)
    acts = random_actions(60, 12, 3)
    ref = rollout_oracle(scn, cfg, acts)
    lin, env_lin = rollout_gpu(scn, cfg, acts)
    gen, env_gen = rollout_gpu(scn, cfg, acts, linear_tracks=False)
    assert env_lin.linear is not None and env_gen.linear is None
    assert "mov_pos" not in env_lin._st and "mov_pos" in env_gen._st
    assert np.abs(lin["mov_pos"] - gen["mov_pos"]).max() < 1e-9
    compare(ref, lin, cfg, "closed form")
    compare(ref, gen, cfg, "table driven")
    alive = ref["alive"]
    assert np.abs(lin["dists"] - gen["dists"])[alive].max() < 1e-4
    assert np.array_equal(lin["done"][alive], gen["done"][alive])
    # the displacement / counter read-back follows the reference's fields too
    d_lin, d_gen = env_lin.get_attr("mov_disp"), env_gen.get_attr("mov_disp")
    assert torch.allclose(d_lin, d_gen, atol=1e-12)
    assert torch.allclose(env_lin.get_attr("mov_counter"), env_gen.get_attr("mov_counter"), atol=1e-9)


@pytest.mark.parametrize("dt", [1.0, 0.5])
def test_closed_form_tracks_wrap_like_the_reference(dt):
    """Short tracks wrap inside the rollout (obstacles.py:199-203: counter and position go back
    to the track start, the counter restarts from 0 -- not from its post-reset value -- so the
    second period is longer than the first)."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    cfg.simulation.t_step_size = dt
    scn = S.moving_obstacles(6, 5, 3, seed=5)
    scn.mov_track[..., 1] = 14  # 14 velocity entries: the first wrap comes after ~12 s
    acts = random_actions(70, 6, 11)
    ref = rollout_oracle(scn, cfg, acts)
    lin, env = rollout_gpu(scn, cfg, acts)
    gen, env_gen = rollout_gpu(scn, cfg, acts, linear_tracks=False)
    assert env.linear is not None and env.linear["first_wrap"] < 30 and env.linear["wrap_period"] < 30
    assert env.linear["wrap_period"] > env.linear["first_wrap"]
    compare(ref, lin, cfg, f"wrap dt={dt}")
    for t in range(acts.shape[0]):
        for m in range(6):
            if ref["alive"][t, m]:
                assert np.abs(lin["mov_pos"][t, m] - ref["mov_pos"][t][m]).max() < 1e-9, (t, m)
    assert np.abs(lin["mov_pos"] - gen["mov_pos"]).max() < 1e-9
    assert torch.allclose(env.get_attr("mov_counter"), env_gen.get_attr("mov_counter"), atol=1e-9)


def test_staged_and_global_capsule_tables_give_identical_results():
    """CTAs whose 32 envs share a path search a shared-memory copy of its capsule tables (bulk async
    copy); CTAs with mixed paths -- and paths longer than AUV_PATH_STAGE_BLOCKS blocks -- search the
    global tables.  Same arithmetic: bit-identical results, whatever the env order."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    n = 256
    scn = S.moving_obstacles(n, 4, 4, seed=8, n_paths=4)  # path-major: 64 consecutive envs per path
    assert (np.diff(scn.path_id) >= 0).all() and len(set(scn.path_id[:64])) == 1
    perm = np.random.RandomState(0).permutation(n)  # mixed: every CTA sees several paths
    mixed = dataclasses.replace(
        scn, path_id=scn.path_id[perm], vessel_init=scn.vessel_init[perm], mov_start=scn.mov_start[perm],
        mov_width=scn.mov_width[perm], mov_track=scn.mov_track[perm], st_pos=scn.st_pos[perm],
        st_radius=scn.st_radius[perm], path_group=0, path_period=0, _bank=scn.bank, _world=None)
    e1 = AUVVecEnv(scn, n, cfg, test_mode=True, auto_reset=False, debug=True)
    e2 = AUVVecEnv(mixed, n, cfg, test_mode=True, auto_reset=False, debug=True)
    o1, o2 = e1.reset().clone(), e2.reset().clone()
    tp = torch.as_tensor(perm, device="cuda")
    assert torch.equal(o1[tp], o2)
    acts = torch.as_tensor(random_actions(40, n, 2), dtype=torch.float32, device="cuda")
    for t in range(40):
        a1, r1, d1, _ = e1.step(acts[t])
        a2, r2, d2, _ = e2.step(acts[t][tp])
        assert torch.equal(a1[tp], a2) and torch.equal(r1[tp], r2) and torch.equal(d1[tp], d2), t
        assert torch.equal(e1.get_attr("nav")[tp][:, :8], e2.get_attr("nav")[:, :8])
        assert torch.equal(e1.get_attr("lidar_dist")[tp], e2.get_attr("lidar_dist"))


def test_long_path_takes_the_global_tables_and_matches_the_oracle():
    """A 2.4 km path has more than 512 projection blocks: no staging, windows of 32 superblocks."""
    cfg = lidar_config()
    wp = np.array([[0.0, 900.0, 1500.0, 2300.0], [0.0, 300.0, -200.0, 100.0]])
    one = S._single(wp, vessel_init=np.array([20.0, -15.0, 0.4]), static=[((120.0, 60.0), 25.0), ((400.0, 130.0), 40.0)])
    assert one.bank.tables[0].blk_dev.shape[0] > 512
    acts = random_actions(80, 1, 4)
    acts[:, :, 0] = np.abs(acts[:, :, 0])
    ref = rollout_oracle(one, cfg, acts)
    gpu, _ = rollout_gpu(one, cfg, acts)
    rep = compare(ref, gpu, cfg, "long path")
    assert rep["arclength_max_abs"] <= 1e-7


def _velocity_rollouts(scn, cfg, acts):
    """Oracle and GPU rollouts in velocity_mode='nearest'.  Per env-step and ray the oracle also records
    whether the ray is decisive: a clear ray with no intersection within the band past sensor_range, or a hit whose runner-up on another obstacle and whose distance
    to sensor_range are both more than twice the range tolerance away, so that FP32 casting cannot report
    another obstacle's velocity.  close[t, m, i]: the ray's two nearest obstacles are both moving, within 15 m."""
    from oracle.sim import cast_ray_runner_up, rays_for_obstacles
    from tests._parity import RANGE_ATOL, RANGE_RTOL

    T, M = acts.shape[:2]
    R = cfg.vessel.n_sensors
    rng = cfg.vessel.sensor_range
    decisive = np.ones((T, M, R), bool)
    close = np.zeros((T, M, R), bool)

    def on_step(t, m, env):
        v = env.vessel
        if not v.nearby:
            return
        p0 = (float(v.state[0]), float(v.state[1]))
        per_ray, _ = rays_for_obstacles(v.nearby, p0, v.heading, v.d_angle, v.n_sensors)
        for i, ang in enumerate(v.sensor_angles + v.heading):
            d, who, other, who2 = cast_ray_runner_up(ang, p0, rng, per_ray[i])
            assert d == v.dists[i]
            band = 2 * (RANGE_ATOL + RANGE_RTOL * d)
            if who is None:  # clear: decisive unless an obstacle is hit just past sensor_range, inside the band
                d_ext = cast_ray_runner_up(ang, p0, rng + 1.0, per_ray[i])[0]
                decisive[t, m, i] = d_ext - rng > band
            else:
                decisive[t, m, i] = other - d > band and rng - d > band
            close[t, m, i] = who2 is not None and not who.static and not who2.static and other - d < 15.0

    ref = rollout_oracle(scn, cfg, acts, on_step=on_step, velocity_mode="nearest")
    gpu, _ = rollout_gpu(scn, cfg, acts, velocity_mode="nearest")
    return ref, gpu, decisive, close


def _check_velocity_channel(ref, gpu, decisive, cfg, label):
    """Velocity components of decisive rays to 1e-5, rewards of decisive env-steps (every ray decisive, collision
    margin above COLLISION_BAND) to the reward tolerance; returns the counts of what is not decisive."""
    from tests._parity import COLLISION_BAND, REWARD_ATOL, REWARD_RTOL

    R = cfg.vessel.n_sensors
    alive = ref["alive"]
    T, M = alive.shape
    assert gpu["obs"].shape[-1] == 6 + 3 * R
    v_ref = ref["obs"][..., 6 + R:].reshape(T, M, 2, R)
    v_gpu = gpu["obs"][..., 6 + R:].reshape(T, M, 2, R)
    err = np.abs(v_gpu - v_ref).max(axis=2)  # [T, M, R]
    rays = alive[..., None] & decisive
    assert err[rays].max() <= 1e-5, (label, "velocity", float(err[rays].max()), np.argwhere(rays & (err > 1e-5))[:5])
    steps = alive & decisive.all(-1) & (np.abs(ref["min_dist"] - cfg.vessel.vessel_width) > COLLISION_BAND)
    rr, rg = ref["reward"][steps], gpu["reward"][steps]
    assert np.all(np.abs(rg - rr) <= REWARD_ATOL + REWARD_RTOL * np.abs(rr)), (label, "reward", float(np.abs(rg - rr).max()))
    rep = dict(label=label, rays=int(alive.sum()) * R, nondecisive_rays=int((alive[..., None] & ~decisive).sum()),
               env_steps=int(alive.sum()), nondecisive_env_steps=int((alive & ~steps).sum()),
               velocity_max_err_decisive=float(err[rays].max()))
    print(rep)
    return rep


def test_velocity_channel_matches_brute_force_sensor_semantics():
    """velocity_mode='nearest': per ray Rz(-angle - pi/2)(dx, dy) of the nearest obstacle hit
    (sensor.py:118-128), (0, 0) for static obstacles and clear rays; max(0, v_y) enters the Colav
    penalty (rewarder.py:199-206); with sensor_use_velocity_observations the 2 R channels follow
    the closeness block as [v_x(0..R-1), v_y(0..R-1)] (environment.py:264-274).  A ray whose two nearest
    obstacles are closer together than the FP32 casting error may legitimately report the other one: the
    oracle's own margin tells these rays apart; they are counted and bounded, every other ray is compared."""
    cfg = lidar_config()
    cfg.vessel.sensor_use_velocity_observations = True
    scn = S.moving_obstacles(10, 14, 6, seed=33)
    # crowd the start areas so that many rays hit moving obstacles
    rs = np.random.RandomState(1)
    for m in range(10):
        for j in range(14):
            ang, dist = rs.uniform(0, 2 * np.pi), rs.uniform(25, 120)
            scn.mov_start[m, j] = scn.vessel_init[m, :2] + dist * np.array([np.cos(ang), np.sin(ang)])
    acts = random_actions(40, 10, 9)
    ref, gpu, decisive, _ = _velocity_rollouts(scn, cfg, acts)
    R = cfg.vessel.n_sensors
    alive = ref["alive"]
    assert np.abs(ref["obs"][..., 6 + R:][alive]).max() > 0.5, "the scenario should exercise the channel"
    rep = _check_velocity_channel(ref, gpu, decisive, cfg, "spread")
    assert rep["nondecisive_rays"] <= 2e-3 * rep["rays"] and rep["nondecisive_env_steps"] <= 0.1 * rep["env_steps"], rep
    gpu0, _ = rollout_gpu(scn, cfg, acts)  # HEAD behaviour stays the default
    assert np.abs(gpu0["obs"][..., 6 + R:]).max() == 0.0
    assert np.abs(gpu["dists"] - ref["dists"])[alive].max() <= 1e-4 + 1e-4 * 150
    assert (np.abs(gpu0["reward"] - gpu["reward"])[alive] > 1e-3).any(), "approaching obstacles must raise the penalty"


def test_velocity_channel_picks_the_nearer_of_two_close_moving_obstacles():
    """Moving obstacles in pairs on one bearing, the second 8-14 m behind the first: many rays see two moving
    obstacles at decisively different but close distances, and must report the nearer one's velocity."""
    cfg = lidar_config()
    cfg.vessel.sensor_use_velocity_observations = True
    scn = S.moving_obstacles(8, 16, 2, seed=34)
    rs = np.random.RandomState(2)
    for m in range(8):
        for j in range(0, 16, 2):
            ang, dist = rs.uniform(0, 2 * np.pi), rs.uniform(20, 100)
            u = np.array([np.cos(ang), np.sin(ang)])
            scn.mov_start[m, j] = scn.vessel_init[m, :2] + dist * u
            scn.mov_start[m, j + 1] = scn.vessel_init[m, :2] + (dist + rs.uniform(8, 14)) * u
    acts = random_actions(30, 8, 10)
    ref, gpu, decisive, close = _velocity_rollouts(scn, cfg, acts)
    rep = _check_velocity_channel(ref, gpu, decisive, cfg, "pairs")
    rays = ref["alive"][..., None] & decisive & close
    rep["close_pair_rays_compared"] = int(rays.sum())
    print(rep)
    assert rep["close_pair_rays_compared"] >= 200, rep
    assert rep["nondecisive_rays"] <= 5e-3 * rep["rays"] and rep["nondecisive_env_steps"] <= 0.2 * rep["env_steps"], rep


def test_steady_state_sample_matches_oracle_config3_shape():
    """The regime bench.py measures: a large batch stepped >= 1000 steps with auto-reset and fresh
    GPU-generated scenarios (ping-pong pool), then the full live state of a sample of envs is
    injected into the oracle and the next 50 steps are compared step by step -- including the
    25-step nearby refresh of every sampled env and at least one auto-reset onto a generated scenario."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    N = 16384
    scn = S.moving_obstacles_template(2 * N, 16, 16, seed=2, n_paths=256, path_period=N)
    env = AUVVecEnv(scn, N, cfg, test_mode=False, auto_reset=True, debug=True)
    env.regenerate_scenarios(seed=5, epoch=1)
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    lo, hi = torch.tensor([-1.0, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    acts = [lo + (hi - lo) * torch.rand((N, 2), device="cuda", generator=gen) for _ in range(16)]
    for t in range(1000):
        env.step(acts[t % 16])
        if t % 10 == 9:
            env.refresh_finished(seed=5)
    rep = live_sample_compare(env, cfg, acts, horizon=50, n_sample=40, start=1000)
    assert rep["resets"] >= 1 and rep["refreshes"] >= 40 and rep["with_records"] >= 10, rep


def test_ring_group_sample_replays_through_auto_resets():
    """A group of an env ring (``groups(4)``: 1024 of 4096 envs, env_offset 3072) strides by the whole ring on
    auto-reset: a finished env moves on to pool scenario (m + 4096) mod M, not (m + 1024).  Its live envs replay
    through the oracle across such resets."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    N = 4096
    scn = S.moving_obstacles_template(2 * N, 16, 16, seed=4, n_paths=64, path_period=N)
    base = AUVVecEnv(scn, N, cfg, test_mode=False, auto_reset=True, debug=True)
    base.regenerate_scenarios(seed=6, epoch=1)
    g = base.groups(4, debug=True)[3]
    assert g.reset_stride == N and g.env_offset == 3 * N // 4 and g.num_envs == N // 4
    g.reset()
    gen = torch.Generator(device="cuda").manual_seed(4)
    lo, hi = torch.tensor([-1.0, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    acts = [lo + (hi - lo) * torch.rand((N // 4, 2), device="cuda", generator=gen) for _ in range(16)]
    for t in range(1100):  # past the first collisions and reward cut-offs
        g.step(acts[t % 16])
    rep = live_sample_compare(g, cfg, acts, horizon=60, n_sample=30, start=1100)
    print(rep)
    assert rep["resets"] >= 2, rep


def test_steady_state_sample_matches_oracle_land_polygons():
    """BASELINE config 4 shape: 131072 envs in one shared world of 512 land polygons; after 300
    steps a sample of live envs (most of them with polygons in range) is replayed by the oracle."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    N = 131072
    scn = S.land_scenarios(N, n_polygons=512, n_moving=0, n_static=0, seed=4, n_paths=512, extent=3000.0)
    env = AUVVecEnv(scn, N, cfg, test_mode=False, auto_reset=True, debug=True)
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(8)
    lo, hi = torch.tensor([0.2, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    acts = [lo + (hi - lo) * torch.rand((N, 2), device="cuda", generator=gen) for _ in range(8)]
    for t in range(300):
        env.step(acts[t % 8])
    rep = live_sample_compare(env, cfg, acts, horizon=30, n_sample=32, start=300, prefer_records=True)
    assert rep["with_records"] >= 20, rep


def test_compact_host_step_is_bit_identical_to_the_dense_copy():
    """step_host / step_async ship head + hit mask + packed non-zero closeness values straight into
    pinned host memory (k_obs_ship) and expand them on the host (auv_compact_expand): the dense array
    they return equals the device observation and the dense D2H copy bit for bit -- through
    auto-resets (the cached first observation replaces the row)."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    cfg.episode.max_timesteps = 9  # time-limit resets inside the rollout
    n = 300  # not a multiple of the 32-env CTAs
    scn = S.moving_obstacles(n, 6, 6, seed=13, n_paths=5)
    rs = np.random.RandomState(3)
    for m in range(0, n, 2):  # crowd every other start area: many hit rays there, none elsewhere
        for j in range(6):
            ang, dist = rs.uniform(0, 2 * np.pi), rs.uniform(20, 100)
            scn.st_pos[m, j] = scn.vessel_init[m, :2] + dist * np.array([np.cos(ang), np.sin(ang)])
    dev = AUVVecEnv(scn, n, cfg, auto_reset=True)
    cmp_ = AUVVecEnv(scn, n, cfg, auto_reset=True, host_chunks=3, host_threads=3, host_transfer="compact")
    dense = AUVVecEnv(scn, n, cfg, auto_reset=True, host_chunks=2, compact_host=False)
    assert cmp_.compact_host and not dense.compact_host and dense.host_transfer == "dense"
    assert AUVVecEnv(scn, n, cfg).host_transfer == "delta"
    for e in (dev, cmp_, dense):
        e.reset()
    acts = random_actions(30, n, 6).astype(np.float32)
    resets = 0
    for t in range(30):
        o1, r1, d1, _ = dev.step(torch.as_tensor(acts[t], device="cuda"))
        if t % 2:
            cmp_.step_async(acts[t])
            o2, r2, d2 = cmp_.step_wait()
        else:
            o2, r2, d2 = cmp_.step_host(acts[t])
        o3, r3, d3 = dense.step_host(acts[t])
        torch.cuda.synchronize()
        a = o1.cpu().numpy()
        assert np.array_equal(a, o2) and np.array_equal(a, o3), t
        assert np.array_equal(r1.cpu().numpy(), r2) and np.array_equal(r2, r3)
        assert np.array_equal(d1.cpu().numpy(), d2) and np.array_equal(d2, d3)
        resets += int(d2.sum())
        assert cmp_.d2h_bytes_per_step < dense.d2h_bytes_per_step
    assert resets > n, "every env should have been auto-reset at least once"
    assert (o2[:, 6:] != 0).any() and (o2[:, 6:] == 0).mean() > 0.5


@pytest.mark.parametrize("gran,velocity", [(8, False), (16, False), (32, False), (16, True)])
def test_delta_host_step_is_bit_identical_to_the_dense_copy(gran, velocity):
    """host_transfer="delta": the dense observation array lives in pinned host memory and the device
    stores only the chunks that changed since the previous step (k_obs_delta against its shadow copy).
    The host array equals the device observation bit for bit at every step -- through auto-resets,
    with an env count that leaves a partial quad at the end, and with the (3, R) velocity layout
    the compact form does not cover -- while fewer bytes cross the link than the dense copy moves."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    cfg.episode.max_timesteps = 9
    kw = {}
    if velocity:
        cfg.vessel.sensor_use_velocity_observations = True
        kw["velocity_mode"] = "nearest"
    n = 301  # n * obs_dim = 301 * 186 is not a multiple of 4: the last quad is partial
    scn = S.moving_obstacles(n, 6, 6, seed=13, n_paths=5)
    rs = np.random.RandomState(3)
    for m in range(0, n, 2):
        for j in range(6):
            ang, dist = rs.uniform(0, 2 * np.pi), rs.uniform(20, 100)
            scn.st_pos[m, j] = scn.vessel_init[m, :2] + dist * np.array([np.cos(ang), np.sin(ang)])
    dev = AUVVecEnv(scn, n, cfg, auto_reset=True, **kw)
    dlt = AUVVecEnv(scn, n, cfg, auto_reset=True, host_chunks=2, host_transfer="delta", delta_gran=gran, **kw)
    assert dlt.host_transfer == "delta" and not dlt.compact_host
    dev.reset()
    dlt.reset()
    acts = random_actions(30, n, 6).astype(np.float32)
    resets = 0
    dense_bytes = n * (dev.obs_dim * 4 + 5)
    for t in range(30):
        o1, r1, d1, _ = dev.step(torch.as_tensor(acts[t], device="cuda"))
        if t % 2:
            dlt.step_async(acts[t])
            o2, r2, d2 = dlt.step_wait()
        else:
            o2, r2, d2 = dlt.step_host(acts[t])
        torch.cuda.synchronize()
        assert np.array_equal(o1.cpu().numpy().view(np.uint32), o2.view(np.uint32)), t
        assert np.array_equal(r1.cpu().numpy(), r2) and np.array_equal(d1.cpu().numpy(), d2)
        resets += int(d2.sum())
        if t % 5 == 4:
            assert 0 < dlt.d2h_bytes_per_step < dense_bytes
    assert resets > n
    assert (o2[:, 6:] != 0).any() and (o2[:, 6:] == 0).mean() > 0.5


def test_env_group_ring_out_of_order_equals_the_whole_env():
    """EnvGroupRing (send / recv): three groups of n envs stepped in whatever order their steps finish
    give, step for step, the rows the whole 3n-env batch gives -- through auto-resets, delta transfer."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    cfg.episode.max_timesteps = 7
    n, G, T = 70, 3, 16
    scn = S.moving_obstacles(G * n, 5, 5, seed=41, n_paths=4)
    ref = AUVVecEnv(scn, G * n, cfg, auto_reset=True)
    ring = ref.ring(G)
    assert len(ring) == G and ring.envs_per_group == n and ring.groups[0].host_transfer == "delta"
    ref.reset()
    ring.reset()
    acts = random_actions(T, G * n, 8).astype(np.float32)
    want = []
    for t in range(T):
        o, r, d, _ = ref.step(torch.as_tensor(acts[t], device="cuda"))
        want.append((o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy()))
    with pytest.raises(RuntimeError):
        ring.recv()
    count = [0] * G
    for g in (2, 0, 1):
        ring.send(g, acts[0, g * n:(g + 1) * n])
    order = []
    while ring.pending:
        g, o, r, d = ring.recv()
        t = count[g]
        order.append(g)
        sl = slice(g * n, (g + 1) * n)
        assert np.array_equal(o, want[t][0][sl]) and np.array_equal(r, want[t][1][sl]) and np.array_equal(d, want[t][2][sl]), (g, t)
        count[g] += 1
        if count[g] < T:
            ring.send(g, acts[count[g], sl])
    assert count == [T] * G and sum(int(w[2].sum()) for w in want) > G * n
    ring.close()


def test_facade_keeps_one_vec_env_alive_across_episodes():
    """AUVEnv.reset(): a random family generates the scenarios of the next `block_size` episodes at once
    and walks through them with reset_envs on ONE AUVVecEnv (device tables, path bank, reset cache built
    once per block); deterministic scenarios replay their single scenario.  Every episode equals what a
    freshly built 1-env AUVVecEnv gives on that scenario of the block."""
    import gym_auv_b200
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    env = gym_auv_b200.make("MovingObstaclesNoRules-v0", cfg)
    env.block_size = 3
    env._vec = None  # drop the block the constructor generated with the default size
    env.vec_env_builds = 0
    acts = random_actions(6, 1, 9).astype(np.float32)
    firsts = []
    for ep in range(5):  # 3 episodes on the first block, 2 on the second
        o = env.reset()
        if ep % 3 == 0:
            block = env.scenario
            assert block.n_scenarios == 3
        assert env.scenario is block
        fresh = AUVVecEnv(block, 1, cfg, auto_reset=False, env_offset=ep % 3)  # env 0 sits on scenario ep % 3
        o_f = fresh.reset()[0].cpu().numpy().astype(np.float64)
        assert np.array_equal(o, o_f), ep
        for t in range(6):
            o, r, d, info = env.step(acts[t, 0])
            of, rf, df, _ = fresh.step(torch.as_tensor(acts[t], device="cuda"))
            assert np.array_equal(o, of[0].cpu().numpy().astype(np.float64)) and r == float(rf.item()), (ep, t)
        assert env.t_step == 6
        firsts.append(o)
        assert len(env.obstacles) > 0 and env.path.length > 100
    assert env.vec_env_builds == 2 and len(env.history) == 4 and env.episode == 6
    assert not np.array_equal(firsts[0], firsts[1])
    fixed = gym_auv_b200.make("TestScenario3-v0", cfg)
    for _ in range(3):
        fixed.reset()
        fixed.step([0.5, 0.1])
    assert fixed.vec_env_builds == 1


def test_vecenv_adapter_history_and_report(tmp_path):
    """B200VecEnv: the SubprocVecEnv surface scripts/run.py:278-475 drives (NumPy in / out, per-env
    info list with terminal_observation, get_attr('history')) with a fresh GPU-generated scenario per
    episode; its history entries add up to the device-side episode statistics, and write_report
    produces the report.txt of reporting.py:37-79."""
    from gym_auv_b200.adapters import B200VecEnv, write_report

    cfg = lidar_config()
    cfg.episode.max_timesteps = 7
    n = 96
    scn = S.moving_obstacles_template(2 * n, 5, 4, seed=1, n_paths=3, path_period=n)
    venv = B200VecEnv(scn, n, cfg, fresh_scenarios=True, refresh_every=3, seed=9)
    obs = venv.reset()
    assert obs.shape == (n, 186) and venv.observation_space.shape == (186,)
    rs = np.random.RandomState(0)
    first_pool = venv.impl.pull_scenarios()
    n_done = 0
    for t in range(25):
        a = rs.uniform([-1, -0.15], [1, 0.15], size=(n, 2)).astype(np.float32)
        obs, rew, done, infos = venv.step(a)
        assert obs.shape == (n, 186) and rew.shape == (n,) and done.dtype == bool and len(infos) == n
        i0 = infos[0]
        assert set(i0) >= {"collision", "reached_goal", "goal_distance", "progress"}
        for i in np.nonzero(done)[0][:3]:
            term = infos[int(i)]["terminal_observation"]
            assert term.shape == (186,) and not np.array_equal(term, obs[i])
        n_done += int(done.sum())
    assert n_done >= 3 * n
    hist = venv.get_attr("history")[0]
    assert len(hist) == n_done
    st = venv.episode_stats(reduce=False)
    assert st["episodes"] == n_done
    assert abs(np.mean([h["reward"] for h in hist]) - st["reward"]) <= 1e-3 * abs(st["reward"])
    assert abs(np.mean([h["timesteps"] for h in hist]) - st["timesteps"]) <= 1e-6
    assert all(h["timesteps"] <= 7 for h in hist)
    path = write_report(hist, str(tmp_path), lastn=50)
    text = open(path).read().splitlines()
    assert text[0] == "# PERFORMANCE METRICS (LAST 50 EPISODES AVG.)"
    assert text[1].split() == ["Episodes", "50"]
    assert [l.split()[0] for l in text[2:4]] == ["Avg.", "Std."] and len(text) == 12
    # fresh scenarios: the pool slots of finished envs were regenerated
    later_pool = venv.impl.pull_scenarios()
    assert (later_pool.st_pos != first_pool.st_pos).any()
    venv.close()


def test_dict_observation_views_on_the_batched_env():
    """use_dict_observation (environment.py:116-137,281-288): 'proprioceptive' [N, 6] and the LiDAR
    image 'lidar' [N, C, R] are zero-copy views of the flat observation; with velocity observations C = 3
    and channels 1-2 carry (v_x, v_y)."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    cfg.vessel.use_dict_observation = True
    cfg.vessel.sensor_use_velocity_observations = True
    scn = S.moving_obstacles(16, 10, 4, seed=4)
    rs = np.random.RandomState(1)
    for m in range(16):
        for j in range(10):
            ang, dist = rs.uniform(0, 2 * np.pi), rs.uniform(25, 110)
            scn.mov_start[m, j] = scn.vessel_init[m, :2] + dist * np.array([np.cos(ang), np.sin(ang)])
    env = AUVVecEnv(scn, 16, cfg, test_mode=True, auto_reset=False, velocity_mode="nearest")
    flat = AUVVecEnv(scn, 16, lidar_config(sensor_use_velocity_observations=True), test_mode=True, auto_reset=False,
                     velocity_mode="nearest")
    o = env.reset()
    f = flat.reset()
    assert set(o) == {"proprioceptive", "lidar"} and o["lidar"].shape == (16, 3, 180)
    assert env.observation_space["lidar"].shape == (3, 180) and env.observation_space["proprioceptive"].shape == (6,)
    a = torch.as_tensor(random_actions(10, 16, 3), dtype=torch.float32, device="cuda")
    for t in range(10):
        o, r, d, _ = env.step(a[t])
        f, rf, df, _ = flat.step(a[t])
        assert torch.equal(o["proprioceptive"], f[:, :6]) and torch.equal(o["lidar"].reshape(16, -1), f[:, 6:])
        assert o["lidar"].data_ptr() == env._out["obs"].data_ptr() + 24  # a view, not a copy
    assert (o["lidar"][:, 1:] != 0).any()


def test_device_path_builder_matches_scipy_tables():
    """auv_pathbank_build (Path.__init__, path.py:19-40, on the GPU) against the host builder
    (SciPy PCHIP): knots and PPoly coefficients to the last bits, the 0.1 m polyline and its
    chord-length prefix sums, the header, and capsules that do contain their part of the polyline."""
    from gym_auv_b200.pathbank import DevicePathBank, PATH_BLOCK, PATH_SUPER, build_path, random_curve_waypoints, HDR_DTYPE

    rng = np.random.RandomState(5)
    wps = [random_curve_waypoints(rng, int(np.floor(4 * rng.rand() + 2)), 800.0) for _ in range(10)]
    wps += [np.array([[0.0, 1100.0], [0.0, 1100.0]]), np.array([[25.0, 25.0], [10.0, 200.0]]),
            np.array([[0.0, 300.0, 300.0, 900.0], [0.0, 0.0, 400.0, 400.0]])]
    bank = DevicePathBank(wps)
    arr = bank.device_arrays("cuda:0")
    torch.cuda.synchronize()
    hdr = arr["hdr"].cpu().numpy().view(HDR_DTYPE)
    V = bank.vcap
    for p, wp in enumerate(wps):
        ref = build_path(wp)
        h = hdr[p]
        n = len(ref.poly)
        assert h["nseg"] == n - 1 and h["v0"] == p * V
        assert abs(h["length"] - ref.length) <= 1e-12 * ref.length
        assert abs(h["end_x"] - ref.end[0]) <= 1e-9 and abs(h["end_y"] - ref.end[1]) <= 1e-9
        pp = arr["pp"][p].cpu().numpy()
        assert np.abs(pp[:, 0] - ref.knots[:-1]).max() <= 1e-12 * ref.length
        assert np.abs(pp[:, 1] - ref.knots[1:]).max() <= 1e-12 * ref.length
        scale = np.abs(ref.coef).max(axis=(0, 2))
        assert np.abs(pp[:, 2:6] - ref.coef[:, 0, :]).max() <= 1e-9 * max(1.0, scale[0])
        assert np.abs(pp[:, 6:10] - ref.coef[:, 1, :]).max() <= 1e-9 * max(1.0, scale[1])
        poly = arr["poly_xy"][p * V:p * V + n].cpu().numpy()
        assert np.abs(poly - ref.poly).max() <= 1e-10
        assert np.abs(arr["poly_cum"][p * V:p * V + n].cpu().numpy() - ref.cum).max() <= 1e-9
        pf = arr["poly_f32"][p * V:p * V + n].cpu().numpy()
        assert np.abs(pf - (ref.poly - ref.origin)).max() <= 1e-4
        # capsules: every covered vertex lies within `dev` of the (rounded) chord
        rel = ref.poly - np.array([h["ox"], h["oy"]])
        for span, ck, dk, off in ((PATH_BLOCK, "blk_chord", "blk_dev", h["b0"]), (PATH_BLOCK * PATH_SUPER, "sb_chord", "sb_dev", h["s0"])):
            nn = (n - 1 + span - 1) // span
            ch = arr[ck][off:off + nn].cpu().numpy().astype(np.float64)
            ax = arr[dk][off:off + nn].cpu().numpy().astype(np.float64)
            for b in range(nn):
                v = rel[b * span:min((b + 1) * span, n - 1) + 1]
                w = v - ch[b, :2]
                t = np.clip((w @ ch[b, 2:]) * ax[b, 0], 0, 1)
                d = np.linalg.norm(w - t[:, None] * ch[b, 2:], axis=1).max()
                assert d <= ax[b, 1], (p, span, b, d, ax[b, 1])
                assert ax[b, 1] <= d + 1e-2  # ... and is not uselessly loose


def test_device_built_bank_steps_like_the_host_built_bank():
    """Same scenarios on a SciPy-built and on a GPU-built path bank: the step agrees to the rounding
    of the tables (positions 1e-9, arclength 1e-7), done / collision flags identical."""
    from gym_auv_b200.pathbank import DevicePathBank
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    scn = S.moving_obstacles(64, 6, 6, seed=31, n_paths=4)
    dscn = dataclasses.replace(scn, _bank=DevicePathBank(scn.waypoints), _world=None)
    e1 = AUVVecEnv(scn, 64, cfg, test_mode=True, auto_reset=False, debug=True)
    e2 = AUVVecEnv(dscn, 64, cfg, test_mode=True, auto_reset=False, debug=True)
    o1, o2 = e1.reset(), e2.reset()
    assert torch.allclose(o1, o2, atol=1e-6)
    a = torch.as_tensor(random_actions(50, 64, 8), dtype=torch.float32, device="cuda")
    for t in range(50):
        o1, r1, d1, i1 = e1.step(a[t])
        o2, r2, d2, i2 = e2.step(a[t])
        assert torch.allclose(o1, o2, atol=1e-6) and torch.allclose(r1, r2, atol=1e-4, rtol=1e-6)
        assert torch.equal(d1, d2) and torch.equal(i1["collision"], i2["collision"])
        assert (e1.get_attr("nav")[:, 0] - e2.get_attr("nav")[:, 0]).abs().max() <= 1e-7
        assert torch.allclose(e1.get_attr("lidar_dist"), e2.get_attr("lidar_dist"), atol=1e-5)


def test_fresh_random_paths_on_the_device_replay_through_the_oracle():
    """regenerate_paths + regenerate_scenarios: a complete MovingObstacles._generate (random curve,
    vessel start, obstacles -- movingobstacles.py:28-95) on the GPU.  The generated curves have the
    shape of RandomCurveThroughOrigin (ends on the circle of radius 400, through the origin), and the
    generated scenarios -- pulled back with their waypoints -- replay through the oracle."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    n = 24
    scn = S.moving_obstacles_template(n, 6, 5, seed=3, n_paths=n, device_paths=True)
    env = AUVVecEnv(scn, n, cfg, test_mode=True, auto_reset=False, debug=True)
    before = [w.copy() for w in scn.bank.waypoints]
    env.regenerate_paths(seed=77, epoch=2)
    env.regenerate_scenarios(seed=77, epoch=2)
    after = scn.bank.waypoints
    assert all(a.shape[1] in (5, 7) for a in after) and any(not np.array_equal(a, b) for a, b in zip(after, before))
    for w in after:
        assert abs(np.hypot(*w[:, 0]) - 400.0) < 1e-9 and np.allclose(w[:, -1], -w[:, 0])
        assert np.abs(w[:, w.shape[1] // 2]).max() == 0.0  # through the origin
        assert np.allclose(w[0, 1:-1] - w[1, 1:-1], (w[0, 1:-1] - w[1, 1:-1]))  # (jitter is one scalar per point)
    host = env.pull_scenarios()
    acts = random_actions(30, n, 12)
    ref = rollout_oracle(host, cfg, acts)
    env.reset()
    a = torch.as_tensor(acts, dtype=torch.float32, device="cuda")
    for t in range(30):
        obs, rew, done, info = env.step(a[t])
        alive = ref["alive"][t]
        o = obs.cpu().numpy()
        assert np.abs(o - ref["obs"][t])[alive].max() <= 1e-4, t
        assert np.abs(rew.cpu().numpy() - ref["reward"][t])[alive].max() <= 1e-3


def test_debug_bounds_build_raises_no_index_violation(tmp_path):
    """compute-sanitizer is not available on every pool, so the kernels carry their own index checks
    (-DAUV_DEBUG_BOUNDS: record / ray / vertex-stage / segment / block indices; a violation raises
    AUV_STATUS_BOUNDS).  The debug library is built here and a crowded rollout -- dense records, several
    shared-memory rounds, land polygons, auto-reset, host step -- is run through it in a subprocess."""
    import subprocess
    import sys

    from gym_auv_b200 import build as B

    lib = str(tmp_path / "libauv_b200_dbg.so")
    cmd = [os.environ.get("NVCC", "nvcc")] + B.NVCC_FLAGS + ["-DAUV_DEBUG_BOUNDS", "-o", lib, B.SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    prog = r"""
import numpy as np, torch
from gym_auv_b200 import lidar_config, scenarios as S
from gym_auv_b200.vec_env import AUVVecEnv
cfg = lidar_config(); cfg.episode.max_timesteps = 12
n = 200
scn = S.land_scenarios(n, n_polygons=40, n_moving=12, n_static=12, seed=2, n_paths=6, extent=900.0)
rs = np.random.RandomState(0)
for m in range(n):
    for j in range(12):
        a, d = rs.uniform(0, 2 * np.pi), rs.uniform(10, 140)
        scn.st_pos[m, j] = scn.vessel_init[m, :2] + d * np.array([np.cos(a), np.sin(a)])
env = AUVVecEnv(scn, n, cfg, auto_reset=True, debug=True, sector_outputs=True, host_chunks=2)
env.reset()
for t in range(40):
    a = rs.uniform([-1, -0.15], [1, 0.15], size=(n, 2)).astype(np.float32)
    if t % 2: env.step(torch.as_tensor(a, device="cuda"))
    else: env.step_host(a)
env.check_status()
assert float(env._scratch["rec_cnt"].float().mean()) > 3
# projection edge cases: the medial line of a hairpin and the centre of a long arc (global tables), cold and warm
from gym_auv_b200.pathbank import build_path
from tests.test_projection_edges import FAMILIES, PATHS, _scenarios
for fam in ("hairpin", "circle_centre_long"):
    key, gen = FAMILIES[fam]
    pts = gen(build_path(PATHS[key]))
    pe = AUVVecEnv(_scenarios(key, "host"), len(pts), cfg, test_mode=True, auto_reset=False, debug=True)
    pe.reset()
    nseg = len(pe.scenarios.bank.tables[0].poly) - 1
    for warm in (-1, 0, -2):
        pe.state.zero_()
        pe.state[0] = torch.as_tensor(pts[:, 0], device="cuda")
        pe.state[1] = torch.as_tensor(pts[:, 1], device="cuda")
        if warm == -2:  # half the path away from the previous answer
            pe._st["prev_seg"].copy_((pe._st["prev_seg"] + nseg // 2) % nseg)
        else:
            pe._st["prev_seg"].fill_(warm)
        pe.step(torch.zeros((len(pts), 2), device="cuda"))
    pe.check_status()
    print(fam, "ok", int(pe._scratch["status"].item()))
print("bounds ok", int(env._scratch["status"].item()))
"""
    env = dict(os.environ, AUV_B200_LIB=lib)
    out = subprocess.run([sys.executable, "-c", prog], capture_output=True, text=True, env=env,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert out.returncode == 0 and "bounds ok 0" in out.stdout, out.stdout[-1500:] + out.stderr[-3000:]


def test_world_grid_broad_phase_equals_the_full_scan():
    """The nearby-list refresh over a shared world of land polygons through the uniform grid over their
    enclosing circles lists exactly the polygons the full scan lists: bit-identical masks, records,
    observations over a rollout with several refreshes."""
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    n = 512
    scn = S.land_scenarios(n, n_polygons=300, n_moving=3, n_static=3, seed=6, n_paths=8, extent=2500.0)
    e1 = AUVVecEnv(scn, n, cfg, test_mode=True, auto_reset=False, debug=True, world_grid=True)
    e2 = AUVVecEnv(scn, n, cfg, test_mode=True, auto_reset=False, debug=True, world_grid=False)
    assert "world_cell_off" in e1._pool and "world_cell_off" not in e2._pool
    o1, o2 = e1.reset(), e2.reset()
    assert torch.equal(o1, o2) and torch.equal(e1._st["nearby_mask"], e2._st["nearby_mask"])
    assert int(e1._st["nearby_mask"].ne(0).sum()) > 0
    a = torch.as_tensor(random_actions(55, n, 5), dtype=torch.float32, device="cuda")
    a[:, :, 0] = a[:, :, 0].abs()
    for t in range(55):
        o1, r1, d1, _ = e1.step(a[t])
        o2, r2, d2, _ = e2.step(a[t])
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2), t
        assert torch.equal(e1._st["nearby_mask"], e2._st["nearby_mask"]), t
        assert torch.equal(e1._scratch["rec_cnt"], e2._scratch["rec_cnt"])
    e1.check_status(), e2.check_status()


def test_realworld_scenario_matches_the_reference_episode_on_gpu():
    """The reference's RealWorldEnv episode (land perimeters incl. one with 230 vertices -- more than
    one vertex stage --, AIS vessel tracks; tests/golden/make_reference_goldens_realworld.py) through the
    loaders and the CUDA step, in a batch of identical worlds."""
    from gym_auv_b200.vec_env import AUVVecEnv
    from tests.test_realworld import GOLD, build_scenario

    cfg = lidar_config()
    scn, _, _ = build_scenario(n=40)
    env = AUVVecEnv(scn, 40, cfg, test_mode=True, auto_reset=False, debug=True)
    obs0 = env.reset().cpu().numpy()
    assert np.abs(obs0 - GOLD["obs0"][None, :]).max() <= 1e-4
    for t, a in enumerate(GOLD["actions"][: len(GOLD["obs"])]):
        act = torch.as_tensor(np.tile(a, (40, 1)), dtype=torch.float32, device="cuda")
        obs, rew, done, info = env.step(act)
        d = env.get_attr("lidar_dist").cpu().numpy()
        ref = GOLD["dists"][t]
        assert (np.abs(d - ref[None, :]) <= 1e-4 + 1e-4 * ref[None, :]).all(), t
        assert np.abs(obs.cpu().numpy() - GOLD["obs"][t][None, :]).max() <= 1e-4
        assert np.abs(rew.cpu().numpy() - GOLD["reward"][t]).max() <= 1e-4 + 1e-4 * abs(GOLD["reward"][t])
        assert int(env._scratch["rec_cnt"][0]) == int(GOLD["n_nearby"][t])
        assert torch.equal(obs[0], obs[39])  # every env of the batch runs the same world
    env.check_status()


def test_c_abi_alone_builds_and_steps_a_batch():
    """INTEGRATION.md section 3: a host that only has the C ABI (here: ctypes + raw device allocations, no
    AUVVecEnv / PathBank / ScenarioSet) builds the path bank from waypoints, samples the scenario pool,
    fills the reset cache, steps with auto-reset and refreshes finished scenarios -- and gets what
    AUVVecEnv gets for the same pool."""
    import ctypes as C

    from gym_auv_b200 import _lib
    from gym_auv_b200.vec_env import AUVVecEnv, make_auv_config, ray_table

    lib = _lib.load()
    dev = torch.device("cuda:0")
    z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
    P_ = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    N, M, P, Km, Ks, R, V = 96, 192, 6, 5, 4, 180, 16384
    conf = lidar_config()
    conf.episode.max_timesteps = 11
    cfg = make_auv_config(conf, "colav", False, True, "reference")
    od = lib.auv_obs_dim(C.byref(cfg))
    # ---- 1. paths
    wp, nwp, status = z((P, 2, 8), torch.float64), z(P, torch.int32), z(1, torch.int32)
    _lib.check(lib.auv_random_curve_waypoints(7, 1, 800.0, None, P, P_(wp), P_(nwp), st), "waypoints")
    pa = dict(hdr=z(P * 64, torch.uint8), poly_xy=z((P * V, 2), torch.float64), poly_cum=z(P * V, torch.float64),
              poly_f32=z((P * V, 2), torch.float32), blk_chord=z((P * V // 32, 4), torch.float32), blk_dev=z((P * V // 32, 2), torch.float32),
              sb_chord=z((P * V // 512, 4), torch.float32), sb_dev=z((P * V // 512, 2), torch.float32), pp=z((P, 999, 12), torch.float64))
    order = ("hdr", "poly_xy", "poly_cum", "poly_f32", "blk_chord", "blk_dev", "sb_chord", "sb_dev", "pp")
    pb = _lib.AuvPathBuild(*[pa[k].data_ptr() for k in order], 1000, V)
    _lib.check(lib.auv_pathbank_build(P_(wp), P_(nwp), None, P, C.byref(pb), P_(status), st), "auv_pathbank_build")
    paths = _lib.AuvPathBank(P, 1000, *[pa[k].data_ptr() for k in order])
    # ---- 2. scenario pool, sampled on the GPU
    mw = 1
    pl = dict(path_id=z(M, torch.int32), vessel_init=z((M, 3), torch.float64), mov_start=z((M, Km, 2), torch.float64),
              mov_width=z((M, Km), torch.float64), mov_track=z((M, Km, 4), torch.int32), mov_pos0=z((M, Km, 2), torch.float64),
              mov_disp0=z((M, Km, 2), torch.float64), mov_counter0=z((M, Km), torch.float64), vel_table=z((M * Km, 2), torch.float64),
              st_pos=z((M, Ks, 2), torch.float64), st_radius=z((M, Ks), torch.float64), st_rec=z((M, Ks, 4), torch.float64),
              mov_lin=z((M, Km, 8), torch.float64), reset_obs=z((M, od), torch.float32), reset_max_progress=z(M, torch.float64),
              reset_mask=z((M, mw), torch.int32))
    first, period = C.c_int32(0), C.c_int32(0)
    _lib.check(lib.auv_linear_wrap(1.0, 1.1, 9999, C.byref(first), C.byref(period)), "auv_linear_wrap")
    pool = _lib.AuvScenarioPool(
        M, Km, Ks, 0, *[pl[k].data_ptr() for k in ("path_id", "vessel_init", "mov_start", "mov_width", "mov_track", "mov_pos0",
                                                   "mov_disp0", "mov_counter0", "vel_table", "st_pos", "st_radius", "st_rec", "mov_lin")],
        1, first.value, period.value, 0, None, None, None, None, None, 0.0, 0.0, 0.0, 0, 0,
        pl["reset_obs"].data_ptr(), pl["reset_max_progress"].data_ptr(), pl["reset_mask"].data_ptr())
    gp = _lib.AuvGenParams(seed=3, epoch=1, post_generate_update=1, t_step_size=1.0, vessel_width=1.255, init_pos_jitter=50.0,
                           mov_disp_std=500.0, mov_width_mean=10.0, mov_speed_lo=1.0, mov_speed_hi=3.0, st_disp_std=250.0,
                           st_radius_mean=30.0, path_group=N // P, path_period=N)
    _lib.check(lib.auv_generate_moving_obstacles(C.byref(gp), C.byref(paths), C.byref(pool), None, M, P_(status), st), "generate")
    # ---- ray table (host constants) and batches
    _, cos_sin, weight, wsum, sector = ray_table(R, 9)
    k64 = np.arange(64) * (2 * np.pi / 64)
    rt = dict(cos_sin=torch.as_tensor(cos_sin).to(dev), weight=torch.as_tensor(weight).to(dev), sector=torch.as_tensor(sector).to(dev),
              unit64=torch.as_tensor(np.stack([np.cos(k64), np.sin(k64)], 1)).to(dev))
    rays = _lib.AuvRayTable(rt["cos_sin"].data_ptr(), rt["weight"].data_ptr(), rt["sector"].data_ptr(), rt["unit64"].data_ptr(), wsum)

    def make_batch(n):
        b = dict(scn_id=torch.arange(n, device=dev, dtype=torch.int32), episode=z(n, torch.int32), state=z((6, n), torch.float64),
                 step_counter=z(n, torch.int32), t_step=z(n, torch.int32), cum_reward=z(n, torch.float64),
                 max_progress=z(n, torch.float64), cte_sum=z(n, torch.float64), nearby_mask=z((n, mw), torch.int32),
                 nav=z((n, 24), torch.float64), rec=z((n, Km + Ks, 80), torch.uint8), rec_cnt=z(n, torch.int32),
                 obst_steps=z(n, torch.int32), prev_seg=torch.full((n,), -1, dtype=torch.int32, device=dev), env_pid=z(n, torch.int32))
        o = dict(obs=z((n, od), torch.float32), reward=z(n, torch.float32), done=z(n, torch.uint8), stats=z(16, torch.float64))
        batch = _lib.AuvBatch(n, mw, 0, 0, b["scn_id"].data_ptr(), b["episode"].data_ptr(), b["state"].data_ptr(),
                              b["step_counter"].data_ptr(), b["t_step"].data_ptr(), b["cum_reward"].data_ptr(),
                              b["max_progress"].data_ptr(), b["cte_sum"].data_ptr(), b["nearby_mask"].data_ptr(), None, None, None,
                              b["nav"].data_ptr(), b["rec"].data_ptr(), b["rec_cnt"].data_ptr(), status.data_ptr(), Km + Ks, 0,
                              b["obst_steps"].data_ptr(), b["prev_seg"].data_ptr(), b["env_pid"].data_ptr())
        out = _lib.AuvStepOut(o["obs"].data_ptr(), o["reward"].data_ptr(), o["done"].data_ptr(), None, None, None, None, None, None,
                              None, None, None, o["stats"].data_ptr(), None, None)
        return b, o, batch, out

    wb, wo, worker, worker_out = make_batch(64)
    # ---- 3. reset cache, 64 scenarios per call
    for f0 in range(0, M, 64):
        _lib.check(lib.auv_reset_cache_fill(C.byref(cfg), C.byref(rays), C.byref(paths), C.byref(pool), C.byref(worker),
                                            C.byref(worker_out), None, f0, min(64, M - f0), st), "auv_reset_cache_fill")
    # ---- 4. run
    b, o, batch, out = make_batch(N)
    _lib.check(lib.auv_reset(C.byref(cfg), C.byref(pool), C.byref(batch), None, st), "auv_reset")
    _lib.check(lib.auv_observe(C.byref(cfg), C.byref(rays), C.byref(paths), C.byref(pool), C.byref(batch), C.byref(out), 1, st), "observe")
    torch.cuda.synchronize()
    assert torch.equal(o["obs"], pl["reset_obs"][:N])  # the cached first observations are what reset() returns
    rs = _lib.AuvRefreshScratch(z(N, torch.int32).data_ptr(), z(64, torch.int32).data_ptr(), z(1, torch.int32).data_ptr(), 64, 0)
    keep = []  # (the scratch tensors above must outlive the calls)
    seen, ids, cnt = z(N, torch.int32), z(64, torch.int32), z(1, torch.int32)
    rs = _lib.AuvRefreshScratch(seen.data_ptr(), ids.data_ptr(), cnt.data_ptr(), 64, 0)
    acts = torch.as_tensor(random_actions(30, N, 1), dtype=torch.float32, device=dev)
    before = pl["st_pos"].clone()
    n_done = 0
    for t in range(30):
        _lib.check(lib.auv_step(C.byref(cfg), C.byref(rays), C.byref(paths), C.byref(pool), C.byref(batch), P_(acts[t]),
                                C.byref(out), st), "auv_step")
        n_done += int(o["done"].sum())
        assert torch.isfinite(o["obs"]).all() and o["obs"].abs().max() <= 1 and torch.isfinite(o["reward"]).all()
        if t % 4 == 3:
            gp.epoch += 1
            _lib.check(lib.auv_refresh_finished(C.byref(cfg), C.byref(rays), C.byref(paths), C.byref(pool), C.byref(batch),
                                                C.byref(worker), C.byref(worker_out), C.byref(rs), C.byref(gp), st), "refresh")
    torch.cuda.synchronize()
    assert int(status.item()) == 0 and n_done >= 2 * N and float(o["stats"][0]) == n_done
    assert (pl["st_pos"] != before).any(), "vacated slots were regenerated"
    assert (b["scn_id"] >= 0).all() and (b["scn_id"] < M).all()
