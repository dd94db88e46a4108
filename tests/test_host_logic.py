"""Host-side logic that needs no GPU: config tree, scenario plug-ins, path bank tables,
ABI library symbols and struct layout."""
import ctypes
import dataclasses
import os
import re

import numpy as np
import pytest

from gym_auv_b200 import Config, effective_reference_config, lidar_config, scenarios as S
from gym_auv_b200.pathbank import PATH_BLOCK, build_path
from oracle import geos_lite as G
from oracle import sim as OS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- config (reference tests/test_config.py + quirk #4) --------------------------------
def test_config_defaults_match_reference_declared_values():
    c = Config()
    assert c.simulation.t_step_size == 1.0 and c.episode.min_goal_distance == 5.0
    assert c.episode.max_timesteps == 10000 and c.episode.min_cumulative_reward == -2000.0
    assert c.vessel.use_lidar is False and c.vessel.n_sensors == 180 and c.vessel.sensor_range == 150.0
    assert c.vessel.vessel_width == 1.255 and c.vessel.sensor_interval_load_obstacles == 25
    assert [f.name for f in c] == ["episode", "simulation", "vessel", "rendering"]


def test_configs_do_not_share_state_unlike_reference():
    a, b = Config(), Config()
    a.simulation.t_step_size = 0.5
    assert b.simulation.t_step_size == 1.0
    e = effective_reference_config()
    assert e.simulation.t_step_size == 0.5 and e.episode.min_goal_distance == 0.1


@pytest.mark.parametrize("use_lidar_velocity", [True, False])
def test_lidar_observation_size(use_lidar_velocity):
    c = lidar_config(sensor_use_velocity_observations=use_lidar_velocity)
    assert c.vessel.lidar_shape == (3 if use_lidar_velocity else 1, 180)
    assert c.vessel.dense_observation_size + c.vessel.n_lidar_observations == 6 + (540 if use_lidar_velocity else 180)


# ---- path bank --------------------------------------------------------------------------
def test_path_table_matches_oracle_path():
    wp = S.random_curve_waypoints(np.random.RandomState(4), 5, 800)
    tab = build_path(wp)
    ora = OS.OraclePath(wp)
    assert tab.length == ora.length
    assert np.array_equal(tab.poly, ora.points)
    assert len(tab.poly) == int(10 * tab.length)
    s = np.linspace(-1, tab.length + 1, 57)
    assert np.allclose(tab(s), ora(s), atol=0, rtol=0)
    # coefficient layout [interval][axis][power] reproduces scipy's evaluation
    j = 417
    t = 0.37 * (tab.knots[j + 1] - tab.knots[j])
    val = ((tab.coef[j, :, 0] * t + tab.coef[j, :, 1]) * t + tab.coef[j, :, 2]) * t + tab.coef[j, :, 3]
    assert np.allclose(val, ora(tab.knots[j] + t), atol=1e-10)
    assert np.allclose(tab.end, ora.end)


def test_path_blocks_bound_their_segments():
    wp = S.random_curve_waypoints(np.random.RandomState(5), 4, 800)
    tab = build_path(wp)
    rel = tab.poly - tab.origin
    nseg = len(tab.poly) - 1
    assert len(tab.blk_dev) == (nseg + PATH_BLOCK - 1) // PATH_BLOCK
    for b in (0, 7, len(tab.blk_dev) - 1):
        lo, hi = b * PATH_BLOCK, min((b + 1) * PATH_BLOCK, nseg)
        a = tab.blk_chord[b, :2].astype(float)
        c = a + tab.blk_chord[b, 2:].astype(float)  # (first vertex, chord vector)
        for k in range(lo, hi + 1):
            d = G.point_segment_distance(rel[k, 0], rel[k, 1], a[0], a[1], c[0], c[1])
            assert d <= tab.blk_dev[b, 1]
        e2 = float(np.sum(tab.blk_chord[b, 2:].astype(float) ** 2))
        assert tab.blk_dev[b, 0] == pytest.approx(1.0 / e2, rel=1e-6)


def test_random_curve_shape():
    for nwp in (2, 3, 4, 5):
        wp = S.random_curve_waypoints(np.random.RandomState(nwp), nwp, 800)
        assert wp.shape == (2, 2 + 3 * (nwp // 2) - (nwp // 2 - 1) * 1) or wp.shape[0] == 2
        assert np.allclose(wp[:, 0], -wp[:, -1])  # end = -start
        assert np.hypot(*wp[:, 0]) == pytest.approx(400.0)


# ---- scenario plug-ins ---------------------------------------------------------------------
def test_moving_obstacles_distribution_and_constraints():
    scn = S.moving_obstacles(48, 17, 11, seed=2, n_paths=6)
    assert scn.k_moving == 17 and scn.k_static == 11 and scn.n_scenarios == 48
    assert scn.mov_width.min() >= 1 and scn.st_radius.min() >= 1
    speed = np.linalg.norm(scn.vel_table, axis=1)
    assert speed.min() >= 1 and speed.max() <= 3
    for m in range(48):
        tab = scn.bank.tables[scn.path_id[m]]
        vp = scn.vessel_init[m, :2]
        assert np.abs(vp - tab(0.0)).max() <= 25.0
        # generate_obstacle's acceptance test (helpers.py:27-33)
        d = np.linalg.norm(scn.st_pos[m] - vp, axis=1) - 1.255 - scn.st_radius[m]
        g = np.linalg.norm(scn.st_pos[m] - tab(tab.length), axis=1) - scn.st_radius[m]
        assert d.min() > 0 and g.min() > 0
        d = np.linalg.norm(scn.mov_start[m] - vp, axis=1) - 1.255 - scn.mov_width[m]
        assert d.min() > 0


def test_initial_obstacle_state_equals_oracle_reset():
    scn = S.moving_obstacles(3, 5, 2, seed=9)
    for dt in (1.0, 0.5):
        pos, disp, counter = scn.initial_obstacle_state(dt)
        for m in range(3):
            env = OS.OracleEnv(scn.describe(m), dict(t_step_size=dt, use_lidar=False))
            mov = [o for o in env.obstacles if not o.static]
            assert np.allclose([o.position for o in mov], pos[m], atol=1e-12)
            assert np.allclose([o.counter for o in mov], counter[m], atol=1e-12)
            assert counter[m, 0] == pytest.approx(0.1 + dt)


def test_debug_scenario_velocity_tables_and_no_post_update():
    scn = S.debug_scenario(seed=1)
    assert scn.k_moving == 10 and not scn.post_generate_update
    assert (scn.mov_track[0, :, 1] == 9999).all() and (scn.mov_track[0, :, 2] == 1).all()
    pos, _, counter = scn.initial_obstacle_state(0.5)
    assert np.allclose(counter, 0.1)


def test_scenario_registry_matches_reference_ids():
    ids = {"TestScenario1-v0", "TestScenario2-v0", "TestScenario3-v0", "TestScenario4-v0", "TestHeadOn-v0",
           "TestCrossing-v0", "TestCrossing1-v0", "DebugScenario-v0", "EmptyScenario-v0",
           "MovingObstaclesNoRules-v0", "PathFollowNoObstacles-v0"}
    assert set(S.SCENARIOS) == ids  # gym_auv/__init__.py:43-121 (uncommented entries)
    assert S.test_scenario1().k_static == 20 and S.test_scenario3().k_static == 21 and S.test_scenario4().k_static == 15


def test_negative_radius_raises_value_error():
    with pytest.raises(ValueError):
        S._single([[0, 10], [0, 10]], static=[((1.0, 1.0), -2.0)])


def test_concat_pads_slots():
    a, b = S.test_scenario3(), S.test_crossing()
    b.post_generate_update = a.post_generate_update
    c = S.concat([a, b])
    assert c.n_scenarios == 2 and c.k_static == 21 and c.k_moving == 1
    assert (c.st_radius[1] == 0).all() and c.mov_width[0, 0] == 0 and c.mov_width[1, 0] == 30


# ---- ABI --------------------------------------------------------------------------------
def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "auv_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(auv_[a-z_0-9]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol(built_lib):
    lib = ctypes.CDLL(built_lib)
    names = _declared_symbols()
    assert {"auv_step", "auv_step_host", "auv_observe", "auv_vessel_step", "auv_obstacle_update", "auv_reset",
            "auv_abi_version", "auv_last_error", "auv_obs_dim", "auv_sizeof", "auv_fma_probe"} <= set(names)
    for n in names:
        assert hasattr(lib, n), f"libauv_b200.so does not export {n}"


def test_binding_layout_and_version(built_lib):
    from gym_auv_b200 import _lib

    lib = _lib.load()  # raises on ABI/layout mismatch
    assert lib.auv_abi_version() == _lib.ABI_VERSION
    assert set(_lib.EXPORTS) == set(_declared_symbols())
    cfg = _lib.AuvConfig(n_sensors=180, use_lidar=1)
    assert lib.auv_obs_dim(ctypes.byref(cfg)) == 186
    cfg.sensor_use_velocity_observations = 1
    assert lib.auv_obs_dim(ctypes.byref(cfg)) == 546
    cfg.use_lidar = 0
    assert lib.auv_obs_dim(ctypes.byref(cfg)) == 6


def test_python_constants_equal_the_header_defines():
    """The host code sizes and indexes device tables with Python copies of the header's constants (pathbank
    builds the capsule tables the kernels search by AUV_PATH_BLOCK / SUPER / SUB): each copy must equal its
    #define, and every status bit must have one."""
    from gym_auv_b200 import _lib, pathbank

    hdr = open(os.path.join(ROOT, "include", "auv_b200.h")).read()
    defines = {k: int(v) for k, v in re.findall(r"^#define (AUV_\w+) +\(?(-?\d+)\)?", hdr, flags=re.M)}
    status = sorted(k[len("AUV_"):] for k in defines if k.startswith("AUV_STATUS_"))
    assert status and status == sorted(k for k in vars(_lib) if k.startswith("STATUS_"))
    mirrors = {f"AUV_{k}": getattr(_lib, k) for k in status + ["ABI_VERSION", "REC_BYTES", "MAX_POLY_VERTS", "NAV_W", "PP_W",
                                                             "PATH_STAGE_BLOCKS"]}
    mirrors.update(AUV_PATH_BLOCK=pathbank.PATH_BLOCK, AUV_PATH_SUPER=pathbank.PATH_SUPER, AUV_PATH_SUB=pathbank.PATH_SUB)
    assert mirrors == {k: defines.get(k) for k in mirrors}


def test_scenario_template_is_the_input_of_gpu_generation():
    scn = S.moving_obstacles_template(64, 5, 3, seed=1, n_paths=4)
    assert scn.n_scenarios == 64 and scn.k_moving == 5 and scn.k_static == 3 and len(scn.waypoints) == 4
    assert scn.vel_table.shape == (64 * 5, 2)  # one constant-velocity entry per (scenario, slot)
    assert np.array_equal(scn.mov_track[..., 0], np.arange(64 * 5).reshape(64, 5))
    assert not (scn.mov_width > 0).any() and not (scn.st_radius > 0).any()  # every slot empty until generated
    scn.validate()
    pos, disp, counter = scn.initial_obstacle_state(1.0)
    assert not disp.any() and not counter.any()


def test_generator_and_pipeline_entry_points_reject_bad_arguments(built_lib):
    from gym_auv_b200 import _lib

    lib = _lib.load()
    assert lib.auv_generate_moving_obstacles(None, None, None, None, 1, None, None) == -1
    gp, paths, pool = _lib.AuvGenParams(seed=1), _lib.AuvPathBank(n_paths=0), _lib.AuvScenarioPool(n_scenarios=4)
    assert lib.auv_generate_moving_obstacles(ctypes.byref(gp), ctypes.byref(paths), ctypes.byref(pool), None, 8, None, None) == -1
    assert b"n_ids" in lib.auv_last_error()
    assert lib.auv_generate_moving_obstacles(ctypes.byref(gp), ctypes.byref(paths), ctypes.byref(pool), None, 4, None, None) == -1
    assert b"path bank" in lib.auv_last_error()
    assert lib.auv_pipeline_graph_state(None) == -1
    assert not lib.auv_pipeline_create(0) and not lib.auv_pipeline_create(99)
    assert ctypes.sizeof(_lib.AuvGenParams) == lib.auv_sizeof(6)


def test_bad_arguments_return_error_codes_not_crashes(built_lib):
    from gym_auv_b200 import _lib

    lib = _lib.load()
    assert lib.auv_vessel_step(None, None, None, None) == -1
    assert b"NULL" in lib.auv_last_error()
    cfg = _lib.AuvConfig(t_step_size=0.0, sensor_interval_load_obstacles=25)
    batch = _lib.AuvBatch(n_envs=4)
    assert lib.auv_vessel_step(ctypes.byref(cfg), ctypes.byref(batch), ctypes.c_void_p(8), None) == -1
    assert b"t_step_size" in lib.auv_last_error()


def test_delta_host_step_rejects_bad_arguments(built_lib):
    """auv_step_host_delta_submit validates its AuvDelta before touching the device: NULL buffers, a chunk size
    other than 8 / 16 / 32 floats and unaligned arrays come back as error codes."""
    from gym_auv_b200 import _lib

    lib = _lib.load()
    assert lib.auv_step_host_delta_submit(None, None, None, None, None, None, None, None, None, None, None, None, None, 1) == -1
    assert b"NULL" in lib.auv_last_error()
    cfg, batch, out = _lib.AuvConfig(t_step_size=1.0), _lib.AuvBatch(n_envs=4), _lib.AuvStepOut()
    p = ctypes.c_void_p(64)
    args = lambda d: (ctypes.byref(cfg), None, None, None, ctypes.byref(batch), p, p, ctypes.byref(out), ctypes.byref(d), p, p,
                      None, None, 1)
    assert lib.auv_step_host_delta_submit(*args(_lib.AuvDelta(None, None, None, 16, 0))) == -1
    assert b"delta buffers" in lib.auv_last_error()
    assert lib.auv_step_host_delta_submit(*args(_lib.AuvDelta(64, 64, None, 12, 0))) == -1
    assert b"gran" in lib.auv_last_error()
    assert lib.auv_step_host_delta_submit(*args(_lib.AuvDelta(64, 72, None, 16, 0))) == -1
    assert b"aligned" in lib.auv_last_error()
    assert ctypes.sizeof(_lib.AuvDelta) == lib.auv_sizeof(11) == 32


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "gym_auv_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn


def test_vec_env_refuses_to_run_without_cuda():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from gym_auv_b200.vec_env import AUVVecEnv

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        AUVVecEnv(S.empty_scenario(), 1, Config(), device="cuda:0")


def test_parity_harness_counts_steps_inside_the_collision_band():
    """tests/_parity.compare skips the bit-exact collision / done comparison where the oracle's minimum
    range is within COLLISION_BAND of the vessel width (FP32 casting may legitimately decide the other
    way) -- and COUNTS those steps.  Forced case: one step inside the band with flipped flags is
    skipped and counted, the same flip outside the band fails."""
    import pytest

    from gym_auv_b200 import lidar_config
    from tests._parity import COLLISION_BAND, compare

    cfg = lidar_config()
    w = cfg.vessel.vessel_width
    T, M, R = 2, 1, cfg.vessel.n_sensors

    def case(min_dist):
        dists = np.full((T, M, R), 150.0)
        dists[1, 0, 7] = min_dist
        ref = dict(alive=np.ones((T, M), bool), state=np.zeros((T, M, 6)), s=np.zeros((T, M)), dists=dists,
                   min_dist=dists.min(axis=2), collision=np.zeros((T, M), bool), reached=np.zeros((T, M), bool),
                   done=np.zeros((T, M), bool), reward=np.zeros((T, M)), obs=np.zeros((T, M, 6 + R)), windows=[[{}] * M] * T)
        gpu = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in ref.items()}
        gpu["collision"][1, 0] = gpu["done"][1, 0] = True  # the FP32 side saw 1.2549 < width
        gpu["windows"] = np.zeros((T, M, 1, 2), int)
        return ref, gpu

    ref, gpu = case(w + 0.5 * COLLISION_BAND)
    rep = compare(ref, gpu, cfg, "inside the band")
    assert rep["collision_skipped_in_band"] == 1 and rep["collision_decisive"] == T * M - 1
    ref, gpu = case(w + 3 * COLLISION_BAND)
    with pytest.raises(AssertionError):
        compare(ref, gpu, cfg, "outside the band")


def test_device_path_slot_capacity_covers_the_random_curve_family():
    """DevicePathBank's default slot (vcap vertices at 10 per metre) holds every RandomCurveThroughOrigin
    (length=800, <= 5 waypoints) curve: PCHIP is monotone per coordinate between knots, so the path length is
    bounded by the L1 length of the waypoint polygon, which for this family is < 4.08 x length."""
    from gym_auv_b200.pathbank import DevicePathBank, build_path, random_curve_waypoints

    rng = np.random.RandomState(5)
    worst = 0.0
    for k in range(300):
        w = random_curve_waypoints(rng, int(np.floor(4 * rng.rand() + 2)), length=800.0)
        l1 = float(np.abs(np.diff(w, axis=1)).sum())
        assert l1 < 4.08 * 800.0
        worst = max(worst, l1)
        if k < 12:
            assert build_path(w).length <= l1 + 1e-9
    bank = DevicePathBank([random_curve_waypoints(rng, 5, length=800.0)])
    assert 10 * 4.08 * 800.0 + 2 <= bank.vcap


def test_env_group_ring_hands_out_groups_in_completion_order():
    """EnvGroupRing.recv returns whichever pending group has finished (not the oldest submission), send appends to
    the pending list, recv without anything in flight raises -- checked with stand-in groups (no GPU)."""
    from gym_auv_b200.vec_env import EnvGroupRing

    class Done:
        def __init__(self):
            self.ready = False

        def query(self):
            return self.ready

    class Group:
        num_envs = 5

        def __init__(self, name):
            self.name, self._async_done, self.wait_seconds, self.sent = name, Done(), 0.0, []

        def step_async(self, actions):
            self.sent.append(actions)
            self._async_done.ready = False

        def step_wait(self):
            return (self.name, len(self.sent)), "rew", "done"

        def reset(self):
            return self.name

        def close(self):
            pass

    groups = [Group("a"), Group("b"), Group("c")]
    ring = EnvGroupRing(groups)
    assert len(ring) == 3 and ring.envs_per_group == 5 and ring.reset() == ["a", "b", "c"]
    with pytest.raises(RuntimeError):
        ring.recv()
    for g in range(3):
        ring.send(g, g)
    assert ring.pending == [0, 1, 2]
    groups[2]._async_done.ready = True  # the last submission finishes first
    g, obs, rew, done = ring.recv()
    assert g == 2 and obs == ("c", 1) and ring.pending == [0, 1]
    ring.send(2, "next")
    groups[0]._async_done.ready = groups[1]._async_done.ready = True
    assert [ring.recv()[0] for _ in range(2)] == [0, 1]  # both ready: submission order
    groups[2]._async_done.ready = True
    assert [r[0] for r in ring.drain()] == [2] and ring.pending == []
    ring.close()
    assert ring.groups == []
