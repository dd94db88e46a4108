"""Episode tracks (AuvStepOut.tracks, ``record_tracks``): the step kernel records, for a sample of the
batch, each step's pose and reward and, when an episode ends, a snapshot of the scenario it ran on --
what ``BaseEnvironment.save_latest_episode`` (environment.py:466-489) keeps as ``path_taken`` and the
obstacles' histories.  CPU tests cover the host assembly, the obstacle-track functions and the ABI
checks; GPU tests cover the recording itself on every step path."""
import ctypes
import os

import numpy as np
import pytest

from gym_auv_b200 import scenarios as S
from gym_auv_b200.vec_env import assemble_episode, pick_finished_row, track_rows

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_stubbed.npz"))


@pytest.fixture(scope="module")
def lib(built_lib):
    from gym_auv_b200 import _lib

    return _lib.load()


# ------------------------------------------------------------------ CPU: host assembly
def _head(ep, steps, finished, collision=0, reached=0, scn=3, upd=None):
    return np.array([ep, steps, finished, collision, reached, scn, steps if upd is None else upd, 0], dtype=np.int32)


def test_finished_row_choice():
    """The finished row with the greater episode number wins; an unfinished row never does, also when it
    holds the greater number; a new episode that has not stepped yet leaves a stale finished row of
    episode - 2 beside the one just finished."""
    assert pick_finished_row(np.stack([_head(0, 5, 0), _head(0, 0, 0)])) is None
    assert pick_finished_row(np.stack([_head(4, 9, 0), _head(3, 7, 1)])) == 1  # episode 4 running
    assert pick_finished_row(np.stack([_head(2, 9, 1), _head(3, 7, 1)])) == 1  # episode 4 not stepped yet
    assert pick_finished_row(np.stack([_head(4, 9, 1), _head(3, 7, 1)])) == 0
    assert pick_finished_row(np.stack([_head(6, 2, 0), _head(1, 7, 1)])) == 1


def test_ring_wrap_truncation_and_step_index():
    T = 8
    pts = np.zeros((T, 4), np.float32)
    for t in range(21):  # 21 steps into a ring of 8: the kernel writes step t at t % T
        pts[t % T] = (t + 1, 10 * (t + 1), 0.01 * (t + 1), -(t + 1))
    rows, idx, trunc = track_rows(_head(0, 21, 1), pts, T)
    assert trunc and list(idx) == list(range(14, 22)) and list(rows[:, 0]) == list(range(14, 22))
    rows, idx, trunc = track_rows(_head(0, 8, 1), pts[:8] * 0 + np.arange(1, 9, dtype=np.float32)[:, None], T)
    assert not trunc and list(idx) == list(range(1, 9))
    snap = np.zeros(4)
    snap[:4] = (0, 1.5, -2.5, 0.25)
    ep = assemble_episode(_head(5, 21, 1, collision=1, scn=0), pts, snap, T, 0, 0, 1.0, None, None)
    assert ep["truncated"] and ep["path_taken"].shape == (8, 2) and list(ep["step_index"]) == list(range(14, 22))
    assert ep["timesteps"] == 21 and ep["collision"] and not ep["reached_goal"] and ep["episode"] == 5
    assert np.array_equal(ep["rewards"], -np.arange(14, 22, dtype=np.float64))
    short = np.zeros((T, 4), np.float32)
    short[:3] = [(1, 2, 3, 4), (5, 6, 7, 8), (9, 10, 11, 12)]
    ep = assemble_episode(_head(2, 3, 1, reached=1, scn=0), short, snap, T, 0, 0, 1.0, None, None)
    assert not ep["truncated"] and "step_index" not in ep and ep["reached_goal"]
    assert np.array_equal(ep["path_taken"], [[1.5, -2.5], [1, 2], [5, 6], [9, 10]])  # row 0: vessel_init exactly
    assert np.array_equal(ep["heading_taken"], [0.25, 3, 7, 11]) and np.array_equal(ep["rewards"], [4, 8, 12])


def test_snapshot_layout_of_static_and_moving_slots():
    """Moving slots come from their 64 B mov_lin record, static slots from their st_rec record; unused
    slots (width / radius <= 0) are dropped."""
    lin = dict(first_wrap=100, wrap_period=50, vel_len=10)
    rec = np.array([[1, 2, 0.5, -0.25, 3.0, 9, 8, 0], [0, 0, 0, 0, 0.0, 0, 0, 0]], float)
    st = np.array([[5, 6, 7, 0], [0, 0, -1, 0]], float)
    snap = np.concatenate([[0, 1, 1, 0], rec.reshape(-1), st.reshape(-1)])
    pts = np.zeros((4, 4), np.float32)
    ep = assemble_episode(_head(0, 2, 1, upd=2), pts, snap, 4, 2, 2, 0.5, lin, None)
    ob = ep["obstacles"]
    assert ob["moving"]["width"].tolist() == [3.0] and ob["moving"]["start"].tolist() == [[9, 8]]
    assert np.array_equal(ob["moving"]["vel_tables"][0], np.repeat([[1.0, -0.5]], 10, axis=0))
    assert ob["static"]["pos"].tolist() == [[5, 6]] and ob["static"]["radius"].tolist() == [7]
    assert np.array_equal(ob["moving_path_taken"][:, 0], [[1, 2], [1.5, 1.75], [2, 1.5]])


# ------------------------------------------------------------------ CPU: obstacle tracks
def test_closed_form_tracks_against_the_stepwise_update(lib):
    """``linear_track_positions`` (the closed form the device evaluates) against ``advance_obstacles``
    iterated one update at a time, across the first wrap and several wrap periods."""
    from gym_auv_b200 import _lib

    dt = 1.0
    scn = S.moving_obstacles(3, 4, 0, seed=5, n_paths=1)
    info = scn.linear_track_info(dt)
    first, period = ctypes.c_int32(0), ctypes.c_int32(0)
    _lib.check(lib.auv_linear_wrap(dt, info["counter0"], info["vel_len"], ctypes.byref(first), ctypes.byref(period)),
               "auv_linear_wrap")
    first, period = int(first.value), int(period.value)
    pos0, _, counter = scn.initial_obstacle_state(dt)
    m = 1
    tr = scn.mov_track[m]
    rec = np.zeros((scn.k_moving, 8))
    rec[:, 0:2] = pos0[m]
    rec[:, 2:4] = dt * scn.vel_table[tr[:, 0]]
    rec[:, 4] = scn.mov_width[m]
    rec[:, 5:7] = scn.mov_start[m]
    horizon = first + 3 * period + 5
    probe = sorted(set(range(0, horizon, 97)) | set(range(first - 3, first + 4)) | set(range(first + period - 3, first + period + 4))
                   | {horizon - 1})
    want = {}
    pos = pos0
    for n in range(horizon):
        if n in probe:
            want[n] = pos[m].copy()
        pos, _, counter = S.advance_obstacles(scn, pos, counter, dt)
    got = S.linear_track_positions(rec, probe, first, period)
    for k, n in enumerate(probe):
        assert np.abs(got[k] - want[n]).max() <= 1e-8, n
    # the closed form itself: exactly pos0 + n d before the wrap, start + ((n - first) mod period + 1) d after
    assert np.array_equal(S.linear_track_positions(rec, [0], first, period)[0], rec[:, 0:2])
    assert np.array_equal(S.linear_track_positions(rec, [first], first, period)[0], rec[:, 5:7] + rec[:, 2:4])


# the golden tracks built with VesselObstacle's construction-time update, which initial_obstacle_state applies
@pytest.mark.parametrize("k", [k for k in range(GOLD["trk_dt"].shape[0]) if bool(GOLD["trk_dt"][k, 1])])
def test_table_tracks_against_reference_golden(k):
    """``table_track_positions`` against the reference-generated VesselObstacle positions (wrap included)."""
    tr = GOLD["trk_traj"][k]
    tr = tr[~np.isnan(tr[:, 0])]
    scn = S._single(np.array([[0.0, 100.0], [0.0, 0.0]]), moving_traj=[(5.0, [(int(t), (x, y)) for t, x, y in tr])])
    got = S.table_track_positions(scn, 0, np.arange(61), float(GOLD["trk_dt"][k, 0]))
    assert np.abs(got[:, 0] - GOLD["trk_pos"][k]).max() <= 1e-9


def test_fma_is_correctly_rounded():
    a = np.array([1.0 + 2.0 ** -30, 3.0, 0.1])
    b = np.array([1.0 - 2.0 ** -30, 7.0, 3.0])
    c = np.array([-1.0, 0.5, -0.3])
    from fractions import Fraction

    got = S._fma(a, b, c)
    for i in range(3):
        assert got[i] == float(Fraction(a[i]) * Fraction(b[i]) + Fraction(c[i]))
    # the closed form's operands (integer update counts, displacements, positions), and sums that nearly cancel
    rng = np.random.default_rng(0)
    n = 4000
    a = rng.integers(0, 2 ** 31, n).astype(np.float64)
    b = rng.normal(0.0, 1.0, n) * np.exp2(rng.integers(-30, 5, n))
    c = rng.normal(0.0, 1000.0, n)
    c[: n // 4] = -(a[: n // 4] * b[: n // 4]) + rng.normal(0.0, 1e-6, n // 4)
    a[-n // 4:] = rng.normal(0.0, 1.0, n // 4)
    b[-n // 4:] = 1.0 + np.exp2(-rng.integers(20, 52, n // 4).astype(np.float64))
    c[-n // 4:] = -a[-n // 4:]
    got = S._fma(a, b, c)
    for i in range(n):
        assert got[i] == float(Fraction(a[i]) * Fraction(b[i]) + Fraction(c[i])), i


# ------------------------------------------------------------------ CPU: ABI
def test_tracks_struct_size(lib):
    from gym_auv_b200 import _lib

    assert ctypes.sizeof(_lib.AuvTracks) == lib.auv_sizeof(12) == 40
    assert _lib.ABI_VERSION == lib.auv_abi_version() == 22


def test_invalid_tracks_are_refused_before_any_device_work(lib):
    """Every step entry point refuses a bad AuvTracks with AUV_EINVAL and a message; the other pointers are
    fake host addresses, so any device work would fail with a CUDA error instead."""
    from gym_auv_b200 import _lib

    cfg = _lib.AuvConfig(t_step_size=1.0, sensor_interval_load_obstacles=25)
    batch, pool, paths = _lib.AuvBatch(n_envs=16), _lib.AuvScenarioPool(), _lib.AuvPathBank()
    p = ctypes.c_void_p(64)
    bad = [
        (_lib.AuvTracks(2, 4, 8, 0, None, 64, 64), b"NULL"),
        (_lib.AuvTracks(2, 4, 8, 0, 64, None, 64), b"NULL"),
        (_lib.AuvTracks(2, 4, 8, 0, 64, 64, None), b"NULL"),
        (_lib.AuvTracks(0, 4, 8, 0, 64, 64, 64), b">= 1"),
        (_lib.AuvTracks(2, 0, 8, 0, 64, 64, 64), b">= 1"),
        (_lib.AuvTracks(2, 4, 0, 0, 64, 64, 64), b">= 1"),
        (_lib.AuvTracks(5, 4, 8, 0, 64, 64, 64), b"n_envs"),
        (_lib.AuvTracks(2, 4, 8, 0, 72, 64, 64), b"points must be 16-byte aligned"),
        (_lib.AuvTracks(2, 4, 8, 0, 64, 68, 64), b"head must be 16-byte aligned"),
        (_lib.AuvTracks(2, 4, 8, 0, 64, 72, 64), b"head must be 16-byte aligned"),
        (_lib.AuvTracks(2, 4, 8, 0, 64, 64, 68), b"snap must be 8-byte aligned"),
    ]
    for tk, msg in bad:
        out = _lib.AuvStepOut(obs=64, reward=64, done=64, tracks=ctypes.addressof(tk))
        calls = [
            lambda: lib.auv_step(ctypes.byref(cfg), None, ctypes.byref(paths), ctypes.byref(pool), ctypes.byref(batch), p,
                                 ctypes.byref(out), None),
            lambda: lib.auv_step_host(ctypes.byref(cfg), None, ctypes.byref(paths), ctypes.byref(pool), ctypes.byref(batch),
                                      p, p, ctypes.byref(out), p, p, p, None),
            lambda: lib.auv_step_host_delta_submit(ctypes.byref(cfg), None, ctypes.byref(paths), ctypes.byref(pool),
                                                   ctypes.byref(batch), p, p, ctypes.byref(out),
                                                   ctypes.byref(_lib.AuvDelta(64, 64, None, 16, 0)), p, p, None, p, 1),
            lambda: lib.auv_step_host_submit(ctypes.byref(cfg), None, ctypes.byref(paths), ctypes.byref(pool),
                                             ctypes.byref(batch), p, p, ctypes.byref(out), p, p, p, None, p, 1),
            lambda: lib.auv_observe(ctypes.byref(cfg), None, ctypes.byref(paths), ctypes.byref(pool), ctypes.byref(batch),
                                    ctypes.byref(out), 0, None),
        ]
        for call in calls:
            assert call() == -1  # AUV_EINVAL
            assert b"tracks" in lib.auv_last_error() and msg in lib.auv_last_error()
    ok = _lib.AuvTracks(4, 5, 8, 0, 64, 64, 64)  # (4 - 1) * 5 < 16: valid, so the check goes on to the next argument
    out = _lib.AuvStepOut(obs=64, reward=64, done=64, seg_tests=64, tracks=ctypes.addressof(ok))
    assert lib.auv_step(ctypes.byref(cfg), None, ctypes.byref(paths), ctypes.byref(pool), ctypes.byref(batch), p,
                        ctypes.byref(out), None) == -1
    assert b"seg_tests" in lib.auv_last_error()


# ------------------------------------------------------------------ GPU
N_ENVS = 4096


def _cfg(max_timesteps=150):
    from gym_auv_b200 import lidar_config

    cfg = lidar_config()
    cfg.episode.max_timesteps = max_timesteps  # several episodes per env within the test
    return cfg


def _actions(n, steps, seed):
    torch = pytest.importorskip("torch")
    gen = torch.Generator(device="cuda").manual_seed(seed)
    lo, hi = torch.tensor([-1.0, -0.15], device="cuda"), torch.tensor([1.0, 0.15], device="cuda")
    return [lo + (hi - lo) * torch.rand((n, 2), device="cuda", generator=gen) for _ in range(steps)]


@pytest.fixture(scope="module")
def paired(lib):
    """Two envs on the same seeded config-3-shaped pool, one recording 64 envs, stepped 600 times with the
    same actions and the device refresh every 8 steps; everything observed along the way."""
    torch = pytest.importorskip("torch")
    from gym_auv_b200.vec_env import AUVVecEnv

    N, cfg = N_ENVS, _cfg()
    scn = S.moving_obstacles_template(2 * N, 16, 16, seed=2, n_paths=64, path_period=N)
    a = AUVVecEnv(scn, N, cfg, auto_reset=True)
    b = AUVVecEnv(scn, N, cfg, auto_reset=True, record_tracks=64)
    for e in (a, b):
        e.regenerate_scenarios(seed=5, epoch=1)
        e.reset()
    tr = torch.as_tensor(b.tracked_envs, device="cuda")
    acts = _actions(N, 16, 7)
    keys = ("obs", "reward", "done", "collision", "reached_goal", "goal_distance", "progress", "terminal_obs",
            "episode_out")
    mism = []
    log = dict(state=[b.state[:, tr].cpu().numpy()], reward=[], done=[], episode_out=[], obst=[], scn=[])
    log["obst"].append(b.obstacle_state()[0][tr].cpu().numpy())
    survivors = {}
    for t in range(600):
        a.step(acts[t % 16])
        b.step(acts[t % 16])
        for k in keys:
            if not torch.equal(a._out[k], b._out[k]):
                mism.append((t, k))
        # the statistics are FP64 atomicAdd sums: their order between CTAs is not fixed, in one env or two
        if not torch.allclose(a._out["stats"], b._out["stats"], rtol=1e-12, atol=0):
            mism.append((t, "stats"))
        for k in ("state", "episode", "t_step", "scn_id", "cum_reward", "obst_steps", "max_progress", "nearby_mask"):
            if not torch.equal(a._st[k], b._st[k]):
                mism.append((t, k))
        log["state"].append(b.state[:, tr].cpu().numpy())
        log["reward"].append(b._out["reward"][tr].cpu().numpy())
        d = b._out["done"][tr].cpu().numpy().astype(bool)
        log["done"].append(d)
        log["episode_out"].append(b._out["episode_out"][tr].cpu().numpy())
        log["obst"].append(b.obstacle_state()[0][tr].cpu().numpy())
        for k in np.nonzero(d)[0][:3]:  # a few late finished episodes, read right away
            if t >= 480 and len(survivors) < 8 and int(b.tracked_envs[k]) not in survivors:
                survivors[int(b.tracked_envs[k])] = (t, b.last_episode(int(b.tracked_envs[k])))
        if t % 8 == 7:
            a.refresh_finished_device(seed=11)
            b.refresh_finished_device(seed=11)
    torch.cuda.synchronize()
    for k in ("state", "reward", "done", "episode_out", "obst"):
        log[k] = np.stack(log[k])
    return dict(a=a, b=b, mism=mism, log=log, survivors=survivors, scn=scn)


def _episodes(done_col):
    """(first step, done step) of each finished episode of one env, steps numbered from 0."""
    ends = np.nonzero(done_col)[0]
    starts = np.concatenate([[0], ends[:-1] + 1])
    return list(zip(starts, ends))


@pytest.mark.gpu
def test_recording_changes_no_result(paired):
    assert paired["mism"] == []
    assert paired["log"]["done"].any(axis=0).sum() >= 32  # most tracked envs finished an episode


@pytest.mark.gpu
def test_points_are_the_state(paired):
    """Each recorded point is float32 of the state after that step, its reward the step's reward; row 0 of
    ``path_taken`` is the scenario's vessel_init, across auto-resets."""
    b, log = paired["b"], paired["log"]
    checked = 0
    for k, e in enumerate(b.tracked_envs):
        done = log["done"][:, k]
        eps = _episodes(done)
        cur_start = eps[-1][1] + 1 if eps else 0
        rec = b.current_episode(int(e))
        n = rec["timesteps"]
        assert n == 600 - cur_start and rec["path_taken"].shape == (n + 1, 2)
        st = log["state"][cur_start:cur_start + n + 1, :, k]  # state after each step of the episode; [0] after reset
        assert np.array_equal(rec["path_taken"][0], st[0, 0:2]) and rec["heading_taken"][0] == st[0, 2]
        assert np.array_equal(rec["path_taken"][1:], st[1:, 0:2].astype(np.float32).astype(np.float64))
        assert np.array_equal(rec["heading_taken"][1:], st[1:, 2].astype(np.float32).astype(np.float64))
        assert np.array_equal(rec["rewards"], log["reward"][cur_start:cur_start + n, k].astype(np.float64))
        last = b.last_episode(int(e))
        if eps:
            s0, s1 = eps[-1]
            m = s1 - s0 + 1
            assert last["timesteps"] == m and last["path_taken"].shape == (m + 1, 2)
            st = log["state"][s0:s1 + 1, :, k]  # [0]: after the reset that started it; the done step's is post-reset
            assert np.array_equal(last["path_taken"][0], st[0, 0:2])
            assert np.array_equal(last["path_taken"][1:m], st[1:m, 0:2].astype(np.float32).astype(np.float64))
            assert np.array_equal(last["rewards"], log["reward"][s0:s1 + 1, k].astype(np.float64))
            checked += 1
        else:
            assert last is None
    assert checked >= 32


@pytest.mark.gpu
def test_finished_episode_survives_the_next_one(paired):
    b, log = paired["b"], paired["log"]
    compared = 0
    for e, (t, early) in paired["survivors"].items():
        k = int(np.nonzero(b.tracked_envs == e)[0][0])
        later = b.last_episode(e)
        if later["episode"] != early["episode"]:
            continue  # finished another one since: compared through test_points_are_the_state
        row = log["episode_out"][t, k]
        assert later["timesteps"] == int(row[1]) and later["collision"] == bool(row[3])
        assert later["reached_goal"] == bool(row[4]) and later["episode"] == int(row[7])
        for key in ("path_taken", "heading_taken", "rewards"):
            assert np.array_equal(later[key], early[key])
        assert np.array_equal(later["obstacles"]["moving_path_taken"], early["obstacles"]["moving_path_taken"])
        compared += 1
    assert compared >= 3


@pytest.mark.gpu
def test_snapshot_survives_the_device_refresh(paired):
    """``moving_path_taken`` equals ``obstacle_state()`` read along the episode, although the refresh has
    since regenerated the pool slot the episode ran on."""
    b, log = paired["b"], paired["log"]
    mov_lin = b._pool["mov_lin"].cpu().numpy()
    regenerated = 0
    for k, e in enumerate(b.tracked_envs):
        eps = _episodes(log["done"][:, k])
        if not eps:
            continue
        s0, s1 = eps[-1]
        m = s1 - s0 + 1
        last = b.last_episode(int(e))
        mp = last["obstacles"]["moving_path_taken"]
        assert mp.shape == (m + 1, 16, 2)
        assert np.array_equal(mp[:m], log["obst"][s0:s1 + 1, k])  # rows 0 .. m-1 (the done step's is post-reset)
        snap_rec = np.concatenate([last["obstacles"]["moving"]["start"], last["obstacles"]["moving"]["width"][:, None]], 1)
        slot = mov_lin[last["scenario"]]
        if not np.array_equal(snap_rec, np.concatenate([slot[:, 5:7], slot[:, 4:5]], 1)):
            regenerated += 1
    assert regenerated >= 8


@pytest.mark.gpu
def test_truncation_keeps_the_last_points(lib):
    torch = pytest.importorskip("torch")
    from gym_auv_b200.vec_env import AUVVecEnv

    scn = S.path_follow_no_obstacles(64, seed=3, n_paths=4)
    env = AUVVecEnv(scn, 64, _cfg(), test_mode=True, auto_reset=True, record_tracks=4, track_capacity=64)
    env.reset()
    zero = torch.zeros((64, 2), device="cuda")
    zero[:, 1] = 0.1  # no thrust: the vessel turns on the spot, the episode cannot end
    states = [env.state[:, env.tracked_envs].cpu().numpy()]
    for _ in range(200):
        _, _, done, _ = env.step(zero)
        assert not bool(done.any())
        states.append(env.state[:, env.tracked_envs].cpu().numpy())
    states = np.stack(states)
    for k, e in enumerate(env.tracked_envs):
        assert env.last_episode(int(e)) is None
        rec = env.current_episode(int(e))
        assert rec["truncated"] and rec["timesteps"] == 200 and rec["path_taken"].shape == (64, 2)
        assert list(rec["step_index"]) == list(range(137, 201))
        assert np.array_equal(rec["path_taken"], states[137:201, 0:2, k].astype(np.float32).astype(np.float64))


def _tracks_of(envs):
    import torch

    torch.cuda.synchronize()
    return [np.concatenate([e._tracks[k].cpu().numpy() for e in envs]) for k in ("points", "head", "snap")]


@pytest.mark.gpu
def test_all_step_paths_record_the_same(lib):
    """``step`` (auv_step), ``step_host`` with the delta transfer, ``step_async`` / ``step_wait`` through
    ``ring(4, record_tracks=4)`` and ``chunks=4`` produce the same track buffers."""
    from gym_auv_b200.vec_env import AUVVecEnv

    N, cfg = 1024, _cfg(100)
    scn = S.moving_obstacles_template(2 * N, 16, 16, seed=6, n_paths=16, path_period=N)
    acts = _actions(N, 8, 3)
    host_acts = [a.cpu().numpy() for a in acts]
    base = AUVVecEnv(scn, N, cfg, auto_reset=True, record_tracks=16, track_capacity=128)
    base.regenerate_scenarios(seed=2, epoch=1)
    chunked = AUVVecEnv(scn, N, cfg, auto_reset=True, record_tracks=16, track_capacity=128, chunks=4, _shared=base._shared_tables())
    hosted = AUVVecEnv(scn, N, cfg, auto_reset=True, record_tracks=16, track_capacity=128, host_transfer="delta",
                       _shared=base._shared_tables())
    ring = base.ring(4, record_tracks=4, track_capacity=128)
    for e in [base, chunked, hosted] + ring.groups:
        e.reset()
    n = ring.envs_per_group
    for t in range(260):
        base.step(acts[t % 8])
        chunked.step(acts[t % 8])
        hosted.step_host(host_acts[t % 8])
        for g in range(4):
            ring.send(g, host_acts[t % 8][g * n:(g + 1) * n])
        ring.drain()
    want = _tracks_of([base])
    assert (want[1][:, :, 2] != 0).any()  # some tracked env finished
    for other in ([chunked], [hosted], ring.groups):
        got = _tracks_of(other)
        for w, g in zip(want, got):
            assert np.array_equal(w, g)


@pytest.mark.gpu
def test_trainer_surface_get_attr_last_episode(lib):
    from gym_auv_b200.adapters import B200VecEnv

    n = 512
    scn = S.moving_obstacles_template(2 * n, 16, 16, seed=1, n_paths=8, path_period=n)
    venv = B200VecEnv(scn, n, _cfg(80), fresh_scenarios=True, record_tracks=8)
    plain = B200VecEnv(scn, n, _cfg(80), fresh_scenarios=True)
    venv.reset()
    plain.reset()
    rng = np.random.RandomState(0)
    for _ in range(120):
        a = rng.uniform([-1, -0.15], [1, 0.15], size=(n, 2)).astype(np.float32)
        venv.step(a)
        plain.step(a)
    eps = venv.get_attr("last_episode")
    tracked = set(int(e) for e in venv.impl.tracked_envs)
    assert len(eps) == n and len(tracked) == 8
    for i, ep in enumerate(eps):
        if i in tracked:
            assert isinstance(ep, dict) and ep["path_taken"].shape == (ep["timesteps"] + 1, 2)
            assert ep["path"].shape == (2, 1000)  # what the facade's self.path(s) gives plot_trajectory: x row, y row
        else:
            assert ep is None
    assert venv.get_attr("last_episode", 1) == [None] and isinstance(venv.get_attr("last_episode", [0])[0], dict)
    assert plain.get_attr("last_episode") == [None] * n


@pytest.mark.gpu
def test_facade_path_taken(lib):
    from gym_auv_b200 import make

    env = make("MovingObstaclesNoRules-v0")
    env.seed(4)
    env.reset()
    rng = np.random.RandomState(1)
    pos = [env.vessel.position.copy()]
    for _ in range(300):
        _, _, done, _ = env.step(rng.uniform([0.2, -0.15], [1, 0.15]))
        pos.append(env.vessel.position.copy())
        if done:
            break
    t = env.t_step
    env.reset()
    pt = env.last_episode["path_taken"]
    assert pt.shape == (t + 1, 2)
    assert np.array_equal(pt[0], pos[0])
    assert np.array_equal(pt[1:], np.asarray(pos[1:t + 1]).astype(np.float32).astype(np.float64))
    assert env.last_episode["obstacles"]["moving_path_taken"].shape[0] == t + 1
    assert env.last_episode["path"].shape == (2, 1000) and not env.last_episode["truncated"]


@pytest.mark.gpu
def test_facade_truncated_test_mode_episode(lib):
    """In test_mode the time limit is off, so an episode can outgrow the track (max_timesteps steps): the
    facade's last_episode then says so and numbers its rows."""
    import torch  # noqa: F401
    from gym_auv_b200 import Config, make

    cfg = Config()
    cfg.episode.max_timesteps = 50
    env = make("PathFollowNoObstacles-v0", cfg, test_mode=True)  # nothing to collide with
    pos = [env.vessel.position.copy()]
    for _ in range(80):
        _, _, done, _ = env.step([0.0, 0.1])  # no thrust: the vessel turns on the spot
        assert not done
        pos.append(env.vessel.position.copy())
    env.reset()
    le = env.last_episode
    assert le["truncated"] and le["path_taken"].shape == (50, 2) and list(le["step_index"]) == list(range(31, 81))
    assert np.array_equal(le["path_taken"], np.asarray(pos[31:81]).astype(np.float32).astype(np.float64))


@pytest.mark.gpu
def test_ray_test_counter_and_tracks_are_exclusive(lib):
    """The ray-test counting kernels do not record: asking for both raises, and an env that records has no
    seg_tests output to read a constant 0 from."""
    from gym_auv_b200.vec_env import AUVVecEnv

    scn = S.path_follow_no_obstacles(8, seed=1, n_paths=2)
    with pytest.raises(ValueError, match="count_ray_tests"):
        AUVVecEnv(scn, 8, _cfg(), debug=True, record_tracks=2)
    env = AUVVecEnv(scn, 8, _cfg(), debug=True, count_ray_tests=False, record_tracks=2)
    with pytest.raises(AttributeError):
        env.get_attr("seg_tests")
    assert env.get_attr("lidar_dist").shape == (8, 180)  # the rest of debug stays
    counted = AUVVecEnv(scn, 8, _cfg(), debug=True)
    counted.reset()
    counted.step(__import__("torch").ones((8, 2), device="cuda"))
    assert counted.get_attr("seg_tests").shape == (1,)


@pytest.mark.gpu
def test_table_driven_obstacle_histories(lib):
    """A pool stepped with the general table-driven obstacle update (linear_tracks=False; the snapshot holds no
    mov_lin records): ``moving_path_taken`` is re-run from the host scenarios and equals ``obstacle_state()``
    read along the episode, for the finished and the running episode."""
    import torch
    from gym_auv_b200.vec_env import AUVVecEnv

    N = 256
    scn = S.moving_obstacles(2 * N, 5, 3, seed=8, n_paths=4)
    env = AUVVecEnv(scn, N, _cfg(60), auto_reset=True, linear_tracks=False, record_tracks=16)
    assert env.linear is None
    env.reset()
    tr = torch.as_tensor(env.tracked_envs, device="cuda")
    acts = _actions(N, 8, 5)
    obst, done = [env.obstacle_state()[0][tr].cpu().numpy()], []
    for t in range(170):
        env.step(acts[t % 8])
        done.append(env._out["done"][tr].cpu().numpy().astype(bool))
        obst.append(env.obstacle_state()[0][tr].cpu().numpy())
    obst, done = np.stack(obst), np.stack(done)
    checked = 0
    for k, e in enumerate(env.tracked_envs):
        eps = _episodes(done[:, k])
        last = env.last_episode(int(e))
        if eps:
            s0, s1 = eps[-1]
            m = s1 - s0 + 1
            used = scn.mov_width[last["scenario"]] > 0
            mp = last["obstacles"]["moving_path_taken"]
            assert mp.shape == (m + 1, int(used.sum()), 2)
            assert np.abs(mp[:m] - obst[s0:s1 + 1, k][:, used]).max() <= 1e-9
            checked += 1
        cur = env.current_episode(int(e))
        s0 = eps[-1][1] + 1 if eps else 0
        used = scn.mov_width[cur["scenario"]] > 0
        assert np.abs(cur["obstacles"]["moving_path_taken"] - obst[s0:, k][:, used]).max() <= 1e-9
    assert checked >= 8
