"""Sub-block capsules (8 segments) of the projection search: the tables contain their segments, both
builders lay them out alike, the device bank's slot size keeps every bulk-copied table 16 B aligned,
and the projection returns the same segment and arclength whether it starts from the previous step's
segment or searches from scratch, with or without sub-block tables."""
import ctypes as C

import numpy as np
import pytest

from gym_auv_b200.pathbank import (HDR_DTYPE, PATH_BLOCK, PATH_SUB, PATH_SUPER, DevicePathBank, PathBank, build_path,
                                   random_curve_waypoints)

torch = pytest.importorskip("torch")


def _contained(rel, nseg, chord, aux, span):
    """Every vertex of node b lies within its deviation of the rounded chord (and the deviation is not loose)."""
    n = (nseg + span - 1) // span
    assert chord.shape[0] >= n and aux.shape[0] >= n
    ch, ax = chord.astype(np.float64), aux.astype(np.float64)
    for b in range(n):
        v = rel[b * span:min((b + 1) * span, nseg) + 1]
        w = v - ch[b, :2]
        t = np.clip((w @ ch[b, 2:]) * ax[b, 0], 0, 1)
        d = np.linalg.norm(w - t[:, None] * ch[b, 2:], axis=1).max()
        assert d <= ax[b, 1], (span, b, d, ax[b, 1])
        assert ax[b, 1] <= d + 1e-2


def _waypoints():
    rng = np.random.RandomState(3)
    wps = [random_curve_waypoints(rng, 5, 400.0), np.array([[0.0, 3.05], [0.0, 0.0]]), np.array([[0.0, 40.0, 41.0], [0.0, 5.0, 30.0]])]
    return wps


def test_sub_capsules_contain_their_segments():
    for wp in _waypoints():
        t = build_path(wp)
        nseg = len(t.poly) - 1
        assert t.sub_chord.shape[0] == (nseg + PATH_SUB - 1) // PATH_SUB
        _contained(t.poly - t.origin, nseg, t.sub_chord, t.sub_dev, PATH_SUB)
    assert any((len(build_path(w).poly) - 1) % PATH_SUB for w in _waypoints())  # a partial last sub-block is covered


def test_host_bank_places_sub_tables_at_four_times_the_first_block():
    tables = [build_path(w) for w in _waypoints()]
    bank = PathBank(tables)
    hdr = bank.header_array()
    per = PATH_BLOCK // PATH_SUB
    assert bank.sub_chord.shape[0] == per * bank.blk_chord.shape[0] == bank.sub_dev.shape[0]
    for p, t in enumerate(tables):
        assert hdr["b0"][p] % 2 == 0 and hdr["s0"][p] % 2 == 0
        j = per * hdr["b0"][p]
        assert np.array_equal(bank.sub_chord[j:j + len(t.sub_chord)], t.sub_chord)
        assert np.array_equal(bank.sub_dev[j:j + len(t.sub_dev)], t.sub_dev)


def test_device_bank_rounds_vcap_to_even_superblock_slots():
    wp = [np.array([[0.0, 100.0], [0.0, 50.0]])]
    span = 2 * PATH_BLOCK * PATH_SUPER
    assert DevicePathBank(wp, vcap=3 * 512).vcap == 2048
    assert DevicePathBank(wp, vcap=40000).vcap % span == 0
    assert DevicePathBank(wp).vcap == 32768


def test_pathbank_build_refuses_odd_superblock_slots(built_lib):
    from gym_auv_b200 import _lib

    lib = _lib.load()
    p = C.c_void_p(256)  # the arguments are checked before any device work
    arrays = [256] * 9
    for vcap, sub in ((1536, (256, 256)), (512, (256, 256)), (2048, (256, None))):
        pb = _lib.AuvPathBuild(*arrays, 1000, vcap, *sub)
        assert lib.auv_pathbank_build(p, p, None, 1, C.byref(pb), None, None) == -1, (vcap, sub)  # AUV_EINVAL


@pytest.mark.gpu
def test_device_sub_tables_match_the_host_builder(built_lib):
    wps = [np.array([[0.0, 60.0, 120.0], [0.0, 40.0, -10.0]]), np.array([[0.0, 3.05], [0.0, 0.0]]),
           np.array([[0.0, 40.0, 41.0], [0.0, 5.0, 30.0]])]  # short enough for 2048-vertex slots
    bank = DevicePathBank(wps, vcap=3 * 512)  # 1.5 superblock slots per path before rounding
    arr = bank.device_arrays("cuda:0")
    torch.cuda.synchronize()
    hdr = arr["hdr"].cpu().numpy().view(HDR_DTYPE)
    per = PATH_BLOCK // PATH_SUB
    sc, sd = arr["sub_chord"].cpu().numpy(), arr["sub_dev"].cpu().numpy()
    for p, wp in enumerate(wps):
        ref = build_path(wp)
        h = hdr[p]
        nseg = int(h["nseg"])
        assert nseg == len(ref.poly) - 1 and h["b0"] % 2 == 0 and h["s0"] % 2 == 0
        n = len(ref.sub_chord)
        j = per * int(h["b0"])
        poly = arr["poly_xy"][p * bank.vcap:p * bank.vcap + nseg + 1].cpu().numpy()
        _contained(poly - np.array([h["ox"], h["oy"]]), nseg, sc[j:j + n], sd[j:j + n], PATH_SUB)
        assert np.abs(sc[j:j + n] - ref.sub_chord).max() <= 1e-4
        assert np.abs(sd[j:j + n] - ref.sub_dev).max() <= 1e-4


def _random_actions(T, M, seed):
    return np.random.RandomState(seed).uniform([-1, -0.15], [1, 0.15], size=(T, M, 2)).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["steps", "displaced", "path_ends", "no_sub_tables", "long_path"])
def test_warm_and_cold_search_give_identical_results(case, built_lib):
    """One env set projects as usual (warm: upper bound from the previous step's segment, sub-block
    pruning); its twin forgets the previous segment before every step, so it searches from scratch.
    The projection is an exact arg-min: segment, arclength and everything downstream are bit-identical.
    'displaced' moves the vessels 3 m (30 segments) along the path between steps,
    'path_ends' warm-starts from the first or the last segment of the path, 'no_sub_tables' steps a bank
    without sub-block tables, 'long_path' has more than AUV_PATH_STAGE_BLOCKS blocks."""
    from gym_auv_b200 import lidar_config, scenarios as S
    from gym_auv_b200.vec_env import AUVVecEnv

    cfg = lidar_config()
    if case == "long_path":
        wp = np.array([[0.0, 900.0, 1500.0, 2300.0], [0.0, 300.0, -200.0, 100.0]])
        scn = S._single(wp, vessel_init=np.array([20.0, -15.0, 0.4]), static=[((120.0, 60.0), 25.0)])
        assert scn.bank.tables[0].blk_dev.shape[0] > 512
        n = 1
    else:
        n = 128
        scn = S.moving_obstacles(n, 4, 4, seed=8, n_paths=4)
    e1 = AUVVecEnv(scn, n, cfg, test_mode=True, auto_reset=False, debug=True)
    e2 = AUVVecEnv(scn, n, cfg, test_mode=True, auto_reset=False, debug=True)
    if case == "no_sub_tables":
        e1.paths.sub_chord = None
        e1.paths.sub_dev = None
    assert torch.equal(e1.reset(), e2.reset())
    nseg = torch.as_tensor(e1._bank["hdr"].cpu().numpy().view(HDR_DTYPE)["nseg"].astype(np.int32), device="cuda")
    acts = torch.as_tensor(_random_actions(40, n, 2), device="cuda")
    warm = 0
    for t in range(40):
        if case == "displaced" and t % 4 == 1:
            chi = e1.get_attr("nav")[:, 1]
            for e in (e1, e2):
                e.state[0] += 3.0 * torch.cos(chi)
                e.state[1] += 3.0 * torch.sin(chi)
        if case == "path_ends" and t > 0:
            ends = nseg[e1._st["env_pid"].long()] - 1
            e1._st["prev_seg"].copy_(torch.where(torch.arange(n, device="cuda") % 2 == t % 2, ends, torch.zeros_like(ends)))
        warm += int((e1._st["prev_seg"] >= 0).sum())
        e2._st["prev_seg"].fill_(-1)
        o1, r1, d1, _ = e1.step(acts[t])
        o2, r2, d2, _ = e2.step(acts[t])
        assert torch.equal(e1._st["prev_seg"], e2._st["prev_seg"]), t
        assert torch.equal(e1.get_attr("nav")[:, :8], e2.get_attr("nav")[:, :8]), t
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2), t
    assert warm >= 30 * n
    e1.check_status()
    e2.check_status()
