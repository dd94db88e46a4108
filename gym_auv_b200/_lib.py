"""ctypes binding of the C ABI in include/auv_b200.h (libauv_b200.so, built in-tree by
``gym_auv_b200/build.py``).  There is NO fallback: if the shared library is missing or
its ABI version differs, importing the compute path raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# AUV_B200_LIB loads a library built elsewhere, e.g. the -DAUV_DEBUG_BOUNDS build of the tests
LIB_PATH = os.environ.get("AUV_B200_LIB", os.path.join(_HERE, "libauv_b200.so"))
ABI_VERSION = 22
REC_BYTES = 80
MAX_POLY_VERTS = 192
STATUS_REC_OVERFLOW = 1
STATUS_GEN_GAVE_UP = 2
STATUS_POLY_TOO_LARGE = 4
STATUS_PATH_TOO_LONG = 8
STATUS_BOUNDS = 16
STATUS_GEN_LAND_BLOCKED = 32
PP_W = 12
PATH_STAGE_BLOCKS = 512
NAV_W = 24
N_STATS = 16
STAT_NAMES = [
    "episodes",
    "reward",
    "reward_sq",
    "progress",
    "collisions",
    "reached_goal",
    "timesteps",
    "cross_track_error",
    "pathlength",
    "steps",
]

# render palette (0xRRGGBB) and frame constants, AUV_RGB_* / AUV_RENDER_* in include/auv_b200.h (rule at AuvRender)
RGB_OWNSHIP = 0xF2C12E
RGB_RAY_HIT = 0xE4572E
RGB_RAY_CLEAR = 0x4F7CAC
RGB_MOVING = 0xD7263D
RGB_STATIC = 0x8E5572
RGB_GOAL = 0x3BB273
RGB_PATH = 0xF4F4F4
RGB_LAND = 0x6B8F3E
RGB_SEA = 0x0B2545
RENDER_SHIP_MIN_PX = 8
RENDER_GOAL_PX = 4
RENDER_PATH_HALF_PX = 1.0
RENDER_RAY_HALF_PX = 0.5
RENDER_MAX_DIM = 4096

OBSERVE_STEP = 0
OBSERVE_RESET = 1
REWARDER_IDS = {"colav": 0, "pathfollow": 1}
CULL_IDS = {"reference": 0, "exact": 1}
VELOCITY_IDS = {"zero": 0, "nearest": 1}

_vp = C.c_void_p


class AuvConfig(C.Structure):
    _fields_ = [
        ("t_step_size", C.c_double),
        ("thrust_max_auv", C.c_double),
        ("moment_max_auv", C.c_double),
        ("vessel_width", C.c_double),
        ("look_ahead_distance", C.c_double),
        ("sensor_range", C.c_double),
        ("min_goal_distance", C.c_double),
        ("min_path_progress", C.c_double),
        ("min_cumulative_reward", C.c_double),
        ("feasibility_width_multiplier", C.c_double),
        ("max_timesteps", C.c_int32),
        ("sensor_interval_load_obstacles", C.c_int32),
        ("n_sensors", C.c_int32),
        ("n_sectors", C.c_int32),
        ("use_lidar", C.c_int32),
        ("sensor_log_transform", C.c_int32),
        ("sensor_use_velocity_observations", C.c_int32),
        ("rewarder", C.c_int32),
        ("test_mode", C.c_int32),
        ("cull_mode", C.c_int32),
        ("auto_reset", C.c_int32),
        ("velocity_mode", C.c_int32),
    ]


class AuvRayTable(C.Structure):
    _fields_ = [("cos_sin", _vp), ("weight", _vp), ("sector", _vp), ("unit64", _vp), ("weight_sum", C.c_double)]


class AuvPathHdr(C.Structure):
    _fields_ = [
        ("v0", C.c_int32),
        ("nseg", C.c_int32),
        ("b0", C.c_int32),
        ("s0", C.c_int32),
        ("ox", C.c_double),
        ("oy", C.c_double),
        ("length", C.c_double),
        ("end_x", C.c_double),
        ("end_y", C.c_double),
        ("extent", C.c_double),
    ]


class AuvPathBank(C.Structure):
    _fields_ = [
        ("n_paths", C.c_int32),
        ("n_knots", C.c_int32),
        ("hdr", _vp),
        ("poly_xy", _vp),
        ("poly_cum", _vp),
        ("poly_f32", _vp),
        ("blk_chord", _vp),
        ("blk_dev", _vp),
        ("sb_chord", _vp),
        ("sb_dev", _vp),
        ("pp", _vp),
        ("sub_chord", _vp),
        ("sub_dev", _vp),
    ]


class AuvScenarioPool(C.Structure):
    _fields_ = [
        ("n_scenarios", C.c_int32),
        ("k_moving", C.c_int32),
        ("k_static", C.c_int32),
        ("n_world", C.c_int32),
        ("path_id", _vp),
        ("vessel_init", _vp),
        ("mov_start", _vp),
        ("mov_width", _vp),
        ("mov_track", _vp),
        ("mov_pos0", _vp),
        ("mov_disp0", _vp),
        ("mov_counter0", _vp),
        ("vel_table", _vp),
        ("st_pos", _vp),
        ("st_radius", _vp),
        ("st_rec", _vp),
        ("mov_lin", _vp),
        ("linear_tracks", C.c_int32),
        ("lin_first_wrap", C.c_int32),
        ("lin_wrap_period", C.c_int32),
        ("reserved0", C.c_int32),
        ("world_circle", _vp),
        ("world_voff", _vp),
        ("world_verts", _vp),
        ("world_cell_off", _vp),
        ("world_cell_items", _vp),
        ("world_grid_x0", C.c_double),
        ("world_grid_y0", C.c_double),
        ("world_grid_cell", C.c_double),
        ("world_grid_nx", C.c_int32),
        ("world_grid_ny", C.c_int32),
        ("reset_obs", _vp),
        ("reset_max_progress", _vp),
        ("reset_mask", _vp),
    ]


class AuvBatch(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32),
        ("mask_words", C.c_int32),
        ("env_offset", C.c_int32),
        ("reset_stride", C.c_int32),
        ("scn_id", _vp),
        ("episode", _vp),
        ("state", _vp),
        ("step_counter", _vp),
        ("t_step", _vp),
        ("cum_reward", _vp),
        ("max_progress", _vp),
        ("cte_sum", _vp),
        ("nearby_mask", _vp),
        ("mov_pos", _vp),
        ("mov_disp", _vp),
        ("mov_counter", _vp),
        ("nav", _vp),
        ("rec", _vp),
        ("rec_cnt", _vp),
        ("status", _vp),
        ("rec_cap", C.c_int32),
        ("reserved1", C.c_int32),
        ("obst_steps", _vp),
        ("prev_seg", _vp),
        ("env_pid", _vp),
    ]


class AuvStepOut(C.Structure):
    _fields_ = [
        ("obs", _vp),
        ("reward", _vp),
        ("done", _vp),
        ("collision", _vp),
        ("reached_goal", _vp),
        ("goal_distance", _vp),
        ("progress", _vp),
        ("lidar_dist", _vp),
        ("windows", _vp),
        ("terminal_obs", _vp),
        ("sector_min_dist", _vp),
        ("sector_feasible_dist", _vp),
        ("stats", _vp),
        ("seg_tests", _vp),
        ("episode_out", _vp),
        ("tracks", _vp),  # const AuvTracks* (host pointer), NULL = no recording
    ]


class AuvTracks(C.Structure):
    _fields_ = [("count", C.c_int32), ("stride", C.c_int32), ("capacity", C.c_int32), ("reserved0", C.c_int32),
                ("points", _vp), ("head", _vp), ("snap", _vp)]


TRACK_HEAD_W = 8  # int32 per row head: episode, steps recorded, finished, collision, reached goal, scenario, obstacle updates, 0


def track_snap_width(k_moving: int, k_static: int) -> int:
    """doubles per snapshot row of AuvTracks.snap: path id, vessel_init, mov_lin records, st_rec records"""
    return 4 + 8 * int(k_moving) + 4 * int(k_static)


class AuvGenParams(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("epoch", C.c_uint32),
        ("post_generate_update", C.c_int32),
        ("t_step_size", C.c_double),
        ("vessel_width", C.c_double),
        ("init_pos_jitter", C.c_double),
        ("mov_disp_std", C.c_double),
        ("mov_width_mean", C.c_double),
        ("mov_speed_lo", C.c_double),
        ("mov_speed_hi", C.c_double),
        ("st_disp_std", C.c_double),
        ("st_radius_mean", C.c_double),
        ("path_group", C.c_int32),
        ("path_period", C.c_int32),
        ("land_clearance", C.c_double),
    ]


class AuvRefreshScratch(C.Structure):
    _fields_ = [("seen_episode", _vp), ("ids", _vp), ("count", _vp), ("capacity", C.c_int32), ("reserved0", C.c_int32)]


class AuvPathBuild(C.Structure):
    _fields_ = [("hdr", _vp), ("poly_xy", _vp), ("poly_cum", _vp), ("poly_f32", _vp), ("blk_chord", _vp), ("blk_dev", _vp),
                ("sb_chord", _vp), ("sb_dev", _vp), ("pp", _vp), ("n_knots", C.c_int32), ("vcap", C.c_int32),
                ("sub_chord", _vp), ("sub_dev", _vp)]


class AuvCompact(C.Structure):
    _fields_ = [("head", _vp), ("mask", _vp), ("vals", _vp), ("counter", _vp), ("words", C.c_int32), ("capacity", C.c_int32)]


class AuvDelta(C.Structure):
    _fields_ = [("obs_host", _vp), ("shadow", _vp), ("shipped", _vp), ("gran", C.c_int32), ("reserved0", C.c_int32)]


class AuvRender(C.Structure):
    _fields_ = [("count", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("reserved0", C.c_int32),
                ("env_ids", _vp), ("half_width", C.c_double)]


EXPORTS = [
    "auv_abi_version",
    "auv_sizeof",
    "auv_last_error",
    "auv_obs_dim",
    "auv_obstacle_update",
    "auv_vessel_step",
    "auv_navigate",
    "auv_observe",
    "auv_reset",
    "auv_step",
    "auv_step_host",
    "auv_fma_probe",
    "auv_timer_create",
    "auv_timer_destroy",
    "auv_step_timed",
    "auv_timer_read",
    "auv_pipeline_create",
    "auv_pipeline_destroy",
    "auv_pipeline_graph_state",
    "auv_step_chunked",
    "auv_step_host_chunked",
    "auv_step_host_submit",
    "auv_generate_moving_obstacles",
    "auv_linear_wrap",
    "auv_pool_pack",
    "auv_obstacle_state",
    "auv_reset_cache_fill",
    "auv_refresh_finished",
    "auv_step_host_compact_submit",
    "auv_step_host_delta_submit",
    "auv_compact_expand",
    "auv_pathbank_build",
    "auv_random_curve_waypoints",
    "auv_render",
]

_lib = None


class AuvLibraryError(RuntimeError):
    pass


def load():
    """Load libauv_b200.so (once).  Raises AuvLibraryError if it is absent or stale."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AuvLibraryError(
            f"{LIB_PATH} not found: build it with `python -m gym_auv_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise AuvLibraryError(f"{LIB_PATH} does not export {name}")
    lib.auv_abi_version.restype = C.c_int
    lib.auv_last_error.restype = C.c_char_p
    lib.auv_obs_dim.argtypes = [C.POINTER(AuvConfig)]
    P = C.POINTER
    lib.auv_obstacle_update.argtypes = [P(AuvConfig), P(AuvScenarioPool), P(AuvBatch), _vp]
    lib.auv_vessel_step.argtypes = [P(AuvConfig), P(AuvBatch), _vp, _vp]
    lib.auv_observe.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), P(AuvStepOut), C.c_int, _vp,
    ]
    lib.auv_navigate.argtypes = [P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp]
    lib.auv_reset.argtypes = [P(AuvConfig), P(AuvScenarioPool), P(AuvBatch), _vp, _vp]
    lib.auv_step.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp, P(AuvStepOut), _vp,
    ]
    lib.auv_step_host.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp, _vp, P(AuvStepOut),
        _vp, _vp, _vp, _vp,
    ]
    lib.auv_pipeline_create.argtypes = [C.c_int]
    lib.auv_pipeline_create.restype = _vp
    lib.auv_pipeline_destroy.argtypes = [_vp]
    lib.auv_pipeline_destroy.restype = None
    lib.auv_pipeline_graph_state.argtypes = [_vp]
    lib.auv_step_chunked.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp, P(AuvStepOut), _vp,
        _vp, C.c_int,
    ]
    lib.auv_step_host_chunked.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp, _vp, P(AuvStepOut),
        _vp, _vp, _vp, _vp, _vp, C.c_int,
    ]
    lib.auv_step_host_submit.argtypes = lib.auv_step_host_chunked.argtypes
    lib.auv_generate_moving_obstacles.argtypes = [P(AuvGenParams), P(AuvPathBank), P(AuvScenarioPool), _vp, C.c_int, _vp, _vp]
    lib.auv_linear_wrap.argtypes = [C.c_double, C.c_double, C.c_int, P(C.c_int32), P(C.c_int32)]
    lib.auv_pool_pack.argtypes = [P(AuvConfig), P(AuvScenarioPool), _vp, C.c_int, _vp]
    lib.auv_obstacle_state.argtypes = [P(AuvConfig), P(AuvScenarioPool), P(AuvBatch), _vp, _vp, _vp, _vp]
    lib.auv_reset_cache_fill.argtypes = [P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch),
                                         P(AuvStepOut), _vp, C.c_int, C.c_int, _vp]
    lib.auv_refresh_finished.argtypes = [P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch),
                                         P(AuvBatch), P(AuvStepOut), P(AuvRefreshScratch), P(AuvGenParams), _vp]
    lib.auv_step_host_compact_submit.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp, _vp, P(AuvStepOut),
        P(AuvCompact), _vp, _vp, _vp, _vp, C.c_int,
    ]
    lib.auv_step_host_delta_submit.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp, _vp, P(AuvStepOut),
        P(AuvDelta), _vp, _vp, _vp, _vp, C.c_int,
    ]
    lib.auv_compact_expand.argtypes = [P(AuvConfig), C.c_int, P(AuvCompact), _vp, _vp, C.c_int]
    lib.auv_pathbank_build.argtypes = [_vp, _vp, _vp, C.c_int, P(AuvPathBuild), _vp, _vp]
    lib.auv_random_curve_waypoints.argtypes = [C.c_uint64, C.c_uint32, C.c_double, _vp, C.c_int, _vp, _vp, _vp]
    lib.auv_render.argtypes = [P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp,
                               P(AuvRender), _vp, _vp]
    lib.auv_timer_create.argtypes = [C.c_int]
    lib.auv_timer_create.restype = _vp
    lib.auv_timer_destroy.argtypes = [_vp]
    lib.auv_timer_destroy.restype = None
    lib.auv_step_timed.argtypes = [
        P(AuvConfig), P(AuvRayTable), P(AuvPathBank), P(AuvScenarioPool), P(AuvBatch), _vp, P(AuvStepOut), _vp,
        _vp, C.c_int,
    ]
    lib.auv_timer_read.argtypes = [_vp, C.c_int, P(C.c_float)]
    lib.auv_fma_probe.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, P(C.c_double)]
    ver = lib.auv_abi_version()
    if ver != ABI_VERSION:
        raise AuvLibraryError(f"ABI mismatch: library {ver}, binding {ABI_VERSION}; rebuild")
    lib.auv_sizeof.argtypes = [C.c_int]
    for i, st in enumerate([AuvConfig, AuvRayTable, AuvPathBank, AuvScenarioPool, AuvBatch, AuvStepOut, AuvGenParams,
                            AuvPathHdr, AuvRefreshScratch, AuvCompact, AuvPathBuild, AuvDelta, AuvTracks, AuvRender]):
        if lib.auv_sizeof(i) != C.sizeof(st):
            raise AuvLibraryError(f"struct layout mismatch for {st.__name__}: C {lib.auv_sizeof(i)} vs ctypes {C.sizeof(st)}")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().auv_last_error().decode("utf-8", "replace")
        raise AuvLibraryError(f"{what} failed (rc={rc}): {msg}")
