/*
 * auv_b200.h -- C ABI of the B200-native batched gym-auv step path.
 *
 * This is the drop-in boundary for the reference's per-step hot path.  The reference
 * (krisbrud/gym-auv) is pure Python: its "FFI" for this path is the gym.Env method
 * surface, so each entry point below names the Python interface it replaces
 * (file:line under gym_auv/ in the reference):
 *
 *   auv_obstacle_update   <- BaseEnvironment._update            environment.py:386-392
 *                            BaseObstacle.update                objects/obstacles.py:44-51
 *                            VesselObstacle._update             objects/obstacles.py:195-215
 *   auv_vessel_step       <- Vessel.step                        objects/vessel/vessel.py:226-247
 *                            odesolver45                        objects/vessel/odesolver.py:2-47
 *                            Vessel._state_dot                  objects/vessel/vessel.py:561-570
 *   auv_navigate          <- Vessel.navigate                    objects/vessel/vessel.py:461-541
 *                            Path.get_closest_arclength etc.    objects/path.py:61-93
 *   auv_observe           <- BaseEnvironment.observe            environment.py:247-290
 *                            Vessel.navigate / Vessel.perceive  vessel.py:461-541 / 249-368
 *                            find_rays_to_simulate_for_obstacles, simulate_sensor
 *                                                               objects/vessel/sensor.py:74-97,140-159
 *                            ColavRewarder/PathFollowRewarder.calculate
 *                                                               objects/rewarder.py:167-241,78-140
 *                            BaseEnvironment._isdone            environment.py:375-384
 *                            BaseEnvironment.reset (auto-reset) environment.py:176-245
 *   auv_step              <- BaseEnvironment.step               environment.py:292-366
 *   auv_step_host         <- the same, called the way a NumPy VecEnv consumer does
 *                            (SubprocVecEnv.step, scripts/run.py:296): host buffers in/out.
 *
 * Rules of the ABI: plain C, plain pointers and sizes, no torch types.  Every pointer in
 * AuvPathBank / AuvScenarioPool / AuvBatch / AuvStepOut is a DEVICE pointer owned by the
 * caller (PyTorch owns the allocations; this library never allocates device memory except
 * the small staging buffers of auv_step_host).  Calls are asynchronous on the given
 * cudaStream_t (passed as void*; NULL = legacy default stream).  Functions return 0 on
 * success, a negative AUV_E* code for bad arguments, or a positive cudaError_t value; the
 * message is available from auv_last_error().  Nothing throws across the boundary.
 */
#ifndef AUV_B200_H
#define AUV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AUV_ABI_VERSION 22

#define AUV_EINVAL (-1)  /* bad argument / NULL pointer / unsupported size */
#define AUV_ENOTSUP (-2) /* feature not built */

#define AUV_REWARDER_COLAV 0      /* rewarder.py:143-241 */
#define AUV_REWARDER_PATHFOLLOW 1 /* rewarder.py:56-140  */

#define AUV_CULL_REFERENCE 0 /* replicate sensor.py:93 seam arithmetic exactly (default) */
#define AUV_CULL_EXACT 1     /* wrap both window ends: every obstacle in range is seen   */

#define AUV_VELOCITY_ZERO 0    /* LiDAR speed measurements are (0, 0): simulate_sensor at HEAD, sensor.py:140-159 */
#define AUV_VELOCITY_NEAREST 1 /* Rz(-angle - pi/2) (dx, dy) of the nearest obstacle a ray hits:
                                  simulate_sensor_brute_force, sensor.py:100-137 (feeds max(0, v_y) in
                                  rewarder.py:199-206 and the 2 R velocity channels of the observation) */

#define AUV_MAX_RAYS 1024
#define AUV_MAX_OBSTACLES 1024 /* moving + static slots per env */
#ifndef AUV_PATH_BLOCK
#define AUV_PATH_BLOCK 32     /* polyline segments per projection block */
#endif
#ifndef AUV_PATH_SUPER
#define AUV_PATH_SUPER 16     /* blocks per projection superblock (8 / 16 / 32 swept: profiles/r1j_variants.txt) */
#endif
#define AUV_PATH_SUB 8        /* polyline segments per sub-block (a block holds AUV_PATH_BLOCK / AUV_PATH_SUB of them) */
#define AUV_NAV_W 24          /* doubles per env in AuvBatch.nav */
#define AUV_REC_BYTES 80      /* bytes per obstacle record in AuvBatch.rec */
#define AUV_MAX_POLY_VERTS 192 /* vertices of one world polygon incl. the closing one */
#define AUV_STATUS_REC_OVERFLOW 1 /* AuvBatch.status bit: more nearby obstacles than rec_cap */
#define AUV_STATUS_GEN_GAVE_UP 2  /* scenario generator: an obstacle was placed after 100000 rejections */
#define AUV_STATUS_PATH_TOO_LONG 8 /* auv_pathbank_build: a path's 0.1 m polyline does not fit its slot (vcap) */
#define AUV_STATUS_BOUNDS 16 /* -DAUV_DEBUG_BOUNDS builds only: an index check of a step kernel failed */
#define AUV_STATUS_POLY_TOO_LARGE 4 /* a world polygon has more than AUV_MAX_POLY_VERTS vertices: it was skipped */
#define AUV_STATUS_GEN_LAND_BLOCKED 32 /* scenario generator: no vessel start clear of land in 4096 draws (last one kept) */
#ifndef AUV_PATH_STAGE_BLOCKS
#define AUV_PATH_STAGE_BLOCKS 512
#endif                            /* paths with at most this many projection blocks (~1.6 km) are searched from a
                                     shared-memory copy of their capsule tables (one bulk async copy per CTA) */
#define AUV_PP_W 12           /* doubles per PCHIP piece record in AuvPathBank.pp */

/* gym_auv/config.py field names (EpisodeConfig/SimulationConfig/VesselConfig).  POD. */
typedef struct AuvConfig {
  double t_step_size;           /* SimulationConfig.t_step_size            config.py:28  */
  double thrust_max_auv;        /* VesselConfig.thrust_max_auv             config.py:39  */
  double moment_max_auv;        /* VesselConfig.moment_max_auv             config.py:40  */
  double vessel_width;          /* VesselConfig.vessel_width               config.py:41  */
  double look_ahead_distance;   /* VesselConfig.look_ahead_distance        config.py:45  */
  double sensor_range;          /* VesselConfig.sensor_range               config.py:64  */
  double min_goal_distance;     /* EpisodeConfig.min_goal_distance         config.py:20  */
  double min_path_progress;     /* EpisodeConfig.min_path_progress         config.py:23  */
  double min_cumulative_reward; /* EpisodeConfig.min_cumulative_reward     config.py:16  */
  double feasibility_width_multiplier; /* VesselConfig.feasibility_width_multiplier config.py:42 */
  int32_t max_timesteps;        /* EpisodeConfig.max_timesteps             config.py:19  */
  int32_t sensor_interval_load_obstacles; /*                               config.py:56  */
  int32_t n_sensors;            /* n_sensors_per_sector * n_sectors        config.py:75  */
  int32_t n_sectors;            /*                                         config.py:58  */
  int32_t use_lidar;            /*                                         config.py:52  */
  int32_t sensor_log_transform; /*                                         config.py:65  */
  int32_t sensor_use_velocity_observations; /* appends 2*n_sensors zeros   config.py:60  */
  int32_t rewarder;             /* AUV_REWARDER_*                                       */
  int32_t test_mode;            /* BaseEnvironment(test_mode=...)    environment.py:32  */
  int32_t cull_mode;            /* AUV_CULL_*                                           */
  int32_t auto_reset;           /* VecEnv semantics: reset done envs inside the step    */
  int32_t velocity_mode;        /* AUV_VELOCITY_*                                       */
} AuvConfig;

/* Per-ray constants, built once on the host from the config (vessel.py:63-68,
 * rewarder.py:203-205, utils/sector_partitioning.py:4-9). */
typedef struct AuvRayTable {
  const double* cos_sin; /* [n_sensors][2]  cos/sin of body angle -pi+(i+1)*2pi/R       */
  const float* weight;   /* [n_sensors]     1/(1+|10*angle_i|)                          */
  const uint8_t* sector; /* [n_sensors]     sector index of ray i                       */
  const double* unit64;  /* [64][2] cos/sin(2 pi k / 64): vertices of buffer(r) (quadsegs 16,
                            obstacles.py:101-106)                                          */
  double weight_sum;     /* sum_i weight[i] (FP64, sequential order)                    */
} AuvRayTable;

/* Path bank: every distinct path (objects/path.py:19-40) tabulated once; envs refer to a
 * path by id.  Polyline = the 0.1 m LineString of path.py:38-40 (FP64), its chord-length
 * prefix sums, and per 32-segment block (and per AUV_PATH_SUPER-block superblock) a capsule
 * (chord + max deviation) used as an exact hierarchical search structure for
 * LineString.project (path.py:93).  PCHIP pieces are scipy PPoly coefficients (path.py:26).
 * Tables are laid out so that every dependent look-up of the step is ONE line: a 64 B header
 * per path, a 96 B record per PCHIP piece (its two knots and eight coefficients). */
typedef struct AuvPathHdr {
  int32_t v0;      /* first polyline vertex in poly_xy / poly_cum                          */
  int32_t nseg;    /* polyline segments (vertices - 1); blocks = ceil(nseg / AUV_PATH_BLOCK),
                      superblocks = ceil(blocks / AUV_PATH_SUPER)                           */
  int32_t b0;      /* first block capsule (even, so the tables can be bulk-copied); the path's
                      sub-block capsules start at (AUV_PATH_BLOCK / AUV_PATH_SUB) * b0       */
  int32_t s0;      /* first superblock capsule (even)                                       */
  double ox, oy;   /* origin the FP32 capsules are relative to                              */
  double length;   /* Path.length                                                           */
  double end_x, end_y; /* Path.end                                                          */
  double extent;   /* max |x - ox| + |y - oy| over the polyline: error bound of the FP32 copy     */
} AuvPathHdr;

typedef struct AuvPathBank {
  int32_t n_paths;
  int32_t n_knots;         /* 1000 */
  const AuvPathHdr* hdr;   /* [n_paths]                                                   */
  const double* poly_xy;   /* [total_vertices][2]                                       */
  const double* poly_cum;  /* [total_vertices] chord-length prefix sum at each vertex   */
  const float* poly_f32;   /* [total_vertices][2] the same vertices relative to the path's origin, FP32:
                              the projection screens segments on these 8 B vertices and evaluates in
                              FP64 only the few that can be the exact minimum                    */
  const float* blk_chord;  /* [total_blocks][4] ax, ay, ex, ey: first vertex and chord vector,
                              relative to the path's origin                             */
  const float* blk_dev;    /* [total_blocks][2] 1/|e|^2 (0 if degenerate), max vertex
                              deviation from the chord + fp pad                         */
  const float* sb_chord;   /* [total_superblocks][4] same layout as blk_chord            */
  const float* sb_dev;     /* [total_superblocks][2] same layout as blk_dev              */
  const double* pp;        /* [n_paths][n_knots-1][AUV_PP_W]: knot j, knot j+1, x: c0..c3,
                              y: c0..c3 (value = ((c0 t + c1) t + c2) t + c3, t = s - knot j),
                              2 unused                                                   */
  const float* sub_chord;  /* [total_blocks * AUV_PATH_BLOCK / AUV_PATH_SUB][4] capsules of AUV_PATH_SUB
                              segments, same layout as blk_chord; a path's table has
                              (AUV_PATH_BLOCK / AUV_PATH_SUB) x its block count entries.  Optional:
                              NULL (with sub_dev) only costs speed, the refine then evaluates
                              every segment of a candidate block                          */
  const float* sub_dev;    /* [total_blocks * AUV_PATH_BLOCK / AUV_PATH_SUB][2] same layout as blk_dev */
} AuvPathBank;

/* Scenario pool: the read-only part of what a scenario plug-in's _generate() produces
 * (envs/movingobstacles.py:28-95, envs/testscenario.py) for M scenarios, plus the state
 * a freshly reset env starts from.  Obstacle slot order: moving first, then static
 * circles (append order of movingobstacles.py:51-90).  width/radius <= 0 marks an
 * unused slot. */
typedef struct AuvScenarioPool {
  int32_t n_scenarios;
  int32_t k_moving;
  int32_t k_static;
  int32_t n_world;             /* shared static polygons (PolygonObstacle), 0 = none     */
  const int32_t* path_id;      /* [M]                                                   */
  const double* vessel_init;   /* [M][3] x, y, psi                                      */
  const double* mov_start;     /* [M][k_moving][2]  trajectory[0] (wrap target)         */
  const double* mov_width;     /* [M][k_moving]                                         */
  const int32_t* mov_track;    /* [M][k_moving][4]  vel_off, vel_len, vel_stride, 0     */
  const double* mov_pos0;      /* [M][k_moving][2]  position right after reset()        */
  const double* mov_disp0;     /* [M][k_moving][2]  last (dx,dy) right after reset()    */
  const double* mov_counter0;  /* [M][k_moving]     waypoint_counter after reset()      */
  const double* vel_table;     /* [n_vel][2] per-second velocities obstacles.py:160-172 */
  const double* st_pos;        /* [M][k_static][2]                                      */
  const double* st_radius;     /* [M][k_static]                                         */
  /* Packed per-slot records the step kernels read (one line per look-up).  Filled from the
   * arrays above by auv_pool_pack, or directly by auv_generate_moving_obstacles. */
  const double* st_rec;        /* [M][k_static][4]  x, y, radius, 0                      */
  const double* mov_lin;       /* [M][k_moving][8]  constant-velocity tracks: position right after
                                  reset() (2), per-step displacement dt*v (2), width, track start (2), 0 */
  /* linear_tracks = 1: every used moving slot follows a constant-velocity track of the same length
   * and the same post-reset counter (the MovingObstacles family, movingobstacles.py:51-75).  The
   * update of obstacles.py:195-215 then has a closed form in the number n of updates since reset:
   *   n <  lin_first_wrap : pos = pos0 + n d
   *   n >= lin_first_wrap : pos = start + ((n - lin_first_wrap) mod lin_wrap_period + 1) d
   * and the step keeps no per-env obstacle state (AuvBatch.mov_* are unused, may be NULL). */
  int32_t linear_tracks;
  int32_t lin_first_wrap;      /* auv_linear_wrap()                                      */
  int32_t lin_wrap_period;
  int32_t reserved0;
  /* static land polygons shared by every scenario of the pool (obstacles.py:116-127):
   * filled, enclosing circle = cached enclosing_circle_of_shape (obstacles.py:235-262).
   * Slots K .. K+n_world-1 of the nearby list / windows output. */
  const double* world_circle;  /* [n_world][3] cx, cy, rho                              */
  const int32_t* world_voff;   /* [n_world+1] first vertex of each closed ring          */
  const double* world_verts;   /* [total][2]  rings, last vertex repeats the first      */
  /* broad phase of the nearby-list refresh over the world (vessel.py:266-273 asks every obstacle):
   * a uniform grid over the enclosing circles -- polygon j is listed in every cell its circle
   * overlaps; a query visits the cells the own-ship's detection disc overlaps and runs the exact
   * distance test only on the polygons listed there.  NULL world_cell_off = test every polygon. */
  const int32_t* world_cell_off;   /* [nx ny + 1] CSR offsets into world_cell_items, cell = iy nx + ix */
  const int32_t* world_cell_items; /* polygon indices                                       */
  double world_grid_x0, world_grid_y0, world_grid_cell; /* origin of cell (0, 0) and the cell size */
  int32_t world_grid_nx, world_grid_ny;
  /* what reset() returns depends on the scenario only: with auto_reset these caches (filled
   * once by running auv_reset + auv_observe(RESET) over the pool) turn the in-step reset of
   * a finished env into a copy */
  const float* reset_obs;            /* [M][obs_dim] first observation of each scenario        */
  const double* reset_max_progress;  /* [M]          Vessel._max_progress after that observe    */
  const uint32_t* reset_mask;        /* [M][mask_words] nearby list loaded by that observe      */
} AuvScenarioPool;

/* Mutable per-env state (SoA).  N = n_envs. */
typedef struct AuvBatch {
  int32_t n_envs;
  int32_t mask_words;     /* ceil((k_moving+k_static+n_world)/32), <= 32               */
  int32_t env_offset;     /* global index of env 0 (multi-GPU shards), used by reset    */
  int32_t reset_stride;   /* a finished env moves from scenario s to (s + reset_stride) mod M;
                             0 = n_envs.  Batches that split one env population (two groups
                             stepped alternately) keep the stride of the whole population       */
  int32_t* scn_id;        /* [N]   scenario each env currently runs                     */
  int32_t* episode;       /* [N]   BaseEnvironment.episode                              */
  double* state;          /* [6][N] x, y, psi, u, v, r   (Vessel._state)                */
  int32_t* step_counter;  /* [N]   Vessel._step_counter                                 */
  int32_t* t_step;        /* [N]   BaseEnvironment.t_step                               */
  double* cum_reward;     /* [N]   BaseEnvironment.cumulative_reward                    */
  double* max_progress;   /* [N]   Vessel._max_progress                                 */
  double* cte_sum;        /* [N]   sum |cross_track_error|*100 over the episode         */
  uint32_t* nearby_mask;  /* [N][mask_words] Vessel._nearby_obstacles membership        */
  double* mov_pos;        /* [N][k_moving][2]                                           */
  double* mov_disp;       /* [N][k_moving][2]                                           */
  double* mov_counter;    /* [N][k_moving]                                              */
  double* nav;            /* [N][AUV_NAV_W] Vessel._last_navi_state_dict (vessel.py:518-539):
                             [0] s, [1] chi, [2] y_e, [3] s_la, [4] look_ahead_heading_error,
                             [5] heading_error, [6] goal_distance, [7] progress;
                             [8..23] = the 128 B hand-over line the casting stage reads in one
                             coalesced load: cos psi, sin psi, reached_goal, y_e, the part of the
                             reward that does not depend on the LiDAR (rewarder.py:216-239 without
                             the closeness term / rewarder.py:118-140), goal_distance, progress,
                             (unused), x, y, psi, cumulative reward, cte sum, t_step, scenario id,
                             record count                                                       */
  /* scratch between the culling stage and the ray-casting stage (opaque to the caller) */
  void* rec;              /* [N][rec_cap][AUV_REC_BYTES] obstacle records, 16-byte aligned       */
  int32_t* rec_cnt;       /* [N] records of each env                                            */
  int32_t* status;        /* [1] or NULL: AUV_STATUS_* bits raised by kernels                   */
  int32_t rec_cap;        /* records per env; >= k_moving+k_static+n_world can never overflow  */
  int32_t reserved1;
  int32_t* obst_steps;    /* [N] obstacle updates since reset (environment.py:386-392 calls)    */
  int32_t* prev_seg;      /* [N] polyline segment the last projection ended on, -1 = none:
                             warm start of the next one (an upper bound only; the search stays exact) */
  int32_t* env_pid;       /* [N] pool.path_id[scn_id[e]], cached by reset                       */
} AuvBatch;

/* Episode tracks of a sample of the batch (the path_taken / obstacle histories of
 * BaseEnvironment.save_latest_episode, environment.py:466-489), recorded by the step kernel.
 * Env e is tracked iff e % stride == 0 && e / stride < count; its track slot is t = e / stride.
 * Each slot has two rows, p = 0 and 1: an episode with counter ep (AuvBatch.episode before any
 * reset in the step) writes row p = ep & 1, so the row of the episode an env just finished stays
 * intact for the whole of its next episode, which writes the other row.  Every AUV_OBSERVE_STEP
 * writes, for each tracked env, the point of the step and rewrites the row's head; the step in
 * which the episode ends also copies the scenario it ran on into the row's snapshot (the pool slot
 * may be regenerated later, auv_refresh_finished).  All buffers are device memory.
 *   points [count][2][capacity] float4: x, y, psi after the step, reward of the step, at index
 *          t_step % capacity (t_step = steps before this one): an episode longer than capacity
 *          keeps its last capacity points
 *   head   [count][2][8] int32: episode counter, steps recorded (t_step + 1), finished flag,
 *          collision, reached goal, scenario id, obstacle updates since reset, 0
 *   snap   [count][2][4 + 8 k_moving + 4 k_static] double: pool path_id, vessel_init (3), then each
 *          moving slot's pool.mov_lin record (8; zeros without linear_tracks) and each static slot's
 *          pool.st_rec record (4) -- valid once the row's finished flag is set */
typedef struct AuvTracks {
  int32_t count;    /* K >= 1 tracked envs                                             */
  int32_t stride;   /* >= 1, (count - 1) * stride < n_envs                             */
  int32_t capacity; /* T >= 1 points kept per episode                                  */
  int32_t reserved0;
  float* points;    /* 16-byte aligned (one float4 store per point)                   */
  int32_t* head;    /* 16-byte aligned (a row is written as two 16-byte stores)        */
  double* snap;     /* 8-byte aligned                                                  */
} AuvTracks;

/* Outputs of one step / observe (all optional except obs/reward/done). */
typedef struct AuvStepOut {
  float* obs;            /* [N][obs_dim]  obs_dim = 6 (+ n_sensors (+ 2 n_sensors))     */
  float* reward;         /* [N]                                                         */
  uint8_t* done;         /* [N]                                                         */
  uint8_t* collision;    /* [N] info["collision"]                                       */
  uint8_t* reached_goal; /* [N] info["reached_goal"]                                    */
  float* goal_distance;  /* [N] info["goal_distance"]                                   */
  float* progress;       /* [N] info["progress"]                                        */
  float* lidar_dist;     /* [N][n_sensors] or NULL: latest distance measurements        */
  int32_t* windows;      /* [N][K+n_world][2] or NULL: culling (a, b) per slot (debug)  */
  float* terminal_obs;   /* [N][obs_dim] or NULL: last obs of a finished episode        */
  float* sector_min_dist;      /* [N][n_sectors] or NULL: closest range per sector (sector map of
                                  utils/sector_partitioning.py:4-9), warp-shuffle min-pooling    */
  float* sector_feasible_dist; /* [N][n_sectors] or NULL: LidarPreprocessor._feasibility_pooling
                                  (sensor.py:251-296) per sector                                  */
  double* stats;         /* [AUV_N_STATS] or NULL: episode-statistic accumulators       */
  unsigned long long* seg_tests; /* [1] or NULL: reference-semantics ray/segment tests  */
  float* episode_out;    /* [N][8] or NULL: the env.history entry (environment.py:476-489) of the
                            episode an env finished in this step (rows of envs with done = 1):
                            reward, timesteps, progress, collision, reached_goal, mean
                            cross-track error, path length, episode number                      */
  const AuvTracks* tracks; /* HOST pointer to the track descriptor, or NULL = no recording: a
                            zero-initialised AuvStepOut records nothing.  Validated by every step
                            entry point before any device work (AUV_EINVAL): NULL buffers, count /
                            stride / capacity < 1, (count - 1) * stride >= n_envs, misaligned
                            points / head / snap, and tracks together with seg_tests (the ray-test
                            counting kernels do not record: set one or the other)              */
} AuvStepOut;

/* indices into AuvStepOut.stats (mirrors env.history keys, environment.py:476-489) */
#define AUV_STAT_EPISODES 0
#define AUV_STAT_REWARD 1
#define AUV_STAT_REWARD_SQ 2
#define AUV_STAT_PROGRESS 3
#define AUV_STAT_COLLISIONS 4
#define AUV_STAT_REACHED_GOAL 5
#define AUV_STAT_TIMESTEPS 6
#define AUV_STAT_CROSS_TRACK 7
#define AUV_STAT_PATHLENGTH 8
#define AUV_STAT_STEPS 9
#define AUV_N_STATS 16

/* observe modes */
#define AUV_OBSERVE_STEP 0  /* observe + reward + done (+ auto-reset): tail of step()    */
#define AUV_OBSERVE_RESET 1 /* observe only: what reset() returns (no reward/done)       */

int auv_abi_version(void);
/* sizeof of the ABI structs, in declaration order (0 AuvConfig, 1 AuvRayTable, 2 AuvPathBank,
 * 3 AuvScenarioPool, 4 AuvBatch, 5 AuvStepOut, 6 AuvGenParams, 7 AuvPathHdr, 8 AuvRefreshScratch, 9 AuvCompact,
 * 10 AuvPathBuild, 11 AuvDelta, 12 AuvTracks) so a binding
 * can verify its layout. */
int auv_sizeof(int which);
const char* auv_last_error(void);
int auv_obs_dim(const AuvConfig* cfg);

int auv_obstacle_update(const AuvConfig* cfg, const AuvScenarioPool* pool, AuvBatch* batch,
                        void* stream);
int auv_vessel_step(const AuvConfig* cfg, AuvBatch* batch, const float* actions /*[N][2]*/,
                    void* stream);
/* Vessel.navigate for every env (fills AuvBatch.nav / max_progress) and, with use_lidar, the
 * culling stage of Vessel.perceive (nearby list, ray windows -> AuvBatch.rec); auv_observe
 * calls it. */
int auv_navigate(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                 const AuvScenarioPool* pool, AuvBatch* batch, void* stream);
int auv_observe(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                const AuvScenarioPool* pool, AuvBatch* batch, AuvStepOut* out, int mode,
                void* stream);
/* Put envs [0,N) whose reset_mask[e] != 0 (or all when NULL) into the post-reset() state
 * of scenario scn_id[e] (does not compute the observation: call auv_observe(RESET)). */
int auv_reset(const AuvConfig* cfg, const AuvScenarioPool* pool, AuvBatch* batch,
              const uint8_t* reset_mask, void* stream);
/* One full env.step() for the whole batch: update -> vessel -> observe/reward/done. */
int auv_step(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
             const AuvScenarioPool* pool, AuvBatch* batch, const float* actions,
             AuvStepOut* out, void* stream);
/* Same with HOST buffers: actions_host -> device, step, obs/reward/done -> host.  The
 * device staging lives in `out` / `actions_dev`; host pointers should be pinned. */
int auv_step_host(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                  const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                  float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                  uint8_t* done_host, void* stream);
/* Chunked step.  Envs are independent (environment.py:292-366 touches one env only), so the
 * batch can be cut into n_chunks env ranges.  auv_step_chunked runs the ranges on the
 * pipeline's own streams (round robin), forking from `stream` and joining back into it.
 * auv_step_host_chunked computes the ranges in order on `stream` and sends each range's
 * observations to the host on the pipeline's copy stream as soon as the range is done, so the
 * D2H of the observations (what bounds the host-buffer step) overlaps the remaining kernels;
 * n_chunks <= 64.  Results are identical to auv_step / auv_step_host; work submitted to
 * `stream` afterwards sees the whole step.  A pipeline holds n_streams (1..16) non-blocking
 * streams + events, no device memory. */
typedef struct AuvPipeline AuvPipeline;
AuvPipeline* auv_pipeline_create(int n_streams);
void auv_pipeline_destroy(AuvPipeline* p);
/* 1: auv_step_host_chunked replays an instantiated CUDA graph (one launch per step; re-captured
 * when an argument changes), 0: nothing captured yet, -1: direct submission (capture was not
 * possible, or AUV_B200_NO_GRAPH is set in the environment). */
int auv_pipeline_graph_state(const AuvPipeline* p);
int auv_step_chunked(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                     const AuvScenarioPool* pool, AuvBatch* batch, const float* actions,
                     AuvStepOut* out, void* stream, AuvPipeline* p, int n_chunks);
int auv_step_host_chunked(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                          const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                          float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                          uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks);
/* auv_step_host_chunked without the final synchronise: the step is only submitted to `stream`;
 * the host buffers are valid once `stream` has drained (VecEnv.step_async / step_wait,
 * stable-baselines' asynchronous interface).  Two env groups on two streams keep the link busy:
 * group A's observations travel while group B is computed. */
int auv_step_host_submit(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                         const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                         float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                         uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks);
/* Lossless COMPACT host step.  The dense observation rows are what bounds the host-buffer step
 * (4 (6 + R) B per env over PCIe) although ~85 % of a row is exactly 0 (rays that read clear).
 * auv_step_host_compact_submit is auv_step_host_submit with the D2H copies replaced by a kernel
 * (k_obs_ship) that writes, straight into PINNED host memory: per env a 32 B head (obs[0..5], the
 * number of non-zero closeness values, their offset in `vals`), the hit mask (one bit per ray) and
 * the non-zero values packed back to back; reward / done go to reward_host / done_host the same way
 * (all host pointers must be pinned, i.e. device-accessible).  Once `stream` has drained,
 * auv_compact_expand scatters them into the caller's dense [N][obs_dim] array with n_threads host
 * threads; prev_mask ([N][words], zero-initialised, owned by the caller together with the dense
 * array) remembers which entries are non-zero so that only changes are touched.  Results are
 * bit-identical to auv_step_host.  Not available with sensor_use_velocity_observations. */
typedef struct AuvCompact {
  float* head;      /* [N][8]       pinned host                                          */
  uint32_t* mask;   /* [N][words]   pinned host                                          */
  float* vals;      /* [capacity]   pinned host                                          */
  int32_t* counter; /* [1]          device                                               */
  int32_t words;    /* ceil(n_sensors / 32)                                              */
  int32_t capacity; /* floats in vals, >= N * words * 32                                 */
} AuvCompact;
int auv_step_host_compact_submit(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                                 const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                                 float* actions_dev, AuvStepOut* out, const AuvCompact* cb, float* reward_host,
                                 uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks);
int auv_compact_expand(const AuvConfig* cfg, int n_envs, const AuvCompact* cb, uint32_t* prev_mask, float* obs_host,
                       int n_threads);
/* Lossless DELTA host step: no host-side work at all.  The caller's dense [N][obs_dim] observation
 * array lives in PINNED host memory and persists from step to step; the device keeps a shadow copy of
 * what that array holds.  After each env range is computed, k_obs_delta compares the new rows with
 * the shadow in chunks of `gran` floats (8, 16 or 32: 32 / 64 / 128 B) and stores ONLY the chunks that
 * differ -- bitwise -- straight into the host array (and the shadow); reward / done are stored whole.
 * ~85 % of a row is 0 step after step (rays that read clear), so ~1/4 of the dense bytes cross the
 * link and the host array is complete the moment the stream drains.  Both arrays must start equal
 * (e.g. zero-filled).  Works with every observation layout (velocity channels included).  Results
 * are bit-identical to auv_step_host.  `shipped` accumulates the number of chunks stored. */
typedef struct AuvDelta {
  float* obs_host;              /* [N][obs_dim] pinned host, 16 B aligned                  */
  float* shadow;                /* [N][obs_dim] device, 16 B aligned                       */
  unsigned long long* shipped;  /* [1] device, cumulative chunks stored (NULL: not counted) */
  int32_t gran;                 /* floats per chunk: 8, 16 or 32                           */
  int32_t ctas;                 /* CTAs of the (link-bound, persistent) kernel; 0 = two per SM */
} AuvDelta;
int auv_step_host_delta_submit(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                               const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                               float* actions_dev, AuvStepOut* out, const AuvDelta* d, float* reward_host,
                               uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks);
/* Per-kernel CUDA-event timing of a step on the launching stream (used by bench.py for the
 * roofline of the dominant kernel).  A timer holds `capacity` slots of 4 events. */
typedef struct AuvTimer AuvTimer;
AuvTimer* auv_timer_create(int capacity);
void auv_timer_destroy(AuvTimer* t);
/* auv_step on ONE stream with events recorded around each of its kernels. */
int auv_step_timed(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                   const AuvScenarioPool* pool, AuvBatch* batch, const float* actions,
                   AuvStepOut* out, void* stream, AuvTimer* t, int slot);
/* after the stream is synchronised: ms[0..2] = k_vessel_nav, k_nav_cull, k_lidar */
int auv_timer_read(AuvTimer* t, int slot, float* ms);
/* GPU-side scenario generation for the MovingObstacles family (SURVEY.md section 8f rank 1):
 * what MovingObstacles._generate (envs/movingobstacles.py:28-95) and helpers.generate_obstacle
 * (utils/helpers.py:5-35) sample per episode -- path choice from the bank, vessel start
 * (path(0) + jitter, heading dir(0) + U(-pi, pi)), per obstacle slot the rejection-sampled
 * position (normal displacement from a uniform arclength in [0.1 L, 0.9 L], clear of the vessel
 * and of the goal), radius / width max(1, Poisson(mean)), and for moving obstacles direction
 * U(0, 2 pi) and speed U(lo, hi) -- for the listed scenarios of the pool, with counter-based
 * Philox4x32-10 streams keyed by (seed; scenario, slot, epoch): same arguments, same scenarios.
 * Every slot of a listed scenario is (re)generated as "used".
 * In a pool with a shared world of land polygons (n_world > 0) every placed object must also be CLEAR OF
 * LAND BY d -- outside every polygon (even-odd rule on the closed ring) and at an FP64 distance > d from
 * every ring: the vessel start by gp->land_clearance (else jitter and heading are redrawn from the same
 * stream; after 4096 draws AUV_STATUS_GEN_LAND_BLOCKED is raised and the last draw kept), a static circle's
 * centre by its radius and a moving obstacle's track start by its width (both redrawn inside the rejection
 * loop above).  Paths, goals and the later course of moving obstacles are not tested.  When no draw is
 * rejected by land the Philox draws are those of a pool without a world. */
typedef struct AuvGenParams {
  uint64_t seed;
  uint32_t epoch;               /* bump to draw a fresh scenario for the same pool slot      */
  int32_t post_generate_update; /* _generate() ends with self._update()  movingobstacles.py:95 */
  double t_step_size;           /* dt of that update                                         */
  double vessel_width;          /* config.py:41                                              */
  double init_pos_jitter;       /* 50    movingobstacles.py:35                               */
  double mov_disp_std;          /* 500   movingobstacles.py:58                               */
  double mov_width_mean;        /* 10    movingobstacles.py:59                               */
  double mov_speed_lo;          /* 1     movingobstacles.py:65                               */
  double mov_speed_hi;          /* 3                                                         */
  double st_disp_std;           /* 250   movingobstacles.py:84                               */
  double st_radius_mean;        /* 30    helpers.py:11                                       */
  /* path of scenario slot m: path_group = 0 -> uniform over the bank (a fresh random curve per
   * episode, movingobstacles.py:28-31); > 0 -> ((m mod path_period) / path_group) mod n_paths, i.e.
   * "paths shared by index" with consecutive slots on the same path (path-major pools: the step
   * kernels then find whole CTAs on one path) */
  int32_t path_group;
  int32_t path_period;
  /* pools with a shared land-polygon world (n_world > 0): the vessel start must be clear of land by
   * land_clearance (0 = only outside every polygon).  See auv_generate_moving_obstacles. */
  double land_clearance;
} AuvGenParams;
/* Writes path_id, vessel_init, mov_start, mov_width, mov_track, vel_table (entry m*Km+j), the
 * post-reset obstacle state mov_pos0/disp0/counter0, st_pos and st_radius of the scenarios
 * ids[0..n_ids) (device array; NULL = scenarios 0..n_ids-1).  The pool's arrays must be writable
 * device memory with vel_table holding n_scenarios * k_moving entries.  The reset cache of those
 * scenarios is stale afterwards: refill it with auv_reset + auv_observe(AUV_OBSERVE_RESET).
 * status (device int or NULL) receives AUV_STATUS_GEN_GAVE_UP and AUV_STATUS_GEN_LAND_BLOCKED.  With
 * n_world > 0 the pool's world_circle / world_voff / world_verts (and, when set, its grid) are read. */
int auv_generate_moving_obstacles(const AuvGenParams* gp, const AuvPathBank* paths, const AuvScenarioPool* pool,
                                  const int32_t* ids, int n_ids, int32_t* status, void* stream);
/* Fill the reset cache (pool.reset_obs / reset_max_progress / reset_mask) of n <= worker->n_envs
 * scenarios -- ids[0..n) (device array) or first..first+n-1 when ids is NULL -- by running
 * reset() + the first observe() (environment.py:176-245) for them on a caller-owned WORKER batch
 * (any AuvBatch / AuvStepOut of at least n envs sharing the pool; its contents are overwritten). */
int auv_reset_cache_fill(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                         const AuvScenarioPool* pool, AuvBatch* worker, AuvStepOut* worker_out, const int32_t* ids,
                         int first, int n, void* stream);
/* Sustained fresh scenarios without a host round trip (the reference draws a new scenario in every
 * reset(), envs/movingobstacles.py:28-95).  Pool of exactly 2 N scenarios: env e alternates between
 * slots e and e + N at every auto-reset, so the slot it is NOT running is free.  One call, all on
 * `stream`: every env whose episode counter moved since the last call lists the slot it vacated
 * (at most `capacity` per call, the rest next time), those slots get freshly generated scenarios
 * (auv_generate_moving_obstacles semantics, Philox streams keyed by gp->seed / gp->epoch -- bump the
 * epoch per call) and their cached first observation is recomputed on the worker batch.  Pools with a
 * shared land-polygon world are refreshed under the same land rule; live->status receives the generator's
 * status bits. */
typedef struct AuvRefreshScratch {
  int32_t* seen_episode; /* [N] episode counter of each env at the last call (zero-initialised)   */
  int32_t* ids;          /* [capacity] pool slots being regenerated (zero-initialised)            */
  int32_t* count;        /* [1]                                                                   */
  int32_t capacity;      /* <= worker->n_envs                                                     */
  int32_t reserved0;
} AuvRefreshScratch;
int auv_refresh_finished(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                         const AuvScenarioPool* pool, const AuvBatch* live, AuvBatch* worker, AuvStepOut* worker_out,
                         const AuvRefreshScratch* rs, const AuvGenParams* gp, void* stream);
/* Device-side construction of path-bank entries (SURVEY.md section 8 f-1): what
 * gym_auv.objects.path.Path.__init__ (path.py:19-40) computes with SciPy -- three rounds of
 * chord-length re-parametrisation through PCHIP resampled at 1000 points, the 0.1 m polyline --
 * plus the tables of AuvPathBank (PPoly piece records, chord-length prefix sums, FP32 polyline,
 * block / superblock capsules, header), one CTA per path, SciPy's / NumPy's evaluation order with
 * explicit round-to-nearest operations.  Slot layout: path p owns vertices [p vcap, (p + 1) vcap),
 * blocks [p vcap / 32, ...), sub-blocks [p vcap / 8, ...), superblocks [p vcap / 512, ...); vcap a multiple
 * of 1024 (so that every path's first block and superblock are even).  sub_chord / sub_dev may be NULL
 * (then they are not built; see AuvPathBank).  A polyline that
 * does not fit raises AUV_STATUS_PATH_TOO_LONG.  waypoints: device [n][2][8] (x row, y row; as passed to
 * the reference's Path()), n_wp: device [n] (2..8), path_ids: device [n] slots to write, NULL = 0..n-1. */
typedef struct AuvPathBuild {
  AuvPathHdr* hdr;
  double* poly_xy;
  double* poly_cum;
  float* poly_f32;
  float* blk_chord;
  float* blk_dev;
  float* sb_chord;
  float* sb_dev;
  double* pp;
  int32_t n_knots; /* 1000 */
  int32_t vcap;
  float* sub_chord;
  float* sub_dev;
} AuvPathBuild;
int auv_pathbank_build(const double* waypoints, const int32_t* n_wp, const int32_t* path_ids, int n,
                       const AuvPathBuild* out, int32_t* status, void* stream);
/* RandomCurveThroughOrigin waypoints (path.py:96-120) with the waypoint count of
 * MovingObstacles._generate (movingobstacles.py:28-31), Philox streams keyed by (seed; path slot, epoch):
 * fills waypoints [n][2][8] / n_wp [n] for auv_pathbank_build. */
int auv_random_curve_waypoints(uint64_t seed, uint32_t epoch, double length, const int32_t* path_ids, int n,
                               double* waypoints, int32_t* n_wp, void* stream);
/* Host helper (no GPU work): first wrap and wrap period, in updates, of a constant-velocity
 * VesselObstacle track (obstacles.py:195-215: counter += dt; floor(counter) >= vel_len - 1 wraps the
 * counter to 0 and the position to the track start).  counter0 = waypoint counter right after
 * reset().  The loop is run literally in FP64, so the integers are the reference's. */
int auv_linear_wrap(double dt, double counter0, int vel_len, int32_t* first_wrap, int32_t* wrap_period);
/* Fill pool.st_rec (and, with pool.linear_tracks, pool.mov_lin) from the unpacked pool arrays for
 * the scenarios ids[0..n_ids) (device array; NULL = scenarios 0..n_ids-1). */
int auv_pool_pack(const AuvConfig* cfg, const AuvScenarioPool* pool, const int32_t* ids, int n_ids, void* stream);
/* Current moving-obstacle positions, last displacements and waypoint counters of every env
 * ([N][k_moving][2], [N][k_moving][2], [N][k_moving]; any may be NULL) -- what
 * VesselObstacle.position / .dx,.dy / .waypoint_counter hold (obstacles.py:195-215).  With
 * pool.linear_tracks they are evaluated from the closed form, otherwise copied from AuvBatch. */
int auv_obstacle_state(const AuvConfig* cfg, const AuvScenarioPool* pool, const AuvBatch* batch, double* pos,
                       double* disp, double* counter, void* stream);
/* Measured FP32 FMA peak helper (roofline denominator): runs `iters` dependent FMAs per
 * thread on a full grid; the caller times it with CUDA events. Returns flop count. */
int auv_fma_probe(float* sink, int blocks, int threads, int iters, void* stream,
                  double* flops_out);

#ifdef __cplusplus
}
#endif
#endif /* AUV_B200_H */
