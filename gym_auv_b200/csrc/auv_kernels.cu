// auv_kernels.cu -- hand-written sm_100a kernels for the gym-auv step path + the C ABI.
//
// Kernel inventory (reference file:line each one replaces is in include/auv_b200.h):
//   k_vessel_nav<DYN,OBST,G>  a group of G lanes per env, FP64: moving-obstacle update (OBST;
//                      closed form for constant-velocity tracks, else per-env state) -> RKF45
//                      vessel step (DYN) -> path projection (exact hierarchical
//                      LineString.project; the path's capsule tables are staged in shared memory
//                      by one bulk async copy per CTA while the RK step runs; warm upper bound
//                      from the previous step's segment) -> navigation record, obs[0..5],
//                      LiDAR-independent part of the reward -> obstacle culling (slots split over
//                      the group): nearby list (every 25 steps), enclosing circles,
//                      reference-exact ray windows, inside tests -> compact per-env obstacle
//                      records in HBM                                          latency / FP64
//   k_lidar<COUNT,VEL,WORLD> one CTA per 32 consecutive envs, every phase with the mapping that fills
//                      its lanes: hand-over lines + obstacle records -> shared memory; WARP PER
//                      RECORD over the CTA's flat record list (analytic edge pick for polygonised
//                      circles, vertices formed on the fly, results merged into the env's range
//                      row by shared-memory atomicMin); WARP PER ENV for closeness / collision /
//                      penalty / observation row / sector pooling / velocity channel; THREAD PER
//                      ENV for reward, done, counters; a warp per finished env for the VecEnv
//                      auto-reset (a COPY of the scenario's cached first observation); TRACK
//                      twins also record the episode tracks of AuvStepOut.tracks    FP32 issue
//   k_obstacle_update / k_vessel_step / k_reset   staged entry points
//   k_pool_pack, k_obstacle_state                  pool packing / obstacle state read-back
//   k_render           top-down RGB frames of a sample of the batch (auv_render.cuh)
//   k_fma_probe        FP32 FMA peak micro-benchmark (roofline denominator)
//
// Precision plan: everything cheap and threshold-sensitive is FP64 (vessel state, RK step,
// obstacle positions, vessel-relative obstacle centres, culling-window integers via an FP32
// fast path with FP64 fallback, projection refine, navigation and reward scalars); the
// O(rays x segments) casting is FP32 on vessel-relative geometry formed in FP64.
#include "auv_device.cuh"
#include "auv_dynamics.cuh"
#include "auv_geometry.cuh"
#include "auv_navigate.cuh"
#include "auv_generate.cuh"
#include "auv_pathbuild.cuh"
#include "../../include/auv_b200.h"

#include <math.h>

namespace auv {

// moving-obstacle update of one (env, slot)   obstacles.py:195-215.  Split into the loads that
// do not depend on each other (one round trip), the velocity lookup (second round trip) and the
// stores, so that callers can keep several slots in flight.  (General, table-driven tracks; pools
// of constant-velocity tracks use the closed form in lin_position.)
struct ObstLoad {
  double w, counter;
  int4 tr;  // vel_off, vel_len, vel_stride, 0
  double2 pos;
};
__device__ __forceinline__ ObstLoad obstacle_load(const AuvScenarioPool& pool, const AuvBatch& batch, long long pe,
                                                  long long ps) {
  ObstLoad o;
  o.w = pool.mov_width[ps];
  o.counter = batch.mov_counter[pe];
  o.tr = reinterpret_cast<const int4*>(pool.mov_track)[ps];
  o.pos = reinterpret_cast<const double2*>(batch.mov_pos)[pe];
  return o;
}
__device__ __forceinline__ void obstacle_finish(const AuvConfig& cfg, const AuvScenarioPool& pool, const AuvBatch& batch,
                                                long long pe, long long ps, ObstLoad o) {
  if (!(o.w > 0.0)) return;
  const double dt = cfg.t_step_size;
  double counter = o.counter + dt;
  int index = (int)floor(counter);
  double2 pos = o.pos;
  if (index >= o.tr.y - 1) {
    counter = 0.0;
    index = 0;
    pos = reinterpret_cast<const double2*>(pool.mov_start)[ps];
  }
  const double2 v = reinterpret_cast<const double2*>(pool.vel_table)[o.tr.x + (long long)index * o.tr.z];
  const double dx = dt * v.x, dy = dt * v.y;
  pos.x += dx;
  pos.y += dy;
  reinterpret_cast<double2*>(batch.mov_pos)[pe] = pos;
  reinterpret_cast<double2*>(batch.mov_disp)[pe] = make_double2(dx, dy);
  batch.mov_counter[pe] = counter;
}
__device__ __forceinline__ void obstacle_update_slot(const AuvConfig& cfg, const AuvScenarioPool& pool,
                                                     const AuvBatch& batch, long long pe, long long ps) {
  obstacle_finish(cfg, pool, batch, pe, ps, obstacle_load(pool, batch, pe, ps));
}

// constant-velocity track after n updates since reset (closed form of obstacles.py:195-215, see
// AuvScenarioPool.linear_tracks): r = the slot's 64 B record in pool.mov_lin
__device__ __forceinline__ double2 lin_position(const AuvScenarioPool& pool, const double2* __restrict__ r, double2 p0,
                                                double2 d, int n) {
  if (n < pool.lin_first_wrap) return make_double2(fma((double)n, d.x, p0.x), fma((double)n, d.y, p0.y));
  const double m = (double)((n - pool.lin_first_wrap) % pool.lin_wrap_period + 1);
  const double sx = r[2].y, sy = r[3].x;
  return make_double2(fma(m, d.x, sx), fma(m, d.y, sy));
}

// ------------------------------------------------------------------------------------
// k_obstacle_update     obstacles.py:195-215 (staged entry point: thread per (env, slot))
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_obstacle_update(AuvConfig cfg, AuvScenarioPool pool,
                                                          AuvBatch batch, int e0, int cnt) {
  const int km = pool.k_moving;
  const long long lid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (lid >= (long long)cnt * km) return;
  const long long gid = lid + (long long)e0 * km;  // envs [e0, e0 + cnt)
  const int e = (int)(gid / km);
  const int j = (int)(gid - (long long)e * km);
  if (j == 0) batch.obst_steps[e] += 1;
  if (!pool.linear_tracks) obstacle_update_slot(cfg, pool, batch, gid, (long long)batch.scn_id[e] * km + j);
}

// Vessel.step only (staged entry point auv_vessel_step)
__global__ void __launch_bounds__(128) k_vessel_step(AuvConfig cfg, AuvBatch batch,
                                                      const float* __restrict__ actions) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = batch.n_envs;
  if (e >= n) return;
  const S6 q = vessel_rk_step(cfg, load_state(batch.state, n, e), reinterpret_cast<const float2*>(actions)[e]);
  store_state(batch.state, n, e, q);
  batch.step_counter[e] += 1;
}

// pack pool.st_rec / pool.mov_lin from the unpacked arrays: thread per (listed scenario, slot)
__global__ void __launch_bounds__(128) k_pool_pack(AuvConfig cfg, AuvScenarioPool pool, const int* __restrict__ ids,
                                                   int n_ids) {
  const int km = pool.k_moving, ks = pool.k_static, per = km + ks;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)n_ids * per) return;
  const int li = (int)(gid / per), slot = (int)(gid - (long long)li * per);
  const int m = ids ? ids[li] : li;
  if (slot < km) {
    if (!pool.linear_tracks) return;
    const long long ps = (long long)m * km + slot;
    double* r = const_cast<double*>(pool.mov_lin) + ps * 8;
    const double w = pool.mov_width[ps];
    const int voff = pool.mov_track[4 * ps];
    const double2 v = w > 0.0 ? reinterpret_cast<const double2*>(pool.vel_table)[voff] : make_double2(0.0, 0.0);
    r[0] = pool.mov_pos0[2 * ps];
    r[1] = pool.mov_pos0[2 * ps + 1];
    r[2] = cfg.t_step_size * v.x;  // dx = dt * vel[idx][0]   obstacles.py:206-207
    r[3] = cfg.t_step_size * v.y;
    r[4] = w;
    r[5] = pool.mov_start[2 * ps];
    r[6] = pool.mov_start[2 * ps + 1];
    r[7] = 0.0;
  } else {
    const long long ps = (long long)m * ks + (slot - km);
    double* r = const_cast<double*>(pool.st_rec) + ps * 4;
    r[0] = pool.st_pos[2 * ps];
    r[1] = pool.st_pos[2 * ps + 1];
    r[2] = pool.st_radius[ps];
    r[3] = 0.0;
  }
}

// VesselObstacle.position / (dx, dy) / waypoint_counter of every (env, slot)
__global__ void __launch_bounds__(128) k_obstacle_state(AuvConfig cfg, AuvScenarioPool pool, AuvBatch batch,
                                                        double* __restrict__ pos, double* __restrict__ disp,
                                                        double* __restrict__ counter) {
  const int km = pool.k_moving;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)batch.n_envs * km) return;
  const int e = (int)(gid / km), j = (int)(gid - (long long)e * km);
  double2 p, d;
  double c;
  if (pool.linear_tracks) {
    const long long ps = (long long)batch.scn_id[e] * km + j;
    const double2* r = reinterpret_cast<const double2*>(pool.mov_lin + ps * 8);
    const int n = batch.obst_steps[e];
    const double w = r[2].x;
    d = r[1];
    p = r[0];
    c = pool.mov_counter0[ps];
    if (w > 0.0) {
      p = lin_position(pool, r, r[0], d, n);
      if (n == 0) d = reinterpret_cast<const double2*>(pool.mov_disp0)[ps];
      // the counter is accumulated literally (counter += dt per update), as the reference does
      const int since = n < pool.lin_first_wrap ? n : (n - pool.lin_first_wrap) % pool.lin_wrap_period;
      if (n >= pool.lin_first_wrap) c = 0.0;
      for (int k = 0; k < since; ++k) c += cfg.t_step_size;
    } else {
      d = make_double2(0.0, 0.0);
    }
  } else {
    p = reinterpret_cast<const double2*>(batch.mov_pos)[gid];
    d = reinterpret_cast<const double2*>(batch.mov_disp)[gid];
    c = batch.mov_counter[gid];
  }
  if (pos) reinterpret_cast<double2*>(pos)[gid] = p;
  if (disp) reinterpret_cast<double2*>(disp)[gid] = d;
  if (counter) counter[gid] = c;
}

// ------------------------------------------------------------------------------------
// Obstacle records: what the culling stage hands to the ray-casting stage (HBM scratch
// owned by the caller, AuvBatch.rec: [N][rec_cap] records of AUV_REC_BYTES bytes).
// ------------------------------------------------------------------------------------
struct __align__(16) ObstRec {
  double cx, cy;         // vessel-relative anchor: circle centre | pentagon rotation centre
  double geo;            // radius | width
  double hx, hy;         // unit heading of a vessel obstacle
  float ecx, ecy, rho;   // enclosing circle, vessel-relative (sensor.py:22-38)
  int a, b;              // culling window (sensor.py:41-97)
  int flags;             // OFLAG_*
  int nv;                // boundary vertices incl. the closing one
  int vbase;             // world polygon: first vertex in pool.world_verts
  float step_len;        // |(dx, dy)| of a vessel obstacle's last update (velocity channel)
  int pad;
};
static_assert(sizeof(ObstRec) == AUV_REC_BYTES, "ObstRec layout");

// reset of one env's mutable state by ONE thread   environment.py:202-212, vessel.py:189-224
__device__ __forceinline__ void reset_env_thread(const AuvScenarioPool& pool, const AuvBatch& batch, int e,
                                                 int scn) {
  const int n = batch.n_envs;
  const int km = pool.k_moving;
  batch.scn_id[e] = scn;
  batch.env_pid[e] = pool.path_id[scn];
  batch.prev_seg[e] = -1;
  batch.obst_steps[e] = 0;
  batch.episode[e] += 1;
  const double* vi = pool.vessel_init + 3ll * scn;
  batch.state[e] = vi[0];
  batch.state[n + e] = vi[1];
  batch.state[2 * n + e] = vi[2];
  batch.state[3 * n + e] = 0.0;
  batch.state[4 * n + e] = 0.0;
  batch.state[5 * n + e] = 0.0;
  batch.step_counter[e] = 0;
  batch.t_step[e] = 0;
  batch.cum_reward[e] = 0.0;
  batch.max_progress[e] = 0.0;
  batch.cte_sum[e] = 0.0;
  if (!pool.linear_tracks)
    for (int j = 0; j < km; ++j) {
      const long long ps = (long long)scn * km + j, pe = (long long)e * km + j;
      reinterpret_cast<double2*>(batch.mov_pos)[pe] = reinterpret_cast<const double2*>(pool.mov_pos0)[ps];
      reinterpret_cast<double2*>(batch.mov_disp)[pe] = reinterpret_cast<const double2*>(pool.mov_disp0)[ps];
      batch.mov_counter[pe] = pool.mov_counter0[ps];
    }
  for (int w = 0; w < batch.mask_words; ++w) batch.nearby_mask[(long long)e * batch.mask_words + w] = 0u;
}

// explicit reset (auv_reset): envs flagged in reset_mask (or all) go back to scenario scn_id[e]
__global__ void __launch_bounds__(128) k_reset(AuvScenarioPool pool, AuvBatch batch,
                                               const uint8_t* __restrict__ reset_mask) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= batch.n_envs) return;
  if (reset_mask != nullptr && reset_mask[e] == 0) return;
  reset_env_thread(pool, batch, e, batch.scn_id[e]);
}

// ------------------------------------------------------------------------------------
// Culling stage ("hierarchical collision detector"), a group of G lanes per env.
//   vessel.py:266-273 nearby list, sensor.py:22-97 windows, obstacles.py:108-113,230-262
//   enclosing circles.  Emits rec[e][0..cnt) and rec_cnt[e].
// ------------------------------------------------------------------------------------
struct SlotGeom {
  bool valid, pent, world;
  double cx, cy, rho, geo, hx, hy;
  float step_len;
  int nv, vbase;
};

// n_upd = obstacle updates since reset (closed-form tracks only)
__device__ __forceinline__ SlotGeom load_slot(const AuvScenarioPool& pool, const AuvBatch& batch, int e, int scn,
                                              int j, double px, double py, int n_upd) {
  SlotGeom g;
  g.valid = g.pent = g.world = false;
  g.cx = g.cy = g.rho = g.geo = 0.0;
  g.hx = 1.0;
  g.hy = 0.0;
  g.step_len = 0.f;
  g.nv = g.vbase = 0;
  const int km = pool.k_moving, ks = pool.k_static, K = km + ks;
  if (j >= K) {  // shared world polygon (PolygonObstacle): cached enclosing circle
    const int wi = j - K;
    const double* c3 = pool.world_circle + 3ll * wi;
    g.vbase = pool.world_voff[wi];
    g.nv = pool.world_voff[wi + 1] - g.vbase;
    g.valid = g.nv >= 4;
    g.world = true;
    g.cx = c3[0] - px;
    g.cy = c3[1] - py;
    g.rho = c3[2];
  } else if (j < km) {  // VesselObstacle: pentagon, enclosing circle of its min-rotated rectangle
    const long long ps = (long long)scn * km + j;
    double w;
    double2 pos, dsp;
    if (pool.linear_tracks) {
      const double2* __restrict__ r = reinterpret_cast<const double2*>(pool.mov_lin + ps * 8);
      const double2 p0 = r[0];
      dsp = r[1];
      w = r[2].x;
      pos = p0;
      if (w > 0.0) {
        pos = lin_position(pool, r, p0, dsp, n_upd);
        if (n_upd == 0) dsp = reinterpret_cast<const double2*>(pool.mov_disp0)[ps];  // update(0.1) of __init__
      }
    } else {
      const long long pe = (long long)e * km + j;
      w = pool.mov_width[ps];
      pos = reinterpret_cast<const double2*>(batch.mov_pos)[pe];
      dsp = reinterpret_cast<const double2*>(batch.mov_disp)[pe];
    }
    if (w > 0.0) {
      g.valid = g.pent = true;
      g.geo = w;
      const double dl2 = dsp.x * dsp.x + dsp.y * dsp.y;
      if (dl2 > 0.0) {
        const double inv = rsqrt(dl2);
        g.hx = dsp.x * inv;
        g.hy = dsp.y * inv;
        g.step_len = (float)(dl2 * inv);
      }
      // obstacles.py:230-262, SURVEY App. A.3: centre = c + R(th)((w/2,0) - c) + pos, c = (5w/18, 0)
      g.cx = (pos.x - px) + w * (5.0 / 18.0) + (w * (2.0 / 9.0)) * g.hx;
      g.cy = (pos.y - py) + (w * (2.0 / 9.0)) * g.hy;
      g.rho = w * 1.1180339887498949;  // sqrt(5)/2
      g.nv = 6;
    }
  } else {  // CircularObstacle: ring = regular n-gon, enclosing circle = (position, radius)
    const double2* __restrict__ r = reinterpret_cast<const double2*>(pool.st_rec + ((long long)scn * ks + (j - km)) * 4);
    const double2 c = r[0];
    const double rad = r[1].x;
    if (rad > 0.0) {
      g.valid = true;
      g.geo = rad;
      g.cx = c.x - px;
      g.cy = c.y - py;
      g.rho = rad;
      g.nv = ngon_sides(rad) + 1;
    }
  }
  return g;
}

// is obstacle slot j within sensor range of the own-ship?  dist(p0, o.boundary) - width < range (vessel.py:266-273):
// decided from the enclosing circle when it can be, else from the exact boundary distance
__device__ __forceinline__ bool slot_is_near(const AuvScenarioPool& pool, const AuvBatch& batch,
                                             const double2* __restrict__ unit64, int e, int scn, int j, double px,
                                             double py, int n_upd, double range, double width) {
  const SlotGeom g = load_slot(pool, batch, e, scn, j, px, py, n_upd);
  if (!g.valid) return false;
  const double dc = sqrt(g.cx * g.cx + g.cy * g.cy);
  if (dc - g.rho - width >= range + 1e-6) return false;  // the boundary lies inside the enclosing circle: distance >= dc - rho
  if (dc + g.rho - width < range - 1e-6) return true;    // ... and distance <= dc + rho
  const double bx0 = g.cx - (g.geo * (2.0 / 9.0)) * g.hx, by0 = g.cy - (g.geo * (2.0 / 9.0)) * g.hy;
  bool in_dummy;
  const double dist = g.world ? world_polygon_distance(reinterpret_cast<const double2*>(pool.world_verts) + g.vbase, g.nv, px,
                                                       py, in_dummy)
                              : boundary_distance(g.pent, g.cx, g.cy, bx0, by0, g.geo, g.hx, g.hy, g.nv, unit64);
  return (dist - width) < range;
}

// Culling stage for one env by its group of G lanes: the lanes take different obstacle slots
// (slot j of a 32-slot word belongs to lane j % G), records are emitted in slot order by a
// ballot prefix.  `store` is false for the padding groups past the end of the env range.
template <int G>
__device__ __forceinline__ void cull_env_group(const AuvConfig& cfg, const AuvScenarioPool& pool,
                                               const AuvBatch& batch, const double2* __restrict__ unit64,
                                               int* __restrict__ windows_out, int e, int scn, double px,
                                               double py, double psi, int step_counter, int n_upd, const int lane,
                                               const unsigned gm, const bool store) {
  const int sub = lane & (G - 1);
  const int R = cfg.n_sensors;
  const int S = pool.k_moving + pool.k_static + pool.n_world;
  const bool refresh = (step_counter % cfg.sensor_interval_load_obstacles) == 0;
  const double range = cfg.sensor_range, width = cfg.vessel_width;
  ObstRec* rec = reinterpret_cast<ObstRec*>(batch.rec) + (long long)e * batch.rec_cap;
  int cnt = 0;
  // ---- nearby list: {o : dist(p0, o.boundary) - width < range}   vessel.py:266-273
  // An env refreshes its list every 25 steps; in the desynchronised steady state that is ~1 of the 8 envs of a
  // warp per step -- but most warps have one.  The warp therefore does its refreshing envs one after the other
  // with ALL 32 lanes on different slots (one round for 32 slots) instead of leaving each to the 4 lanes of its
  // group (8 rounds during which the other groups wait).
  const int K = pool.k_moving + pool.k_static;
  const bool grid = pool.world_cell_off != nullptr && pool.n_world > 0;  // world slots through the broad phase
  const int S_scan = grid ? K : S;
  const unsigned rmask = __ballot_sync(AUV_FULL, refresh && sub == 0 && store);
  for (unsigned rm = rmask; rm; rm &= rm - 1) {  // uniform in the warp
    const int src = __ffs(rm) - 1;
    const int eb = __shfl_sync(AUV_FULL, e, src), sb = __shfl_sync(AUV_FULL, scn, src);
    const int nb = __shfl_sync(AUV_FULL, n_upd, src);
    const double pxb = __shfl_sync(AUV_FULL, px, src), pyb = __shfl_sync(AUV_FULL, py, src);
    for (int base = 0; base < S; base += 32) {
      unsigned word = 0u;
      if (base < S_scan) {
        const int j = base + lane;
        word = __ballot_sync(AUV_FULL, j < S_scan && slot_is_near(pool, batch, unit64, eb, sb, j, pxb, pyb, nb, range, width));
      }
      if (lane == src) batch.nearby_mask[(long long)eb * batch.mask_words + (base >> 5)] = word;
    }
  }
  if (rmask) __syncwarp();
  if (refresh) {
    if (grid) {
      // uniform grid over the world's enclosing circles: only the polygons listed in the cells that the
      // detection disc's bounding box overlaps can be near; the exact test is the same
      __syncwarp(gm);
      const double rq = range + width + 1e-3, cell = pool.world_grid_cell;
      const int ix0 = max(0, (int)floor((px - rq - pool.world_grid_x0) / cell));
      const int ix1 = min(pool.world_grid_nx - 1, (int)floor((px + rq - pool.world_grid_x0) / cell));
      const int iy0 = max(0, (int)floor((py - rq - pool.world_grid_y0) / cell));
      const int iy1 = min(pool.world_grid_ny - 1, (int)floor((py + rq - pool.world_grid_y0) / cell));
      for (int iy = iy0; iy <= iy1; ++iy)
        for (int ix = ix0; ix <= ix1; ++ix) {
          const int c = iy * pool.world_grid_nx + ix;
          const int i0 = pool.world_cell_off[c], i1 = pool.world_cell_off[c + 1];
          for (int it = i0 + sub; it < i1; it += G) {
            const int j = K + pool.world_cell_items[it];
            if (store && slot_is_near(pool, batch, unit64, e, scn, j, px, py, n_upd, range, width))
              atomicOr(batch.nearby_mask + (long long)e * batch.mask_words + (j >> 5), 1u << (j & 31));
          }
        }
    }
    __syncwarp(gm);
  }
  for (int base = 0; base < S; base += 32) {
    const unsigned* mw = batch.nearby_mask + (long long)e * batch.mask_words + (base >> 5);
    const unsigned word = refresh ? __ldcg(mw) : *mw;
    // ---- one record per nearby obstacle: lane `sub` takes the (sub + t G)-th set bit of the word
    //      ("by rank"), so the groups of a warp run the expensive window arithmetic together
    if (windows_out != nullptr && store) {
      for (int j = base + sub; j < min(S, base + 32); j += G)
        reinterpret_cast<int2*>(windows_out)[(long long)e * S + j] = make_int2(0, 0);
      __syncwarp(gm);
    }
    const int nw = __popc(word);
    for (int r = sub; r < nw; r += G) {
      unsigned wv = word;
      for (int t = 0; t < r; ++t) wv &= wv - 1;
      const int j = base + __ffs(wv) - 1;
      const SlotGeom g = load_slot(pool, batch, e, scn, j, px, py, n_upd);
      int wa = 0, wb = 0;
      bool allrays = false, inside = false;
      double bx0 = 0.0, by0 = 0.0;
      if (g.valid) {
        int lo, hi;
        cull_bounds(g.cx, g.cy, g.rho, psi, R, lo, hi);
        window_from_bounds(lo, hi, R, cfg.cull_mode, wa, wb, allrays);
        bx0 = g.cx - (g.geo * (2.0 / 9.0)) * g.hx;
        by0 = g.cy - (g.geo * (2.0 / 9.0)) * g.hy;
        if (g.cx * g.cx + g.cy * g.cy <= g.rho * g.rho) {  // filled boundaries: own-ship inside => range 0
          if (g.pent)
            inside = vessel_inside_pentagon(bx0, by0, g.geo, g.hx, g.hy);
          else if (g.world)
            world_polygon_distance(reinterpret_cast<const double2*>(pool.world_verts) + g.vbase, g.nv, px, py, inside);
        }
      }
      if (!store) continue;
      if (windows_out != nullptr) reinterpret_cast<int2*>(windows_out)[(long long)e * S + j] = make_int2(wa, wb);
      const int idx = cnt + r;
      AUV_CHECK(batch.status, j >= 0 && j < S && idx >= 0);
      if (idx >= batch.rec_cap) {  // cannot happen when rec_cap >= number of slots
        if (batch.status != nullptr) atomicOr(batch.status, AUV_STATUS_REC_OVERFLOW);
        continue;
      }
      ObstRec q;
      q.cx = g.pent ? bx0 : g.cx;
      q.cy = g.pent ? by0 : g.cy;
      q.geo = g.geo;
      q.hx = g.hx;
      q.hy = g.hy;
      q.ecx = (float)g.cx;
      q.ecy = (float)g.cy;
      q.rho = (float)g.rho;
      q.a = wa;  // a nearby bit is only ever set for a valid slot; an invalid one would leave an
      q.b = wb;  // empty window (0, 0) that no ray tests
      q.flags = (g.pent ? (OFLAG_FILLED | OFLAG_PENTAGON) : 0) | (g.world ? (OFLAG_FILLED | OFLAG_WORLD) : 0) |
                (inside ? OFLAG_INSIDE : 0) | (allrays ? OFLAG_ALLRAYS : 0);
      q.nv = g.valid ? g.nv : 1;
      q.vbase = g.vbase;
      q.step_len = g.step_len;
      q.pad = 0;
      rec[idx] = q;
    }
    cnt = min(cnt + nw, batch.rec_cap);
  }
  if (store && sub == 0) {
    batch.rec_cnt[e] = cnt;
    batch.nav[(long long)e * AUV_NAV_W + NAV_CNT] = (double)cnt;
  }
}

// ---- reset cache (pool.reset_*) and sustained scenario refresh, all on the device
// worker env w takes the k-th listed scenario (padded with repeats: recomputing is idempotent)
__global__ void __launch_bounds__(128) k_worker_fill(AuvBatch wb, const int* __restrict__ ids, int first, int n,
                                                     const int* __restrict__ n_dev) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= wb.n_envs) return;
  if (n_dev != nullptr) n = min(n, *n_dev);
  const int k = n > 0 ? min(w, n - 1) : 0;
  wb.scn_id[w] = ids ? ids[k] : first + k;
}
// one warp per worker env: its first observation, max progress and nearby list become the
// cached reset of its scenario (environment.py:176-245 computed once per scenario)
__global__ void __launch_bounds__(128) k_cache_scatter(AuvScenarioPool pool, AuvBatch wb, const float* __restrict__ wobs,
                                                       int obs_dim, int use_lidar, int n, const int* __restrict__ n_dev) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (n_dev != nullptr) n = min(n, *n_dev);
  if (w >= n || w >= wb.n_envs) return;
  const int m = wb.scn_id[w];
  float* dst = const_cast<float*>(pool.reset_obs) + (long long)m * obs_dim;
  const float* src = wobs + (long long)w * obs_dim;
  for (int k = lane; k < obs_dim; k += 32) dst[k] = src[k];
  if (lane == 0) const_cast<double*>(pool.reset_max_progress)[m] = wb.max_progress[w];
  if (use_lidar)
    for (int k = lane; k < wb.mask_words; k += 32)
      const_cast<uint32_t*>(pool.reset_mask)[(long long)m * wb.mask_words + k] = wb.nearby_mask[(long long)w * wb.mask_words + k];
}
// envs that finished an episode since the last call list the pool slot they vacated: with a
// ping-pong pool of 2 N scenarios env e alternates between slots e and e + N
__global__ void __launch_bounds__(128) k_refresh_collect(AuvBatch live, int n_scenarios, int* __restrict__ seen,
                                                         int* __restrict__ ids, int* __restrict__ count, int capacity) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= live.n_envs) return;
  const int ep = live.episode[e];
  if (ep == seen[e]) return;
  const int k = atomicAdd(count, 1);
  if (k >= capacity) return;  // stays listed as unseen: picked up by the next call
  seen[e] = ep;
  ids[k] = (int)(((long long)live.scn_id[e] + (live.reset_stride > 0 ? live.reset_stride : live.n_envs)) % n_scenarios);
}

// table-driven moving-obstacle update of one env by its group of G lanes (two slots in flight per lane)
template <int G>
__device__ __noinline__ void obstacle_update_group(const AuvConfig& cfg, const AuvScenarioPool& pool, const AuvBatch& batch,
                                                   int e, int scn, int sub, bool store) {
  if (!store) return;
  const int km = pool.k_moving;
  const long long pe0 = (long long)e * km, ps0 = (long long)scn * km;
  for (int j = sub; j < km; j += 2 * G) {
    const bool two = j + G < km;
    const ObstLoad a = obstacle_load(pool, batch, pe0 + j, ps0 + j);
    const ObstLoad b = obstacle_load(pool, batch, pe0 + (two ? j + G : j), ps0 + (two ? j + G : j));
    obstacle_finish(cfg, pool, batch, pe0 + j, ps0 + j, a);
    if (two) obstacle_finish(cfg, pool, batch, pe0 + j + G, ps0 + j + G, b);
  }
}

// ---- bulk async copy (TMA, 1-D) + mbarrier: a CTA's copy of its path's capsule tables
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "AUV_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra AUV_DONE;\n"
      "bra AUV_WAIT;\n"
      "AUV_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// BaseEnvironment._update (OBST) + Vessel.step (DYN) + the path projection of Vessel.navigate, a
// group of G lanes per env (k_nav_cull below, the same mapping, does the rest of Vessel.navigate and
// the culling stage).  The scalar FP64 chains (RK step, PCHIP, navigation features) are
// computed redundantly by the lanes of a group; the table searches (path projection, obstacle
// slots) are split over them, which shortens the per-warp critical path ~G-fold and gives the
// SM G times more warps to hide the remaining load latency with (thread-per-env had N/32 warps:
// 3 per scheduler at 65536 envs, one long dependent chain each -- profiles/earlier).
// When every env of the CTA follows the same path (scenario pools are laid out path-major, so this
// is the normal case) the path's capsule tables -- <= 13 KB -- are copied to shared memory by
// ONE bulk async copy (cp.async.bulk + mbarrier) issued before the RK step and awaited after it:
// the ~50 capsule tests per env then read shared memory instead of four dependent rounds of
// global loads.  CTAs with mixed paths (or a path with more than AUV_PATH_STAGE_BLOCKS blocks)
// search the global tables; the arithmetic is the same.
#define AUV_NAV_G 4
#define AUV_NAV_THREADS 128  // a multiple of 128: one 32-env sub-block (4 warps) per 128 threads
#define AUV_NAV_MINB (1024 / AUV_NAV_THREADS)  // 64 registers: 32 warps per SM (6 / 7 / 8 CTAs of 128: 0.106 / 0.101 / 0.096 ms)
constexpr int NAV_STAGE_SB = (AUV_PATH_STAGE_BLOCKS + AUV_PATH_SUPER - 1) / AUV_PATH_SUPER;
constexpr int NAV_SUBBLOCKS = AUV_NAV_THREADS / 128;
// shared memory of one sub-block: its path's capsule tables
struct __align__(16) NavStage {
  float4 chord[AUV_PATH_STAGE_BLOCKS];
  float2 aux[AUV_PATH_STAGE_BLOCKS];
  float4 sbc[NAV_STAGE_SB];
  float2 sba[NAV_STAGE_SB];
};
// Two launches: k_vessel_nav stops after the projection, k_nav_cull does navigation + culling.  Same total
// kernel time as one launch (0.104 ms), but three kernels per env range interleave better across the step's
// two streams: 0.180 -> 0.172 ms per step
template <bool DYN, bool OBST, int G>
__global__ void __launch_bounds__(AUV_NAV_THREADS, AUV_NAV_MINB) k_vessel_nav(const __grid_constant__ AuvConfig cfg,
                                                                const __grid_constant__ AuvPathBank paths,
                                                                const __grid_constant__ AuvScenarioPool pool,
                                                                const __grid_constant__ AuvBatch batch,
                                                                const double2* __restrict__ unit64,
                                                                int* __restrict__ windows_out,
                                                                const float* __restrict__ actions,
                                                                float* __restrict__ obs_out, int obs_dim, int e0, int e1) {
  extern __shared__ __align__(16) unsigned char nav_smem[];
  NavStage* stages = reinterpret_cast<NavStage*>(nav_smem);
  __shared__ __align__(8) unsigned long long s_bar[NAV_SUBBLOCKS];
  __shared__ int s_pid[AUV_NAV_THREADS / 32];
  const int lane = threadIdx.x & 31, sub = lane & (G - 1);
  const int sbk = threadIdx.x >> 7, tsb = threadIdx.x & 127;  // sub-block of 32 envs, thread within it
  NavStage& st = stages[sbk];
  const unsigned gm = group_mask<G>(lane);
  const int eraw = e0 + (blockIdx.x * AUV_NAV_THREADS + threadIdx.x) / G;  // envs [e0, e1)
  const bool store = eraw < e1;
  const int e = store ? eraw : e1 - 1;  // padding groups shadow the last env and store nothing
  const int n = batch.n_envs;
  // ---- first round of loads: everything that is indexed by the env alone
  const int scn = batch.scn_id[e];
  const int pid = batch.env_pid[e];
  const int prev_seg = batch.prev_seg[e];
  int step_counter = batch.step_counter[e];
  int n_upd = batch.obst_steps[e];
  S6 y = load_state(batch.state, n, e);
  float2 act = make_float2(0.f, 0.f);
  if (DYN) act = reinterpret_cast<const float2*>(actions)[e];
  if (tsb == 0) mbar_init(&s_bar[sbk], 1);
  {  // does the whole sub-block follow one path?
    int same;
    __match_all_sync(AUV_FULL, pid, &same);
    if (lane == 0) s_pid[threadIdx.x >> 5] = same ? pid : -1;
  }
  __syncthreads();
  // ---- second round: the path's header line
  const AuvPathHdr h = paths.hdr[pid];
  const int nblk = (h.nseg + AUV_PATH_BLOCK - 1) / AUV_PATH_BLOCK;
  const int nsb = (nblk + AUV_PATH_SUPER - 1) / AUV_PATH_SUPER;
  bool staged = s_pid[4 * sbk] >= 0 && nblk <= AUV_PATH_STAGE_BLOCKS;
#pragma unroll
  for (int w = 1; w < 4; ++w) staged = staged && s_pid[4 * sbk + w] == s_pid[4 * sbk];
  if (staged && tsb == 0) {
    const unsigned nb2 = (unsigned)(nblk + 1) & ~1u, ns2 = (unsigned)(nsb + 1) & ~1u;  // tables are padded to even counts
    mbar_expect_tx(&s_bar[sbk], nb2 * 24u + ns2 * 24u);
    bulk_g2s(st.chord, reinterpret_cast<const float4*>(paths.blk_chord) + h.b0, nb2 * 16u, &s_bar[sbk]);
    bulk_g2s(st.aux, reinterpret_cast<const float2*>(paths.blk_dev) + h.b0, nb2 * 8u, &s_bar[sbk]);
    bulk_g2s(st.sbc, reinterpret_cast<const float4*>(paths.sb_chord) + h.s0, ns2 * 16u, &s_bar[sbk]);
    bulk_g2s(st.sba, reinterpret_cast<const float2*>(paths.sb_dev) + h.s0, ns2 * 8u, &s_bar[sbk]);
  }
  if (OBST) {
    ++n_upd;
    if (store && sub == 0) batch.obst_steps[e] = n_upd;
    if (!pool.linear_tracks) {  // table-driven tracks (out of line: pools of constant-velocity tracks never get here)
      obstacle_update_group<G>(cfg, pool, batch, e, scn, sub, store);
      __syncwarp();  // the updated obstacles are visible to the group
    }
  }
  if (DYN) {
    y = vessel_rk_step(cfg, y, act);
    ++step_counter;
    if (store && sub == 0) {
      store_state(batch.state, n, e, y);
      batch.step_counter[e] = step_counter;
    }
  }
  PathTabs T;
  if (staged) {
    mbar_wait(&s_bar[sbk], 0);
    T.sbc = st.sbc;
    T.sba = st.sba;
    T.chord = st.chord;
    T.aux = st.aux;
  } else {
    T.sbc = reinterpret_cast<const float4*>(paths.sb_chord) + h.s0;
    T.sba = reinterpret_cast<const float2*>(paths.sb_dev) + h.s0;
    T.chord = reinterpret_cast<const float4*>(paths.blk_chord) + h.b0;
    T.aux = reinterpret_cast<const float2*>(paths.blk_dev) + h.b0;
  }
  int seg;
  const double s = project_group<G>(paths, h, T, y.x, y.y, prev_seg, lane, gm, seg, batch.status);
  AUV_CHECK(batch.status, seg >= 0 && seg < h.nseg && (!staged || (nblk <= AUV_PATH_STAGE_BLOCKS && nsb <= NAV_STAGE_SB)));
  if (store && sub == 0) {
    batch.prev_seg[e] = seg;
    batch.nav[(long long)e * AUV_NAV_W + NAV_S] = s;  // the arclength, handed to k_nav_cull
  }
}

// second half of the navigation stage as its own launch: Vessel.navigate + the culling stage
template <int G>
__global__ void __launch_bounds__(128, 8) k_nav_cull(const __grid_constant__ AuvConfig cfg, const __grid_constant__ AuvPathBank paths,
                                                     const __grid_constant__ AuvScenarioPool pool,
                                                     const __grid_constant__ AuvBatch batch, const double2* __restrict__ unit64,
                                                     int* __restrict__ windows_out, float* __restrict__ obs_out, int obs_dim,
                                                     int e0, int e1) {
  const int lane = threadIdx.x & 31, sub = lane & (G - 1);
  const unsigned gm = group_mask<G>(lane);
  const int eraw = e0 + (blockIdx.x * 128 + threadIdx.x) / G;
  const bool store = eraw < e1;
  const int e = store ? eraw : e1 - 1;
  const int n = batch.n_envs;
  const int scn = batch.scn_id[e];
  const int pid = batch.env_pid[e];
  const int step_counter = batch.step_counter[e];
  const int n_upd = batch.obst_steps[e];
  const S6 y = load_state(batch.state, n, e);
  const double s = batch.nav[(long long)e * AUV_NAV_W + NAV_S];
  const AuvPathHdr h = paths.hdr[pid];
  __syncwarp();  // every lane has read s before the group's leader overwrites the record
  navigate_env(cfg, paths, h, batch, pid, e, scn, s, y.x, y.y, y.psi, y.u, y.v, y.r,
               obs_out ? obs_out + (long long)e * obs_dim : nullptr, store && sub == 0);
  if (cfg.use_lidar)
    cull_env_group<G>(cfg, pool, batch, unit64, windows_out, e, scn, y.x, y.y, y.psi, step_counter, n_upd, lane, gm, store);
}

// ------------------------------------------------------------------------------------
// k_lidar: one CTA per block of E (<= 32) consecutive envs, four phases that each use the
// mapping that fills the lanes:
//   1. the envs' hand-over lines (E x 128 B, coalesced) and obstacle records (contiguous per env)
//      go to shared memory; every ray of every env starts at sensor_range
//   2. WARP PER RECORD over the CTA's flat record list (warps never idle on an env with nothing
//      in range, and a warp's record has one boundary type: no divergence): lanes over the
//      record's candidate rays, analytic edge pick / staged vertex chain, results merged into
//      the env's range row in shared memory by atomicMin on the bit pattern
//   3. WARP PER ENV over the range rows: closeness, collision, penalty, observation row
//      (8-byte vector stores), optional per-ray / per-sector outputs
//   4. THREAD PER ENV: reward, done, counters, statistics -- one warp does the scalar tail of all
//      E envs at once, its outputs leave coalesced; finished envs are then auto-reset by a warp
//      each (copy of the cached first observation)
// ------------------------------------------------------------------------------------
#define AUV_LIDAR_THREADS 256
#define AUV_LIDAR_RCAP 96  // records per shared-memory round
#define AUV_LIDAR_MAX_ENVS 32  // envs per CTA (<= 32: one warp scans their record counts)

struct LidarArgs {
  AuvConfig cfg;
  AuvRayTable rays;
  AuvPathBank paths;
  AuvScenarioPool pool;
  AuvBatch batch;
  AuvStepOut out;
  const void* pad0;  // keeps the fields below 16-byte aligned, as before AuvStepOut.tracks (vector parameter loads)
  int mode;       // AUV_OBSERVE_STEP | AUV_OBSERVE_RESET
  int obs_dim;
  int e0, e1;     // envs [e0, e1) of the batch are processed by this launch
  int envs_per_cta;  // E: 32 unless the ray count makes the range rows too large
  int vmax;       // staged vertices per warp (float2): AUV_MAX_POLY_VERTS with world polygons, else 16
  float pen_clear_ray;     // range * exp(-0.1 range): penalty term of a ray that reads sensor_range
  float inv_log_range;     // 1 / log(1 + range)
  double clear_closeness;  // -range * exp(-0.1 range): closeness reward when every ray is clear
  double inv_weight_sum;   // 1 / sum of the ray weights
  double feas_width;       // vessel_width * feasibility_width_multiplier (sensor.py:166-168)
  AuvTracks trk;           // copy of *out.tracks (TRACK instantiations only; zeros otherwise)
};

// dynamic shared memory of a CTA; every part is 16-byte aligned
struct LidarSmem {
  double* hand;     // [E][16]   hand-over lines
  void* sdist;      // [E][rpad] float ranges, or (VEL) u64 keys = range bits << 32 | record index
  ObstRec* rec;     // [RCAP]    records of the round
  int* rec_env;     // [RCAP]    local env | (record index in its env << 8)
  float2* verts;    // [warps][vmax]
  float2* unit;     // [64]      cos/sin(2 pi k / 64) in FP32
  int* off;         // [E + 1]   exclusive scan of the envs' record counts
  float* pen;       // [E]       sum of w_i (penalty_i - clear penalty) over hit rays
  int* flag;        // [E]       bit 0 collision, bit 1 auto-reset pending, (TRACK) bit 2 tracked env
                    //           finished, bit 3 parity of its episode
  int* next;        // [E]       scenario the env resets onto
};
__host__ __device__ constexpr size_t lidar_smem_bytes_for(int E, int rpad, int vmax, int vel) {
  return (size_t)E * 16 * 8 + (size_t)E * rpad * (vel ? 8 : 4) + AUV_LIDAR_RCAP * sizeof(ObstRec) + AUV_LIDAR_RCAP * 4 +
         (size_t)(AUV_LIDAR_THREADS / 32) * vmax * 8 + 64 * 8 + 48 * 4 + 32 * 4 + 32 * 4 + 32 * 4;
}
__device__ __forceinline__ LidarSmem lidar_carve(unsigned char* p, int E, int rpad, int vmax, int vel) {
  LidarSmem s;
  s.hand = reinterpret_cast<double*>(p);
  p += (size_t)E * 16 * 8;
  s.sdist = p;
  p += (size_t)E * rpad * (vel ? 8 : 4);
  s.rec = reinterpret_cast<ObstRec*>(p);
  p += AUV_LIDAR_RCAP * sizeof(ObstRec);
  s.rec_env = reinterpret_cast<int*>(p);
  p += AUV_LIDAR_RCAP * 4;
  s.verts = reinterpret_cast<float2*>(p);
  p += (size_t)(AUV_LIDAR_THREADS / 32) * vmax * 8;
  s.unit = reinterpret_cast<float2*>(p);
  p += 64 * 8;
  s.off = reinterpret_cast<int*>(p);
  p += 48 * 4;
  s.pen = reinterpret_cast<float*>(p);
  p += 32 * 4;
  s.flag = reinterpret_cast<int*>(p);
  p += 32 * 4;
  s.next = reinterpret_cast<int*>(p);
  return s;
}

// range of the ray (c, s) against one regular n-gon ring inscribed in the circle (ecx, ecy, rho),
// n = nn >= 16 sides, vertex k at polar angle 2 pi k / nn (unit table u64 = cos/sin(2 pi k / 64)).
// The ray's line meets the circle at polar angles theta + g (far side) and theta + pi - g (near
// side), g = asin(-hc / rho); between circle and polygon lies the circular segment of exactly one
// edge, so the polygon crossing is on the edge whose angular span contains that angle.  The
// neighbour on the nearer side is tested too (FP32 error of asinf near span boundaries).  With the
// own-ship outside the circle the near side alone decides: a line that does not cross the edge under
// its entry point leaves the circle through the same circular segment.  Vertices are formed on the
// fly from the FP32 centre (rounded once from the FP64 vessel-relative centre).
__device__ __forceinline__ float cast_ngon(float ecx, float ecy, float rho, int nn, const float2* __restrict__ u64,
                                           float c, float s, float theta, float tc, float hc, float best, float rangef) {
  const float g = asinf(fminf(fmaxf(-hc / rho, -1.f), 1.f));
  const float invd = (float)nn * 0.15915494309189535f;
  const int sh = 6 - (31 - __clz(nn));  // unit table stride 64 / nn
  const bool outside = tc * tc + hc * hc > rho * rho * 1.0001f + 1e-3f;
#pragma unroll
  for (int sol = 0; sol < 2; ++sol) {
    if (sol == 1 && outside) break;
    const float p = (sol == 0 ? theta + 3.14159265358979f - g : theta + g) * invd;
    const float kf = floorf(p);
    const int k0 = (int)kf;
    const int first = (p - kf < 0.5f) ? k0 - 1 : k0;  // edges (first, first+1), (first+1, first+2)
    float xp, yp;
    {
      const float2 un = u64[(first & (nn - 1)) << sh];
      const float vx = fmaf(rho, un.x, ecx), vy = fmaf(rho, un.y, ecy);
      xp = vx * c + vy * s;
      yp = vy * c - vx * s;
    }
#pragma unroll
    for (int w = 1; w <= 2; ++w) {
      const float2 un = u64[((first + w) & (nn - 1)) << sh];
      const float vx = fmaf(rho, un.x, ecx), vy = fmaf(rho, un.y, ecy);
      const float xc = vx * c + vy * s;
      const float yc = vy * c - vx * s;
      if ((yp <= 0.f && yc >= 0.f) || (yp >= 0.f && yc <= 0.f)) {
        const float t = xp + (xc - xp) * (yp / (yp - yc));
        if (t >= 0.f && t <= rangef) best = fminf(best, t);
      }
      xp = xc;
      yp = yc;
    }
  }
  return best;
}

// range of the ray (c, s) against a staged closed vertex chain vp[0..nq)
__device__ __forceinline__ float cast_chain(const float2* __restrict__ vp, int nq, float c, float s, float best,
                                            float rangef) {
  float2 v = vp[0];
  float xp = v.x * c + v.y * s;
  float yp = v.y * c - v.x * s;
  for (int k = 1; k < nq; ++k) {
    v = vp[k];
    const float xc = v.x * c + v.y * s;
    const float yc = v.y * c - v.x * s;
    if ((yp <= 0.f && yc >= 0.f) || (yp >= 0.f && yc <= 0.f)) {
      const float t = xp + (xc - xp) * (yp / (yp - yc));
      if (t >= 0.f && t <= rangef) best = fminf(best, t);
    }
    xp = xc;
    yp = yc;
  }
  return best;
}

// range row access: plain floats, or (velocity mode) 64-bit keys that carry the record index of
// the nearest hit -- ranges are >= 0, so both order like the values; ties go to the lower record
// index = the earlier obstacle of the nearby list (min((distance, i)), sensor.py:113-117)
template <bool VEL>
__device__ __forceinline__ float range_get(const void* row, int i) {
  if (VEL) return __uint_as_float((unsigned)(reinterpret_cast<const unsigned long long*>(row)[i] >> 32));
  return reinterpret_cast<const float*>(row)[i];
}
template <bool VEL>
__device__ __forceinline__ void range_min(void* row, int i, float d, int slot) {
  if (VEL)
    atomicMin(reinterpret_cast<unsigned long long*>(row) + i,
              ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)min(slot, 255));
  else
    atomicMin(reinterpret_cast<int*>(row) + i, __float_as_int(d));
}

#define AUV_LIDAR_MINB 5  // 48 registers (4 / 5 / 6 CTAs per SM: 0.0807 / 0.0767 / 0.101 ms)
// A world polygon with more vertices than a warp's vertex stage holds, cast chain by chain
// (consecutive chains share their end vertex).  Cold: land perimeters of thousands of vertices only.
template <bool VEL>
__device__ __noinline__ void cast_long_polygon(const double2* __restrict__ wv, int nq, int vmax, float2* wverts, double px,
                                               double py, double cpsi, double spsi, const double2* __restrict__ cos_sin,
                                               float ecx, float ecy, float rho, void* row, int slot, int lane, int n1, int n2,
                                               int lo1, int lo2, float rangef) {
  const float slack = rho * 1e-5f + 1e-4f;
  const int tot = n1 + n2;
  for (int v0 = 0; v0 < nq - 1; v0 += vmax - 1) {
    const int nqc = min(nq - v0, vmax);
    __syncwarp();
    for (int k = lane; k < nqc; k += 32) {
      const double2 w = wv[v0 + k];
      wverts[k] = make_float2((float)(w.x - px), (float)(w.y - py));
    }
    __syncwarp();
    for (int u = lane; u < tot; u += 32) {
      const int i = u < n1 ? lo1 + u : lo2 + (u - n1);
      const float cur = range_get<VEL>(row, i);
      const double2 cs = cos_sin[i];
      const float c = (float)(cs.x * cpsi - cs.y * spsi), sn = (float)(cs.y * cpsi + cs.x * spsi);
      const float tc = ecx * c + ecy * sn;
      const float hc = ecy * c - ecx * sn;
      if (fabsf(hc) > rho + slack || tc + rho + slack < 0.f || tc - rho - slack > cur) continue;
      const float got = cast_chain(wverts, nqc, c, sn, cur, rangef);
      if (got < cur) range_min<VEL>(row, i, got, slot);
    }
  }
}

// TRACK: record the episode tracks of AuvStepOut.tracks (instantiated with COUNT = false only)
template <bool COUNT, bool VEL, bool WORLD, bool TRACK = false>
__global__ void __launch_bounds__(AUV_LIDAR_THREADS, AUV_LIDAR_MINB) k_lidar(const __grid_constant__ LidarArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int NW = AUV_LIDAR_THREADS / 32;
  const AuvConfig& cfg = A.cfg;
  const AuvBatch& batch = A.batch;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int R = cfg.n_sensors;
  const int rpad = cfg.use_lidar ? ((R + 31) & ~31) : 32;
  const int E = A.envs_per_cta;
  const int env0 = A.e0 + blockIdx.x * E;
  const int ne = min(E, A.e1 - env0);
  const LidarSmem sm = lidar_carve(smem_raw, E, rpad, A.vmax, VEL ? 1 : 0);
  const float rangef = (float)cfg.sensor_range;
  const float widthf = (float)cfg.vessel_width;
  const int n = batch.n_envs;
#define HAND(el, k) sm.hand[(el) * 16 + ((k) - NAV_HAND)]

  // ---- phase 1: hand-over lines, unit table, range rows
  for (int k = tid; k < ne * 16; k += AUV_LIDAR_THREADS)
    sm.hand[k] = batch.nav[(long long)(env0 + (k >> 4)) * AUV_NAV_W + NAV_HAND + (k & 15)];
  if (cfg.use_lidar) {
    if (tid < 64) {
      const double2 un = reinterpret_cast<const double2*>(A.rays.unit64)[tid];
      sm.unit[tid] = make_float2((float)un.x, (float)un.y);
    }
    if (VEL) {
      const unsigned long long key0 = ((unsigned long long)__float_as_uint(rangef) << 32) | 255ull;
      for (int k = tid; k < ne * rpad; k += AUV_LIDAR_THREADS) reinterpret_cast<unsigned long long*>(sm.sdist)[k] = key0;
    } else {
      for (int k = tid; k < ne * rpad / 4; k += AUV_LIDAR_THREADS)
        reinterpret_cast<float4*>(sm.sdist)[k] = make_float4(rangef, rangef, rangef, rangef);
    }
  }
  __syncthreads();
  unsigned long long ntests = 0;
  if (cfg.use_lidar) {
    if (warp == 0) {  // exclusive scan of the record counts (E <= 32)
      const int c = lane < ne ? (int)HAND(lane, NAV_CNT) : 0;
      const int incl = warp_incl_scan(c, lane);
      sm.off[lane + 1] = incl;
      if (lane == 0) sm.off[0] = 0;
    }
    __syncthreads();
    const int total = sm.off[ne];
    const double2* __restrict__ unit = reinterpret_cast<const double2*>(A.rays.unit64);
    const double2* __restrict__ cos_sin = reinterpret_cast<const double2*>(A.rays.cos_sin);
    const float dth_f = (float)(2.0 * AUV_PI / (double)R);
    float2* wverts = sm.verts + (size_t)warp * A.vmax;
    for (int r0 = 0; r0 < total; r0 += AUV_LIDAR_RCAP) {
      const int nr = min(AUV_LIDAR_RCAP, total - r0);
      // ---- records of the round: 16-byte pieces, the env of a record by bisection of the scan
      for (int k = tid; k < nr * 5; k += AUV_LIDAR_THREADS) {
        const int r = r0 + k / 5, piece = k - (k / 5) * 5;
        int lo = 0, hi = ne - 1;  // last env with off[env] <= r
        while (lo < hi) {
          const int mid = (lo + hi + 1) >> 1;
          if (sm.off[mid] <= r) lo = mid; else hi = mid - 1;
        }
        const int idx = r - sm.off[lo];
        AUV_CHECK(batch.status, lo >= 0 && lo < ne && idx >= 0 && idx < batch.rec_cap && k < AUV_LIDAR_RCAP * 5);
        const uint4* g = reinterpret_cast<const uint4*>(reinterpret_cast<const ObstRec*>(batch.rec) +
                                                        (long long)(env0 + lo) * batch.rec_cap + idx);
        reinterpret_cast<uint4*>(sm.rec)[k] = g[piece];
        if (piece == 0) sm.rec_env[r - r0] = lo | (idx << 8);
      }
      __syncthreads();
      // ---- phase 2: warp per record
      for (int rr = warp; rr < nr; rr += NW) {
        const ObstRec& q = sm.rec[rr];
        const int el = sm.rec_env[rr] & 255, slot = sm.rec_env[rr] >> 8;
        const int fl = q.flags, nq = q.nv;
        AUV_CHECK(batch.status, rr < AUV_LIDAR_RCAP && el >= 0 && el < ne && slot >= 0 && slot < batch.rec_cap);
        // candidate rays of the record (sensor.py:93-95): i in I1 = [a,b) or i-R in [a,b), i.e.
        // I2 = [a+R, b+R), both clipped to [0,R).  An obstacle whose window is wider than R is
        // listed -- and tested -- twice upstream: the min does not care, so the part of I2 that
        // repeats I1 is dropped here (and counted in COUNT mode below).
        int n1, n2 = 0, lo1 = 0, lo2 = 0;
        if (fl & OFLAG_ALLRAYS) {
          n1 = R;
        } else {
          lo1 = max(q.a, 0);
          const int hi1 = min(q.b, R);
          n1 = max(0, hi1 - lo1);
          lo2 = max(q.a + R, 0);
          if (n1 > 0) lo2 = max(lo2, hi1);
          n2 = max(0, min(q.b + R, R) - lo2);
        }
        const int tot = n1 + n2;
        if (COUNT) {  // reference-semantics ray/segment tests of this record (bench / parity only)
          for (int i = lane; i < R; i += 32) {
            const int hits = ((q.a <= i && i < q.b) ? 1 : 0) + ((q.a <= i - R && i - R < q.b) ? 1 : 0);
            if ((fl & OFLAG_ALLRAYS) || hits > 0) ntests += (unsigned)((nq - 1) * max(hits, 1));
          }
        }
        if (tot == 0) continue;
        void* row = VEL ? (void*)(reinterpret_cast<unsigned long long*>(sm.sdist) + (size_t)el * rpad)
                        : (void*)(reinterpret_cast<float*>(sm.sdist) + (size_t)el * rpad);
        if (fl & OFLAG_INSIDE) {  // own-ship inside a filled boundary: every candidate ray reads 0
          for (int u = lane; u < tot; u += 32) range_min<VEL>(row, u < n1 ? lo1 + u : lo2 + (u - n1), 0.f, slot);
          continue;
        }
        const bool world = WORLD && (fl & OFLAG_WORLD);  // pools without land polygons run the instantiation without this path
        const bool ngon = !(fl & OFLAG_PENTAGON) && !world && nq > 16;
        if (!ngon) {
          if (nq > A.vmax) {
            // a world polygon with more vertices than the stage holds (land perimeters of any length): cast chain
            // by chain, out of line -- the hot loop below stays as small as it was without them
            if (world)
              cast_long_polygon<VEL>(reinterpret_cast<const double2*>(A.pool.world_verts) + q.vbase, nq, A.vmax, wverts,
                                     HAND(el, NAV_X), HAND(el, NAV_Y), HAND(el, NAV_COSPSI), HAND(el, NAV_SINPSI), cos_sin,
                                     q.ecx, q.ecy, q.rho, row, slot, lane, n1, n2, lo1, lo2, rangef);
            else if (lane == 0 && batch.status != nullptr)  // cannot happen (pentagon 6, small n-gon <= 9 vertices)
              atomicOr(batch.status, AUV_STATUS_POLY_TOO_LARGE);
            continue;
          }
          // stage the vertices: vessel-relative, formed in FP64, stored FP32
          __syncwarp();
          if (world) {
            const double px = HAND(el, NAV_X), py = HAND(el, NAV_Y);
            const double2* wv = reinterpret_cast<const double2*>(A.pool.world_verts) + q.vbase;
            for (int k = lane; k < nq; k += 32) {
              const double2 w = wv[k];
              wverts[k] = make_float2((float)(w.x - px), (float)(w.y - py));
            }
          } else if (fl & OFLAG_PENTAGON) {
            if (lane < 6) {
              double vx, vy;
              pent_vertex(lane == 5 ? 0 : lane, q.cx, q.cy, q.geo, q.hx, q.hy, vx, vy);
              wverts[lane] = make_float2((float)vx, (float)vy);
            }
          } else {  // small polygonised circle (2 / 4 / 8 sides) incl. the closing vertex
            const int ne_ = nq - 1, sh = 6 - (31 - __clz(ne_));
            if (lane < nq) {
              const double2 un = __ldg(&unit[(lane == ne_ ? 0 : lane) << sh]);
              wverts[lane] = make_float2((float)(q.cx + q.geo * un.x), (float)(q.cy + q.geo * un.y));
            }
          }
          __syncwarp();
        }
        const double cpsi = HAND(el, NAV_COSPSI), spsi = HAND(el, NAV_SINPSI);
        const float psi_m_pi = (float)(HAND(el, NAV_PSI) - AUV_PI);
        const float ecx = q.ecx, ecy = q.ecy, rho = q.rho;
        const float slack = rho * 1e-5f + 1e-4f;
        AUV_CHECK(batch.status, tot <= R && (n1 == 0 || (lo1 >= 0 && lo1 + n1 <= R)) && (n2 == 0 || (lo2 >= 0 && lo2 + n2 <= R)) &&
                                    (ngon || nq <= A.vmax));
        for (int u = lane; u < tot; u += 32) {
          const int i = u < n1 ? lo1 + u : lo2 + (u - n1);
          AUV_CHECK(batch.status, i >= 0 && i < R && i < rpad);
          const float cur = range_get<VEL>(row, i);
          // ray direction in the world frame, formed in FP64 (vessel.py:317)
          const double2 cs = cos_sin[i];
          const float c = (float)(cs.x * cpsi - cs.y * spsi), sn = (float)(cs.y * cpsi + cs.x * spsi);
          const float tc = ecx * c + ecy * sn;
          const float hc = ecy * c - ecx * sn;
          if (fabsf(hc) > rho + slack || tc + rho + slack < 0.f || tc - rho - slack > cur) continue;
          float got;
          if (ngon) {
            // world angle of ray i; only selects which polygon edge the analytic pick looks at
            const float theta = fmaf((float)(i + 1), dth_f, psi_m_pi);
            got = cast_ngon(ecx, ecy, rho, nq - 1, sm.unit, c, sn, theta, tc, hc, cur, rangef);
          } else {
            got = cast_chain(wverts, nq, c, sn, cur, rangef);
          }
          if (got < cur) range_min<VEL>(row, i, got, slot);
        }
      }
      __syncthreads();
    }
  }
  if (COUNT) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ntests += __shfl_xor_sync(AUV_FULL, ntests, o);
    if (lane == 0 && ntests) atomicAdd(A.out.seg_tests, ntests);
  }

  // ---- phase 3: warp per env -- closeness / collision / penalty / observation in one pass over the rays
  //      (vessel.py:88-95,356-359; rewarder.py:199-214; zeros without nearby obstacles: vessel.py:275-305)
  if (cfg.use_lidar) {
    const bool pooling = A.out.sector_min_dist != nullptr || A.out.sector_feasible_dist != nullptr;
    const bool vel_obs = cfg.sensor_use_velocity_observations != 0;
    const bool vec2 = (A.obs_dim & 1) == 0;  // rows and obs + 6 are 8-byte aligned
    const double2* __restrict__ cos_sin = reinterpret_cast<const double2*>(A.rays.cos_sin);
    for (int el = warp; el < ne; el += NW) {
      const int e = env0 + el;
      float* obs = A.out.obs + (long long)e * A.obs_dim;
      const int cnt = sm.off[el + 1] - sm.off[el];
      const void* row = VEL ? (const void*)(reinterpret_cast<const unsigned long long*>(sm.sdist) + (size_t)el * rpad)
                            : (const void*)(reinterpret_cast<const float*>(sm.sdist) + (size_t)el * rpad);
      float extra = 0.f;
      bool collision = false;
      if (cnt > 0) {
        const double cpsi = HAND(el, NAV_COSPSI), spsi = HAND(el, NAV_SINPSI);
        const ObstRec* grec = reinterpret_cast<const ObstRec*>(batch.rec) + (long long)e * batch.rec_cap;
        for (int k = lane; k < (R + 1) / 2; k += 32) {
          float cl2[2] = {0.f, 0.f};
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int i = 2 * k + h;
            if (i >= R) continue;
            const float d = range_get<VEL>(row, i);
            float vxr = 0.f, vyr = 0.f;
            if (d < rangef) {
              if (cfg.sensor_log_transform)  // log(1 + d) by the hardware log2: |error| < 1e-6 of a value in [0, 5]
                cl2[h] = 1.f - fminf(fmaxf(__logf(1.f + d) * A.inv_log_range, 0.f), 1.f);
              else
                cl2[h] = 1.f - fminf(fmaxf(d / rangef, 0.f), 1.f);
              cl2[h] = fminf(fmaxf(cl2[h], -1.f), 1.f);
              if (VEL) {
                // sensor.py:118-128: Rz(-theta - pi/2) (dx, dy) of the nearest obstacle hit by the ray
                const int slot = (int)(reinterpret_cast<const unsigned long long*>(row)[i] & 255ull);
                const ObstRec& q = grec[slot];
                if (q.flags & OFLAG_PENTAGON) {
                  const double2 cs = cos_sin[i];
                  const double c = cs.x * cpsi - cs.y * spsi, sn = cs.y * cpsi + cs.x * spsi;
                  const double dx = (double)q.step_len * q.hx, dy = (double)q.step_len * q.hy;
                  vxr = (float)(-sn * dx + c * dy);
                  vyr = (float)(-c * dx - sn * dy);
                }
              }
              extra += A.rays.weight[i] * (rangef * __expf(-0.1f * d + fmaxf(0.f, vyr)) - A.pen_clear_ray);
              collision = collision || (d < widthf);
            }
            if (vel_obs) {
              obs[6 + R + i] = fminf(fmaxf(vxr, -1.f), 1.f);
              obs[6 + 2 * R + i] = fminf(fmaxf(vyr, -1.f), 1.f);
            }
            if (!vec2) obs[6 + i] = cl2[h];
          }
          if (vec2) {
            if (2 * k + 1 < R)
              reinterpret_cast<float2*>(obs + 6)[k] = make_float2(cl2[0], cl2[1]);
            else
              obs[6 + 2 * k] = cl2[0];
          }
        }
        collision = __any_sync(AUV_FULL, collision);
        extra = warp_sum(extra);
      } else {
        if (vec2) {
          float2* o2 = reinterpret_cast<float2*>(obs + 6);
          for (int k = lane; k < R / 2; k += 32) o2[k] = make_float2(0.f, 0.f);
          if ((R & 1) && lane == 0) obs[6 + R - 1] = 0.f;
        } else {
          for (int i = lane; i < R; i += 32) obs[6 + i] = 0.f;
        }
        if (vel_obs)
          for (int k = lane; k < 2 * R; k += 32) obs[6 + R + k] = 0.f;
      }
      if (lane == 0) {
        sm.pen[el] = extra;
        sm.flag[el] = collision ? 1 : 0;
      }
      if (A.out.lidar_dist != nullptr)
        for (int i = lane; i < R; i += 32) A.out.lidar_dist[(long long)e * R + i] = range_get<VEL>(row, i);

      // ---- optional sector pooling (utils/sector_partitioning.py:4-9; sensor.py:215-296)
      if (pooling) {
        const int ns = cfg.n_sectors;
        float* prow = reinterpret_cast<float*>(sm.verts + (size_t)warp * A.vmax);  // vertex stage is free again
        float* ssec = prow;                // [32] sector minima
        __syncwarp();
        ssec[lane] = rangef;
        __syncwarp();
        // min-pooling: segmented warp-shuffle reduction keyed by the ray's sector id
        for (int i0 = 0; i0 < R; i0 += 32) {
          const int i = i0 + lane;
          float d = i < R ? range_get<VEL>(row, i) : INFINITY;
          const int sid = i < R ? (int)A.rays.sector[i] : -1 - lane;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const float od = __shfl_down_sync(AUV_FULL, d, o);
            const int os = __shfl_down_sync(AUV_FULL, sid, o);
            if (lane + o < 32 && os == sid) d = fminf(d, od);
          }
          const int ps = __shfl_up_sync(AUV_FULL, sid, 1);
          const bool head = i < R && (lane == 0 || ps != sid);
          if (head && sid < 32) ssec[sid] = fminf(ssec[sid], d);  // one head per sector per iteration
          __syncwarp();
        }
        if (A.out.sector_min_dist != nullptr && lane < ns) A.out.sector_min_dist[(long long)e * ns + lane] = ssec[lane];
        if (A.out.sector_feasible_dist != nullptr) {
          // the pooling routine reads plain float ranges: velocity mode keeps keys, so it gets a copy
          const float* frow;
          if (VEL) {
            float* tmp = reinterpret_cast<float*>(const_cast<void*>(row));  // compact the keys in place (row is done)
            __syncwarp();
            for (int i0 = 0; i0 < R; i0 += 32) {
              const int i = i0 + lane;
              const float d = i < R ? range_get<VEL>(row, i) : 0.f;
              __syncwarp();
              if (i < R) tmp[i] = d;
              __syncwarp();
            }
            frow = tmp;
          } else {
            frow = reinterpret_cast<const float*>(row);
          }
          if (lane < ns) {
            int lo = 0, hi = R;
            for (int k = 0; k < R; ++k) {  // the sector table is monotone
              const int sd = A.rays.sector[k];
              if (sd < lane) lo = k + 1;
              if (sd <= lane) hi = k + 1;
            }
            A.out.sector_feasible_dist[(long long)e * ns + lane] =
                hi > lo ? feasibility_pooling(frow + lo, hi - lo, A.feas_width, 2.0 * AUV_PI / (double)R) : rangef;
          }
        }
        __syncwarp();
      }
    }
  }
  __syncthreads();

  // ---- phase 4: thread per env -- reward (rewarder.py) + done (environment.py:375-384) + counters;
  //      k_vessel_nav computed everything that does not depend on the LiDAR.  obs[0..5] is its too.
  if (warp == 0 && lane < ne) {
    const int el = lane, e = env0 + el;
    const bool collision = cfg.use_lidar && (sm.flag[el] & 1);
    const double progress = HAND(el, NAV_H_PROGRESS), goal_dist = HAND(el, NAV_H_GOAL);
    const bool reached = HAND(el, NAV_REACHED) != 0.0;
    int fl = 0;
    if (A.mode == AUV_OBSERVE_RESET) {  // explicit reset observe: info mirrors a fresh env
      if (A.out.collision) A.out.collision[e] = collision;
      if (A.out.reached_goal) A.out.reached_goal[e] = reached;
      if (A.out.goal_distance) A.out.goal_distance[e] = (float)goal_dist;
      if (A.out.progress) A.out.progress[e] = (float)progress;
    } else {
      double reward = HAND(el, NAV_REWARD_BASE);
      if (collision) {
        reward = -10000.0 * (1.0 - 0.5);
      } else if (cfg.rewarder == AUV_REWARDER_COLAV) {
        // without LiDAR every ray keeps its reset value sensor_range (vessel.py:206-208)
        const float pen = (float)A.rays.weight_sum * A.pen_clear_ray + sm.pen[el];
        const double closeness_reward = cfg.use_lidar ? -(double)pen * A.inv_weight_sum : A.clear_closeness;
        reward += 0.5 * closeness_reward;
        if (reward < 0.0) reward *= 2.0;
      }
      const double y_e = HAND(el, NAV_H_YE);
      const double cum = HAND(el, NAV_CUM) + reward;
      const int t_step = (int)HAND(el, NAV_TSTEP);
      const bool done = collision || reached || (!cfg.test_mode && t_step >= cfg.max_timesteps - 1) ||
                        (!cfg.test_mode && cum < cfg.min_cumulative_reward);
      const double cte_sum = HAND(el, NAV_CTE) + fabs(y_e);
      const bool do_reset = done && cfg.auto_reset;
      const int scn = (int)HAND(el, NAV_SCN);
      A.out.reward[e] = (float)reward;
      A.out.done[e] = done;
      if (A.out.collision) A.out.collision[e] = collision;
      if (A.out.reached_goal) A.out.reached_goal[e] = reached;
      if (A.out.goal_distance) A.out.goal_distance[e] = (float)goal_dist;
      if (A.out.progress) A.out.progress[e] = (float)progress;
      if (done && A.out.episode_out != nullptr) {  // env.history entry of the finished episode
        float4* eo = reinterpret_cast<float4*>(A.out.episode_out + 8ll * e);
        eo[0] = make_float4((float)cum, (float)(t_step + 1), (float)progress, collision ? 1.f : 0.f);
        eo[1] = make_float4(reached ? 1.f : 0.f, (float)(cte_sum / (double)(t_step + 1)),
                            (float)A.paths.hdr[batch.env_pid[e]].length, (float)batch.episode[e]);
      }
      if (TRACK && e % A.trk.stride == 0 && e / A.trk.stride < A.trk.count) {
        // episode track: the point of this step and the row's head (row = parity of the episode,
        // read before the auto-reset below moves the counter on)
        const int ep = batch.episode[e];
        const long long row = 2ll * (e / A.trk.stride) + (ep & 1);
        reinterpret_cast<float4*>(A.trk.points)[row * A.trk.capacity + t_step % A.trk.capacity] =
            make_float4((float)HAND(el, NAV_X), (float)HAND(el, NAV_Y), (float)HAND(el, NAV_PSI), (float)reward);
        int4* hd = reinterpret_cast<int4*>(A.trk.head + 8 * row);
        hd[0] = make_int4(ep, t_step + 1, done ? 1 : 0, collision ? 1 : 0);
        hd[1] = make_int4(reached ? 1 : 0, scn, batch.obst_steps[e], 0);
        if (done) fl = 4 | ((ep & 1) << 3);  // snapshot of the finished scenario in the bulk part
      }
      if (!do_reset) {
        batch.cum_reward[e] = cum;
        batch.t_step[e] = t_step + 1;
        batch.cte_sum[e] = cte_sum;
      } else {
        // ---- VecEnv auto-reset, scalar part.  The first observation of an episode depends on the
        // scenario only, so it was computed once per pool scenario (pool.reset_*) and the reset
        // is a copy: no navigation / culling / casting on the step path.
        const int next = (int)(((long long)scn + (batch.reset_stride > 0 ? batch.reset_stride : n)) % A.pool.n_scenarios);
        const int npid = A.pool.path_id[next];
        if (A.out.stats != nullptr) {  // env.history entry, environment.py:476-489
          double* st = A.out.stats;
          atomicAdd(st + AUV_STAT_EPISODES, 1.0);
          atomicAdd(st + AUV_STAT_REWARD, cum);
          atomicAdd(st + AUV_STAT_REWARD_SQ, cum * cum);
          atomicAdd(st + AUV_STAT_PROGRESS, progress);
          atomicAdd(st + AUV_STAT_COLLISIONS, collision ? 1.0 : 0.0);
          atomicAdd(st + AUV_STAT_REACHED_GOAL, reached ? 1.0 : 0.0);
          atomicAdd(st + AUV_STAT_TIMESTEPS, (double)(t_step + 1));
          atomicAdd(st + AUV_STAT_CROSS_TRACK, cte_sum / (double)(t_step + 1));
          atomicAdd(st + AUV_STAT_PATHLENGTH, A.paths.hdr[batch.env_pid[e]].length);
        }
        batch.scn_id[e] = next;
        batch.env_pid[e] = npid;
        batch.prev_seg[e] = -1;
        batch.obst_steps[e] = 0;
        batch.episode[e] += 1;
        const double* vi = A.pool.vessel_init + 3ll * next;
        batch.state[e] = vi[0];
        batch.state[n + e] = vi[1];
        batch.state[2ll * n + e] = vi[2];
        batch.state[3ll * n + e] = 0.0;
        batch.state[4ll * n + e] = 0.0;
        batch.state[5ll * n + e] = 0.0;
        batch.step_counter[e] = 0;
        batch.t_step[e] = 0;
        batch.cum_reward[e] = 0.0;
        batch.cte_sum[e] = 0.0;
        batch.max_progress[e] = A.pool.reset_max_progress[next];
        sm.next[el] = next;
        fl |= 2;
      }
    }
    sm.flag[el] = fl;
  }
  __syncthreads();
  // ---- auto-reset, bulk part (a warp per finished env): terminal obs out, cached first obs in,
  //      obstacle state (table-driven tracks only) and nearby list of the next scenario
  //      (TRACK) and the snapshot of the scenario a tracked env finished: its pool slot still holds it
  for (int el = warp; el < ne; el += NW) {
    if (TRACK) {
      const int tf = sm.flag[el];
      if (!(tf & 6)) continue;
      if (tf & 4) {
        const int e = env0 + el, scn = (int)HAND(el, NAV_SCN);
        const int km = A.pool.k_moving, ks = A.pool.k_static, w = 4 + 8 * km + 4 * ks;
        double* sn = A.trk.snap + (2ll * (e / A.trk.stride) + ((tf >> 3) & 1)) * w;
        for (int k = lane; k < w; k += 32) {
          double v;
          if (k == 0) v = (double)A.pool.path_id[scn];
          else if (k < 4) v = A.pool.vessel_init[3ll * scn + (k - 1)];
          else if (k < 4 + 8 * km) v = A.pool.mov_lin ? A.pool.mov_lin[8ll * km * scn + (k - 4)] : 0.0;
          else v = A.pool.st_rec[4ll * ks * scn + (k - 4 - 8 * km)];
          sn[k] = v;
        }
      }
      if (!(tf & 2)) continue;
    } else if (!(sm.flag[el] & 2)) {
      continue;
    }
    const int e = env0 + el, next = sm.next[el];
    const int km = A.pool.k_moving;
    float* obs = A.out.obs + (long long)e * A.obs_dim;
    const float* robs = A.pool.reset_obs + (long long)next * A.obs_dim;
    float* tobs = A.out.terminal_obs ? A.out.terminal_obs + (long long)e * A.obs_dim : nullptr;
    for (int k = lane; k < A.obs_dim; k += 32) {
      if (tobs) tobs[k] = obs[k];
      obs[k] = robs[k];
    }
    if (!A.pool.linear_tracks)
      for (int j = lane; j < km; j += 32) {
        const long long ps = (long long)next * km + j, pe = (long long)e * km + j;
        reinterpret_cast<double2*>(batch.mov_pos)[pe] = reinterpret_cast<const double2*>(A.pool.mov_pos0)[ps];
        reinterpret_cast<double2*>(batch.mov_disp)[pe] = reinterpret_cast<const double2*>(A.pool.mov_disp0)[ps];
        batch.mov_counter[pe] = A.pool.mov_counter0[ps];
      }
    if (cfg.use_lidar)
      for (int w = lane; w < batch.mask_words; w += 32)
        batch.nearby_mask[(long long)e * batch.mask_words + w] = A.pool.reset_mask[(long long)next * batch.mask_words + w];
  }
#undef HAND
}

// ------------------------------------------------------------------------------------
// k_obs_ship: lossless compact transfer of a step's results to the host.  ~85 % of the closeness
// block of an observation is exactly 0 (clear rays), and the dense [N][6 + R] float rows are what
// bounds the host-buffer step (49 MB per 65536 envs over PCIe).  One CTA per 32 envs turns its rows
// into: a 32 B head per env (obs[0..5], count, offset), the hit mask (one bit per ray) and the
// non-zero values packed back to back -- and writes all three, plus reward / done, STRAIGHT into
// pinned host memory with coalesced stores (the packed block of a CTA is contiguous and 128 B
// aligned): the kernel's own stores are the transfer, its exact size is decided on the device,
// and the whole step stays one replayable CUDA graph.  auv_compact_expand scatters on the host.
// ------------------------------------------------------------------------------------
#define AUV_SHIP_THREADS 256
#define AUV_SHIP_ENVS 32
__global__ void __launch_bounds__(AUV_SHIP_THREADS) k_obs_ship(const float* __restrict__ obs, int obs_dim, int R, int words,
                                                              int e0, int e1, const float* __restrict__ reward,
                                                              const uint8_t* __restrict__ done, float* __restrict__ head_h,
                                                              uint32_t* __restrict__ mask_h, float* __restrict__ vals_h,
                                                              int* __restrict__ counter, int capacity,
                                                              float* __restrict__ reward_h, uint8_t* __restrict__ done_h) {
  extern __shared__ __align__(16) unsigned char ship_smem[];
  const int rpad = words * 32;
  float* s_vals = reinterpret_cast<float*>(ship_smem);                       // [E][rpad] packed per env
  uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_vals + AUV_SHIP_ENVS * rpad);  // [E][words]
  int* s_off = reinterpret_cast<int*>(s_mask + AUV_SHIP_ENVS * words);       // [E + 1]
  __shared__ int s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int env0 = e0 + blockIdx.x * AUV_SHIP_ENVS;
  const int ne = min(AUV_SHIP_ENVS, e1 - env0);
  // ---- pack: warp per env
  for (int el = warp; el < ne; el += AUV_SHIP_THREADS / 32) {
    const float* row = obs + (long long)(env0 + el) * obs_dim + 6;
    int run = 0;
    for (int w = 0; w < words; ++w) {
      const int i = w * 32 + lane;
      const float v = i < R ? row[i] : 0.f;
      const unsigned m = __ballot_sync(AUV_FULL, v != 0.f);
      if (v != 0.f) s_vals[el * rpad + run + __popc(m & ((1u << lane) - 1u))] = v;
      if (lane == 0) s_mask[el * words + w] = m;
      run += __popc(m);
    }
    if (lane == 0) s_off[el + 1] = run;  // counts for now
  }
  __syncthreads();
  if (warp == 0) {  // exclusive scan of the counts; one reservation per CTA, padded to 32 floats (128 B)
    const int c = lane < ne ? s_off[lane + 1] : 0;
    const int incl = warp_incl_scan(c, lane);
    __syncwarp();
    s_off[lane + 1] = incl;
    if (lane == 0) s_off[0] = 0;
    const int total = __shfl_sync(AUV_FULL, incl, 31);
    if (lane == 0) s_base = total > 0 ? atomicAdd(counter, (total + 31) & ~31) : 0;
  }
  __syncthreads();
  const int base = s_base, total = s_off[ne];
  // ---- ship: head, mask, reward, done (contiguous per CTA), packed values (flat, coalesced)
  for (int k = tid; k < ne * 8; k += AUV_SHIP_THREADS) {
    const int el = k >> 3, f = k & 7;
    float v;
    if (f < 6) v = obs[(long long)(env0 + el) * obs_dim + f];
    else if (f == 6) v = __int_as_float(s_off[el + 1] - s_off[el]);
    else v = __int_as_float(base + s_off[el]);
    head_h[(long long)env0 * 8 + k] = v;
  }
  for (int k = tid; k < ne * words; k += AUV_SHIP_THREADS) mask_h[(long long)env0 * words + k] = s_mask[k];
  if (tid < ne) {
    reward_h[env0 + tid] = reward[env0 + tid];
    done_h[env0 + tid] = done[env0 + tid];
  }
  if (base + total <= capacity)
    for (int k = tid; k < total; k += AUV_SHIP_THREADS) {
      int lo = 0, hi = ne - 1;  // env of packed value k: last env with off <= k
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s_off[mid] <= k) lo = mid; else hi = mid - 1;
      }
      vals_h[base + k] = s_vals[lo * rpad + (k - s_off[lo])];
    }
}

// ------------------------------------------------------------------------------------
// Delta transfer (auv_step_host_delta_submit): the dense observation array of the caller lives
// in pinned host memory and keeps its content between steps; `shadow` is the device's copy of
// what it holds.  A thread owns one 16 B quad of the flat [N * obs_dim] array, a chunk is `g4`
// consecutive quads (2 / 4 / 8: 32 / 64 / 128 B) of one warp; a chunk is stored -- to the host
// array and to the shadow -- iff any of its words differs bitwise.  The stores of a chunk are one
// contiguous, aligned run, so the link sees whole 32 / 64 / 128 B writes.
// ------------------------------------------------------------------------------------
#define AUV_DELTA_THREADS 64
#define AUV_DELTA_UNROLL 2
// The kernel is bound by the host link, not by the SMs: it runs as a SMALL persistent grid (two
// CTAs of 64 threads x 40 registers per SM: one fits into the registers five k_lidar
// CTAs leave over) that strides over the range, so that its warps -- stalled on the link's write
// queue most of the time -- leave the SMs to the step kernels of the next env range / env group
// running beside it.  (One CTA per 256 quads, the first version, filled every
// CTA slot of the GPU with stalled warps: the step kernels of the other stream waited for it.)
__global__ void __launch_bounds__(AUV_DELTA_THREADS, 24) k_obs_delta(const float* __restrict__ obs, float* __restrict__ shadow,
                                                                float* __restrict__ obs_h, long long f0, long long f1, int g4,
                                                                const float* __restrict__ reward,
                                                                const uint8_t* __restrict__ done, float* __restrict__ reward_h,
                                                                uint8_t* __restrict__ done_h, int e0, int e1,
                                                                unsigned long long* __restrict__ shipped) {
  const int lane = threadIdx.x & 31;
  const long long nthreads = (long long)gridDim.x * AUV_DELTA_THREADS;
  const long long gtid = (long long)blockIdx.x * AUV_DELTA_THREADS + threadIdx.x;
  for (long long e = e0 + gtid; e < e1; e += nthreads) {
    reward_h[e] = reward[e];
    done_h[e] = done[e];
  }
  const long long qfull = f1 >> 2, qend = (f1 + 3) >> 2;  // quads wholly inside the range / touched by it (f0 is a multiple of 4)
  const unsigned cm = (g4 >= 32 ? 0xffffffffu : ((1u << g4) - 1u)) << (lane & ~(g4 - 1));
  unsigned count = 0u;
  // qb = the quad of lane 0: the trip count is uniform in the warp
  for (long long qb = (f0 >> 2) + gtid - lane; qb < qend; qb += nthreads * AUV_DELTA_UNROLL) {
    uint4 cur[AUV_DELTA_UNROLL], old[AUV_DELTA_UNROLL];
#pragma unroll
    for (int u = 0; u < AUV_DELTA_UNROLL; ++u) {
      const long long q = qb + u * nthreads + lane;
      cur[u] = old[u] = make_uint4(0u, 0u, 0u, 0u);
      if (q < qfull) {
        cur[u] = __ldcs(reinterpret_cast<const uint4*>(obs) + q);
        old[u] = __ldcs(reinterpret_cast<const uint4*>(shadow) + q);
      }
    }
#pragma unroll
    for (int u = 0; u < AUV_DELTA_UNROLL; ++u) {
      const long long q = qb + u * nthreads + lane;
      const bool full = q < qfull, part = !full && q < qend;
      bool changed = (cur[u].x != old[u].x) | (cur[u].y != old[u].y) | (cur[u].z != old[u].z) | (cur[u].w != old[u].w);
      if (part)
        for (long long i = q << 2; i < f1; ++i) changed |= __float_as_uint(obs[i]) != __float_as_uint(shadow[i]);
      const unsigned any = __ballot_sync(AUV_FULL, changed);
      const bool ship = (any & cm) != 0u;
      if (ship) {
        if (full) {
          reinterpret_cast<uint4*>(obs_h)[q] = cur[u];
          reinterpret_cast<uint4*>(shadow)[q] = cur[u];
        } else if (part) {
          for (long long i = q << 2; i < f1; ++i) obs_h[i] = shadow[i] = obs[i];
        }
      }
      count += __popc(__ballot_sync(AUV_FULL, ship && (full || part) && (lane & (g4 - 1)) == 0));
    }
  }
  if (shipped != nullptr && lane == 0 && count) atomicAdd(shipped, (unsigned long long)count);
}

// ------------------------------------------------------------------------------------
// FP32 FMA peak probe: 8 independent FMA chains per thread
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_fma_probe(float* sink, int iters) {
  float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
  float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
  const float m = 0.999f, c = 1e-3f;
  for (int i = 0; i < iters; ++i) {
    a0 = fmaf(a0, m, c);
    a1 = fmaf(a1, m, c);
    a2 = fmaf(a2, m, c);
    a3 = fmaf(a3, m, c);
    a4 = fmaf(a4, m, c);
    a5 = fmaf(a5, m, c);
    a6 = fmaf(a6, m, c);
    a7 = fmaf(a7, m, c);
  }
  const float r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (r == 12345.678f) sink[0] = r;  // never true; keeps the chains alive
}

}  // namespace auv

#include "auv_render.cuh"

// ======================================================================================
// C ABI
// ======================================================================================
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>

static thread_local char g_err[512] = "";

static int set_err(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}
static int cuda_check(cudaError_t e, const char* where) {
  if (e == cudaSuccess) return 0;
  snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
  return (int)e;
}

extern "C" {

static int check_pool_tracks(const AuvScenarioPool* pool, const AuvBatch* batch);

int auv_abi_version(void) { return AUV_ABI_VERSION; }
int auv_sizeof(int which) {
  switch (which) {
    case 0: return (int)sizeof(AuvConfig);
    case 1: return (int)sizeof(AuvRayTable);
    case 2: return (int)sizeof(AuvPathBank);
    case 3: return (int)sizeof(AuvScenarioPool);
    case 4: return (int)sizeof(AuvBatch);
    case 5: return (int)sizeof(AuvStepOut);
    case 6: return (int)sizeof(AuvGenParams);
    case 7: return (int)sizeof(AuvPathHdr);
    case 8: return (int)sizeof(AuvRefreshScratch);
    case 9: return (int)sizeof(AuvCompact);
    case 10: return (int)sizeof(AuvPathBuild);
    case 11: return (int)sizeof(AuvDelta);
    case 12: return (int)sizeof(AuvTracks);
    case 13: return (int)sizeof(AuvRender);
    default: return AUV_EINVAL;
  }
}
const char* auv_last_error(void) { return g_err; }

int auv_obs_dim(const AuvConfig* cfg) {
  if (!cfg) return AUV_EINVAL;
  int d = 6;
  if (cfg->use_lidar) {
    d += cfg->n_sensors;
    if (cfg->sensor_use_velocity_observations) d += 2 * cfg->n_sensors;
  }
  return d;
}

static int check_cfg(const AuvConfig* cfg) {
  if (!cfg) return set_err(AUV_EINVAL, "cfg is NULL");
  if (cfg->use_lidar && (cfg->n_sensors <= 0 || cfg->n_sensors > AUV_MAX_RAYS))
    return set_err(AUV_EINVAL, "n_sensors out of range");
  if (!(cfg->t_step_size > 0.0)) return set_err(AUV_EINVAL, "t_step_size must be > 0");
  if (cfg->sensor_interval_load_obstacles <= 0)
    return set_err(AUV_EINVAL, "sensor_interval_load_obstacles must be > 0");
  if (cfg->use_lidar && (cfg->n_sectors <= 0 || cfg->n_sectors > 32))
    return set_err(AUV_EINVAL, "n_sectors must be in 1..32");
  return 0;
}

static int launch_obstacle_update(const AuvConfig* cfg, const AuvScenarioPool* pool, const AuvBatch* batch,
                                  int e0, int cnt, void* stream) {
  const long long total = (long long)cnt * pool->k_moving;
  if (total == 0) return 0;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  auv::k_obstacle_update<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(*cfg, *pool, *batch, e0, cnt);
  return cuda_check(cudaGetLastError(), "k_obstacle_update");
}

int auv_obstacle_update(const AuvConfig* cfg, const AuvScenarioPool* pool, AuvBatch* batch,
                        void* stream) {
  if (int rc = check_cfg(cfg)) return rc;
  if (!pool || !batch) return set_err(AUV_EINVAL, "pool/batch is NULL");
  if (batch->n_envs <= 0) return set_err(AUV_EINVAL, "n_envs must be > 0");
  if (!batch->obst_steps) return set_err(AUV_EINVAL, "batch.obst_steps is NULL");
  if (int rc = check_pool_tracks(pool, batch)) return rc;
  return launch_obstacle_update(cfg, pool, batch, 0, batch->n_envs, stream);
}

int auv_vessel_step(const AuvConfig* cfg, AuvBatch* batch, const float* actions, void* stream) {
  if (int rc = check_cfg(cfg)) return rc;
  if (!batch || !actions) return set_err(AUV_EINVAL, "batch/actions is NULL");
  if (batch->n_envs <= 0) return set_err(AUV_EINVAL, "n_envs must be > 0");
  const int threads = 128;
  const int blocks = (batch->n_envs + threads - 1) / threads;
  auv::k_vessel_step<<<blocks, threads, 0, (cudaStream_t)stream>>>(*cfg, *batch, actions);
  return cuda_check(cudaGetLastError(), "k_vessel_step");
}

int auv_reset(const AuvConfig* cfg, const AuvScenarioPool* pool, AuvBatch* batch,
              const uint8_t* reset_mask, void* stream) {
  if (int rc = check_cfg(cfg)) return rc;
  if (!pool || !batch) return set_err(AUV_EINVAL, "pool/batch is NULL");
  if (batch->n_envs <= 0) return set_err(AUV_EINVAL, "n_envs must be > 0");
  if (!batch->obst_steps || !batch->prev_seg || !batch->env_pid)
    return set_err(AUV_EINVAL, "batch.obst_steps / prev_seg / env_pid is NULL");
  if (int rc = check_pool_tracks(pool, batch)) return rc;
  const int threads = 128;
  const int blocks = (batch->n_envs + threads - 1) / threads;
  auv::k_reset<<<blocks, threads, 0, (cudaStream_t)stream>>>(*pool, *batch, reset_mask);
  return cuda_check(cudaGetLastError(), "k_reset");
}

static int check_pool_tracks(const AuvScenarioPool* pool, const AuvBatch* batch) {
  if (pool->k_static > 0 && !pool->st_rec) return set_err(AUV_EINVAL, "pool.st_rec is NULL (auv_pool_pack)");
  if (pool->k_moving > 0) {
    if (pool->linear_tracks) {
      if (!pool->mov_lin) return set_err(AUV_EINVAL, "pool.mov_lin is NULL with linear_tracks (auv_pool_pack)");
      if (pool->lin_first_wrap <= 0 || pool->lin_wrap_period <= 0)
        return set_err(AUV_EINVAL, "pool.lin_first_wrap / lin_wrap_period not set (auv_linear_wrap)");
    } else if (!batch->mov_pos || !batch->mov_disp || !batch->mov_counter) {
      return set_err(AUV_EINVAL, "batch.mov_pos / mov_disp / mov_counter is NULL with table-driven tracks");
    }
  }
  return 0;
}

static int check_batch(const AuvConfig* cfg, const AuvScenarioPool* pool, const AuvBatch* batch) {
  if (batch->n_envs <= 0) return set_err(AUV_EINVAL, "n_envs must be > 0");
  if (!batch->nav) return set_err(AUV_EINVAL, "batch.nav is NULL");
  if (pool->n_world < 0) return set_err(AUV_EINVAL, "n_world < 0");
  const int slots = pool->k_moving + pool->k_static + pool->n_world;
  if (slots > AUV_MAX_OBSTACLES) return set_err(AUV_EINVAL, "too many obstacle slots");
  if (batch->mask_words * 32 < slots) return set_err(AUV_EINVAL, "mask_words too small");
  if (pool->n_world > 0 && (!pool->world_circle || !pool->world_voff || !pool->world_verts))
    return set_err(AUV_EINVAL, "world arrays are NULL");
  if (cfg->use_lidar && (!batch->rec_cnt || (slots > 0 && (!batch->rec || batch->rec_cap <= 0))))
    return set_err(AUV_EINVAL, "batch.rec / rec_cnt / rec_cap missing");
  if (!batch->obst_steps || !batch->prev_seg || !batch->env_pid)
    return set_err(AUV_EINVAL, "batch.obst_steps / prev_seg / env_pid is NULL");
  if (int rc = check_pool_tracks(pool, batch)) return rc;
  return 0;
}

// AuvStepOut.tracks (NULL = no recording): checked before any device work
static int check_tracks(const AuvStepOut* out, const AuvBatch* batch) {
  const AuvTracks* t = out->tracks;
  if (t == nullptr) return 0;
  if (!t->points || !t->head || !t->snap) return set_err(AUV_EINVAL, "tracks: points / head / snap is NULL");
  if (t->count < 1 || t->stride < 1 || t->capacity < 1)
    return set_err(AUV_EINVAL, "tracks: count, stride and capacity must be >= 1");
  if ((long long)(t->count - 1) * t->stride >= (long long)batch->n_envs)
    return set_err(AUV_EINVAL, "tracks: (count - 1) * stride must be < n_envs");
  if ((size_t)t->points & 15u) return set_err(AUV_EINVAL, "tracks: points must be 16-byte aligned");
  if ((size_t)t->head & 15u) return set_err(AUV_EINVAL, "tracks: head must be 16-byte aligned");
  if ((size_t)t->snap & 7u) return set_err(AUV_EINVAL, "tracks: snap must be 8-byte aligned");
  if (out->seg_tests != nullptr) return set_err(AUV_EINVAL, "tracks cannot be recorded together with out.seg_tests");
  return 0;
}

static int check_observe_args(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                              const AuvScenarioPool* pool, AuvBatch* batch, AuvStepOut* out, int mode) {
  if (int rc = check_cfg(cfg)) return rc;
  if (!paths || !pool || !batch || !out) return set_err(AUV_EINVAL, "NULL argument");
  if (int rc = check_tracks(out, batch)) return rc;
  if (cfg->use_lidar && (!rays || !rays->unit64 || !rays->cos_sin || !rays->weight || !rays->sector))
    return set_err(AUV_EINVAL, "ray table is NULL with use_lidar");
  if (!out->obs) return set_err(AUV_EINVAL, "out.obs is NULL");
  if (mode == AUV_OBSERVE_STEP && (!out->reward || !out->done))
    return set_err(AUV_EINVAL, "out.reward/out.done is NULL");
  if (mode == AUV_OBSERVE_STEP && cfg->auto_reset &&
      (!pool->reset_obs || !pool->reset_max_progress || (cfg->use_lidar && !pool->reset_mask)))
    return set_err(AUV_EINVAL, "auto_reset needs the pool's cached first observations (pool.reset_*)");
  return check_batch(cfg, pool, batch);
}

static int nav_configure(size_t smem) {
  if (smem <= 48 * 1024) return 0;
  static std::atomic<size_t> configured[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  if (smem <= configured[dev].load(std::memory_order_acquire)) return 0;
  const void* fns[3] = {(const void*)auv::k_vessel_nav<true, true, AUV_NAV_G>, (const void*)auv::k_vessel_nav<true, false, AUV_NAV_G>,
                        (const void*)auv::k_vessel_nav<false, false, AUV_NAV_G>};
  for (int i = 0; i < 3; ++i)
    if (int rc = cuda_check(cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                            "cudaFuncSetAttribute(k_vessel_nav)"))
      return rc;
  configured[dev].store(smem, std::memory_order_release);
  return 0;
}

static int launch_vessel_nav(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                             const AuvScenarioPool* pool, AuvBatch* batch, AuvStepOut* out,
                             const float* actions, void* stream, int e0 = 0, int cnt = -1, bool with_obstacles = false,
                             cudaEvent_t between = nullptr /* recorded between the two launches (auv_step_timed) */) {
  if ((paths->sub_chord == nullptr) != (paths->sub_dev == nullptr))
    return set_err(AUV_EINVAL, "paths: sub_chord and sub_dev are both set or both NULL");
  if (cnt < 0) cnt = batch->n_envs - e0;
  const int per_cta = AUV_NAV_THREADS / AUV_NAV_G;  // envs per CTA
  const int blocks = (cnt + per_cta - 1) / per_cta;
  const size_t nsm = sizeof(auv::NavStage) * auv::NAV_SUBBLOCKS;
  if (int rc = nav_configure(nsm)) return rc;
  const double2* unit = rays ? reinterpret_cast<const double2*>(rays->unit64) : nullptr;
  int* win = out ? out->windows : nullptr;
  float* obs = out ? out->obs : nullptr;
  const int od = auv_obs_dim(cfg);
  cudaStream_t s = (cudaStream_t)stream;
  if (actions && with_obstacles && pool->k_moving > 0)
    auv::k_vessel_nav<true, true, AUV_NAV_G><<<blocks, AUV_NAV_THREADS, nsm, s>>>(*cfg, *paths, *pool, *batch, unit, win, actions, obs, od, e0, e0 + cnt);
  else if (actions)
    auv::k_vessel_nav<true, false, AUV_NAV_G><<<blocks, AUV_NAV_THREADS, nsm, s>>>(*cfg, *paths, *pool, *batch, unit, win, actions, obs, od, e0, e0 + cnt);
  else
    auv::k_vessel_nav<false, false, AUV_NAV_G><<<blocks, AUV_NAV_THREADS, nsm, s>>>(*cfg, *paths, *pool, *batch, unit, win, nullptr, obs, od, e0, e0 + cnt);
  if (int rc = cuda_check(cudaGetLastError(), "k_vessel_nav")) return rc;
  if (between != nullptr) cudaEventRecord(between, s);
  auv::k_nav_cull<AUV_NAV_G><<<(cnt + 31) / 32, 128, 0, s>>>(*cfg, *paths, *pool, *batch, unit, win, obs, od, e0, e0 + cnt);
  return cuda_check(cudaGetLastError(), "k_nav_cull");
}

// the dynamic shared-memory opt-in of k_lidar is per device and per function; it is made once,
// outside any stream capture (auv_step_host_submit calls lidar_configure before capturing)
static std::atomic<size_t> g_lidar_smem_configured[64];
static int lidar_configure(size_t smem) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  if (smem <= g_lidar_smem_configured[dev].load(std::memory_order_acquire)) return 0;
  const void* fns[12] = {(const void*)auv::k_lidar<false, false, false>, (const void*)auv::k_lidar<true, false, false>,
                         (const void*)auv::k_lidar<false, true, false>,  (const void*)auv::k_lidar<true, true, false>,
                         (const void*)auv::k_lidar<false, false, true>,  (const void*)auv::k_lidar<true, false, true>,
                         (const void*)auv::k_lidar<false, true, true>,   (const void*)auv::k_lidar<true, true, true>,
                         (const void*)auv::k_lidar<false, false, false, true>, (const void*)auv::k_lidar<false, true, false, true>,
                         (const void*)auv::k_lidar<false, false, true, true>,  (const void*)auv::k_lidar<false, true, true, true>};
  for (int i = 0; i < 12; ++i)
    if (int rc = cuda_check(cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                            "cudaFuncSetAttribute(k_lidar)"))
      return rc;
  size_t seen = g_lidar_smem_configured[dev].load(std::memory_order_relaxed);
  while (seen < smem && !g_lidar_smem_configured[dev].compare_exchange_weak(seen, smem, std::memory_order_release)) {
  }
  return 0;
}
static int lidar_vmax(const AuvScenarioPool* pool) { return pool->n_world > 0 ? AUV_MAX_POLY_VERTS : 16; }
static int lidar_velocity(const AuvConfig* cfg) { return cfg->use_lidar && cfg->velocity_mode == AUV_VELOCITY_NEAREST; }
static int lidar_rpad(const AuvConfig* cfg) { return cfg->use_lidar ? ((cfg->n_sensors + 31) & ~31) : 32; }
// envs per CTA: 32 unless the range rows would not leave room for several CTAs per SM
static int lidar_envs_per_cta(const AuvConfig* cfg) {
  int e = AUV_LIDAR_MAX_ENVS;
  const size_t row = (size_t)lidar_rpad(cfg) * (lidar_velocity(cfg) ? 8 : 4);
  while (e > 1 && row * e > 40 * 1024) e >>= 1;
  return e;
}
static size_t lidar_smem_bytes(const AuvConfig* cfg, const AuvScenarioPool* pool) {
  return auv::lidar_smem_bytes_for(lidar_envs_per_cta(cfg), lidar_rpad(cfg), lidar_vmax(pool), lidar_velocity(cfg));
}

static int launch_lidar(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                        const AuvScenarioPool* pool, AuvBatch* batch, AuvStepOut* out, int mode,
                        void* stream, int e0 = 0, int cnt = -1) {
  if (cnt < 0) cnt = batch->n_envs - e0;
  auv::LidarArgs args;
  args.cfg = *cfg;
  if (rays) args.rays = *rays; else memset(&args.rays, 0, sizeof(args.rays));
  args.paths = *paths;
  args.pool = *pool;
  args.batch = *batch;
  args.out = *out;
  args.mode = mode;
  args.obs_dim = auv_obs_dim(cfg);
  args.e0 = e0;
  args.e1 = e0 + cnt;
  args.envs_per_cta = lidar_envs_per_cta(cfg);
  args.vmax = lidar_vmax(pool);
  args.clear_closeness = -cfg->sensor_range * exp(-0.1 * cfg->sensor_range);
  args.pen_clear_ray = (float)(-args.clear_closeness);
  args.inv_log_range = (float)(1.0 / log1p(cfg->sensor_range));
  args.inv_weight_sum = (rays && rays->weight_sum > 0.0) ? 1.0 / rays->weight_sum : 0.0;
  args.feas_width = cfg->vessel_width * cfg->feasibility_width_multiplier;
  const bool track = out->tracks != nullptr;  // validated by check_tracks: never together with seg_tests
  if (track) args.trk = *out->tracks; else memset(&args.trk, 0, sizeof(args.trk));
  const size_t smem = lidar_smem_bytes(cfg, pool);
  if (int rc = lidar_configure(smem)) return rc;
  const int blocks = (cnt + args.envs_per_cta - 1) / args.envs_per_cta;
  cudaStream_t s = (cudaStream_t)stream;
  const bool count = out->seg_tests != nullptr, vel = lidar_velocity(cfg) != 0;
  const bool world = pool->n_world > 0;  // the instantiation with the land-polygon path only when there is land
#define AUV_LAUNCH_LIDAR(C, V, W) auv::k_lidar<C, V, W><<<blocks, AUV_LIDAR_THREADS, smem, s>>>(args)
#define AUV_LAUNCH_LIDAR_TRACK(V, W) auv::k_lidar<false, V, W, true><<<blocks, AUV_LIDAR_THREADS, smem, s>>>(args)
  if (track) {
    if (world && vel) AUV_LAUNCH_LIDAR_TRACK(true, true);
    else if (world) AUV_LAUNCH_LIDAR_TRACK(false, true);
    else if (vel) AUV_LAUNCH_LIDAR_TRACK(true, false);
    else AUV_LAUNCH_LIDAR_TRACK(false, false);
  } else if (world) {
    if (count && vel) AUV_LAUNCH_LIDAR(true, true, true);
    else if (count) AUV_LAUNCH_LIDAR(true, false, true);
    else if (vel) AUV_LAUNCH_LIDAR(false, true, true);
    else AUV_LAUNCH_LIDAR(false, false, true);
  } else {
    if (count && vel) AUV_LAUNCH_LIDAR(true, true, false);
    else if (count) AUV_LAUNCH_LIDAR(true, false, false);
    else if (vel) AUV_LAUNCH_LIDAR(false, true, false);
    else AUV_LAUNCH_LIDAR(false, false, false);
  }
#undef AUV_LAUNCH_LIDAR
#undef AUV_LAUNCH_LIDAR_TRACK
  return cuda_check(cudaGetLastError(), "k_lidar");
}

int auv_navigate(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                 const AuvScenarioPool* pool, AuvBatch* batch, void* stream) {
  if (int rc = check_cfg(cfg)) return rc;
  if (!paths || !pool || !batch) return set_err(AUV_EINVAL, "NULL argument");
  if (cfg->use_lidar && (!rays || !rays->unit64)) return set_err(AUV_EINVAL, "ray table is NULL with use_lidar");
  if (int rc = check_batch(cfg, pool, batch)) return rc;
  return launch_vessel_nav(cfg, rays, paths, pool, batch, nullptr, nullptr, stream);
}

int auv_observe(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                const AuvScenarioPool* pool, AuvBatch* batch, AuvStepOut* out, int mode,
                void* stream) {
  if (int rc = check_observe_args(cfg, rays, paths, pool, batch, out, mode)) return rc;
  if (int rc = launch_vessel_nav(cfg, rays, paths, pool, batch, out, nullptr, stream)) return rc;
  return launch_lidar(cfg, rays, paths, pool, batch, out, mode, stream);
}

int auv_step(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
             const AuvScenarioPool* pool, AuvBatch* batch, const float* actions, AuvStepOut* out,
             void* stream) {
  if (!actions) return set_err(AUV_EINVAL, "actions is NULL");
  if (int rc = check_observe_args(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP)) return rc;
  // the moving-obstacle update (environment.py:386-392) runs inside the vessel/navigation kernel
  if (int rc = launch_vessel_nav(cfg, rays, paths, pool, batch, out, actions, stream, 0, -1, true)) return rc;
  return launch_lidar(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP, stream);
}

// ---- chunked step: the batch is cut into env ranges, each range runs its three kernels (and,
// for the host-buffer variant, its copies) on its own stream.  The thread-per-env culling kernel
// is latency-bound at low occupancy and the warp-per-env casting kernel is issue-bound, so ranges
// in different stages fill each other's idle issue slots; with host buffers the D2H of range c
// overlaps the kernels of range c+1.  Envs are independent: no ordering is needed between ranges.
#define AUV_PIPE_MAX_STREAMS 16
#define AUV_PIPE_MAX_CHUNKS 64
struct AuvPipeline {
  int n_streams;
  cudaStream_t st[AUV_PIPE_MAX_STREAMS];
  cudaEvent_t fork, join[AUV_PIPE_MAX_STREAMS];
  cudaEvent_t chunk[AUV_PIPE_MAX_CHUNKS];  // "range c computed" (host-buffer variant)
  // the host-buffer step as an instantiated CUDA graph: one launch per step instead of
  // ~5 driver calls per range (re-captured whenever an argument changes)
  cudaGraphExec_t gexec;
  unsigned long long gkey;
  int graph_state;  // 0 none, 1 valid, -1 capture not possible (direct submission)
};

AuvPipeline* auv_pipeline_create(int n_streams) {
  if (n_streams <= 0 || n_streams > AUV_PIPE_MAX_STREAMS) {
    set_err(AUV_EINVAL, "n_streams out of range");
    return nullptr;
  }
  AuvPipeline* p = new AuvPipeline;
  p->n_streams = n_streams;
  p->gexec = nullptr;
  p->gkey = 0;
  p->graph_state = 0;
  bool ok = cudaEventCreateWithFlags(&p->fork, cudaEventDisableTiming) == cudaSuccess;
  int made = 0;
  for (; ok && made < n_streams; ++made) {
    ok = cudaStreamCreateWithFlags(&p->st[made], cudaStreamNonBlocking) == cudaSuccess &&
         cudaEventCreateWithFlags(&p->join[made], cudaEventDisableTiming) == cudaSuccess;
  }
  for (int c = 0; ok && c < AUV_PIPE_MAX_CHUNKS; ++c)
    ok = cudaEventCreateWithFlags(&p->chunk[c], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    cuda_check(cudaGetLastError(), "auv_pipeline_create");
    delete p;  // leaks the few objects created before the failure; the context is unusable anyway
    return nullptr;
  }
  return p;
}
void auv_pipeline_destroy(AuvPipeline* p) {
  if (!p) return;
  for (int i = 0; i < p->n_streams; ++i) {
    cudaStreamDestroy(p->st[i]);
    cudaEventDestroy(p->join[i]);
  }
  for (int c = 0; c < AUV_PIPE_MAX_CHUNKS; ++c) cudaEventDestroy(p->chunk[c]);
  cudaEventDestroy(p->fork);
  if (p->gexec) cudaGraphExecDestroy(p->gexec);
  delete p;
}

int auv_pipeline_graph_state(const AuvPipeline* p) { return p ? p->graph_state : AUV_EINVAL; }

static int chunk_size(int n, int n_chunks) {
  int c = (n + n_chunks - 1) / n_chunks;
  return (c + 255) / 256 * 256;  // whole CTAs of every kernel (k_vessel_nav: up to 1024 threads = 256 envs)
}

// device-resident variant: every range on its own stream (round robin)
static int step_chunked(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                        const AuvScenarioPool* pool, AuvBatch* batch, const float* actions, AuvStepOut* out,
                        void* stream, AuvPipeline* p, int n_chunks) {
  if (!p) return set_err(AUV_EINVAL, "pipeline is NULL");
  if (n_chunks <= 0) return set_err(AUV_EINVAL, "n_chunks must be > 0");
  if (int rc = check_observe_args(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const int n = batch->n_envs;
  const int cs = chunk_size(n, n_chunks);
  if (int rc = cuda_check(cudaEventRecord(p->fork, s), "fork")) return rc;
  int used = 0;
  for (int c = 0, e0 = 0; e0 < n; ++c, e0 += cs) {
    const int cnt = n - e0 < cs ? n - e0 : cs;
    cudaStream_t cst = p->st[c % p->n_streams];
    void* vs = (void*)cst;
    if (c < p->n_streams) {
      if (int rc = cuda_check(cudaStreamWaitEvent(cst, p->fork, 0), "wait fork")) return rc;
      used = c + 1;
    }
    if (int rc = launch_vessel_nav(cfg, rays, paths, pool, batch, out, actions, vs, e0, cnt, true)) return rc;
    if (int rc = launch_lidar(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP, vs, e0, cnt)) return rc;
  }
  for (int i = 0; i < used; ++i) {
    if (int rc = cuda_check(cudaEventRecord(p->join[i], p->st[i]), "join record")) return rc;
    if (int rc = cuda_check(cudaStreamWaitEvent(s, p->join[i], 0), "join wait")) return rc;
  }
  return 0;
}

// host-buffer variant: the ranges are computed IN ORDER on one stream and their observations
// leave on the pipeline's copy stream as soon as each range is done, so the link is busy from
// the end of the first range to the end of the step (the step is bound by the D2H of the
// observations: ~49 MB per step at 65536 envs x 186 floats)
static int launch_obs_ship(const AuvConfig* cfg, const AuvStepOut* out, const AuvCompact* cb, float* reward_host,
                           uint8_t* done_host, int e0, int cnt, cudaStream_t s) {
  const int R = cfg->use_lidar ? cfg->n_sensors : 0;
  const int words = cb->words;
  const size_t smem = (size_t)AUV_SHIP_ENVS * words * 32 * 4 + (size_t)AUV_SHIP_ENVS * words * 4 + (AUV_SHIP_ENVS + 1) * 4 + 16;
  static std::atomic<size_t> configured[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  if (smem > 48 * 1024 && smem > configured[dev].load()) {
    if (int rc = cuda_check(cudaFuncSetAttribute(auv::k_obs_ship, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                            "cudaFuncSetAttribute(k_obs_ship)"))
      return rc;
    configured[dev].store(smem);
  }
  const int blocks = (cnt + AUV_SHIP_ENVS - 1) / AUV_SHIP_ENVS;
  auv::k_obs_ship<<<blocks, AUV_SHIP_THREADS, smem, s>>>(out->obs, auv_obs_dim(cfg), R, words, e0, e0 + cnt, out->reward, out->done,
                                                        cb->head, cb->mask, cb->vals, cb->counter, cb->capacity, reward_host,
                                                        done_host);
  return cuda_check(cudaGetLastError(), "k_obs_ship");
}

static int launch_obs_delta(const AuvConfig* cfg, const AuvStepOut* out, const AuvDelta* d, float* reward_host,
                            uint8_t* done_host, int e0, int cnt, cudaStream_t s) {
  const long long od = auv_obs_dim(cfg);
  const long long f0 = od * e0, f1 = od * (e0 + cnt);  // e0 is a multiple of 256 envs: f0 is 1 KB aligned
  const long long quads = (f1 - f0 + 3) / 4;
  static std::atomic<int> sms[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  int n_sm = sms[dev].load();
  if (n_sm == 0) {
    if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm <= 0) n_sm = 148;
    sms[dev].store(n_sm);
  }
  long long blocks = 2 * n_sm;
  const long long need = (quads + AUV_DELTA_THREADS - 1) / AUV_DELTA_THREADS;
  if (blocks > need) blocks = need;
  if (blocks < 1) blocks = 1;
  auv::k_obs_delta<<<(int)blocks, AUV_DELTA_THREADS, 0, s>>>(out->obs, d->shadow, d->obs_host, f0, f1, d->gran / 4, out->reward,
                                                            out->done, reward_host, done_host, e0, e0 + cnt, d->shipped);
  return cuda_check(cudaGetLastError(), "k_obs_delta");
}

static int enqueue_host_step(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                             const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                             float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                             uint8_t* done_host, cudaStream_t s, cudaStream_t ds, AuvPipeline* p, int n_chunks,
                             const AuvCompact* cb = nullptr, const AuvDelta* dl = nullptr) {
  const int n = batch->n_envs;
  const int cs = chunk_size(n, n_chunks);
  const size_t od = (size_t)auv_obs_dim(cfg);
  if (int rc = cuda_check(cudaMemcpyAsync(actions_dev, actions_host, (size_t)n * 2 * sizeof(float), cudaMemcpyHostToDevice, s),
                          "H2D actions"))
    return rc;
  if (cb != nullptr)
    if (int rc = cuda_check(cudaMemsetAsync(cb->counter, 0, sizeof(int32_t), s), "compact counter")) return rc;
  for (int c = 0, e0 = 0; e0 < n; ++c, e0 += cs) {
    const int cnt = n - e0 < cs ? n - e0 : cs;
    if (int rc = launch_vessel_nav(cfg, rays, paths, pool, batch, out, actions_dev, (void*)s, e0, cnt, true)) return rc;
    if (int rc = launch_lidar(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP, (void*)s, e0, cnt)) return rc;
    if (ds != s) {
      if (int rc = cuda_check(cudaEventRecord(p->chunk[c], s), "range done")) return rc;
      if (int rc = cuda_check(cudaStreamWaitEvent(ds, p->chunk[c], 0), "copy stream wait")) return rc;
    }
    if (dl != nullptr) {  // delta transfer: changed chunks of the dense rows, stored by the kernel
      if (int rc = launch_obs_delta(cfg, out, dl, reward_host, done_host, e0, cnt, ds)) return rc;
    } else if (cb != nullptr) {  // compact transfer: the kernel's own stores into pinned host memory
      if (int rc = launch_obs_ship(cfg, out, cb, reward_host, done_host, e0, cnt, ds)) return rc;
    } else if (int rc = cuda_check(cudaMemcpyAsync(obs_host + od * e0, out->obs + od * e0, (size_t)cnt * od * sizeof(float),
                                                   cudaMemcpyDeviceToHost, ds), "D2H obs"))
      return rc;
  }
  if (cb == nullptr && dl == nullptr) {
    if (int rc = cuda_check(cudaMemcpyAsync(reward_host, out->reward, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, ds),
                            "D2H reward"))
      return rc;
    if (int rc = cuda_check(cudaMemcpyAsync(done_host, out->done, (size_t)n, cudaMemcpyDeviceToHost, ds), "D2H done"))
      return rc;
  }
  if (ds != s) {
    if (int rc = cuda_check(cudaEventRecord(p->join[0], ds), "join record")) return rc;
    return cuda_check(cudaStreamWaitEvent(s, p->join[0], 0), "join wait");
  }
  return 0;
}

static unsigned long long fnv1a(unsigned long long h, const void* data, size_t n) {
  const unsigned char* b = (const unsigned char*)data;
  for (size_t i = 0; i < n; ++i) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}

static int step_host_chunked(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                             const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                             float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                             uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks,
                             const AuvCompact* cb = nullptr, const AuvDelta* dl = nullptr) {
  if (!p) return set_err(AUV_EINVAL, "pipeline is NULL");
  if (n_chunks <= 0 || n_chunks > AUV_PIPE_MAX_CHUNKS) return set_err(AUV_EINVAL, "n_chunks out of range");
  if (int rc = check_observe_args(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP)) return rc;
  cudaStream_t s = (cudaStream_t)stream, ds = p->st[0];
  if (p->graph_state >= 0 && p->n_streams >= 2) {
    unsigned long long key = 1469598103934665603ull;
    key = fnv1a(key, cfg, sizeof(*cfg));
    if (rays) key = fnv1a(key, rays, sizeof(*rays));
    key = fnv1a(key, paths, sizeof(*paths));
    key = fnv1a(key, pool, sizeof(*pool));
    key = fnv1a(key, batch, sizeof(*batch));
    key = fnv1a(key, out, sizeof(*out));
    if (out->tracks) key = fnv1a(key, out->tracks, sizeof(*out->tracks));
    const void* ptrs[6] = {actions_host, actions_dev, obs_host, reward_host, done_host, (const void*)(size_t)n_chunks};
    key = fnv1a(key, ptrs, sizeof(ptrs));
    if (cb) key = fnv1a(key, cb, sizeof(*cb));
    if (dl) key = fnv1a(key, dl, sizeof(*dl));
    if (p->graph_state == 0 || key != p->gkey) {
      if (p->gexec) {
        cudaGraphExecDestroy(p->gexec);
        p->gexec = nullptr;
      }
      p->graph_state = 0;
      // one-time function attributes are set outside the capture
      if (int rc0 = lidar_configure(lidar_smem_bytes(cfg, pool))) return rc0;
      if (int rc0 = nav_configure(sizeof(auv::NavStage) * auv::NAV_SUBBLOCKS)) return rc0;
      cudaStream_t cs = p->st[1];
      cudaGraph_t graph = nullptr;
      int rc = 0;
      if (cudaStreamBeginCapture(cs, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
        rc = enqueue_host_step(cfg, rays, paths, pool, batch, actions_host, actions_dev, out, obs_host, reward_host,
                               done_host, cs, ds, p, n_chunks, cb, dl);
        const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
        if (rc == 0 && ce == cudaSuccess && graph != nullptr &&
            cudaGraphInstantiate(&p->gexec, graph, 0) == cudaSuccess) {
          p->graph_state = 1;
          p->gkey = key;
        }
        if (graph) cudaGraphDestroy(graph);
      }
      if (p->graph_state != 1) {
        cudaGetLastError();    // clear; fall back to direct submission from now on
        p->graph_state = -1;
        if (rc) return rc;
      }
    }
    if (p->graph_state == 1) return cuda_check(cudaGraphLaunch(p->gexec, s), "cudaGraphLaunch");
  }
  return enqueue_host_step(cfg, rays, paths, pool, batch, actions_host, actions_dev, out, obs_host, reward_host, done_host,
                           s, ds, p, n_chunks, cb, dl);
}

int auv_step_chunked(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                     const AuvScenarioPool* pool, AuvBatch* batch, const float* actions, AuvStepOut* out,
                     void* stream, AuvPipeline* p, int n_chunks) {
  if (!actions) return set_err(AUV_EINVAL, "actions is NULL");
  return step_chunked(cfg, rays, paths, pool, batch, actions, out, stream, p, n_chunks);
}

int auv_step_host_submit(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                         const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                         float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                         uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks) {
  if (!cfg || !batch || !out || !actions_host || !actions_dev || !obs_host || !reward_host || !done_host)
    return set_err(AUV_EINVAL, "NULL argument");
  return step_host_chunked(cfg, rays, paths, pool, batch, actions_host, actions_dev, out, obs_host, reward_host,
                           done_host, stream, p, n_chunks);
}

int auv_step_host_compact_submit(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                                 const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                                 float* actions_dev, AuvStepOut* out, const AuvCompact* cb, float* reward_host,
                                 uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks) {
  if (!cfg || !batch || !out || !actions_host || !actions_dev || !cb || !reward_host || !done_host)
    return set_err(AUV_EINVAL, "NULL argument");
  if (!cb->head || !cb->mask || !cb->vals || !cb->counter) return set_err(AUV_EINVAL, "compact buffers are NULL");
  if (cfg->sensor_use_velocity_observations) return set_err(AUV_ENOTSUP, "compact transfer with velocity observations");
  const int R = cfg->use_lidar ? cfg->n_sensors : 0;
  if (cb->words != (R + 31) / 32 || cb->words <= 0) return set_err(AUV_EINVAL, "compact.words must be ceil(n_sensors / 32) >= 1");
  if ((long long)cb->capacity < (long long)batch->n_envs * cb->words * 32)
    return set_err(AUV_EINVAL, "compact.capacity must be >= n_envs * words * 32");
  return step_host_chunked(cfg, rays, paths, pool, batch, actions_host, actions_dev, out, nullptr, reward_host, done_host,
                           stream, p, n_chunks, cb);
}

int auv_step_host_delta_submit(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                               const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                               float* actions_dev, AuvStepOut* out, const AuvDelta* d, float* reward_host,
                               uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks) {
  if (!cfg || !batch || !out || !actions_host || !actions_dev || !d || !reward_host || !done_host)
    return set_err(AUV_EINVAL, "NULL argument");
  if (!d->obs_host || !d->shadow) return set_err(AUV_EINVAL, "delta buffers are NULL");
  if (d->gran != 8 && d->gran != 16 && d->gran != 32) return set_err(AUV_EINVAL, "delta.gran must be 8, 16 or 32");
  if (((size_t)d->obs_host | (size_t)d->shadow | (size_t)out->obs) & 15u)
    return set_err(AUV_EINVAL, "delta: obs_host, shadow and out->obs must be 16 B aligned");
  return step_host_chunked(cfg, rays, paths, pool, batch, actions_host, actions_dev, out, nullptr, reward_host, done_host,
                           stream, p, n_chunks, nullptr, d);
}

int auv_compact_expand(const AuvConfig* cfg, int n_envs, const AuvCompact* cb, uint32_t* prev_mask, float* obs_host,
                       int n_threads) {
  if (!cfg || !cb || !prev_mask || !obs_host || n_envs <= 0) return set_err(AUV_EINVAL, "bad auv_compact_expand arguments");
  const int od = auv_obs_dim(cfg), words = cb->words;
  const float* head = cb->head;
  const uint32_t* mask = cb->mask;
  const float* vals = cb->vals;
  if (n_threads < 1) n_threads = 1;
#pragma omp parallel for num_threads(n_threads) schedule(static)
  for (int e = 0; e < n_envs; ++e) {
    float* row = obs_host + (size_t)e * od;
    const float* h = head + (size_t)e * 8;
    for (int k = 0; k < 6; ++k) row[k] = h[k];
    int off;
    memcpy(&off, h + 7, sizeof(int));
    const float* v = vals + off;
    uint32_t* pm = prev_mask + (size_t)e * words;
    const uint32_t* nm = mask + (size_t)e * words;
    float* cl = row + 6;
    for (int w = 0; w < words; ++w) {
      uint32_t clear = pm[w] & ~nm[w];  // rays that read clear again
      while (clear) {
        cl[w * 32 + __builtin_ctz(clear)] = 0.f;
        clear &= clear - 1;
      }
      uint32_t set = nm[w];
      while (set) {
        cl[w * 32 + __builtin_ctz(set)] = *v++;
        set &= set - 1;
      }
      pm[w] = nm[w];
    }
  }
  return 0;
}

int auv_step_host_chunked(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                          const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                          float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                          uint8_t* done_host, void* stream, AuvPipeline* p, int n_chunks) {
  if (int rc = auv_step_host_submit(cfg, rays, paths, pool, batch, actions_host, actions_dev, out, obs_host, reward_host,
                                    done_host, stream, p, n_chunks))
    return rc;
  return cuda_check(cudaStreamSynchronize((cudaStream_t)stream), "sync");
}

#define AUV_TIMER_EVENTS 4
struct AuvTimer {
  int capacity;
  cudaEvent_t* ev;  // [capacity][AUV_TIMER_EVENTS]
};

AuvTimer* auv_timer_create(int capacity) {
  if (capacity <= 0) return nullptr;
  AuvTimer* t = new AuvTimer;
  t->capacity = capacity;
  t->ev = new cudaEvent_t[(size_t)capacity * AUV_TIMER_EVENTS];
  for (int i = 0; i < capacity * AUV_TIMER_EVENTS; ++i)
    if (cudaEventCreate(&t->ev[i]) != cudaSuccess) {
      for (int k = 0; k < i; ++k) cudaEventDestroy(t->ev[k]);
      delete[] t->ev;
      delete t;
      return nullptr;
    }
  return t;
}
void auv_timer_destroy(AuvTimer* t) {
  if (!t) return;
  for (int i = 0; i < t->capacity * AUV_TIMER_EVENTS; ++i) cudaEventDestroy(t->ev[i]);
  delete[] t->ev;
  delete t;
}
int auv_step_timed(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                   const AuvScenarioPool* pool, AuvBatch* batch, const float* actions, AuvStepOut* out,
                   void* stream, AuvTimer* t, int slot) {
  if (!t || slot < 0 || slot >= t->capacity) return set_err(AUV_EINVAL, "bad timer/slot");
  if (!actions) return set_err(AUV_EINVAL, "actions is NULL");
  if (int rc = check_observe_args(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  cudaEvent_t* e = t->ev + AUV_TIMER_EVENTS * slot;
  cudaEventRecord(e[0], s);
  if (int rc = launch_vessel_nav(cfg, rays, paths, pool, batch, out, actions, stream, 0, -1, true, e[1])) return rc;
  cudaEventRecord(e[2], s);
  if (int rc = launch_lidar(cfg, rays, paths, pool, batch, out, AUV_OBSERVE_STEP, stream)) return rc;
  return cuda_check(cudaEventRecord(e[3], s), "cudaEventRecord");
}
int auv_timer_read(AuvTimer* t, int slot, float* ms) {
  if (!t || !ms || slot < 0 || slot >= t->capacity) return set_err(AUV_EINVAL, "bad timer/slot");
  cudaEvent_t* e = t->ev + AUV_TIMER_EVENTS * slot;
  for (int k = 0; k < AUV_TIMER_EVENTS - 1; ++k)
    if (int rc = cuda_check(cudaEventElapsedTime(&ms[k], e[k], e[k + 1]), "cudaEventElapsedTime")) return rc;
  return 0;
}

int auv_step_host(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                  const AuvScenarioPool* pool, AuvBatch* batch, const float* actions_host,
                  float* actions_dev, AuvStepOut* out, float* obs_host, float* reward_host,
                  uint8_t* done_host, void* stream) {
  if (!cfg || !batch || !out || !actions_host || !actions_dev || !obs_host || !reward_host || !done_host)
    return set_err(AUV_EINVAL, "NULL argument");
  if (int rc = check_tracks(out, batch)) return rc;  // before the copy of the actions
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)batch->n_envs;
  if (int rc = cuda_check(cudaMemcpyAsync(actions_dev, actions_host, n * 2 * sizeof(float),
                                          cudaMemcpyHostToDevice, s), "H2D actions"))
    return rc;
  if (int rc = auv_step(cfg, rays, paths, pool, batch, actions_dev, out, stream)) return rc;
  const size_t od = (size_t)auv_obs_dim(cfg);
  if (int rc = cuda_check(cudaMemcpyAsync(obs_host, out->obs, n * od * sizeof(float),
                                          cudaMemcpyDeviceToHost, s), "D2H obs"))
    return rc;
  if (int rc = cuda_check(cudaMemcpyAsync(reward_host, out->reward, n * sizeof(float),
                                          cudaMemcpyDeviceToHost, s), "D2H reward"))
    return rc;
  if (int rc = cuda_check(cudaMemcpyAsync(done_host, out->done, n, cudaMemcpyDeviceToHost, s), "D2H done"))
    return rc;
  return cuda_check(cudaStreamSynchronize(s), "sync");
}

static int check_gen_world(const AuvGenParams* gp, const AuvScenarioPool* pool) {
  if (pool->n_world < 0) return set_err(AUV_EINVAL, "n_world < 0");
  if (pool->n_world == 0) return 0;
  if (!pool->world_circle || !pool->world_voff || !pool->world_verts) return set_err(AUV_EINVAL, "world arrays are NULL");
  if (pool->world_cell_off &&
      (!pool->world_cell_items || pool->world_grid_nx <= 0 || pool->world_grid_ny <= 0 || !(pool->world_grid_cell > 0.0)))
    return set_err(AUV_EINVAL, "world grid: NULL items or empty grid");
  if (!(gp->land_clearance >= 0.0)) return set_err(AUV_EINVAL, "land_clearance must be >= 0");
  return 0;
}

// both launches of the generator (auv_generate.cuh): per scenario, then per (scenario, obstacle slot)
static int launch_generate(const AuvGenParams* gp, const AuvPathBank* paths, const AuvScenarioPool* pool,
                           const int32_t* ids, int n_ids, const int32_t* n_ids_dev, int32_t* status, cudaStream_t s) {
  const int threads = 128;
  auv::k_generate_scenario_heads<<<(unsigned)((n_ids + threads - 1) / threads), threads, 0, s>>>(*gp, *paths, *pool, ids, n_ids,
                                                                                               n_ids_dev, status);
  if (int rc = cuda_check(cudaGetLastError(), "k_generate_scenario_heads")) return rc;
  const long long total = (long long)n_ids * (pool->k_moving + pool->k_static);
  if (total == 0) return 0;
  // programmatic dependent launch: the slot grid is dispatched while the per-scenario grid runs and waits for
  // its results on the device (griddepcontrol.wait), so the split costs no launch gap
  cudaLaunchConfig_t lc = {};
  lc.gridDim = dim3((unsigned)((total + threads - 1) / threads));
  lc.blockDim = dim3(threads);
  lc.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = at;
  lc.numAttrs = 1;
  return cuda_check(cudaLaunchKernelEx(&lc, auv::k_generate_moving_obstacles, *gp, *paths, *pool, ids, n_ids, n_ids_dev, status),
                    "k_generate_moving_obstacles");
}

int auv_generate_moving_obstacles(const AuvGenParams* gp, const AuvPathBank* paths, const AuvScenarioPool* pool,
                                  const int32_t* ids, int n_ids, int32_t* status, void* stream) {
  if (!gp || !paths || !pool) return set_err(AUV_EINVAL, "NULL argument");
  if (n_ids <= 0 || (!ids && n_ids > pool->n_scenarios)) return set_err(AUV_EINVAL, "n_ids out of range");
  if (paths->n_paths <= 0) return set_err(AUV_EINVAL, "empty path bank");
  if (pool->k_moving < 0 || pool->k_static < 0) return set_err(AUV_EINVAL, "negative slot count");
  if (!pool->path_id || !pool->vessel_init) return set_err(AUV_EINVAL, "pool.path_id / vessel_init is NULL");
  if (pool->k_moving > 0 && (!pool->mov_start || !pool->mov_width || !pool->mov_track || !pool->vel_table ||
                             !pool->mov_pos0 || !pool->mov_disp0 || !pool->mov_counter0))
    return set_err(AUV_EINVAL, "moving-obstacle arrays are NULL");
  if (pool->k_static > 0 && (!pool->st_pos || !pool->st_radius)) return set_err(AUV_EINVAL, "static-obstacle arrays are NULL");
  if (int rc = check_gen_world(gp, pool)) return rc;
  return launch_generate(gp, paths, pool, ids, n_ids, nullptr, status, (cudaStream_t)stream);
}

int auv_linear_wrap(double dt, double counter0, int vel_len, int32_t* first_wrap, int32_t* wrap_period) {
  if (!(dt > 0.0) || vel_len < 2 || !first_wrap || !wrap_period) return set_err(AUV_EINVAL, "bad auv_linear_wrap arguments");
  const int limit = 1 << 30;
  // obstacles.py:195-215, literally: counter += dt; index = floor(counter); index >= len - 1 wraps
  double c = counter0;
  int n = 0;
  for (;;) {
    ++n;
    c += dt;
    if ((int)floor(c) >= vel_len - 1) break;
    if (n >= limit) return set_err(AUV_EINVAL, "track never wraps");
  }
  *first_wrap = n;
  c = 0.0;
  n = 0;
  for (;;) {
    ++n;
    c += dt;
    if ((int)floor(c) >= vel_len - 1) break;
    if (n >= limit) return set_err(AUV_EINVAL, "track never wraps");
  }
  *wrap_period = n;
  return 0;
}

int auv_pool_pack(const AuvConfig* cfg, const AuvScenarioPool* pool, const int32_t* ids, int n_ids, void* stream) {
  if (int rc = check_cfg(cfg)) return rc;
  if (!pool) return set_err(AUV_EINVAL, "pool is NULL");
  if (n_ids <= 0 || (!ids && n_ids > pool->n_scenarios)) return set_err(AUV_EINVAL, "n_ids out of range");
  if (pool->k_static > 0 && (!pool->st_rec || !pool->st_pos || !pool->st_radius))
    return set_err(AUV_EINVAL, "static-obstacle arrays are NULL");
  if (pool->k_moving > 0 && pool->linear_tracks &&
      (!pool->mov_lin || !pool->mov_pos0 || !pool->mov_start || !pool->mov_width || !pool->mov_track || !pool->vel_table))
    return set_err(AUV_EINVAL, "moving-obstacle arrays are NULL");
  const long long total = (long long)n_ids * (pool->k_moving + pool->k_static);
  if (total == 0) return 0;
  const int threads = 128;
  auv::k_pool_pack<<<(unsigned)((total + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(*cfg, *pool, ids, n_ids);
  return cuda_check(cudaGetLastError(), "k_pool_pack");
}

int auv_obstacle_state(const AuvConfig* cfg, const AuvScenarioPool* pool, const AuvBatch* batch, double* pos,
                       double* disp, double* counter, void* stream) {
  if (int rc = check_cfg(cfg)) return rc;
  if (!pool || !batch) return set_err(AUV_EINVAL, "pool/batch is NULL");
  if (batch->n_envs <= 0) return set_err(AUV_EINVAL, "n_envs must be > 0");
  if (!batch->obst_steps) return set_err(AUV_EINVAL, "batch.obst_steps is NULL");
  if (int rc = check_pool_tracks(pool, batch)) return rc;
  const long long total = (long long)batch->n_envs * pool->k_moving;
  if (total == 0) return 0;
  const int threads = 128;
  auv::k_obstacle_state<<<(unsigned)((total + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(*cfg, *pool, *batch, pos,
                                                                                                         disp, counter);
  return cuda_check(cudaGetLastError(), "k_obstacle_state");
}

// first observation of the listed scenarios -> pool.reset_* (at most worker->n_envs per call)
static int reset_cache_fill(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                            const AuvScenarioPool* pool, AuvBatch* worker, AuvStepOut* wout, const int32_t* ids, int first,
                            int n, const int32_t* n_dev, void* stream) {
  if (n <= 0 || n > worker->n_envs) return set_err(AUV_EINVAL, "n must be in 1..worker.n_envs");
  if (!pool->reset_obs || !pool->reset_max_progress || (cfg->use_lidar && !pool->reset_mask))
    return set_err(AUV_EINVAL, "pool.reset_* is NULL");
  if (int rc = check_observe_args(cfg, rays, paths, pool, worker, wout, AUV_OBSERVE_RESET)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const int wn = worker->n_envs, threads = 128;
  auv::k_worker_fill<<<(wn + threads - 1) / threads, threads, 0, s>>>(*worker, ids, first, n, n_dev);
  if (int rc = cuda_check(cudaGetLastError(), "k_worker_fill")) return rc;
  if (int rc = auv_reset(cfg, pool, worker, nullptr, stream)) return rc;
  if (int rc = auv_observe(cfg, rays, paths, pool, worker, wout, AUV_OBSERVE_RESET, stream)) return rc;
  auv::k_cache_scatter<<<(n * 32 + threads - 1) / threads, threads, 0, s>>>(*pool, *worker, wout->obs, auv_obs_dim(cfg),
                                                                          cfg->use_lidar, n, n_dev);
  return cuda_check(cudaGetLastError(), "k_cache_scatter");
}

int auv_reset_cache_fill(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                         const AuvScenarioPool* pool, AuvBatch* worker, AuvStepOut* worker_out, const int32_t* ids,
                         int first, int n, void* stream) {
  if (!cfg || !paths || !pool || !worker || !worker_out) return set_err(AUV_EINVAL, "NULL argument");
  if (!ids && (first < 0 || first + n > pool->n_scenarios)) return set_err(AUV_EINVAL, "scenario range out of bounds");
  return reset_cache_fill(cfg, rays, paths, pool, worker, worker_out, ids, first, n, nullptr, stream);
}

int auv_refresh_finished(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths,
                         const AuvScenarioPool* pool, const AuvBatch* live, AuvBatch* worker, AuvStepOut* worker_out,
                         const AuvRefreshScratch* rs, const AuvGenParams* gp, void* stream) {
  if (!cfg || !paths || !pool || !live || !worker || !worker_out || !rs || !gp) return set_err(AUV_EINVAL, "NULL argument");
  if (!rs->seen_episode || !rs->ids || !rs->count || rs->capacity <= 0 || rs->capacity > worker->n_envs)
    return set_err(AUV_EINVAL, "refresh scratch: NULL array or capacity not in 1..worker.n_envs");
  if (pool->n_scenarios != 2 * (live->reset_stride > 0 ? live->reset_stride : live->n_envs))
    return set_err(AUV_EINVAL, "refresh needs a pool of exactly 2 * reset_stride (default n_envs) scenarios");
  if (int rc = check_gen_world(gp, pool)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 128;
  if (int rc = cuda_check(cudaMemsetAsync(rs->count, 0, sizeof(int32_t), s), "memset")) return rc;
  auv::k_refresh_collect<<<(live->n_envs + threads - 1) / threads, threads, 0, s>>>(*live, pool->n_scenarios, rs->seen_episode,
                                                                                    rs->ids, rs->count, rs->capacity);
  if (int rc = cuda_check(cudaGetLastError(), "k_refresh_collect")) return rc;
  if (int rc = launch_generate(gp, paths, pool, rs->ids, rs->capacity, rs->count, live->status, s)) return rc;
  return reset_cache_fill(cfg, rays, paths, pool, worker, worker_out, rs->ids, 0, rs->capacity, rs->count, stream);
}

int auv_pathbank_build(const double* waypoints, const int32_t* n_wp, const int32_t* path_ids, int n,
                       const AuvPathBuild* out, int32_t* status, void* stream) {
  if (!waypoints || !n_wp || !out || n <= 0) return set_err(AUV_EINVAL, "bad auv_pathbank_build arguments");
  if (!out->hdr || !out->poly_xy || !out->poly_cum || !out->poly_f32 || !out->blk_chord || !out->blk_dev || !out->sb_chord ||
      !out->sb_dev || !out->pp)
    return set_err(AUV_EINVAL, "AuvPathBuild holds a NULL array");
  if (out->n_knots != auv::PB_NK) return set_err(AUV_EINVAL, "n_knots must be 1000");
  if ((out->sub_chord == nullptr) != (out->sub_dev == nullptr))
    return set_err(AUV_EINVAL, "AuvPathBuild: sub_chord and sub_dev are both set or both NULL");
  if (out->vcap <= 0 || out->vcap % (2 * AUV_PATH_BLOCK * AUV_PATH_SUPER) != 0)
    return set_err(AUV_EINVAL, "vcap must be a positive multiple of 2 * AUV_PATH_BLOCK * AUV_PATH_SUPER");
  const size_t smem = auv::pathbuild_smem_bytes();
  static std::atomic<int> configured[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  if (!configured[dev].load()) {
    if (int rc = cuda_check(cudaFuncSetAttribute(auv::k_path_build, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                            "cudaFuncSetAttribute(k_path_build)"))
      return rc;
    configured[dev].store(1);
  }
  auv::PathBuildOut o;
  o.hdr = out->hdr;
  o.poly_xy = out->poly_xy;
  o.poly_cum = out->poly_cum;
  o.poly_f32 = out->poly_f32;
  o.blk_chord = out->blk_chord;
  o.blk_dev = out->blk_dev;
  o.sb_chord = out->sb_chord;
  o.sb_dev = out->sb_dev;
  o.pp = out->pp;
  o.vcap = out->vcap;
  o.sub_chord = out->sub_chord;
  o.sub_dev = out->sub_dev;
  auv::k_path_build<<<n, auv::PB_THREADS, smem, (cudaStream_t)stream>>>(waypoints, n_wp, path_ids, n, o, status);
  return cuda_check(cudaGetLastError(), "k_path_build");
}

int auv_random_curve_waypoints(uint64_t seed, uint32_t epoch, double length, const int32_t* path_ids, int n,
                               double* waypoints, int32_t* n_wp, void* stream) {
  if (!waypoints || !n_wp || n <= 0 || !(length > 0.0)) return set_err(AUV_EINVAL, "bad auv_random_curve_waypoints arguments");
  auv::k_random_curve_waypoints<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(seed, epoch, length, path_ids, n, waypoints, n_wp);
  return cuda_check(cudaGetLastError(), "k_random_curve_waypoints");
}

int auv_fma_probe(float* sink, int blocks, int threads, int iters, void* stream, double* flops_out) {
  if (!sink || blocks <= 0 || threads <= 0 || threads > 256 || iters <= 0)
    return set_err(AUV_EINVAL, "bad probe arguments");
  auv::k_fma_probe<<<blocks, threads, 0, (cudaStream_t)stream>>>(sink, iters);
  if (flops_out) *flops_out = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
  return cuda_check(cudaGetLastError(), "k_fma_probe");
}

int auv_render(const AuvConfig* cfg, const AuvRayTable* rays, const AuvPathBank* paths, const AuvScenarioPool* pool,
               const AuvBatch* batch, const float* obs, const AuvRender* r, uint8_t* frames, void* stream) {
  if (!cfg || !rays || !paths || !pool || !batch || !r || !frames || !r->env_ids)
    return set_err(AUV_EINVAL, "auv_render: NULL argument");
  if (int rc = check_cfg(cfg)) return rc;
  if (cfg->use_lidar && (!obs || !rays->cos_sin)) return set_err(AUV_EINVAL, "auv_render: obs / rays.cos_sin is NULL with use_lidar");
  if (r->count < 1) return set_err(AUV_EINVAL, "auv_render: count must be >= 1");
  if (r->width < 1 || r->width > AUV_RENDER_MAX_DIM || r->height < 1 || r->height > AUV_RENDER_MAX_DIM)
    return set_err(AUV_EINVAL, "auv_render: width and height must be in 1..4096");
  if (!(isfinite(r->half_width) && r->half_width > 0.0)) return set_err(AUV_EINVAL, "auv_render: half_width must be finite and > 0");
  if (batch->n_envs <= 0) return set_err(AUV_EINVAL, "n_envs must be > 0");
  if (!batch->state || !batch->scn_id || !batch->obst_steps || !batch->env_pid)
    return set_err(AUV_EINVAL, "auv_render: batch.state / scn_id / obst_steps / env_pid is NULL");
  if (!paths->hdr || !paths->poly_xy || !paths->blk_chord || !paths->blk_dev)
    return set_err(AUV_EINVAL, "auv_render: path bank arrays are NULL");
  if (pool->k_moving < 0 || pool->k_static < 0 || pool->n_world < 0) return set_err(AUV_EINVAL, "negative slot count");
  if (pool->k_static > 0 && (!pool->st_rec || !rays->unit64)) return set_err(AUV_EINVAL, "auv_render: pool.st_rec / rays.unit64 is NULL");
  if (int rc = check_pool_tracks(pool, batch)) return rc;
  if (pool->k_moving > 0 && (pool->linear_tracks ? !pool->mov_disp0 : !pool->mov_width))
    return set_err(AUV_EINVAL, "auv_render: pool.mov_disp0 / mov_width is NULL");
  if (pool->n_world > 0) {
    if (!pool->world_circle || !pool->world_voff || !pool->world_verts) return set_err(AUV_EINVAL, "world arrays are NULL");
    if (pool->world_cell_off &&
        (!pool->world_cell_items || pool->world_grid_nx <= 0 || pool->world_grid_ny <= 0 || !(pool->world_grid_cell > 0.0)))
      return set_err(AUV_EINVAL, "world grid: NULL items or empty grid");
  }
  auv::RenderArgs a;
  a.cfg = *cfg;
  a.rays = *rays;
  a.paths = *paths;
  a.pool = *pool;
  a.batch = *batch;
  a.obs = obs;
  a.env_ids = r->env_ids;
  a.frames = frames;
  a.half_width = r->half_width;
  a.obs_dim = auv_obs_dim(cfg);
  a.width = r->width;
  a.height = r->height;
  a.tiles_x = (r->width + AUV_RENDER_TILE - 1) / AUV_RENDER_TILE;
  const int tiles_y = (r->height + AUV_RENDER_TILE - 1) / AUV_RENDER_TILE;
  auv::k_render<<<dim3((unsigned)r->count, (unsigned)(a.tiles_x * tiles_y)), AUV_RENDER_THREADS, 0, (cudaStream_t)stream>>>(a);
  return cuda_check(cudaGetLastError(), "k_render");
}

}  // extern "C"
