// auv_generate.cuh -- GPU-side scenario generation for the MovingObstacles family:
// what MovingObstacles._generate (envs/movingobstacles.py:28-95) and helpers.generate_obstacle
// (utils/helpers.py:5-35) sample per episode, batched in two launches -- one thread per scenario for the
// path and vessel start, then one per (scenario, obstacle slot) --, counter-based Philox4x32-10 streams
// (SURVEY.md section 8f rank 1).  In a pool with a shared land-polygon world every placed object must also
// be clear of land (land_clear below; DESIGN.md section 6b); without a world the draws are unchanged.  The reference mixes a
// seeded RandomState with the global unseeded np.random (SURVEY quirk B10), so its streams
// cannot be reproduced; parity here is distributional + the acceptance rule, and every
// generated scenario can be pulled back to the host and replayed through the oracle.
#pragma once
#include "auv_device.cuh"
#include "auv_navigate.cuh"
#include "../../include/auv_b200.h"

namespace auv {

// Philox4x32-10 (Salmon et al., SC'11): counter (c0..c3), key (k0, k1)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// one independent stream per (scenario, slot, epoch); doubles with 53 random bits in [0, 1)
struct GenRng {
  uint2 key;
  unsigned scenario, slot, epoch, draw;
  uint4 buf;
  int have;  // doubles left in buf (2 per Philox call)
  __device__ __forceinline__ GenRng(unsigned long long seed, unsigned scenario_, unsigned slot_, unsigned epoch_)
      : key(make_uint2((unsigned)seed, (unsigned)(seed >> 32))), scenario(scenario_), slot(slot_), epoch(epoch_),
        draw(0), buf(make_uint4(0, 0, 0, 0)), have(0) {}
  __device__ __forceinline__ double u01() {
    if (have == 0) {
      buf = philox4x32_10(make_uint4(scenario, slot, epoch, draw++), key);
      have = 2;
    }
    const unsigned a = have == 2 ? buf.x : buf.z, b = have == 2 ? buf.y : buf.w;
    --have;
    return (double)(((unsigned long long)(a >> 5) << 26) | (unsigned long long)(b >> 6)) * (1.0 / 9007199254740992.0);
  }
  __device__ __forceinline__ double normal() {  // Box-Muller
    const double u1 = 1.0 - u01(), u2 = u01();
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
  }
  __device__ __forceinline__ int poisson(double lam) {  // Knuth's product method (lam <= ~500)
    const double L = exp(-lam);
    int k = 0;
    double p = 1.0;
    do {
      ++k;
      p *= u01();
    } while (p > L);
    return k - 1;
  }
};

#define AUV_GEN_SLOT_VESSEL 0xFFFFu
#define AUV_GEN_SLOT_PATH 0xFFFEu
#define AUV_GEN_MAX_TRIES 100000
#define AUV_GEN_VESSEL_TRIES 4096  // vessel-start draws before AUV_STATUS_GEN_LAND_BLOCKED

__device__ __forceinline__ void gen_path_point(const AuvPathBank& pb, int pid, double L, double s, double& x, double& y,
                                               double& dir) {
  PchipOut a, b;
  pchip_eval2(pb, pid, L, s, s, a, b);
  x = a.px;
  y = a.py;
  dir = atan2(a.dy, a.dx);  // Path.get_direction, path.py:72-82
}

// ---- "clear of land by d": (px, py) is outside every world polygon (even-odd rule on the closed ring) and its
// FP64 distance to every ring is > d.  Not world_polygon_distance: that is the step's FP32 culling test.
// Polygon j alone; the ring is read from global memory, so any perimeter length is accepted.  The crossing and
// distance tests are written without divisions (the division slow path is a call, which makes the
// rejection loops spill); they decide as oracle.geos_lite.point_in_ring / point_ring_distance do up to rounding.
__device__ __forceinline__ bool land_polygon_clear(const AuvScenarioPool& pool, int j, double px, double py, double d) {
  const double cx = pool.world_circle[3 * j], cy = pool.world_circle[3 * j + 1], rr = pool.world_circle[3 * j + 2] + d;
  if ((px - cx) * (px - cx) + (py - cy) * (py - cy) > rr * rr) return true;  // enclosing circle out of reach
  const double2* v = reinterpret_cast<const double2*>(pool.world_verts);
  const int k1 = pool.world_voff[j + 1];
  const double d2 = d * d;
  bool inside = false;
  double2 a = v[pool.world_voff[j]];
  for (int k = pool.world_voff[j] + 1; k < k1; ++k) {
    const double2 b = v[k];
    const double ex = b.x - a.x, ey = b.y - a.y, qx = a.x - px, qy = a.y - py;
    const double cr = qx * ey - qy * ex;  // (a - p) x (b - a): its sign tells on which side of the edge p lies
    if ((a.y > py) != (b.y > py)) {  // crossing number: the edge crosses the horizontal through p ...
      if (cr == 0.0) return false;   // ... at p itself (on the boundary = inside)
      if ((cr > 0.0) == (ey > 0.0)) inside = !inside;  // ... right of p
    }
    // point-segment distance (GEOS Distance::pointToSegment), squared and compared with d^2
    const double len2 = ex * ex + ey * ey, t = -(qx * ex + qy * ey);  // t = (p - a).(b - a)
    double dist2;
    if (t <= 0.0 || len2 == 0.0) {
      dist2 = qx * qx + qy * qy;
    } else if (t >= len2) {
      dist2 = (b.x - px) * (b.x - px) + (b.y - py) * (b.y - py);
    } else {
      dist2 = -1.0;  // interior foot: |cr|^2 / len2 <= d^2
      if (cr * cr <= d2 * len2) return false;
    }
    if (dist2 >= 0.0 && dist2 <= d2) return false;  // early exit: within d of this edge
    a = b;
  }
  return !inside;
}

// the whole world: the cells of the pool's uniform grid that the disc of radius d overlaps (cell ranges computed
// as World.grid computes a circle's), or every polygon when the pool has no grid
__device__ __forceinline__ bool land_clear(const AuvScenarioPool& pool, double px, double py, double d) {
  if (pool.n_world <= 0) return true;
  if (pool.world_cell_off == nullptr) {
    for (int j = 0; j < pool.n_world; ++j)
      if (!land_polygon_clear(pool, j, px, py, d)) return false;
    return true;
  }
  const double cell = pool.world_grid_cell;
  const double fx0 = floor((px - d - pool.world_grid_x0) / cell), fx1 = floor((px + d - pool.world_grid_x0) / cell);
  const double fy0 = floor((py - d - pool.world_grid_y0) / cell), fy1 = floor((py + d - pool.world_grid_y0) / cell);
  const int nx = pool.world_grid_nx, ny = pool.world_grid_ny;
  if (!(fx1 >= 0.0 && fy1 >= 0.0 && fx0 <= (double)(nx - 1) && fy0 <= (double)(ny - 1))) return true;  // off the grid
  const int ix0 = (int)fmax(fx0, 0.0), ix1 = (int)fmin(fx1, (double)(nx - 1));
  const int iy0 = (int)fmax(fy0, 0.0), iy1 = (int)fmin(fy1, (double)(ny - 1));
  for (int iy = iy0; iy <= iy1; ++iy)
    for (int ix = ix0; ix <= ix1; ++ix) {
      const int c = iy * nx + ix;
      for (int it = pool.world_cell_off[c]; it < pool.world_cell_off[c + 1]; ++it)
        if (!land_polygon_clear(pool, pool.world_cell_items[it], px, py, d)) return false;
    }
  return true;
}

// Both generator kernels are launched with 128 threads.  __maxnreg__ instead of __launch_bounds__(128): with the
// latter ptxas kept the rejection loops at 48-64 registers and spilled what lives across the calls of the
// FP64 division / trig slow paths.
// Launch 1 of 2, thread per listed scenario: path choice and the vessel start, written to pool.path_id /
// vessel_init.  ids == nullptr: scenarios [0, n_ids); n_ids_dev: list length decided on the device
// (auv_refresh_finished).
__global__ void __maxnreg__(128) k_generate_scenario_heads(const __grid_constant__ AuvGenParams gp,
                                                                  const __grid_constant__ AuvPathBank pb,
                                                                  const __grid_constant__ AuvScenarioPool pool,
                                                                  const int* __restrict__ ids, int n_ids,
                                                                  const int* __restrict__ n_ids_dev,
                                                                  int* __restrict__ status) {
  asm volatile("griddepcontrol.launch_dependents;");  // let k_generate_moving_obstacles be dispatched now
  if (n_ids_dev != nullptr) n_ids = min(n_ids, *n_ids_dev);
  const int li = blockIdx.x * blockDim.x + threadIdx.x;
  if (li >= n_ids) return;
  const int m = ids ? ids[li] : li;
  GenRng rp(gp.seed, (unsigned)m, AUV_GEN_SLOT_PATH, gp.epoch);
  // path choice: uniform over the bank (movingobstacles.py:28-31 draws a fresh curve), or -- path-major
  // pools -- the path the slot is laid out for: consecutive groups of path_group scenarios share a path
  const double upath = rp.u01();
  const int pid = gp.path_group > 0 ? (int)(((long long)m % gp.path_period) / gp.path_group) % pb.n_paths
                                    : min(pb.n_paths - 1, (int)(upath * pb.n_paths));
  GenRng rv(gp.seed, (unsigned)m, AUV_GEN_SLOT_VESSEL, gp.epoch);
  double x0, y0, dir0;
  gen_path_point(pb, pid, pb.hdr[pid].length, 0.0, x0, y0, dir0);
  // movingobstacles.py:34-38: init_state = path(0) + 50 (rand(2) - 0.5); angle = dir(0) + 2 pi (rand - 0.5);
  // in a world the start must be clear of land by land_clearance: redraw from the same stream
  double vx, vy, vpsi;
  for (int tries = 1;; ++tries) {
    vx = x0 + gp.init_pos_jitter * (rv.u01() - 0.5);
    vy = y0 + gp.init_pos_jitter * (rv.u01() - 0.5);
    vpsi = princip(dir0 + 2.0 * AUV_PI * (rv.u01() - 0.5));
    if (land_clear(pool, vx, vy, gp.land_clearance)) break;
    if (tries >= AUV_GEN_VESSEL_TRIES) {  // keep the last draw
      if (status) atomicOr(status, AUV_STATUS_GEN_LAND_BLOCKED);
      break;
    }
  }
  const_cast<int*>(pool.path_id)[m] = pid;
  double* wv = const_cast<double*>(pool.vessel_init);
  wv[3ll * m + 0] = vx;
  wv[3ll * m + 1] = vy;
  wv[3ll * m + 2] = vpsi;
}

// Launch 2 of 2, thread per (listed scenario, obstacle slot): slots [0, Km) moving, [Km, Km+Ks) static; the
// path and vessel start are read back from what k_generate_scenario_heads wrote.
__global__ void __maxnreg__(128) k_generate_moving_obstacles(const __grid_constant__ AuvGenParams gp,
                                                                    const __grid_constant__ AuvPathBank pb,
                                                                    const __grid_constant__ AuvScenarioPool pool,
                                                                    const int* __restrict__ ids, int n_ids,
                                                                    const int* __restrict__ n_ids_dev,
                                                                    int* __restrict__ status) {
  // launched as a programmatic dependent of k_generate_scenario_heads: wait until it has completed and its
  // writes are visible (a no-op after an ordinary launch)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int km = pool.k_moving, ks = pool.k_static, per = km + ks;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n_ids_dev != nullptr) n_ids = min(n_ids, *n_ids_dev);
  if (gid >= (long long)n_ids * per) return;
  const int li = (int)(gid / per), slot = (int)(gid - (long long)li * per);
  const int m = ids ? ids[li] : li;
  const int pid = pool.path_id[m];
  const double L = pb.hdr[pid].length;
  const double vx = pool.vessel_init[3ll * m], vy = pool.vessel_init[3ll * m + 1];
  // ---- helpers.generate_obstacle: rejection until clear of the vessel and of the goal (and, in a world, the
  // centre / track start clear of land by the radius / width)
  const bool moving = slot < km;
  const double disp_std = moving ? gp.mov_disp_std : gp.st_disp_std;
  const double mean = moving ? gp.mov_width_mean : gp.st_radius_mean;
  double gx, gy, gdir;
  gen_path_point(pb, pid, L, L, gx, gy, gdir);
  GenRng r(gp.seed, (unsigned)m, (unsigned)slot, gp.epoch);
  double ox = 0.0, oy = 0.0, rad = 1.0;
  int tries = 0;
  for (;; ++tries) {
    const double disp = disp_std * r.normal();
    const double s = (0.1 + 0.8 * r.u01()) * L;
    double px, py, pdir;
    gen_path_point(pb, pid, L, s, px, py, pdir);
    const double ang = princip(pdir - 0.5 * AUV_PI);
    double sa, ca;
    sincos(ang, &sa, &ca);
    ox = px + disp * ca;
    oy = py + disp * sa;
    rad = fmax(1.0, (double)r.poisson(mean));
    const double dv = sqrt((ox - vx) * (ox - vx) + (oy - vy) * (oy - vy)) - gp.vessel_width - rad;
    const double dg = sqrt((ox - gx) * (ox - gx) + (oy - gy) * (oy - gy)) - rad;
    if (fmin(dv, dg) > 0.0 && land_clear(pool, ox, oy, rad)) break;
    if (tries >= AUV_GEN_MAX_TRIES) {
      if (status) atomicOr(status, AUV_STATUS_GEN_GAVE_UP);
      break;
    }
  }
  if (moving) {
    // movingobstacles.py:51-75: direction = rand 2 pi, speed ~ U(1, 3), 10000-point linear track
    const double phi = 2.0 * AUV_PI * r.u01();
    const double speed = gp.mov_speed_lo + (gp.mov_speed_hi - gp.mov_speed_lo) * r.u01();
    double sp, cp;
    sincos(phi, &sp, &cp);
    const double ux = speed * cp, uy = speed * sp;
    const long long ps = (long long)m * km + slot;
    const_cast<double*>(pool.mov_start)[2 * ps] = ox;
    const_cast<double*>(pool.mov_start)[2 * ps + 1] = oy;
    const_cast<double*>(pool.mov_width)[ps] = rad;
    reinterpret_cast<int4*>(const_cast<int*>(pool.mov_track))[ps] = make_int4((int)ps, 9999, 0, 0);
    const_cast<double*>(pool.vel_table)[2 * ps] = ux;
    const_cast<double*>(pool.vel_table)[2 * ps + 1] = uy;
    // state right after reset(): update(0.1) in VesselObstacle.__init__ (obstacles.py:192-193) and
    // one more _update() at the end of _generate (movingobstacles.py:95)
    const double h2 = gp.post_generate_update ? gp.t_step_size : 0.0;
    const double last = gp.post_generate_update ? gp.t_step_size : 0.1;
    const_cast<double*>(pool.mov_pos0)[2 * ps] = (ox + 0.1 * ux) + h2 * ux;
    const_cast<double*>(pool.mov_pos0)[2 * ps + 1] = (oy + 0.1 * uy) + h2 * uy;
    const_cast<double*>(pool.mov_disp0)[2 * ps] = last * ux;
    const_cast<double*>(pool.mov_disp0)[2 * ps + 1] = last * uy;
    const_cast<double*>(pool.mov_counter0)[ps] = 0.1 + h2;
    if (pool.mov_lin != nullptr) {  // packed record of the closed-form update (auv_pool_pack layout)
      double* q = const_cast<double*>(pool.mov_lin) + ps * 8;
      q[0] = (ox + 0.1 * ux) + h2 * ux;
      q[1] = (oy + 0.1 * uy) + h2 * uy;
      q[2] = gp.t_step_size * ux;
      q[3] = gp.t_step_size * uy;
      q[4] = rad;
      q[5] = ox;
      q[6] = oy;
      q[7] = 0.0;
    }
  } else {
    const long long ps = (long long)m * ks + (slot - km);
    const_cast<double*>(pool.st_pos)[2 * ps] = ox;
    const_cast<double*>(pool.st_pos)[2 * ps + 1] = oy;
    const_cast<double*>(pool.st_radius)[ps] = rad;
    double* q = const_cast<double*>(pool.st_rec) + ps * 4;
    q[0] = ox;
    q[1] = oy;
    q[2] = rad;
    q[3] = 0.0;
  }
}

}  // namespace auv
