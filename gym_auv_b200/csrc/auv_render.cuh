// auv_render.cuh -- k_render: top-down RGB frames of live envs.  The frame rule (camera, layers, colours) is
// stated once, at AuvRender in include/auv_b200.h.  Included by auv_kernels.cu after the step kernels: it
// reuses load_slot / lin_position (obstacle geometry at the env's current obstacle state), pent_vertex,
// ngon_sides and the ray table as they are.
//
// Mapping: one CTA per (frame, 32 x 32 pixel tile), 256 threads, 4 pixels per thread.  Each pixel keeps the
// index of the first layer found to contain it (0 own-ship ... 8 sea).  Per drawable kind the CTA builds a
// display list in shared memory from the candidates whose bounds meet the tile (obstacle slots by enclosing
// circle, world polygons through the pool's grid cells under the tile, path blocks by their capsules, rays by
// a segment test), at most one chunk of candidates at a time, then every pixel tests the listed shapes of a
// layer above the one it already has.  No pixel walks all slots, all polygons or the whole polyline.
// Precision (DESIGN section 3): camera-relative geometry is formed in FP64 and rounded once; pixel tests are
// FP32.  Output bytes are plain stores (no atomics): the result is a union per layer, so the order in which
// the shared-memory lists are filled cannot change a byte.
#pragma once

namespace auv {

#define AUV_RENDER_TILE 32
#define AUV_RENDER_THREADS 256
#define AUV_RENDER_PPT (AUV_RENDER_TILE * AUV_RENDER_TILE / AUV_RENDER_THREADS)  // pixels per thread
#define AUV_RENDER_CHUNK 256     // candidates tested per round of a display list
#define AUV_RENDER_PATH_CHUNK 64 // path blocks per round (their vertices are staged)
#define AUV_RENDER_WORLD_LIST 512

// colour index -> 0xRRGGBB (an immediate per case: no constant-bank table)
__device__ __forceinline__ uint32_t render_rgb(int layer) {
  switch (layer) {
    case 0: return AUV_RGB_OWNSHIP;
    case 1: return AUV_RGB_RAY_HIT;
    case 2: return AUV_RGB_RAY_CLEAR;
    case 3: return AUV_RGB_MOVING;
    case 4: return AUV_RGB_STATIC;
    case 5: return AUV_RGB_GOAL;
    case 6: return AUV_RGB_PATH;
    case 7: return AUV_RGB_LAND;
    default: return AUV_RGB_SEA;
  }
}
#define RL_SHIP 0
#define RL_RAY_HIT 1
#define RL_RAY_CLEAR 2
#define RL_MOVING 3
#define RL_STATIC 4
#define RL_GOAL 5
#define RL_PATH 6
#define RL_LAND 7
#define RL_SEA 8

struct RenderArgs {
  AuvConfig cfg;
  AuvRayTable rays;
  AuvPathBank paths;
  AuvScenarioPool pool;
  AuvBatch batch;
  const float* obs;
  const int32_t* env_ids;
  uint8_t* frames;
  double half_width;
  int obs_dim, width, height, tiles_x;
};

// pixel-centre rectangle of a tile, camera frame (FP64)
struct TileRect {
  double x0, x1, y0, y1;
};

// does the segment a -> b meet the rectangle grown by g?  (Liang-Barsky clip: exact for the grown rectangle,
// which contains every point within g of the original one)
__device__ __forceinline__ bool seg_meets_rect(double ax, double ay, double bx, double by, const TileRect& t, double g) {
  const double dx = bx - ax, dy = by - ay;
  const double p[4] = {-dx, dx, -dy, dy};
  const double q[4] = {ax - (t.x0 - g), (t.x1 + g) - ax, ay - (t.y0 - g), (t.y1 + g) - ay};
  double t0 = 0.0, t1 = 1.0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (p[k] == 0.0) {
      if (q[k] < 0.0) return false;
    } else {
      const double r = q[k] / p[k];
      if (p[k] < 0.0) t0 = fmax(t0, r);
      else t1 = fmin(t1, r);
    }
  }
  return t0 <= t1;
}

__device__ __forceinline__ bool disc_meets_rect(double cx, double cy, double r, const TileRect& t, double g) {
  const double dx = fmax(fmax(t.x0 - cx, cx - t.x1), 0.0), dy = fmax(fmax(t.y0 - cy, cy - t.y1), 0.0);
  const double rr = r + g;
  return dx * dx + dy * dy <= rr * rr;
}

// is p within sqrt(h2) of the segment a-b?  (no division: the perpendicular case compares cross^2 with h2 |e|^2)
__device__ __forceinline__ bool seg_within(float px, float py, float ax, float ay, float bx, float by, float h2) {
  const float ex = bx - ax, ey = by - ay, wx = px - ax, wy = py - ay;
  const float dot = wx * ex + wy * ey, len2 = ex * ex + ey * ey;
  if (dot <= 0.f) return wx * wx + wy * wy <= h2;
  if (dot >= len2) {
    const float ux = px - bx, uy = py - by;
    return ux * ux + uy * uy <= h2;
  }
  const float cr = wx * ey - wy * ex;
  return cr * cr <= h2 * len2;
}

// inside the convex pentagon v[0..4] (either orientation; the boundary counts as inside)
__device__ __forceinline__ bool in_pentagon(const float2* v, float px, float py) {
  bool pos = true, neg = true;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const float2 a = v[k], b = v[k == 4 ? 0 : k + 1];
    const float cr = (b.x - a.x) * (py - a.y) - (b.y - a.y) * (px - a.x);
    pos = pos && cr >= 0.f;
    neg = neg && cr <= 0.f;
  }
  return pos || neg;
}

// inside the filled regular n-gon of circumradius r with vertices r unit[k 64 / n] (counter-clockwise), q relative
// to its centre: decided by the circumcircle / incircle where it can be, else by the edge whose angular sector
// holds q and its two neighbours (inside a convex polygon <=> inside all three of those half-planes)
__device__ __forceinline__ bool in_ngon(const float2* unit, float qx, float qy, float r, int n) {
  const float d2 = qx * qx + qy * qy;
  if (d2 > r * r) return false;
  const float ri = r * cospif(1.f / (float)n);
  if (d2 < ri * ri * 0.9999f) return true;
  const int sh = 6 - (31 - __clz(n));  // unit table stride 64 / n
  const int k0 = (int)floorf(atan2f(qy, qx) * ((float)n * 0.15915494309189535f)) & (n - 1);
#pragma unroll
  for (int t = -1; t <= 1; ++t) {
    const int k = (k0 + t) & (n - 1);
    const float2 ua = unit[k << sh], ub = unit[((k + 1) & (n - 1)) << sh];
    const float ax = r * ua.x, ay = r * ua.y, bx = r * ub.x, by = r * ub.y;
    if ((bx - ax) * (qy - ay) - (by - ay) * (qx - ax) < 0.f) return false;
  }
  return true;
}

// even-odd rule on the closed ring v[0..nv) (last vertex repeats the first), the crossing test of point_in_ring
__device__ __forceinline__ bool in_ring(const float2* v, int nv, float px, float py) {
  bool in = false;
  float2 a = v[0];
  for (int k = 1; k < nv; ++k) {
    const float2 b = v[k];
    if ((a.y > py) != (b.y > py)) {
      const float xint = a.x + (py - a.y) * (b.x - a.x) / (b.y - a.y);
      if (xint > px) in = !in;
    }
    a = b;
  }
  return in;
}

// CTA barrier: does some pixel of the tile still lack a layer at or above `layer` + 1?
__device__ __forceinline__ bool tile_needs(const int (&best)[AUV_RENDER_PPT], int layer) {
  bool nd = false;
#pragma unroll
  for (int k = 0; k < AUV_RENDER_PPT; ++k) nd = nd || best[k] > layer;
  return __syncthreads_or(nd) != 0;
}

// shade the world polygons listed in s_list[0 .. *s_cnt) (a polygon may be listed twice: the union does not
// change), one at a time with its vertices staged in s_wv, then empty the list.  Called by the whole CTA.
__device__ __forceinline__ void land_flush(int (&best)[AUV_RENDER_PPT], const float (&px)[AUV_RENDER_PPT],
                                           const float (&py)[AUV_RENDER_PPT], const AuvScenarioPool& pool, double x,
                                           double y, const int* s_list, float2* s_wv, int* s_cnt) {
  const int n = *s_cnt;
  for (int li = 0; li < n; ++li) {
    if (!tile_needs(best, RL_LAND)) break;  // (also the barrier before s_wv is overwritten)
    const int wi = s_list[li];
    const int vb = pool.world_voff[wi], nv = pool.world_voff[wi + 1] - vb;
    for (int v = threadIdx.x; v < nv; v += AUV_RENDER_THREADS) {
      const double2 q = reinterpret_cast<const double2*>(pool.world_verts)[vb + v];
      s_wv[v] = make_float2((float)(q.x - x), (float)(q.y - y));
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < AUV_RENDER_PPT; ++k)
      if (best[k] > RL_LAND && in_ring(s_wv, nv, px[k], py[k])) best[k] = RL_LAND;
  }
  __syncthreads();
  if (threadIdx.x == 0) *s_cnt = 0;
  __syncthreads();
}

// launched with AUV_RENDER_THREADS threads; __maxnreg__ rather than __launch_bounds__ for the reason given at
// k_generate_scenario_heads (the FP64 division / trig slow paths spilled at the 64 registers ptxas chose)
__global__ void __maxnreg__(128) k_render(const __grid_constant__ RenderArgs A) {
  __shared__ float2 s_unit[64];
  __shared__ float2 s_ship[5];
  __shared__ float4 s_item[AUV_RENDER_CHUNK];                        // rays (ex, ey, -, hit) | circles (cx, cy, r, n)
  __shared__ float2 s_pent[AUV_RENDER_CHUNK][5];                     // moving obstacles
  __shared__ float2 s_pv[AUV_RENDER_PATH_CHUNK][AUV_PATH_BLOCK + 1]; // path block vertices
  __shared__ float4 s_pch[AUV_RENDER_PATH_CHUNK];                    // path block chord (camera frame)
  __shared__ float2 s_pdev[AUV_RENDER_PATH_CHUNK];                   // 1/|e|^2, deviation
  __shared__ int s_pblk[AUV_RENDER_PATH_CHUNK];
  __shared__ int s_list[AUV_RENDER_WORLD_LIST];                      // world polygons
  __shared__ float2 s_wv[AUV_MAX_POLY_VERTS];
  __shared__ int s_cnt;

  const int tid = threadIdx.x;
  const int f = blockIdx.x;
  const int W = A.width, H = A.height;
  const int r0 = (blockIdx.y / A.tiles_x) * AUV_RENDER_TILE, c0 = (blockIdx.y % A.tiles_x) * AUV_RENDER_TILE;
  const int col = c0 + (tid & (AUV_RENDER_TILE - 1));
  uint8_t* frame = A.frames + (size_t)f * H * W * 3;
  const int e = A.env_ids[f];
  const AuvBatch& batch = A.batch;
  const int N = batch.n_envs;
  if (e < 0 || e >= N) {  // an id outside the batch is never read: the frame is zeros
#pragma unroll
    for (int k = 0; k < AUV_RENDER_PPT; ++k) {
      const int row = r0 + (tid >> 5) + k * (AUV_RENDER_THREADS / AUV_RENDER_TILE);
      if (row < H && col < W) {
        uint8_t* px = frame + ((size_t)row * W + col) * 3;
        px[0] = px[1] = px[2] = 0;
      }
    }
    return;
  }
  const double s = 2.0 * A.half_width / (double)W;
  const double x = batch.state[e], y = batch.state[N + e], psi = batch.state[2 * N + e];
  const int scn = batch.scn_id[e], n_upd = batch.obst_steps[e];
  const AuvConfig& cfg = A.cfg;
  const AuvScenarioPool& pool = A.pool;

  // pixel centres, camera frame
  float px[AUV_RENDER_PPT], py[AUV_RENDER_PPT];
  int best[AUV_RENDER_PPT];
  const float pyc = (float)(((double)col + 0.5 - 0.5 * W) * s);
#pragma unroll
  for (int k = 0; k < AUV_RENDER_PPT; ++k) {
    const int row = r0 + (tid >> 5) + k * (AUV_RENDER_THREADS / AUV_RENDER_TILE);
    px[k] = (float)((0.5 * H - (double)row - 0.5) * s);
    py[k] = pyc;
    best[k] = (row < H && col < W) ? RL_SEA : -1;  // -1: outside the frame, never drawn
  }
  const int r1 = min(r0 + AUV_RENDER_TILE, H), c1 = min(c0 + AUV_RENDER_TILE, W);
  TileRect rect;
  rect.x0 = (0.5 * H - (double)(r1 - 1) - 0.5) * s;
  rect.x1 = (0.5 * H - (double)r0 - 0.5) * s;
  rect.y0 = ((double)c0 + 0.5 - 0.5 * W) * s;
  rect.y1 = ((double)(c1 - 1) + 0.5 - 0.5 * W) * s;
  const double pad = 0.01 * s;  // covers the FP32 rounding of the pixel tests

  // ---- 1 own-ship
  double cpsi, spsi;
  sincos(psi, &spsi, &cpsi);
  if (tid < 5) {
    double vx, vy;
    pent_vertex(tid, 0.0, 0.0, fmax(cfg.vessel_width, AUV_RENDER_SHIP_MIN_PX * s), cpsi, spsi, vx, vy);
    s_ship[tid] = make_float2((float)vx, (float)vy);
  }
  if (tid < 64 && A.rays.unit64 != nullptr) {
    const double2 u = reinterpret_cast<const double2*>(A.rays.unit64)[tid];
    s_unit[tid] = make_float2((float)u.x, (float)u.y);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < AUV_RENDER_PPT; ++k)
    if (best[k] > RL_SHIP && in_pentagon(s_ship, px[k], py[k])) best[k] = RL_SHIP;

  // ---- 2 LiDAR rays (channel 0 of the observation row)
  if (cfg.use_lidar && tile_needs(best, RL_SHIP)) {
    const int R = cfg.n_sensors;
    const double range = cfg.sensor_range, log_range = log1p(range);
    const float* row = A.obs + (size_t)e * A.obs_dim + 6;
    const double2* cs = reinterpret_cast<const double2*>(A.rays.cos_sin);
    const float h = (float)(AUV_RENDER_RAY_HALF_PX * s), h2 = h * h;
    for (int base = 0; base < R; base += AUV_RENDER_CHUNK) {
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      const int i = base + tid;
      if (i < R) {
        const double c = (double)row[i];
        const double d = c == 0.0 ? range : (cfg.sensor_log_transform ? expm1((1.0 - c) * log_range) : (1.0 - c) * range);
        const double2 a = cs[i];
        const double ex = d * (cpsi * a.x - spsi * a.y), ey = d * (spsi * a.x + cpsi * a.y);
        if (seg_meets_rect(0.0, 0.0, ex, ey, rect, AUV_RENDER_RAY_HALF_PX * s + pad))
          s_item[atomicAdd(&s_cnt, 1)] = make_float4((float)ex, (float)ey, 0.f, c > 0.0 ? 1.f : 0.f);
      }
      __syncthreads();
      const int n = s_cnt;
      for (int li = 0; li < n; ++li) {
        const float4 it = s_item[li];
        const int layer = it.w != 0.f ? RL_RAY_HIT : RL_RAY_CLEAR;
#pragma unroll
        for (int k = 0; k < AUV_RENDER_PPT; ++k)
          if (best[k] > layer && seg_within(px[k], py[k], 0.f, 0.f, it.x, it.y, h2)) best[k] = layer;
      }
      __syncthreads();
    }
  }

  // ---- 3 moving obstacles
  const int km = pool.k_moving, ks = pool.k_static;
  if (km > 0 && tile_needs(best, RL_RAY_CLEAR)) {
    for (int base = 0; base < km; base += AUV_RENDER_CHUNK) {
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      const int j = base + tid;
      if (j < km) {
        const SlotGeom g = load_slot(pool, batch, e, scn, j, x, y, n_upd);
        if (g.valid && disc_meets_rect(g.cx, g.cy, g.rho, rect, pad)) {
          const int li = atomicAdd(&s_cnt, 1);
          const double bx0 = g.cx - (g.geo * (2.0 / 9.0)) * g.hx, by0 = g.cy - (g.geo * (2.0 / 9.0)) * g.hy;
#pragma unroll
          for (int v = 0; v < 5; ++v) {
            double vx, vy;
            pent_vertex(v, bx0, by0, g.geo, g.hx, g.hy, vx, vy);
            s_pent[li][v] = make_float2((float)vx, (float)vy);
          }
        }
      }
      __syncthreads();
      const int n = s_cnt;
      for (int li = 0; li < n; ++li)
#pragma unroll
        for (int k = 0; k < AUV_RENDER_PPT; ++k)
          if (best[k] > RL_MOVING && in_pentagon(s_pent[li], px[k], py[k])) best[k] = RL_MOVING;
      __syncthreads();
    }
  }

  // ---- 4 static circles
  if (ks > 0 && tile_needs(best, RL_MOVING)) {
    for (int base = 0; base < ks; base += AUV_RENDER_CHUNK) {
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      const int j = base + tid;
      if (j < ks) {
        const SlotGeom g = load_slot(pool, batch, e, scn, km + j, x, y, n_upd);
        if (g.valid && disc_meets_rect(g.cx, g.cy, g.rho, rect, pad))
          s_item[atomicAdd(&s_cnt, 1)] = make_float4((float)g.cx, (float)g.cy, (float)g.geo, __int_as_float(g.nv - 1));
      }
      __syncthreads();
      const int n = s_cnt;
      for (int li = 0; li < n; ++li) {
        const float4 it = s_item[li];
#pragma unroll
        for (int k = 0; k < AUV_RENDER_PPT; ++k)
          if (best[k] > RL_STATIC && in_ngon(s_unit, px[k] - it.x, py[k] - it.y, it.z, __float_as_int(it.w)))
            best[k] = RL_STATIC;
      }
      __syncthreads();
    }
  }

  // ---- 5 goal, 6 path
  const AuvPathHdr hdr = A.paths.hdr[batch.env_pid[e]];
  {
    const float gx = (float)(hdr.end_x - x), gy = (float)(hdr.end_y - y);
    const float gr = (float)(AUV_RENDER_GOAL_PX * s), gr2 = gr * gr;
#pragma unroll
    for (int k = 0; k < AUV_RENDER_PPT; ++k) {
      const float dx = px[k] - gx, dy = py[k] - gy;
      if (best[k] > RL_GOAL && dx * dx + dy * dy <= gr2) best[k] = RL_GOAL;
    }
  }
  if (tile_needs(best, RL_GOAL)) {
    const double ox = hdr.ox - x, oy = hdr.oy - y;
    const int nblk = (hdr.nseg + AUV_PATH_BLOCK - 1) / AUV_PATH_BLOCK;
    const float h = (float)(AUV_RENDER_PATH_HALF_PX * s), h2 = h * h;
    const double2* __restrict__ pv = reinterpret_cast<const double2*>(A.paths.poly_xy) + hdr.v0;
    for (int base = 0; base < nblk; base += AUV_RENDER_PATH_CHUNK) {
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      const int b = base + tid;
      if (tid < AUV_RENDER_PATH_CHUNK && b < nblk) {
        const float4 ch = reinterpret_cast<const float4*>(A.paths.blk_chord)[hdr.b0 + b];
        const float2 dv = reinterpret_cast<const float2*>(A.paths.blk_dev)[hdr.b0 + b];
        const double ax = ox + (double)ch.x, ay = oy + (double)ch.y;
        if (seg_meets_rect(ax, ay, ax + (double)ch.z, ay + (double)ch.w, rect, (double)dv.y + AUV_RENDER_PATH_HALF_PX * s + pad)) {
          const int li = atomicAdd(&s_cnt, 1);
          s_pblk[li] = b;
          s_pch[li] = make_float4((float)ax, (float)ay, ch.z, ch.w);
          s_pdev[li] = dv;
        }
      }
      __syncthreads();
      const int n = s_cnt;
      for (int idx = tid; idx < n * (AUV_PATH_BLOCK + 1); idx += AUV_RENDER_THREADS) {
        const int li = idx / (AUV_PATH_BLOCK + 1), v = idx - li * (AUV_PATH_BLOCK + 1);
        const int sv = s_pblk[li] * AUV_PATH_BLOCK + v;
        if (sv <= hdr.nseg) {
          const double2 q = pv[sv];
          s_pv[li][v] = make_float2((float)(q.x - x), (float)(q.y - y));
        }
      }
      __syncthreads();
      for (int li = 0; li < n; ++li) {
        const float4 ch = s_pch[li];
        const float2 dv = s_pdev[li];
        const float reach = dv.y + h + (float)pad, reach2 = reach * reach;
        const int nseg = min(AUV_PATH_BLOCK, hdr.nseg - s_pblk[li] * AUV_PATH_BLOCK);
#pragma unroll
        for (int k = 0; k < AUV_RENDER_PPT; ++k) {
          if (best[k] <= RL_PATH || pt_chord_d2_f(px[k], py[k], ch, dv.x) > reach2) continue;
          for (int sg = 0; sg < nseg; ++sg) {
            const float2 a = s_pv[li][sg], bq = s_pv[li][sg + 1];
            if (seg_within(px[k], py[k], a.x, a.y, bq.x, bq.y, h2)) {
              best[k] = RL_PATH;
              break;
            }
          }
        }
      }
      __syncthreads();
    }
  }

  // ---- 7 land: world polygons through the grid cells under the tile (or every polygon without a grid)
  if (pool.n_world > 0 && tile_needs(best, RL_PATH)) {
    const int K = km + ks;
    const bool grid = pool.world_cell_off != nullptr;
    int ix0 = 0, iy0 = 0, nxr = 1, cells = 1;
    if (grid) {
      const double cell = pool.world_grid_cell;
      ix0 = max(0, (int)floor((x + rect.x0 - pad - pool.world_grid_x0) / cell));
      const int ix1 = min(pool.world_grid_nx - 1, (int)floor((x + rect.x1 + pad - pool.world_grid_x0) / cell));
      iy0 = max(0, (int)floor((y + rect.y0 - pad - pool.world_grid_y0) / cell));
      const int iy1 = min(pool.world_grid_ny - 1, (int)floor((y + rect.y1 + pad - pool.world_grid_y0) / cell));
      nxr = ix1 - ix0 + 1;
      cells = (ix1 < ix0 || iy1 < iy0) ? 0 : nxr * (iy1 - iy0 + 1);
    }
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    for (int ci = 0; ci < cells; ++ci) {
      int i0 = 0, i1 = pool.n_world;
      if (grid) {
        const int c = (iy0 + ci / nxr) * pool.world_grid_nx + ix0 + ci % nxr;
        i0 = pool.world_cell_off[c];
        i1 = pool.world_cell_off[c + 1];
      }
      for (int it = i0; it < i1; it += AUV_RENDER_CHUNK) {
        // the list may only grow by a chunk when a chunk still fits: every thread reads the count (stable since the
        // previous barrier) before any thread appends, so the flush decision is the same in the whole CTA
        const int listed = s_cnt;
        __syncthreads();
        if (listed > AUV_RENDER_WORLD_LIST - AUV_RENDER_CHUNK) land_flush(best, px, py, pool, x, y, s_list, s_wv, &s_cnt);
        if (it + tid < i1) {
          const int wi = grid ? pool.world_cell_items[it + tid] : it + tid;
          const SlotGeom g = load_slot(pool, batch, e, scn, K + wi, x, y, n_upd);
          if (g.valid && g.nv <= AUV_MAX_POLY_VERTS && disc_meets_rect(g.cx, g.cy, g.rho, rect, pad))
            s_list[atomicAdd(&s_cnt, 1)] = wi;
        }
        __syncthreads();
      }
    }
    land_flush(best, px, py, pool, x, y, s_list, s_wv, &s_cnt);
  }

#pragma unroll
  for (int k = 0; k < AUV_RENDER_PPT; ++k) {
    if (best[k] < 0) continue;
    const int row = r0 + (tid >> 5) + k * (AUV_RENDER_THREADS / AUV_RENDER_TILE);
    const uint32_t rgb = render_rgb(best[k]);
    uint8_t* p = frame + ((size_t)row * W + col) * 3;
    p[0] = (uint8_t)(rgb >> 16);
    p[1] = (uint8_t)(rgb >> 8);
    p[2] = (uint8_t)rgb;
  }
}

}  // namespace auv
