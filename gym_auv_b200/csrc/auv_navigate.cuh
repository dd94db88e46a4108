// auv_navigate.cuh -- path projection (exact hierarchical LineString.project), PCHIP
// evaluation and Vessel.navigate, one thread per env (FP64).
#pragma once
#include "auv_device.cuh"
#include "../../include/auv_b200.h"

namespace auv {

// ------------------------------------------------------------------------------------
// Path projection + navigation features, a group of G lanes per env (FP64)
//   path.py:61-93 (PCHIP eval, LineString.project), vessel.py:461-541 (navigate)
// The result is the env's navigation record nav[e][AUV_NAV_W] in HBM; the warp-per-env
// LiDAR kernel reads it back (one 96 B coalesced load).
// ------------------------------------------------------------------------------------
#define NAV_S 0
#define NAV_CHI 1
#define NAV_YE 2
#define NAV_SLA 3
#define NAV_LA_ERR 4
#define NAV_HEAD_ERR 5
#define NAV_GOAL 6
#define NAV_PROGRESS 7
// [8..23]: the 128 B hand-over line of the casting stage (k_lidar reads exactly these 16 doubles)
#define NAV_HAND 8
#define NAV_COSPSI 8
#define NAV_SINPSI 9
#define NAV_REACHED 10
#define NAV_H_YE 11
#define NAV_REWARD_BASE 12
#define NAV_H_GOAL 13
#define NAV_H_PROGRESS 14
#define NAV_X 16
#define NAV_Y 17
#define NAV_PSI 18
#define NAV_CUM 19
#define NAV_CTE 20
#define NAV_TSTEP 21
#define NAV_SCN 22
#define NAV_CNT 23

// scipy PPoly evaluation (extrapolate=True): interval j with x[j] <= s < x[j+1], clamped.
// One PCHIP piece is one 96 B record (its two knots + 8 coefficients), so an evaluation is a
// single round of loads: the knots are nearly uniform, the record of the uniform guess almost
// always is the right one; its own knots tell, and the neighbour is fetched when it is not.
struct PchipOut {
  double px, py, dx, dy;
};
struct PPiece {
  double2 k, a, b, c, d;  // (knot j, knot j+1), x: (c0, c1), (c2, c3), y: (c0, c1), (c2, c3)
};
__device__ __forceinline__ PPiece pp_load(const double* __restrict__ base, int j) {
  const double2* __restrict__ r = reinterpret_cast<const double2*>(base + (long long)j * AUV_PP_W);
  PPiece p;
  p.k = r[0];
  p.a = r[1];
  p.b = r[2];
  p.c = r[3];
  p.d = r[4];
  return p;
}
__device__ __forceinline__ void pp_settle(const double* __restrict__ base, int nk, double s, int& j, PPiece& p) {
  while (j > 0 && s < p.k.x) p = pp_load(base, --j);
  while (j < nk - 2 && s >= p.k.y) p = pp_load(base, ++j);
}
__device__ __forceinline__ void pp_eval(const PPiece& p, double s, PchipOut& o) {
  const double t = s - p.k.x;
  o.px = ((p.a.x * t + p.a.y) * t + p.b.x) * t + p.b.y;
  o.py = ((p.c.x * t + p.c.y) * t + p.d.x) * t + p.d.y;
  o.dx = (3.0 * p.a.x * t + 2.0 * p.a.y) * t + p.b.x;
  o.dy = (3.0 * p.c.x * t + 2.0 * p.c.y) * t + p.d.x;
}
// two evaluations, both records in flight together.  L = Path.length (last knot).
__device__ __forceinline__ void pchip_eval2(const AuvPathBank& pb, int pid, double L, double s1, double s2,
                                            PchipOut& o1, PchipOut& o2) {
  const int nk = pb.n_knots;
  const double* __restrict__ base = pb.pp + (long long)pid * (nk - 1) * AUV_PP_W;
  const double per = (double)(nk - 1) / L;  // pieces per metre: the uniform guess (settled against the record's own knots)
  int j1 = max(0, min(nk - 2, (int)(s1 * per)));
  int j2 = max(0, min(nk - 2, (int)(s2 * per)));
  PPiece p1 = pp_load(base, j1), p2 = pp_load(base, j2);
  pp_settle(base, nk, s1, j1, p1);
  pp_settle(base, nk, s2, j2, p2);
  pp_eval(p1, s1, o1);
  pp_eval(p2, s2, o2);
}

// exact squared distance from P to segment AB (GEOS Distance::pointToSegment, squared;
// the r<=0 / r>=1 tests are done on the numerator, no division)
__device__ __forceinline__ double seg_d2(double px, double py, double2 A, double2 B) {
  const double ex = B.x - A.x, ey = B.y - A.y;
  const double wx = px - A.x, wy = py - A.y;
  const double len2 = ex * ex + ey * ey;
  const double num = wx * ex + wy * ey;
  if (len2 == 0.0 || num <= 0.0) return wx * wx + wy * wy;
  if (num >= len2) {
    const double zx = px - B.x, zy = py - B.y;
    return zx * zx + zy * zy;
  }
  const double cr = wx * ey - wy * ex;
  return cr * cr / len2;
}

// the same distance as the exact fraction num / den (den > 0): candidates are compared by cross-multiplication,
// one division for the winner instead of one per segment (FP64 divisions are ~20 instructions each)
__device__ __forceinline__ void seg_d2_frac(double px, double py, double2 A, double2 B, double& num, double& den) {
  const double ex = B.x - A.x, ey = B.y - A.y;
  const double wx = px - A.x, wy = py - A.y;
  const double len2 = ex * ex + ey * ey;
  const double t = wx * ex + wy * ey;
  den = 1.0;
  if (len2 == 0.0 || t <= 0.0) {
    num = wx * wx + wy * wy;
  } else if (t >= len2) {
    const double zx = px - B.x, zy = py - B.y;
    num = zx * zx + zy * zy;
  } else {
    const double cr = wx * ey - wy * ex;
    num = cr * cr;
    den = len2;
  }
}

// ---- sub-warp groups: G consecutive lanes (G = 4, 8, 16 or 32) work on one env
template <int G>
__device__ __forceinline__ unsigned group_mask(int lane) {
  return G == 32 ? AUV_FULL : (((1u << G) - 1u) << (lane & ~(G - 1)));
}
template <int G>
__device__ __forceinline__ float group_min(unsigned gm, float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(gm, v, o));
  return v;
}
// bits of the group's lanes (bit k = lane k of the group) for which pred holds
template <int G>
__device__ __forceinline__ unsigned group_ballot(unsigned gm, int lane, bool pred) {
  const unsigned b = __ballot_sync(gm, pred);
  return G == 32 ? b : ((b >> (lane & ~(G - 1))) & ((1u << G) - 1u));
}

// capsule tables of one path: the global arrays, or the CTA's shared-memory copy of them
struct PathTabs {
  const float4* sbc;    // superblock chords
  const float2* sba;    // superblock (1/|e|^2, deviation)
  const float4* chord;  // block chords
  const float2* aux;    // block (1/|e|^2, deviation)
};

constexpr int kSubPerBlk = AUV_PATH_BLOCK / AUV_PATH_SUB;  // sub-blocks of a block

// GEOS LengthIndexOfPoint::indexOf (LineString.project) restated as an exact four-level
// search, executed by a GROUP of G lanes per env.  Level 3 = superblocks of AUV_PATH_SUPER
// blocks, level 2 = blocks of 32 segments, level 1 = sub-blocks of AUV_PATH_SUB segments; each
// node is a capsule (chord, max deviation) that contains its part of the polyline, so
//   dist(P, node) in [dc - dev, dc + dev],  dc = dist(P, chord)   (FP32, padded).
// An upper bound `ub` of the minimum distance comes either from the segment the previous step's
// projection ended on (WARM: the own-ship moves < 1 m per step, so the exact FP64 distance to a few
// segments around it is within millimetres of the answer -- it is only used as a bound, the search
// below stays exhaustive) or, without one (first step of an episode), from pass A over the
// superblock capsules and pass B over the block capsules of the surviving superblocks.  Pass C
// tests the sub-block capsules of every block whose lower bound does not exceed `ub` and refines
// the surviving sub-blocks in FP64 (a segment d along the path from the foot point is ~d^2 / 2r farther
// away at cross-track distance r, so these are the one or two sub-blocks around it).  In every pass the lanes of
// the group take different nodes / segments, so one round of loads covers G of them, and bounds are
// shared by shuffle-min; all bounds are compared in the squared domain.  Every loop pops the next set
// bit of a mask that is uniform in the group ("by rank"): the groups of a warp then run their r-th
// live node together instead of serialising over node indices.  The arg-min is lexicographic in
// (distance, segment index), which is GEOS's "first minimum wins" independent of visiting order.
// Every lane returns the same arclength; seg_out = the winning segment.
#ifdef AUV_NOINLINE_PROJECT
#define AUV_PROJECT_INLINE __noinline__
#else
#define AUV_PROJECT_INLINE __forceinline__
#endif
#ifdef AUV_NOINLINE_NAVIGATE
#define AUV_NAVIGATE_INLINE __noinline__
#else
#define AUV_NAVIGATE_INLINE __forceinline__
#endif
// Upper bound of the distance without a previous segment (first step of an episode): pass A over
// the superblock capsules, pass B over the block capsules of the superblocks that survive it.
// Cold: kept out of line so that the hot path of the kernel stays small (the step kernel is
// instruction-cache bound otherwise: 130 KB of SASS before this split).
template <int G>
__device__ __noinline__ float project_cold_bound(const PathTabs& T, const int nblk, const int nsb, const float qx,
                                                 const float qy, const float pad, const int lane, const unsigned gm) {
  constexpr int KB = AUV_PATH_SUPER / G;
  const int sub = lane & (G - 1);
  const float up = 1.f + 4e-6f, dn2 = (1.f - 4e-6f) * (1.f - 4e-6f);
  float ub = INFINITY;
#define AUV_TIGHTEN(d2, dv)                                         \
  if ((d2) < ub * ub) ub = fminf(ub, sqrtf(d2) * up + (dv) + pad);
#define AUV_PRUNED(d2, dv) ((d2) * dn2 > (ub + (dv) + pad) * (ub + (dv) + pad))
  for (int g0 = 0; g0 < nsb; g0 += G) {
    const int i = min(g0 + sub, nsb - 1);
    const float2 ax = T.sba[i];
    const float d2 = pt_chord_d2_f(qx, qy, T.sbc[i], ax.x);
    AUV_TIGHTEN(d2, ax.y)
  }
  ub = group_min<G>(gm, ub);
  for (int sb = 0; sb < nsb; ++sb) {
    const float2 a0 = T.sba[sb];
    if (AUV_PRUNED(pt_chord_d2_f(qx, qy, T.sbc[sb], a0.x), a0.y)) continue;  // uniform in the group
    const int be = min(nblk, (sb + 1) * AUV_PATH_SUPER);
#pragma unroll 1
    for (int k = 0; k < KB; ++k) {
      const int i = min(sb * AUV_PATH_SUPER + k * G + sub, be - 1);
      const float2 ax = T.aux[i];
      const float d2 = pt_chord_d2_f(qx, qy, T.chord[i], ax.x);
      AUV_TIGHTEN(d2, ax.y)
    }
    ub = group_min<G>(gm, ub);
  }
#undef AUV_TIGHTEN
#undef AUV_PRUNED
  return ub;
}

template <int G>
__device__ AUV_PROJECT_INLINE double project_group(const AuvPathBank& pb, const AuvPathHdr& h, const PathTabs& T,
                                                   const double px, const double py, const int prev_seg,
                                                   const int lane, const unsigned gm, int& seg_out, int* status = nullptr) {
  constexpr int KB = AUV_PATH_SUPER / G;  // blocks of a superblock per lane
  constexpr int SPL = AUV_PATH_SUB > G ? AUV_PATH_SUB / G : 1;  // segments of a sub-block per lane
  static_assert(G >= kSubPerBlk, "one lane per sub-block of a block");
  const int sub = lane & (G - 1);
  const int nseg = h.nseg;
  const int nblk = (nseg + AUV_PATH_BLOCK - 1) / AUV_PATH_BLOCK;
  const int nsb = (nblk + AUV_PATH_SUPER - 1) / AUV_PATH_SUPER;
  const float qx = (float)(px - h.ox), qy = (float)(py - h.oy);
  const float pad = 1e-6f * (fabsf(qx) + fabsf(qy)) + 1e-6f;
  const float4* chord = T.chord;
  const float2* aux = T.aux;
  const float4* sbc = T.sbc;
  const float2* sba = T.sba;
  const double2* __restrict__ poly = reinterpret_cast<const double2*>(pb.poly_xy) + h.v0;
  const float4* __restrict__ subc = reinterpret_cast<const float4*>(pb.sub_chord) + kSubPerBlk * h.b0;
  const float2* __restrict__ subd = reinterpret_cast<const float2*>(pb.sub_dev) + kSubPerBlk * h.b0;
  const float up = 1.f + 4e-6f, dn2 = (1.f - 4e-6f) * (1.f - 4e-6f);
  float ub = INFINITY;
#define AUV_TIGHTEN(d2, dv)                                         \
  if ((d2) < ub * ub) ub = fminf(ub, sqrtf(d2) * up + (dv) + pad);
#define AUV_PRUNED(d2, dv) ((d2) * dn2 > (ub + (dv) + pad) * (ub + (dv) + pad))
  const bool warm = prev_seg >= 0 && prev_seg < nseg;  // uniform in the group
  if (warm) {
    // lanes look at segments prev-3, prev, prev+3, prev+6 (...): an actual segment's exact distance
    // (FP64; rounding to FP32 is covered by `up`)
    const int k = min(max(prev_seg + (sub - 1) * 3, 0), nseg - 1);
    ub = sqrtf(group_min<G>(gm, (float)seg_d2(px, py, poly[k], poly[k + 1]))) * up + pad;
  } else {
    ub = project_cold_bound<G>(T, nblk, nsb, qx, qy, pad, lane, gm);  // first step of an episode: out of line
  }
  double best_num = INFINITY, best_den = 1.0;  // smallest squared distance so far, as a fraction
  int best_seg = 0x7fffffff;
  // superblocks in windows of 32 (one bit each); the lanes test different superblocks
  for (int w0 = 0; w0 < nsb; w0 += 32) {
    const int wn = min(32, nsb - w0);
    unsigned live = 0u;
#pragma unroll
    for (int k = 0; k < 32 / G; ++k) {
      if (k * G >= wn) break;  // (uniform in the group; in the warp too when its envs share a path)
      const int t = k * G + sub;
      const int i = min(w0 + t, nsb - 1);
      const float2 a0 = sba[i];
      live |= group_ballot<G>(gm, lane, t < wn && !AUV_PRUNED(pt_chord_d2_f(qx, qy, sbc[i], a0.x), a0.y)) << (k * G);
    }
    // pass C: exact refine of the blocks that can still hold the minimum
    for (unsigned rest = live; rest;) {
      const int t = __ffs(rest) - 1;
      rest &= rest - 1;
      const int sb = w0 + t;
      const int be = min(nblk, (sb + 1) * AUV_PATH_SUPER);
      unsigned cand = 0u;  // bit = block offset inside the superblock, uniform in the group
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        const int b = sb * AUV_PATH_SUPER + k * G + sub;
        const int i = min(b, be - 1);
        const float4 ch = chord[i];
        const float2 ax = aux[i];
        cand |= group_ballot<G>(gm, lane, b < be && !AUV_PRUNED(pt_chord_d2_f(qx, qy, ch, ax.x), ax.y)) << (k * G);
      }
      while (cand) {
        const int b = sb * AUV_PATH_SUPER + __ffs(cand) - 1;
        cand &= cand - 1;
        const int se = min(nseg, (b + 1) * AUV_PATH_BLOCK);
        AUV_CHECK(status, b >= 0 && b < nblk && sb < nsb);
        // the block's sub-block capsules, one per lane (without sub-block tables every sub-block is refined)
        unsigned subs = (1u << kSubPerBlk) - 1u;  // bit = sub-block offset inside the block, uniform in the group
        if (pb.sub_chord != nullptr) {
          const int j = b * kSubPerBlk + min(sub, kSubPerBlk - 1);
          const float4 ch = subc[j];
          const float2 ax = subd[j];
          subs = group_ballot<G>(gm, lane, sub < kSubPerBlk && j * AUV_PATH_SUB < nseg &&
                                               !AUV_PRUNED(pt_chord_d2_f(qx, qy, ch, ax.x), ax.y));
        }
        // (screening segments in FP32 first was measured slower: far from the path many segments tie within the
        // FP32 error bound, and the divergent FP64 re-evaluation costs more than evaluating all of them)
        while (subs) {
          const int j = b * kSubPerBlk + __ffs(subs) - 1;
          subs &= subs - 1;
          const int je = j * AUV_PATH_SUB + AUV_PATH_SUB;
          const int k0 = j * AUV_PATH_SUB + sub * SPL;  // this lane's consecutive segments
          double2 v[SPL + 1];
#pragma unroll
          for (int u = 0; u <= SPL; ++u) v[u] = poly[min(k0 + u, se)];
#pragma unroll
          for (int u = 0; u < SPL; ++u) {
            if (k0 + u < min(se, je)) {
              double num, den;
              seg_d2_frac(px, py, v[u], v[u + 1], num, den);
              // a lane's segments come in increasing order over the whole search: strictly smaller only
              if (num * best_den < best_num * den) {
                best_num = num;
                best_den = den;
                best_seg = k0 + u;
              }
            }
          }
        }
      }
    }
  }
#undef AUV_TIGHTEN
#undef AUV_PRUNED
  double best_d2 = best_num / best_den;
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) {  // lexicographic (distance, segment) arg-min over the group
    const double od = __shfl_xor_sync(gm, best_d2, o);
    const int oi = __shfl_xor_sync(gm, best_seg, o);
    if (od < best_d2 || (od == best_d2 && oi < best_seg)) {
      best_d2 = od;
      best_seg = oi;
    }
  }
  // a bound that pruned every segment would leave best_seg = 0x7fffffff: flag it, and keep the debug build's read in bounds
  AUV_CHECK(status, best_seg >= 0 && best_seg < nseg);
#ifdef AUV_DEBUG_BOUNDS
  best_seg = min(max(best_seg, 0), nseg - 1);
#endif
  seg_out = best_seg;
  // segmentNearestMeasure of the winning segment
  const double2 A = poly[best_seg], B = poly[best_seg + 1];
  const double start = pb.poly_cum[h.v0 + best_seg];
  const double ex = B.x - A.x, ey = B.y - A.y;
  const double len2 = ex * ex + ey * ey;
  if (len2 == 0.0) return start;
  const double r = ((px - A.x) * ex + (py - A.y) * ey) / len2;
  if (r <= 0.0) return start;
  const double seglen = sqrt(len2);
  if (r <= 1.0) return start + r * seglen;
  return start + seglen;
}

// Vessel.navigate (vessel.py:461-541) for env e; writes nav[e][:] and max_progress[e], the
// navigation part of the observation (vessel.py:518-539, clipped: environment.py:276-280) and
// the LiDAR-independent part of the reward (rewarder.py:78-140,167-241).
// `s` is the projected arclength (project_group); every lane of the env's group computes the
// same scalars, `store` is true for the one lane that writes them.
__device__ AUV_NAVIGATE_INLINE void navigate_env(const AuvConfig& cfg, const AuvPathBank& pb, const AuvPathHdr& h,
                                             const AuvBatch& batch, int pid, int e, int scn, const double s, double px,
                                             double py, double psi, double vu, double vv, double vr,
                                             float* __restrict__ obs_row, const bool store) {
  const double L = h.length;
  const double s_la = fmin(L, s + cfg.look_ahead_distance);
  PchipOut at_s, at_la;
  pchip_eval2(pb, pid, L, s, s_la, at_s, at_la);
  const double p_x = at_s.px, p_y = at_s.py, d_x = at_s.dx, d_y = at_s.dy;
  const double l_x = at_la.px, l_y = at_la.py, ldx = at_la.dx, ldy = at_la.dy;
  const double chi = (double)atan2f((float)d_y, (float)d_x);  // diagnostic only (nav[NAV_CHI])
  // cross-track error = second row of Rz(-chi) applied to (path(s) - p); cos/sin(chi) are the
  // normalised derivative (no trig needed)
  const double dn = sqrt(d_x * d_x + d_y * d_y);
  const double idn = dn > 0.0 ? 1.0 / dn : 0.0;
  const double cc = dn > 0.0 ? d_x * idn : 1.0, sc = d_y * idn;
  const double y_e = -sc * (p_x - px) + cc * (p_y - py);
  // heading errors feed float32 observations and cos() in the reward: FP32 atan2 (~2e-7 rad)
  const double la_err = princip((double)atan2f((float)ldy, (float)ldx) - psi);
  const double head_err = princip((double)atan2f((float)(l_y - py), (float)(l_x - px)) - psi);
  const double progress = s / L;
  const double gx = h.end_x - px, gy = h.end_y - py;
  const double goal = sqrt(gx * gx + gy * gy);
  const bool reached = (goal <= cfg.min_goal_distance) || (progress >= cfg.min_path_progress);
  double sp, cp;
  sincos(psi, &sp, &cp);
  const double cos_he = (double)cosf((float)head_err);
  const double maxprog = fmax(progress, batch.max_progress[e]);  // vessel.py:507
  // ---- reward without the closeness term.  Colav (rewarder.py:216-239):
  //   r = 0.5 path + 0.5 closeness - living - 10|r| + slow, x2 if negative (k_lidar adds closeness);
  // PathFollow (rewarder.py:118-140): r = path - living - 10|r| + slow.
  const double cte = y_e * 0.01;  // y_e / 100 to within 1 ulp; feeds a float32 observation and exp()
  const double speed2 = vu * vu + vv * vv;
  const double speed = sqrt(speed2);
  double path_reward = (1.0 + cos_he * speed * 0.5) * (1.0 + (double)__expf((float)(-5.0 * fabs(cte)))) - 1.0;
  const double living = 0.5 * (2.0 * 0.05 + 1.0);
  double base;
  if (cfg.rewarder == AUV_REWARDER_COLAV) {
    if (progress < maxprog) path_reward = fmin(path_reward, 0.0);
    base = 0.5 * path_reward - living - 10.0 * fabs(vr) + (speed2 < 0.04 * 0.04 ? -2.0 : 0.0);
  } else {
    base = path_reward - living - 10.0 * fabs(vr) + (speed2 < 0.1 * 0.1 ? -2.0 : 0.0);
  }
  if (!store) return;
  batch.max_progress[e] = maxprog;
  // the 192 B record leaves as 12 x 16 B stores (indices: NAV_* above)
  double2* o = reinterpret_cast<double2*>(batch.nav + (long long)e * AUV_NAV_W);
  o[0] = make_double2(s, chi);                                // NAV_S, NAV_CHI
  o[1] = make_double2(y_e, s_la);                             // NAV_YE, NAV_SLA
  o[2] = make_double2(la_err, head_err);                      // NAV_LA_ERR, NAV_HEAD_ERR
  o[3] = make_double2(goal, progress);                        // NAV_GOAL, NAV_PROGRESS
  o[4] = make_double2(cp, sp);                                // NAV_COSPSI, NAV_SINPSI
  o[5] = make_double2(reached ? 1.0 : 0.0, y_e);              // NAV_REACHED, NAV_H_YE
  o[6] = make_double2(base, goal);                            // NAV_REWARD_BASE, NAV_H_GOAL
  o[7] = make_double2(progress, 0.0);                         // NAV_H_PROGRESS, unused
  o[8] = make_double2(px, py);                                // NAV_X, NAV_Y
  o[9] = make_double2(psi, batch.cum_reward[e]);              // NAV_PSI, NAV_CUM
  o[10] = make_double2(batch.cte_sum[e], (double)batch.t_step[e]);  // NAV_CTE, NAV_TSTEP
  o[11] = make_double2((double)scn, 0.0);                     // NAV_SCN, NAV_CNT (the culling stage overwrites it)
  if (obs_row != nullptr) {  // [u, v, r, look-ahead heading error, heading error, cross-track / 100]
    obs_row[0] = (float)fmin(fmax(vu, -1.0), 1.0);
    obs_row[1] = (float)fmin(fmax(vv, -1.0), 1.0);
    obs_row[2] = (float)fmin(fmax(vr, -1.0), 1.0);
    obs_row[3] = (float)fmin(fmax(la_err, -1.0), 1.0);
    obs_row[4] = (float)fmin(fmax(head_err, -1.0), 1.0);
    obs_row[5] = (float)fmin(fmax(cte, -1.0), 1.0);
  }
}

}  // namespace auv
