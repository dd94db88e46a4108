// auv_pathbuild.cuh -- device-side construction of the path bank (SURVEY.md section 8 f-1):
// what gym_auv.objects.path.Path.__init__ (path.py:19-40) computes with SciPy, one CTA per path:
//   3 x { chord-length parameter of the current points -> PCHIP (Fritsch-Carlson slopes) ->
//         resample at linspace(0, arc[-1], 1000) }
//   -> PPoly knots / coefficients, the 0.1 m polyline with its chord-length prefix sums, the FP32
//      copy, and the capsule tables of the projection search (sub-blocks, blocks, superblocks) -- the layout of
//      AuvPathBank.
// The arithmetic follows SciPy's evaluation order (scipy.interpolate.PchipInterpolator:
// _find_derivatives / _edge_case, CubicHermiteSpline coefficients, _ppoly.evaluate_poly1's power
// sum) and NumPy's linspace / cumsum, every operation an explicit round-to-nearest intrinsic (no
// FMA contraction), so knots and coefficients agree with the host builder to the last bits.
// k_random_curve_waypoints draws RandomCurveThroughOrigin (path.py:96-120) with Philox streams.
#pragma once
#include "auv_device.cuh"
#include "auv_generate.cuh"
#include "../../include/auv_b200.h"

namespace auv {

#define PB_MUL(a, b) __dmul_rn((a), (b))
#define PB_ADD(a, b) __dadd_rn((a), (b))
#define PB_SUB(a, b) __dsub_rn((a), (b))
#define PB_DIV(a, b) __ddiv_rn((a), (b))
constexpr int PB_NK = 1000;  // knots (path.py:28)
constexpr int PB_THREADS = 256;

__device__ __forceinline__ double pb_sign(double v) { return v > 0.0 ? 1.0 : (v < 0.0 ? -1.0 : 0.0); }

// scipy PchipInterpolator._edge_case
__device__ __forceinline__ double pb_edge(double h0, double h1, double m0, double m1) {
  double d = PB_DIV(PB_SUB(PB_MUL(PB_ADD(PB_MUL(2.0, h0), h1), m0), PB_MUL(h0, m1)), PB_ADD(h0, h1));
  const bool mask = pb_sign(d) != pb_sign(m0);
  const bool mask2 = (pb_sign(m0) != pb_sign(m1)) && (fabs(d) > PB_MUL(3.0, fabs(m0)));
  if (mask) d = 0.0;
  else if (mask2) d = PB_MUL(3.0, m0);
  return d;
}

// PPoly value at x on interval j (scipy _ppoly.evaluate_poly1, dx = 0: power sum, not Horner)
__device__ __forceinline__ double pb_eval(const double* __restrict__ c, double s) {  // c = c0..c3 of the interval
  double res = PB_MUL(c[3], 1.0);
  double z = s;
  res = PB_ADD(res, PB_MUL(c[2], z));
  z = PB_MUL(z, s);
  res = PB_ADD(res, PB_MUL(c[1], z));
  z = PB_MUL(z, s);
  res = PB_ADD(res, PB_MUL(c[0], z));
  return res;
}

// interval of x in the knot vector kn[0..n): kn[j] <= x < kn[j+1], the last interval closed on the
// right, out-of-range clamped (scipy find_interval with extrapolate)
__device__ __forceinline__ int pb_interval(const double* __restrict__ kn, int n, double x) {
  if (!(x > kn[0])) return 0;
  if (x >= kn[n - 1]) return n - 2;
  int lo = 0, hi = n - 1;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (x < kn[mid]) hi = mid; else lo = mid;
  }
  return lo;
}

// numpy.linspace(0, stop, num)[i]
__device__ __forceinline__ double pb_linspace(double stop, int num, int i) {
  if (i == num - 1) return stop;
  const double step = PB_DIV(stop, (double)(num - 1));
  return PB_MUL((double)i, step);
}

// One CTA per path.  Dynamic shared memory: arc[1000], pts[2][1000], d[2][1000], coef[2][999][4].
struct PathBuildOut {
  AuvPathHdr* hdr;
  double* poly_xy;
  double* poly_cum;
  float* poly_f32;
  float* blk_chord;
  float* blk_dev;
  float* sb_chord;
  float* sb_dev;
  double* pp;
  int vcap;  // vertices per path slot (a multiple of 2 * AUV_PATH_BLOCK * AUV_PATH_SUPER)
  float* sub_chord;  // NULL: no sub-block tables
  float* sub_dev;
};
__host__ __device__ constexpr size_t pathbuild_smem_bytes() {
  return sizeof(double) * (PB_NK + 2 * PB_NK + 2 * PB_NK + 2 * (PB_NK - 1) * 4) + 64;
}

__device__ __forceinline__ void pb_capsules(const double2* __restrict__ poly, double ox, double oy, int nseg, int span,
                                            double extent1, float4* __restrict__ chord, float2* __restrict__ aux) {
  const int nn = (nseg + span - 1) / span;
  for (int b = threadIdx.x; b < nn; b += PB_THREADS) {
    const int first = b * span, last = min(first + span, nseg);
    const double rax = poly[first].x - ox, ray = poly[first].y - oy;
    const float4 ch = make_float4((float)rax, (float)ray, (float)((poly[last].x - ox) - rax), (float)((poly[last].y - oy) - ray));
    const double ax = (double)ch.x, ay = (double)ch.y, ex = (double)ch.z, ey = (double)ch.w;
    const double len2 = PB_ADD(PB_MUL(ex, ex), PB_MUL(ey, ey));
    const float inv = len2 > 0.0 ? (float)PB_DIV(1.0, len2) : 0.f;
    double dev = 0.0;
    for (int k = 0; k <= span; ++k) {
      const int v = min(first + k, last);
      const double wx = (poly[v].x - ox) - ax, wy = (poly[v].y - oy) - ay;
      double t = PB_MUL(PB_ADD(PB_MUL(wx, ex), PB_MUL(wy, ey)), (double)inv);
      t = fmin(fmax(t, 0.0), 1.0);
      const double rx = PB_SUB(wx, PB_MUL(t, ex)), ry = PB_SUB(wy, PB_MUL(t, ey));
      dev = fmax(dev, sqrt(PB_ADD(PB_MUL(rx, rx), PB_MUL(ry, ry))));
    }
    dev = PB_ADD(dev, PB_MUL(8.0 * 1.1920928955078125e-07, extent1));
    chord[b] = ch;
    aux[b] = make_float2(inv, nextafterf((float)dev, INFINITY));
  }
}

__global__ void __launch_bounds__(PB_THREADS) k_path_build(const double* __restrict__ waypoints, const int* __restrict__ n_wp,
                                                           const int* __restrict__ path_ids, int n_paths_listed,
                                                           PathBuildOut out, int* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char pb_smem[];
  double* arc = reinterpret_cast<double*>(pb_smem);   // [1000] knots of the current round
  double* pts = arc + PB_NK;                           // [2][1000] points of the current round
  double* der = pts + 2 * PB_NK;                       // [2][1000] PCHIP derivatives
  double* coef = der + 2 * PB_NK;                      // [2][999][4]
  __shared__ double s_extent;
  const int li = blockIdx.x;
  if (li >= n_paths_listed) return;
  const int p = path_ids ? path_ids[li] : li;
  const int tid = threadIdx.x;
  int n = n_wp[li];
  for (int k = tid; k < n; k += PB_THREADS) {
    pts[k] = waypoints[(long long)li * 16 + k];
    pts[PB_NK + k] = waypoints[(long long)li * 16 + 8 + k];
  }
  __syncthreads();
  for (int round = 0; round < 3; ++round) {
    // ---- chord-length parameter (np.cumsum: sequential)
    if (tid == 0) {
      double a = 0.0;
      arc[0] = 0.0;
      for (int k = 1; k < n; ++k) {
        const double dx = PB_SUB(pts[k], pts[k - 1]), dy = PB_SUB(pts[PB_NK + k], pts[PB_NK + k - 1]);
        a = PB_ADD(a, sqrt(PB_ADD(PB_MUL(dx, dx), PB_MUL(dy, dy))));
        arc[k] = a;
      }
    }
    __syncthreads();
    // ---- PCHIP derivatives (scipy PchipInterpolator._find_derivatives), per axis
    for (int idx = tid; idx < 2 * n; idx += PB_THREADS) {
      const int ax = idx / n, k = idx - ax * n;
      const double* y = pts + ax * PB_NK;
      double d;
      if (n == 2) {
        d = PB_DIV(PB_SUB(y[1], y[0]), PB_SUB(arc[1], arc[0]));
      } else if (k == 0) {
        const double h0 = PB_SUB(arc[1], arc[0]), h1 = PB_SUB(arc[2], arc[1]);
        d = pb_edge(h0, h1, PB_DIV(PB_SUB(y[1], y[0]), h0), PB_DIV(PB_SUB(y[2], y[1]), h1));
      } else if (k == n - 1) {
        const double h0 = PB_SUB(arc[n - 1], arc[n - 2]), h1 = PB_SUB(arc[n - 2], arc[n - 3]);
        d = pb_edge(h0, h1, PB_DIV(PB_SUB(y[n - 1], y[n - 2]), h0), PB_DIV(PB_SUB(y[n - 2], y[n - 3]), h1));
      } else {
        const double hm = PB_SUB(arc[k], arc[k - 1]), hk = PB_SUB(arc[k + 1], arc[k]);
        const double mm = PB_DIV(PB_SUB(y[k], y[k - 1]), hm), mk = PB_DIV(PB_SUB(y[k + 1], y[k]), hk);
        if (pb_sign(mk) != pb_sign(mm) || mk == 0.0 || mm == 0.0) {
          d = 0.0;
        } else {
          const double w1 = PB_ADD(PB_MUL(2.0, hk), hm), w2 = PB_ADD(hk, PB_MUL(2.0, hm));
          const double wh = PB_DIV(PB_ADD(PB_DIV(w1, mm), PB_DIV(w2, mk)), PB_ADD(w1, w2));
          d = PB_DIV(1.0, wh);
        }
      }
      der[ax * PB_NK + k] = d;
    }
    __syncthreads();
    // ---- cubic Hermite -> PPoly coefficients (scipy CubicHermiteSpline.__init__)
    for (int idx = tid; idx < 2 * (n - 1); idx += PB_THREADS) {
      const int ax = idx / (n - 1), k = idx - ax * (n - 1);
      const double* y = pts + ax * PB_NK;
      const double* dd = der + ax * PB_NK;
      const double dxr = PB_SUB(arc[k + 1], arc[k]);
      const double slope = PB_DIV(PB_SUB(y[k + 1], y[k]), dxr);
      const double t = PB_DIV(PB_SUB(PB_ADD(dd[k], dd[k + 1]), PB_MUL(2.0, slope)), dxr);
      double* c = coef + ((size_t)ax * (PB_NK - 1) + k) * 4;
      c[0] = PB_DIV(t, dxr);
      c[1] = PB_SUB(PB_DIV(PB_SUB(slope, dd[k]), dxr), t);
      c[2] = dd[k];
      c[3] = y[k];
    }
    __syncthreads();
    if (round == 2) break;
    // ---- resample at linspace(arc[0], arc[-1], 1000) into registers, then replace the points
    double nx[(PB_NK + PB_THREADS - 1) / PB_THREADS], ny[(PB_NK + PB_THREADS - 1) / PB_THREADS];
    const double stop = arc[n - 1];
#pragma unroll
    for (int r = 0; r < (PB_NK + PB_THREADS - 1) / PB_THREADS; ++r) {
      const int i = tid + r * PB_THREADS;
      if (i < PB_NK) {
        const double x = pb_linspace(stop, PB_NK, i);
        const int j = pb_interval(arc, n, x);
        const double s = PB_SUB(x, arc[j]);
        nx[r] = pb_eval(coef + (size_t)j * 4, s);
        ny[r] = pb_eval(coef + ((size_t)(PB_NK - 1) + j) * 4, s);
      }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < (PB_NK + PB_THREADS - 1) / PB_THREADS; ++r) {
      const int i = tid + r * PB_THREADS;
      if (i < PB_NK) {
        pts[i] = nx[r];
        pts[PB_NK + i] = ny[r];
      }
    }
    n = PB_NK;
    __syncthreads();
  }
  // ---- the final spline: knots = arc (n = 1000 unless the path never left round 0), coefficients
  //      (callers always pass >= 2 waypoints; after round 0 n is 1000)
  const double L = arc[n - 1];
  const int n_poly = (int)PB_MUL(10.0, L);  // int(10 * length), path.py:38
  if (tid == 0 && (n_poly > out.vcap || n_poly < 2) && status != nullptr) atomicOr(status, AUV_STATUS_PATH_TOO_LONG);
  double* pp = out.pp + (size_t)p * (PB_NK - 1) * AUV_PP_W;
  for (int k = tid; k < PB_NK - 1; k += PB_THREADS) {
    double* r = pp + (size_t)k * AUV_PP_W;
    r[0] = arc[k];
    r[1] = arc[k + 1];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      r[2 + q] = coef[(size_t)k * 4 + q];
      r[6 + q] = coef[((size_t)(PB_NK - 1) + k) * 4 + q];
    }
    r[10] = r[11] = 0.0;
  }
  __syncthreads();
  if (n_poly > out.vcap || n_poly < 2) return;
  // ---- 0.1 m polyline: spline(linspace(0, L, n_poly))   path.py:38-40
  const size_t v0 = (size_t)p * out.vcap;
  double2* poly = reinterpret_cast<double2*>(out.poly_xy) + v0;
  for (int i = tid; i < n_poly; i += PB_THREADS) {
    const double x = pb_linspace(L, n_poly, i);
    const int j = pb_interval(arc, PB_NK, x);
    const double s = PB_SUB(x, arc[j]);
    poly[i] = make_double2(pb_eval(coef + (size_t)j * 4, s), pb_eval(coef + ((size_t)(PB_NK - 1) + j) * 4, s));
  }
  __syncthreads();
  const double ox = poly[0].x, oy = poly[0].y;
  // ---- chord-length prefix sums (np.cumsum: sequential) and the extent, FP32 copy in parallel
  if (tid == 0) {
    double a = 0.0;
    out.poly_cum[v0] = 0.0;
    for (int k = 1; k < n_poly; ++k) {
      const double dx = PB_SUB(poly[k].x, poly[k - 1].x), dy = PB_SUB(poly[k].y, poly[k - 1].y);
      a = PB_ADD(a, sqrt(PB_ADD(PB_MUL(dx, dx), PB_MUL(dy, dy))));
      out.poly_cum[v0 + k] = a;
    }
  }
  double ext_sum = 0.0, ext_max = 0.0;
  float2* pf = reinterpret_cast<float2*>(out.poly_f32) + v0;
  for (int i = tid; i < n_poly; i += PB_THREADS) {
    const double rx = poly[i].x - ox, ry = poly[i].y - oy;
    pf[i] = make_float2((float)rx, (float)ry);
    ext_sum = fmax(ext_sum, fabs(rx) + fabs(ry));
    ext_max = fmax(ext_max, fmax(fabs(rx), fabs(ry)));
  }
  // block reduction of the two maxima through the (now free) derivative scratch
  der[tid] = ext_sum;
  der[PB_THREADS + tid] = ext_max;
  __syncthreads();
  if (tid == 0) {
    double a = 0.0, b = 0.0;
    for (int k = 0; k < PB_THREADS; ++k) {
      a = fmax(a, der[k]);
      b = fmax(b, der[PB_THREADS + k]);
    }
    s_extent = a;
    der[0] = b;
  }
  __syncthreads();
  const double extent1 = der[0] + 1.0;  // float(np.abs(rel).max()) + 1.0
  const int nseg = n_poly - 1;
  const int bcap = out.vcap / AUV_PATH_BLOCK, scap = bcap / AUV_PATH_SUPER;
  pb_capsules(poly, ox, oy, nseg, AUV_PATH_BLOCK, extent1, reinterpret_cast<float4*>(out.blk_chord) + (size_t)p * bcap,
              reinterpret_cast<float2*>(out.blk_dev) + (size_t)p * bcap);
  pb_capsules(poly, ox, oy, nseg, AUV_PATH_BLOCK * AUV_PATH_SUPER, extent1,
              reinterpret_cast<float4*>(out.sb_chord) + (size_t)p * scap, reinterpret_cast<float2*>(out.sb_dev) + (size_t)p * scap);
  if (out.sub_chord != nullptr) {
    const int ucap = out.vcap / AUV_PATH_SUB;
    pb_capsules(poly, ox, oy, nseg, AUV_PATH_SUB, extent1, reinterpret_cast<float4*>(out.sub_chord) + (size_t)p * ucap,
                reinterpret_cast<float2*>(out.sub_dev) + (size_t)p * ucap);
  }
  if (tid == 0) {
    AuvPathHdr h;
    h.v0 = (int)v0;
    h.nseg = nseg;
    h.b0 = p * bcap;
    h.s0 = p * scap;
    h.ox = ox;
    h.oy = oy;
    h.length = L;
    const int j = PB_NK - 2;  // spline(L): last interval
    const double s = PB_SUB(L, arc[j]);
    h.end_x = pb_eval(coef + (size_t)j * 4, s);
    h.end_y = pb_eval(coef + ((size_t)(PB_NK - 1) + j) * 4, s);
    h.extent = s_extent;
    out.hdr[p] = h;
  }
}

// RandomCurveThroughOrigin waypoints (path.py:96-120) + the waypoint count of
// MovingObstacles._generate (movingobstacles.py:28-31: nwp = floor(4 rand + 2)), thread per path
__global__ void __launch_bounds__(128) k_random_curve_waypoints(unsigned long long seed, unsigned epoch, double length,
                                                                const int* __restrict__ path_ids, int n,
                                                                double* __restrict__ waypoints, int* __restrict__ n_wp) {
  const int li = blockIdx.x * blockDim.x + threadIdx.x;
  if (li >= n) return;
  const int p = path_ids ? path_ids[li] : li;
  GenRng r(seed, (unsigned)p, 0xFFFDu, epoch);
  const int nwaypoints = (int)floor(4.0 * r.u01() + 2.0);
  const double a0 = 2.0 * AUV_PI * (r.u01() - 0.5);
  double sa, ca;
  sincos(a0, &sa, &ca);
  const double sx = 0.5 * length * ca, sy = 0.5 * length * sa;
  const int half = nwaypoints / 2;
  // after round k the list is [start, p1_0.., origin, ..p2_0, end]: the k-th inserted pair sits k+1 from the ends
  double* wx = waypoints + (long long)li * 16;
  double* wy = wx + 8;
  const int total = 3 + 2 * half;
  wx[0] = sx;
  wy[0] = sy;
  wx[total - 1] = -sx;
  wy[total - 1] = -sy;
  for (int k = 0; k < half; ++k) {
    const double f = (double)(half - k) / (double)(half + 1), sc = length / (double)(half + 1);
    const double j1 = sc * (r.u01() - 0.5), j2 = sc * (r.u01() - 0.5);  // ONE scalar jitter for both coordinates
    wx[1 + k] = f * sx + j1;
    wy[1 + k] = f * sy + j1;
    wx[total - 2 - k] = f * -sx + j2;
    wy[total - 2 - k] = f * -sy + j2;
  }
  wx[1 + half] = 0.0;
  wy[1 + half] = 0.0;
  for (int k = total; k < 8; ++k) wx[k] = wy[k] = 0.0;
  n_wp[li] = total;
}

}  // namespace auv
