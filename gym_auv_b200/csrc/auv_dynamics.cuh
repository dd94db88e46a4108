// auv_dynamics.cuh -- 3-DOF vessel model + Fehlberg step (FP64, registers).
#pragma once
#include "auv_device.cuh"
#include "../../include/auv_b200.h"

namespace auv {

// ------------------------------------------------------------------------------------
// k_vessel_step     vessel.py:226-247,561-578; odesolver.py:2-47; constants.py:33-72
// ------------------------------------------------------------------------------------
struct S6 {
  double x, y, psi, u, v, r;
};

// nu_dot = M^-1 (tau - D nu - N(nu) nu) and eta_dot = Rz(psi) nu with cos/sin(psi) supplied.
// Inlined, as rot_cs below: out of line was measured at 0.104 -> 0.126 ms (the S6 structs go through the stack)
__device__ __forceinline__ S6 state_dot_cs(const S6& s, double cp, double sp, double tau_u, double tau_r) {
  // M = [[25.8,0,0],[0,33.8,1.0948],[0,1.0948,2.76]]   (constants.py:33-36)
  constexpr double m11 = 33.8, m12 = 23.8 * 0.046, m22 = 2.76;
  constexpr double det = m11 * m22 - m12 * m12;
  constexpr double i00 = 1.0 / 25.8, i11 = m22 / det, i12 = -m12 / det, i22 = m11 / det;
  S6 d;
  d.x = cp * s.u - sp * s.v;
  d.y = sp * s.u + cp * s.v;
  d.psi = s.r;
  // tau - D nu - N(nu) nu   (constants.py:39-43, 63-72)
  const double f1 = (tau_u - 2.0 * s.u) - 2.0 * s.u;
  const double f2 = (0.0 - (7.0 * s.v - 2.5425 * s.r)) - (7.0 * s.v + (23.8 * s.u + 0.1) * s.r);
  const double f3 = (tau_r - (-2.5425 * s.v + 1.422 * s.r)) - (0.1 * s.v + (23.8 * 0.046 * s.u + 0.5) * s.r);
  d.u = i00 * f1;
  d.v = i11 * f2 + i12 * f3;
  d.r = i12 * f2 + i22 * f3;
  return d;
}

// cos/sin(psi0 + d) from cos/sin(psi0) by the angle-addition formulas; sin d / cos d from their
// Taylor series (|d| <= 0.5: truncation < 1e-17).  The Fehlberg stages evaluate Rz at
// psi0 + h * (combination of yaw rates), a small offset from the step's initial heading, so one
// FP64 sincos per step replaces six (+ six fmod in princip); results agree with
// sincos(princip(psi0 + d)) to ~2e-16.  Larger offsets take the direct route.
__device__ __forceinline__ void rot_cs(double c0, double s0, double psi0, double d, double& c, double& s) {
  if (fabs(d) > 0.5) {
    sincos(princip(psi0 + d), &s, &c);
    return;
  }
  const double z = d * d;
  double sd = -1.0 / 1307674368000.0;            // -z^7/15!
  sd = fma(sd, z, 1.0 / 6227020800.0);           //  z^6/13!
  sd = fma(sd, z, -1.0 / 39916800.0);
  sd = fma(sd, z, 1.0 / 362880.0);
  sd = fma(sd, z, -1.0 / 5040.0);
  sd = fma(sd, z, 1.0 / 120.0);
  sd = fma(sd, z, -1.0 / 6.0);
  sd = fma(sd * z, d, d);
  double cd = 1.0 / 20922789888000.0;            //  z^8/16!
  cd = fma(cd, z, -1.0 / 87178291200.0);         // -z^7/14!
  cd = fma(cd, z, 1.0 / 479001600.0);
  cd = fma(cd, z, -1.0 / 3628800.0);
  cd = fma(cd, z, 1.0 / 40320.0);
  cd = fma(cd, z, -1.0 / 720.0);
  cd = fma(cd, z, 1.0 / 24.0);
  cd = fma(cd, z, -0.5);
  cd = fma(cd, z, 1.0);
  c = c0 * cd - s0 * sd;
  s = s0 * cd + c0 * sd;
}

#define S6_STAGE(out, y, EXPR, dpsi)   \
  out.x = y.x + (EXPR(x));             \
  out.y = y.y + (EXPR(y));             \
  dpsi = (EXPR(psi));                  \
  out.psi = y.psi + dpsi;              \
  out.u = y.u + (EXPR(u));             \
  out.v = y.v + (EXPR(v));             \
  out.r = y.r + (EXPR(r));

// one Fehlberg step for one env (vessel.py:226-247, odesolver.py:13-46): returns the 5th-order
// solution q.  The tableau fractions are folded into per-step coefficients (h * a/b) instead of
// the reference's h*k*a/b evaluation order: ~100 FP64 divisions fewer per step, results differ
// by a few ulp (tests/test_gpu_parity.py::test_vessel_step_matches_reference_goldens).
__device__ __forceinline__ S6 vessel_rk_step(const AuvConfig& cfg, const S6& y, float2 a) {
  if (isnan(a.x) || isnan(a.y)) a = make_float2(0.f, 0.f);  // environment.py:314-315
  const double tau_u = fmin(fmax((double)a.x, 0.0), 1.0) * cfg.thrust_max_auv;
  const double tau_r = fmin(fmax((double)a.y, -1.0), 1.0) * cfg.moment_max_auv;
  const double h = cfg.t_step_size;
  double c0, s0, c, s, dpsi;
  sincos(princip(y.psi), &s0, &c0);
  // The derivatives do not depend on x, y, so no stage needs the x/y parts of earlier k's: they
  // are folded into the result as soon as they exist (b-weights in the tableau's order), which
  // takes 2 x 5 doubles out of the live set of this register-bound kernel.
  S6 t, k1, k2, k3, k4, k5, k6, q;
  const double b1 = h * (16.0 / 135.0), b3 = h * (6656.0 / 12825.0), b4 = h * (28561.0 / 56430.0),
               b5 = h * (9.0 / 50.0), b6 = h * (2.0 / 55.0);
  k1 = state_dot_cs(y, c0, s0, tau_u, tau_r);
  double ax = b1 * k1.x, ay = b1 * k1.y;
  const double a21 = h * (1.0 / 4.0);
#define E2(f) a21 * k1.f
  S6_STAGE(t, y, E2, dpsi)
  rot_cs(c0, s0, y.psi, dpsi, c, s);
  k2 = state_dot_cs(t, c, s, tau_u, tau_r);
  const double a31 = h * (3.0 / 32.0), a32 = h * (9.0 / 32.0);
#define E3(f) a31 * k1.f + a32 * k2.f
  S6_STAGE(t, y, E3, dpsi)
  rot_cs(c0, s0, y.psi, dpsi, c, s);
  k3 = state_dot_cs(t, c, s, tau_u, tau_r);
  ax += b3 * k3.x;
  ay += b3 * k3.y;
  const double a41 = h * (1932.0 / 2197.0), a42 = h * (7200.0 / 2197.0), a43 = h * (7296.0 / 2197.0);
#define E4(f) a41 * k1.f - a42 * k2.f + a43 * k3.f
  S6_STAGE(t, y, E4, dpsi)
  rot_cs(c0, s0, y.psi, dpsi, c, s);
  k4 = state_dot_cs(t, c, s, tau_u, tau_r);
  ax += b4 * k4.x;
  ay += b4 * k4.y;
  const double a51 = h * (439.0 / 216.0), a52 = h * 8.0, a53 = h * (3680.0 / 513.0), a54 = h * (845.0 / 4104.0);
#define E5(f) a51 * k1.f - a52 * k2.f + a53 * k3.f - a54 * k4.f
  S6_STAGE(t, y, E5, dpsi)
  rot_cs(c0, s0, y.psi, dpsi, c, s);
  k5 = state_dot_cs(t, c, s, tau_u, tau_r);
  ax -= b5 * k5.x;
  ay -= b5 * k5.y;
  const double a61 = h * (8.0 / 27.0), a62 = h * 2.0, a63 = h * (3544.0 / 2565.0), a64 = h * (1859.0 / 4104.0),
               a65 = h * (11.0 / 40.0);
#define E6(f) -a61 * k1.f + a62 * k2.f - a63 * k3.f + a64 * k4.f - a65 * k5.f
  S6_STAGE(t, y, E6, dpsi)
  rot_cs(c0, s0, y.psi, dpsi, c, s);
  k6 = state_dot_cs(t, c, s, tau_u, tau_r);
  ax += b6 * k6.x;
  ay += b6 * k6.y;
#define EQ(f) b1 * k1.f + b3 * k3.f + b4 * k4.f - b5 * k5.f + b6 * k6.f
  q.x = y.x + ax;
  q.y = y.y + ay;
  q.psi = y.psi + (EQ(psi));
  q.u = y.u + (EQ(u));
  q.v = y.v + (EQ(v));
  q.r = y.r + (EQ(r));
  q.psi = princip(q.psi);
  return q;
}

__device__ __forceinline__ S6 load_state(const double* st, int n, int e) {
  S6 y;
  y.x = st[e];
  y.y = st[n + e];
  y.psi = st[2 * n + e];
  y.u = st[3 * n + e];
  y.v = st[4 * n + e];
  y.r = st[5 * n + e];
  return y;
}
__device__ __forceinline__ void store_state(double* st, int n, int e, const S6& q) {
  st[e] = q.x;
  st[n + e] = q.y;
  st[2 * n + e] = q.psi;
  st[3 * n + e] = q.u;
  st[4 * n + e] = q.v;
  st[5 * n + e] = q.r;
}

}  // namespace auv
