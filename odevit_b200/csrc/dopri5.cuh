// Dormand-Prince 5(4) with Shampine's dense output (torchdiffeq _impl/dopri5.py, rk_common.py, interp.py, misc.py): the
// tableau and the per-image step-control arithmetic shared by the multi-kernel adaptive solve (solve_adaptive.cu) and the
// adaptive mode of the on-chip-state kernel (solve_resident.cu).  Time, dt and the error norms are fp64; stage values
// fp32.
#pragma once
#include <cmath>

#include "host.h"

namespace odevit {

// a[m] = beta[m - 1], b = c_sol[:6]
inline const Tableau kDopri5 = {
    6,
    {{0},
     {(float)(1. / 5)},
     {(float)(3. / 40), (float)(9. / 40)},
     {(float)(44. / 45), (float)(-56. / 15), (float)(32. / 9)},
     {(float)(19372. / 6561), (float)(-25360. / 2187), (float)(64448. / 6561), (float)(-212. / 729)},
     {(float)(9017. / 3168), (float)(-355. / 33), (float)(46732. / 5247), (float)(49. / 176), (float)(-5103. / 18656)}},
    {(float)(35. / 384), 0.f, (float)(500. / 1113), (float)(125. / 192), (float)(-2187. / 6784), (float)(11. / 84)}};
// error weights c_sol - c_error over k1..k7, and the dense-output midpoint weights c_mid / 2
constexpr float kDopri5Err[7] = {(float)(35. / 384 - 1951. / 21600), 0.f, (float)(500. / 1113 - 22642. / 50085),
                                 (float)(125. / 192 - 451. / 720), (float)(-2187. / 6784 + 12231. / 42400),
                                 (float)(11. / 84 - 649. / 6300), (float)(-1. / 60)};
constexpr float kDopri5Mid[7] = {(float)(6025192743. / 30085553152. / 2), 0.f,
                                 (float)(51252292925. / 65400821598. / 2), (float)(-2691868925. / 45128329728. / 2),
                                 (float)(187940372067. / 1594534317056. / 2), (float)(-1776094331. / 19743644256. / 2),
                                 (float)(11237099. / 235043384. / 2)};

// Why an image stopped (the status of odevit_solve_adaptive_resident is this + 1)
constexpr int kErrMax = 0, kErrNonFinite = 1, kErrUnderflow = 2;

// misc._select_initial_step (order 4), from s0 = sum (y0 / sc)^2 and s1 = sum (f0 / sc)^2 over the image's nel elements:
// h0 (the probe is y0 + h0 f0) and d1
__device__ __forceinline__ void dp5_probe_step(double s0, double s1, double nel, double& h0, double& d1) {
  const double d0 = sqrt(s0 / nel);
  d1 = sqrt(s1 / nel);
  h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
}
// ... and the first dt from s2 = sum ((f1 - f0) / sc)^2 at the probe
__device__ __forceinline__ double dp5_first_step(double s2, double nel, double h0, double d1) {
  const double d2 = sqrt(s2 / nel) / h0;
  const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : pow(0.01 / fmax(d1, d2), 1.0 / 5.0);
  return fmin(100.0 * h0, h1);
}
// _optimal_step_size(dt, ratio, safety 0.9, ifactor 10, dfactor 0.2, order 5)
__device__ __forceinline__ double dp5_next_step(double dt, double ratio) {
  if (ratio == 0.0) return dt * 10.0;
  return dt * fmin(10.0, fmax(0.9 * pow(ratio, -1.0 / 5.0), ratio < 1.0 ? 1.0 : 0.2));
}
// interp._interp_fit of an accepted step: y0 + x cd + x^2 cc + x^3 cb + x^4 ca at x = (t - t0) / dt.  m = sum_l
// c_mid[l] k_l (k1 = f0, k7 = f1).
struct Dp5Quartic {
  float a0, ca, cb, cc, cd;
  Dp5Quartic() = default;
  __device__ __forceinline__ Dp5Quartic(float y0, float y1, float f0, float f1, float m, float dt) {
    const float ym = fmaf(dt, m, y0);
    a0 = y0;
    ca = 2.f * dt * (f1 - f0) - 8.f * (y1 + y0) + 16.f * ym;
    cb = dt * (5.f * f0 - 3.f * f1) + 18.f * y0 + 14.f * y1 - 32.f * ym;
    cc = dt * (f1 - 4.f * f0) - 11.f * y0 - 5.f * y1 + 16.f * ym;
    cd = dt * f0;
  }
  __device__ __forceinline__ float at(float x) const {
    const float x2 = x * x, x3 = x2 * x, x4 = x3 * x;
    return a0 + x * cd + x2 * cc + x3 * cb + x4 * ca;
  }
};

}  // namespace odevit
