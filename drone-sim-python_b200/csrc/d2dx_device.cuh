// Device-side fp64 building blocks shared by every d2dx kernel (sm_100a).
// Each function names the reference code it evaluates (paths relative to the reference's src/).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/d2dx.h"
#include "d2dx_math.cuh"

namespace d2dx {

// elementary functions used on the hot path: the straight-line versions of d2dx_math.cuh, or (-DD2DX_USE_LIBM)
// CUDA's libdevice for A/B comparison
#ifdef D2DX_USE_LIBM
__device__ __forceinline__ void sincos_b(double x, double& s, double& c) { ::sincos(x, &s, &c); }   // bounded argument
__device__ __forceinline__ void sincos_any(double x, double& s, double& c) { ::sincos(x, &s, &c); }
__device__ __forceinline__ double atan2_f(double y, double x) { return ::atan2(y, x); }
__device__ __forceinline__ double atan_f(double v) { return ::atan(v); }
__host__ __device__ __forceinline__ double sqrt_f(double v) { return ::sqrt(v); }
__host__ __device__ __forceinline__ double rsqrt_f(double v) { return 1.0 / ::sqrt(v); }
__host__ __device__ __forceinline__ double rcp_f(double v) { return 1.0 / v; }
__host__ __device__ __forceinline__ double div_f(double a, double b) { return a / b; }
#else
__device__ __forceinline__ void sincos_b(double x, double& s, double& c) { fm::sincos(x, s, c); }
// libdevice's Payne-Hanek path for huge phases, out of line and by value: its scratch array stays in ITS frame, the caller
// keeps no address-taken locals (a by-reference call put a stack frame and STL / LDL pairs into every rollout kernel)
struct SinCos { double s, c; };
static __device__ __noinline__ SinCos sincos_slow(double x) { SinCos r; ::sincos(x, &r.s, &r.c); return r; }
__device__ __forceinline__ void sincos_any(double x, double& s, double& c) {
  // the straight-line path runs unconditionally (its block joins the caller's: the scheduler may interleave it with independent
  // work); |x| >= 1e5 -- decided on the high word, 0x40F86A00 = hi(1e5) -- is redone out of line afterwards
  fm::sincos(x, s, c);
  if ((__double2hiint(x) & 0x7fffffff) >= 0x40F86A00) { const SinCos r = sincos_slow(x); s = r.s; c = r.c; }
}
__device__ __forceinline__ double atan2_f(double y, double x) { return fm::atan2(y, x); }
__device__ __forceinline__ double atan_f(double v) { return fm::atan(v); }
// host instances (plain IEEE operations) exist so that the Riccati reductions below can be compiled for the CPU and checked
// against scipy.linalg.solve_continuous_are without a GPU (csrc/host_check.cu, tests/test_care_math.py)
#ifdef __CUDA_ARCH__
__host__ __device__ __forceinline__ double sqrt_f(double v) { return fm::sqrt(v); }
__host__ __device__ __forceinline__ double rsqrt_f(double v) { return fm::rsqrt(v); }
__host__ __device__ __forceinline__ double rcp_f(double v) { return fm::rcp(v); }
__host__ __device__ __forceinline__ double div_f(double a, double b) { return fm::div(a, b); }
#else
__host__ __device__ __forceinline__ double sqrt_f(double v) { return ::sqrt(v); }
__host__ __device__ __forceinline__ double rsqrt_f(double v) { return 1.0 / ::sqrt(v); }
__host__ __device__ __forceinline__ double rcp_f(double v) { return 1.0 / v; }
__host__ __device__ __forceinline__ double div_f(double a, double b) { return a / b; }
#endif
#endif

constexpr double kPi = 3.141592653589793;        // np.pi
constexpr double kTwoPi = 6.283185307179586;     // 2*np.pi
constexpr double kG = 9.81;                      // d2d/dynamic.py:9, d2d/guidance.py:39

// norm_mpi_pi, d2d/utils.py:7: (v + pi) % (2 pi) - pi with NumPy's floored float modulo
// (npy_remainder: fmod, then += b when the signs differ).  The three branches are bit-identical to
// fmod for |a| < 4 pi (a - 2pi is exact there by Sterbenz) and skip CUDA's iterative fmod.
static __device__ __noinline__ double wrap_2pi_slow(double a) {
  double m;
  if (a >= 0.0 && a < kTwoPi) m = a;
  else if (a >= kTwoPi && a < 2.0 * kTwoPi) m = a - kTwoPi;
  else if (a < 0.0 && a > -kTwoPi) m = a + kTwoPi;
  else {
    m = fmod(a, kTwoPi);
    if (m != 0.0) { if (m < 0.0) m += kTwoPi; } else m = 0.0;
  }
  return m;
}
// The three cases a feedback error or an integrated heading produces are decided on the HIGH WORD of a = v + pi by the integer
// pipe (the rollout kernels are bound by the fp64 pipe) and cost one DADD with a selected addend:
//   |a| < 2 pi for certain (|hi| < hi(2 pi) = 0x401921FB):  a >= 0 -> a;   a < 0 -> a + 2 pi (npy_remainder's sign fix)
//   2 pi < a < 4 pi for certain (0x401921FB < hi < 0x402921FB):  a - 2 pi  (exact by Sterbenz = fmod)
// everything else -- hi(a) equal to a boundary word, a = -0.0 (remainder +0.0), larger magnitudes, NaN -- is not `fast`.
__device__ __forceinline__ double wrap_2pi_fast(double a, bool& fast) {
  const int h = __double2hiint(a);
  const unsigned am = h & 0x7fffffff;
  const bool lap1 = static_cast<unsigned>(h - 0x401921FC) < 0x000FFFFFu;          // h in [0x401921FC, 0x402921FB)
  fast = (am < 0x401921FBu && !(h < 0 && am == 0)) || lap1;
  return a + (lap1 ? -kTwoPi : (h < 0 ? kTwoPi : 0.0));
}
__device__ __forceinline__ double wrap_pi(double v) {
  const double a = v + kPi;
  bool fast;
  const double m = wrap_2pi_fast(a, fast);
  return (fast ? m : wrap_2pi_slow(a)) - kPi;
}
// for callers with their own exact fallback: ok &= fast, the value is only meaningful when ok stays true
__device__ __forceinline__ double wrap_pi_or_flag(double v, bool& ok) {
  bool fast;
  const double m = wrap_2pi_fast(v + kPi, fast);
  ok = ok && fast;
  return m - kPi;
}

// np.clip with plain compare-and-select (fmin/fmax expand to ~8 instructions each on sm_100a because of their
// NaN-quieting semantics; a NaN input still comes out as NaN here, like np.clip)
__device__ __forceinline__ double clip(double v, double lo, double hi) {
  const double t = v < lo ? lo : v;
  return t > hi ? hi : t;
}
// clip(v, -s, s) for s >= 0: one compare on |v| and the sign copied back (NaN passes through, like np.clip).
// (Deciding these saturations on the integer pipe -- high-word keys with an out-of-line exact path, or full 64-bit integer
//  compares -- was measured in round 2: each fp64 compare saved costs more ALU issue slots than it frees on the fp64 pipe;
//  the rollout kernel ran 1.5 - 7 % slower.  profiles/README.md.)
__device__ __forceinline__ double clip_sym(double v, double s) {
  const double m = fabs(v) > s ? s : fabs(v);
  return copysign(m, v);
}

// flat output and its three time derivatives, Trajectory.get -> (4,2), d2d/trajectory.py:88-122
struct FlatOut { double y0x, y0y, y1x, y1y, y2x, y2y, y3x, y3y; };

// PolynomialOne.get, d2d/trajectory.py:74-82: Horner over all 8 slots of derivative row d, with the
// separate multiply and add of `v *= t; v += c`; rows d >= 1 are arr(d, pow+d) * coefs[0][pow+d]
// (:70-72), an exact small integer times the stored coefficient, so they are rebuilt on the fly.
template <int D, typename LD>
__device__ __forceinline__ double poly_row(LD c0, double t) {
  double v = 0.0;   // coefs[D][7] .. coefs[D][8-D] are structural zeros for D >= 1
  bool first = true;
#pragma unroll
  for (int j = 7 - D; j >= 0; --j) {
    const int n = j + D;
    const double f = (D == 0) ? 1.0 : (D == 1) ? double(n) : (D == 2) ? double(n * (n - 1)) : double(n * (n - 1) * (n - 2));
    const double c = (D == 0) ? c0(n) : __dmul_rn(f, c0(n));
    if (first) { v = c; first = false; }
    else v = __dadd_rn(__dmul_rn(v, t), c);
  }
  return v;
}

// One trajectory segment evaluated at time t.  `P(k)` returns parameter slot k (include/d2dx.h).
template <bool WANT3, typename LD>
__device__ __forceinline__ void segment_eval(int type, LD P, double t, FlatOut& Y, const d2dx_traj_table* tt = nullptr) {
  Y.y2x = Y.y2y = Y.y3x = Y.y3y = 0.0;
  switch (type) {
    case D2DX_SEG_TABLE: {           // TrajTabulated.get, d2d/trajectory_factory.py:162-171
      const int first = (int)P(1), n = (int)P(2);
      const double* tm = tt->tab_time + first;
      int lo = 0, hi = n;            // np.argmin(t > sol_time): first row with sol_time >= t, 0 when there is none
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (t > tm[mid]) lo = mid + 1; else hi = mid; }
      const int idx = first + (lo < n ? lo : 0);
      Y.y0x = tt->tab_x[idx]; Y.y0y = tt->tab_y[idx];
      Y.y1x = tt->tab_vx[idx]; Y.y1y = tt->tab_vy[idx];
    } break;
    case D2DX_SEG_LINE: {            // TrajectoryLine.get, d2d/trajectory.py:136-141
      const double dt = t - P(0);
      Y.y1x = P(3); Y.y1y = P(4);
      Y.y0x = __dadd_rn(P(1), __dmul_rn(Y.y1x, dt));
      Y.y0y = __dadd_rn(P(2), __dmul_rn(Y.y1y, dt));
    } break;
    case D2DX_SEG_CIRCLE: {          // TrajectoryCircle.get, d2d/trajectory.py:153-160
      const double r = P(3), om = P(4);
      const double alpha = __dadd_rn(__dmul_rn(t - P(0), om), P(5));
      double sa, ca;
      sincos_any(alpha, sa, ca);
      const double w1 = __dmul_rn(om, r), w2 = __dmul_rn(__dmul_rn(om, om), r);
      Y.y0x = __dadd_rn(P(1), __dmul_rn(r, ca)); Y.y0y = __dadd_rn(P(2), __dmul_rn(r, sa));
      Y.y1x = -w1 * sa; Y.y1y = w1 * ca;
      Y.y2x = -w2 * ca; Y.y2y = -w2 * sa;
      if (WANT3) { const double w3 = __dmul_rn(om * om * om, r); Y.y3x = w3 * sa; Y.y3y = -w3 * ca; }
    } break;
    case D2DX_SEG_SLALOM: {          // TrajSlalom.get, d2d/trajectory_factory.py:133-145 (a=10, om=1)
      const double dt = t - P(0);
      Y.y1x = P(3); Y.y1y = P(4);
      Y.y0x = __dadd_rn(P(1), __dmul_rn(Y.y1x, dt));
      Y.y0y = __dadd_rn(P(2), __dmul_rn(Y.y1y, dt));
      const double alpha = __dadd_rn(dt, P(5));
      double s, c;
      sincos_any(alpha, s, c);
      Y.y0y = __dadd_rn(Y.y0y, 10.0 * s);
      Y.y1y = __dadd_rn(Y.y1y, 10.0 * c);
      Y.y2y = -10.0 * s;
      if (WANT3) Y.y3y = -10.0 * c;
    } break;
    case D2DX_SEG_POLY: {            // MinSnapPoly.get, d2d/trajectory.py:185-187
      const double dt = t - P(0);
      auto cx = [&](int k) { return P(1 + k); };
      auto cy = [&](int k) { return P(9 + k); };
      Y.y0x = poly_row<0>(cx, dt); Y.y0y = poly_row<0>(cy, dt);
      Y.y1x = poly_row<1>(cx, dt); Y.y1y = poly_row<1>(cy, dt);
      Y.y2x = poly_row<2>(cx, dt); Y.y2y = poly_row<2>(cy, dt);
      if (WANT3) { Y.y3x = poly_row<3>(cx, dt); Y.y3y = poly_row<3>(cy, dt); }
    } break;
    default: {                       // D2DX_SEG_SI_LINE / D2DX_SEG_SI_CIRCLE: SpaceIndexedTraj.get, d2d/trajectory.py:231-241
      double l0, l1, l2, l3 = 0.0;   // lambda(t) and its derivatives: polynomial (PolynomialOne / AffineOne / CstOne) or SinOne (:26-38)
      if (P(16) == 0.0) {
        auto cl = [&](int k) { return P(5 + k); };
        const double td = t - P(14);  // time origin of the polynomial piece (0 for PolynomialOne / AffineOne; the knot of a FooOne piece)
        l0 = poly_row<0>(cl, td); l1 = poly_row<1>(cl, td); l2 = poly_row<2>(cl, td);
        if (WANT3) l3 = poly_row<3>(cl, td);
      } else {
        const double a = P(6), om = P(7);
        double sa, ca;
        sincos_any(__dmul_rn(om, t - P(8)), sa, ca);
        const double asa = __dmul_rn(a, sa), aca = __dmul_rn(a, ca);
        l0 = __dadd_rn(P(5), asa); l1 = __dmul_rn(om, aca); l2 = -(om * om) * asa;
        if (WANT3) l3 = -(om * om * om) * aca;
      }
      l0 = clip(l0, 0.0, 1.0);       // :233 "protect ourself against unruly dynamics"
      if (type == D2DX_SEG_SI_LINE) {
        const double gx = P(3), gy = P(4);      // dg/dlambda of the line geometry; higher ones vanish
        Y.y0x = __dadd_rn(P(1), __dmul_rn(gx, l0)); Y.y0y = __dadd_rn(P(2), __dmul_rn(gy, l0));
        Y.y1x = l1 * gx; Y.y1y = l1 * gy;
        Y.y2x = l2 * gx; Y.y2y = l2 * gy;
        if (WANT3) { Y.y3x = l3 * gx; Y.y3y = l3 * gy; }
      } else {                        // circle geometry g(lambda) = TrajectoryCircle.get(lambda), chain rule of :235-238
        const double r = P(3), om = P(4);
        double sa, ca;
        sincos_any(__dadd_rn(__dmul_rn(l0 - P(0), om), P(13)), sa, ca);
        const double w1 = __dmul_rn(om, r), w2 = __dmul_rn(__dmul_rn(om, om), r), w3 = __dmul_rn(om * om * om, r);
        const double g1x = -w1 * sa, g1y = w1 * ca, g2x = -w2 * ca, g2y = -w2 * sa, g3x = w3 * sa, g3y = -w3 * ca;
        Y.y0x = __dadd_rn(P(1), __dmul_rn(r, ca)); Y.y0y = __dadd_rn(P(2), __dmul_rn(r, sa));
        Y.y1x = l1 * g1x; Y.y1y = l1 * g1y;
        const double l1s = l1 * l1;
        Y.y2x = l2 * g1x + l1s * g2x; Y.y2y = l2 * g1y + l1s * g2y;
        if (WANT3) {
          const double m = 3.0 * l1 * l2, l1c = l1s * l1;
          Y.y3x = l3 * g1x + m * g2x + l1c * g3x; Y.y3y = l3 * g1y + m * g2y + l1c * g3y;
        }
      }
    } break;
  }
}

// CompositeTraj.get, d2d/trajectory.py:202-208: which segment is active and at which local time.
// Plain trajectories (traj_dur <= 0) evaluate their only segment at t.
__device__ __forceinline__ int composite_locate(const d2dx_traj_table& tt, int b, double t, double& t_eval) {
  const double dur = tt.traj_dur[b];
  const int first = tt.first_seg[b];
  if (!(dur > 0.0)) { t_eval = t; return first; }
  const double lapse = fmod(t - tt.traj_t0[b], dur);
  const int n = tt.n_segs[b];
  int k = 0;                                   // np.argmax of an all-False mask is 0
  for (int j = 0; j < n; ++j) if (tt.seg_end[first + j] > lapse) { k = j; break; }
  t_eval = lapse;
  return first + k;
}

// Aircraft.cont_dyn, d2d/dynamic.py:14-23
struct AcPar { double wx, wy, n_inv_tau_phi, n_inv_tau_v; };   // -1/tau as the reference forms it

__device__ __forceinline__ void cont_dyn(const AcPar& a, double psi, double phi, double v, double phi_c,
                                         double v_c, double& dx, double& dy, double& dpsi, double& dphi, double& dv) {
  double s, c, sp, cp;
  sincos_b(psi, s, c);
  sincos_b(phi, sp, cp);
  dx = v * c + a.wx;
  dy = v * s + a.wy;
  dpsi = kG * sp * rcp_f(v * cp);            // g / v * tan(phi)
  dphi = a.n_inv_tau_phi * (phi - phi_c);
  dv = a.n_inv_tau_v * (v - v_c);
}

// Reference formulation of one control step (every stage with full-range sin / cos): used for the single-call
// entry points' odd inputs and as the fallback of rk4_step when a stage leaves the fast path's validity range.
// Arguments and result travel by value (registers): nothing of the caller's state has its address taken.
struct State5 { double x, y, psi, phi, v; };
static __device__ __noinline__ State5 rk4_step_generic(const AcPar a, const State5 X, double phi_c, double v_c, double dt, int nsub) {
  const double h = dt / nsub, hh = 0.5 * h, h6 = h / 6.0;
  double x = X.x, y = X.y, psi = X.psi, phi = X.phi, v = X.v;
  for (int s = 0; s < nsub; ++s) {
    double k1[5], k2[5], k3[5], k4[5];
    cont_dyn(a, psi, phi, v, phi_c, v_c, k1[0], k1[1], k1[2], k1[3], k1[4]);
    cont_dyn(a, psi + hh * k1[2], phi + hh * k1[3], v + hh * k1[4], phi_c, v_c, k2[0], k2[1], k2[2], k2[3], k2[4]);
    cont_dyn(a, psi + hh * k2[2], phi + hh * k2[3], v + hh * k2[4], phi_c, v_c, k3[0], k3[1], k3[2], k3[3], k3[4]);
    cont_dyn(a, psi + h * k3[2], phi + h * k3[3], v + h * k3[4], phi_c, v_c, k4[0], k4[1], k4[2], k4[3], k4[4]);
    x += h6 * (k1[0] + 2.0 * k2[0] + 2.0 * k3[0] + k4[0]);
    y += h6 * (k1[1] + 2.0 * k2[1] + 2.0 * k3[1] + k4[1]);
    psi += h6 * (k1[2] + 2.0 * k2[2] + 2.0 * k3[2] + k4[2]);
    phi += h6 * (k1[3] + 2.0 * k2[3] + 2.0 * k3[3] + k4[3]);
    v += h6 * (k1[4] + 2.0 * k2[4] + 2.0 * k3[4] + k4[4]);
  }
  State5 r;
  r.x = x; r.y = y; r.psi = wrap_pi(psi); r.phi = phi; r.v = v;
  return r;
}
__device__ __forceinline__ void rk4_generic_inplace(const AcPar& a, double* X, double phi_c, double v_c, double dt, int nsub) {
  State5 in;
  in.x = X[0]; in.y = X[1]; in.psi = X[2]; in.phi = X[3]; in.v = X[4];
  const State5 r = rk4_step_generic(a, in, phi_c, v_c, dt, nsub);
  X[0] = r.x; X[1] = r.y; X[2] = r.psi; X[3] = r.phi; X[4] = r.v;
}

// The bank and air-speed loops are first-order lags with the input held, phi' = -(phi - phi_c) / tau: every RK4 stage value and
// the step itself are phi_c + (phi - phi_c) * (a polynomial in z = -h / tau) -- the same numbers the four stage derivatives
// produce, up to rounding.  A caller whose step length and time constants are fixed for the launch computes the factors once
// (lag_coef) and passes them: 5 fp64 instructions per lag and sub-step instead of 15.
struct LagCoef { double f2, f3, f4, ff, v2, v3, v4, vf; };
__device__ __forceinline__ void lag_coef(double h, double n_inv_tau, double& c2, double& c3, double& c4, double& cf) {
  const double z = h * n_inv_tau;
  c2 = fma(0.5, z, 1.0);                      // stage 2: phi + h/2 k1
  c3 = fma(0.5 * z, c2, 1.0);                 // stage 3: phi + h/2 k2
  c4 = fma(z, c3, 1.0);                       // stage 4: phi + h k3
  cf = fma(z * (1.0 / 6.0), (1.0 + 2.0 * c2) + (2.0 * c3 + c4), 1.0);      // phi + h/6 (k1 + 2 k2 + 2 k3 + k4)
}
__device__ __forceinline__ LagCoef lag_coef(double h, const AcPar& a) {
  LagCoef L;
  lag_coef(h, a.n_inv_tau_phi, L.f2, L.f3, L.f4, L.ff);
  lag_coef(h, a.n_inv_tau_v, L.v2, L.v3, L.v4, L.vf);
  return L;
}

#ifdef D2DX_USE_LIBM
template <bool ONE = false, bool LAG = false>
__device__ __forceinline__ void rk4_step(const AcPar& a, double* X, double phi_c, double v_c, double dt, int nsub, const LagCoef* = nullptr) {
  rk4_generic_inplace(a, X, phi_c, v_c, dt, nsub);
}
#else
// g tan(phi) / v with one reciprocal through the Pade ratio of d2dx_math.cuh (|phi| <= 1.15, checked by the caller)
__device__ __forceinline__ double turn_rate(double phi, double v) {
  double tn, td;
  fm::tan_ratio(phi, tn, td);
  return kG * tn * rcp_f(v * td);
}

// heading of an RK4 stage by angle addition: sin / cos of psi0 + d from (s0, c0) = sin / cos psi0, |d| < 0.1
__device__ __forceinline__ void stage_heading(double s0, double c0, double d, double& s, double& c) {
  double sd, cd;
  fm::sincos_small(d, sd, cd);
  s = fma(c0, sd, s0 * cd);
  c = fma(-s0, sd, c0 * cd);
}

// |x| below a validity threshold given by its HIGH WORD (integer pipe; NaN compares false).  The thresholds of the fast RK4 path
// are safety margins, not sharp limits: 0x3FB99999 = just under 0.1, 0x3FF26666 = just under 1.15.
__device__ __forceinline__ bool abs_below(double x, int thr_hi) { return (__double2hiint(x) & 0x7fffffff) < thr_hi; }
constexpr int kHiIncr = 0x3FB99999, kHiBank = 0x3FF26666;

// Fixed-step stand-in for Aircraft.disc_dyn (d2d/dynamic.py:25-28): nsub classical RK4 sub-steps of cont_dyn
// (:14-23) with the input held, then psi wrapped once (:27).  Straight-line fast path: the four stage headings share
// one full sincos (stages 2-4 by angle addition of the increment h psi_dot), tan(phi) is a Pade ratio folded into
// the 1/v reciprocal.  Validity (|increment| < 0.1, |phi| <= 1.15) is accumulated in one flag; if it is ever violated
// the control step is redone with rk4_step_generic.
// ONE = the caller guarantees nsub == 1 (the Monte-Carlo rollouts): no sub-step loop, so no loop-carried register copies.
template <bool ONE = false, bool LAG = false>
__device__ __forceinline__ void rk4_step(const AcPar& a, double* X, double phi_c, double v_c, double dt, int nsub, const LagCoef* L = nullptr) {
  // h = dt / nsub and h / 6 as written in the oracle cost two IEEE divisions (~40 instructions) per control step; the
  // reciprocal forms differ by at most one ulp of h (1e-16 relative on one step length), far inside the 1e-9 parity bound
  const double h = (ONE || nsub == 1) ? dt : dt * (1.0 / nsub), hh = 0.5 * h, h6 = h * (1.0 / 6.0);
  double x = X[0], y = X[1], psi = X[2], phi = X[3], v = X[4];
  bool fast_ok = true;                       // every stage increment < 0.1 rad and every bank angle <= 1.15 rad
  const int n_sub = ONE ? 1 : nsub;
#pragma unroll
  for (int sub = 0; sub < n_sub; ++sub) {
    double s1, c1, s, c, d;
    sincos_b(psi, s1, c1);
    if constexpr (LAG) {                     // the two lags in closed form (L: the factors of THIS h)
      const double df = phi - phi_c, dv = v - v_c;
      const double k1x = v * c1 + a.wx, k1y = v * s1 + a.wy, k1p = turn_rate(phi, v);
      fast_ok = fast_ok && abs_below(phi, kHiBank);
      double ph = fma(df, L->f2, phi_c), vv = fma(dv, L->v2, v_c);
      d = hh * k1p; fast_ok = fast_ok && abs_below(d, kHiIncr) && abs_below(ph, kHiBank);
      stage_heading(s1, c1, d, s, c);
      const double k2x = vv * c + a.wx, k2y = vv * s + a.wy, k2p = turn_rate(ph, vv);
      ph = fma(df, L->f3, phi_c); vv = fma(dv, L->v3, v_c);
      d = hh * k2p; fast_ok = fast_ok && abs_below(d, kHiIncr) && abs_below(ph, kHiBank);
      stage_heading(s1, c1, d, s, c);
      const double k3x = vv * c + a.wx, k3y = vv * s + a.wy, k3p = turn_rate(ph, vv);
      ph = fma(df, L->f4, phi_c); vv = fma(dv, L->v4, v_c);
      d = h * k3p; fast_ok = fast_ok && abs_below(d, kHiIncr) && abs_below(ph, kHiBank);
      stage_heading(s1, c1, d, s, c);
      const double k4x = vv * c + a.wx, k4y = vv * s + a.wy, k4p = turn_rate(ph, vv);
      x += h6 * (k1x + 2.0 * k2x + 2.0 * k3x + k4x);
      y += h6 * (k1y + 2.0 * k2y + 2.0 * k3y + k4y);
      psi += h6 * (k1p + 2.0 * k2p + 2.0 * k3p + k4p);
      phi = fma(df, L->ff, phi_c); v = fma(dv, L->vf, v_c);
    } else {
      // stage 1
      const double k1x = v * c1 + a.wx, k1y = v * s1 + a.wy, k1p = turn_rate(phi, v);
      const double k1f = a.n_inv_tau_phi * (phi - phi_c), k1v = a.n_inv_tau_v * (v - v_c);
      fast_ok = fast_ok && abs_below(phi, kHiBank);
      // stage 2
      double ph = phi + hh * k1f, vv = v + hh * k1v;
      d = hh * k1p; fast_ok = fast_ok && abs_below(d, kHiIncr) && abs_below(ph, kHiBank);
      stage_heading(s1, c1, d, s, c);
      const double k2x = vv * c + a.wx, k2y = vv * s + a.wy, k2p = turn_rate(ph, vv);
      const double k2f = a.n_inv_tau_phi * (ph - phi_c), k2v = a.n_inv_tau_v * (vv - v_c);
      // stage 3
      ph = phi + hh * k2f; vv = v + hh * k2v;
      d = hh * k2p; fast_ok = fast_ok && abs_below(d, kHiIncr) && abs_below(ph, kHiBank);
      stage_heading(s1, c1, d, s, c);
      const double k3x = vv * c + a.wx, k3y = vv * s + a.wy, k3p = turn_rate(ph, vv);
      const double k3f = a.n_inv_tau_phi * (ph - phi_c), k3v = a.n_inv_tau_v * (vv - v_c);
      // stage 4
      ph = phi + h * k3f; vv = v + h * k3v;
      d = h * k3p; fast_ok = fast_ok && abs_below(d, kHiIncr) && abs_below(ph, kHiBank);
      stage_heading(s1, c1, d, s, c);
      const double k4x = vv * c + a.wx, k4y = vv * s + a.wy, k4p = turn_rate(ph, vv);
      const double k4f = a.n_inv_tau_phi * (ph - phi_c), k4v = a.n_inv_tau_v * (vv - v_c);
      x += h6 * (k1x + 2.0 * k2x + 2.0 * k3x + k4x);
      y += h6 * (k1y + 2.0 * k2y + 2.0 * k3y + k4y);
      psi += h6 * (k1p + 2.0 * k2p + 2.0 * k3p + k4p);
      phi += h6 * (k1f + 2.0 * k2f + 2.0 * k3f + k4f);
      v += h6 * (k1v + 2.0 * k2v + 2.0 * k3v + k4v);
    }
  }
  psi = wrap_pi_or_flag(psi, fast_ok);       // a heading outside the wrap's three common cases also goes the generic way
  if (!fast_ok) {                            // NaN compares false: also caught
    rk4_generic_inplace(a, X, phi_c, v_c, dt, nsub);
    return;
  }
  X[0] = x; X[1] = y; X[2] = psi; X[3] = phi; X[4] = v;
}
#endif

// DiffFlatness.state_and_input_from_output, d2d/guidance.py:23-47
struct FlatState { double x, y, psi, phi, va, inv_va, u_phi, u_v, vadot, psidot, z /* tan(phi) */, cpsi, spsi; };

__device__ __forceinline__ void flatness(const FlatOut& Y, double wx, double wy, double tau_v, FlatState& r) {
  const double vax = Y.y1x - wx, vay = Y.y1y - wy;
  const double va2 = vax * vax + vay * vay;
  const double inv_va = rsqrt_f(va2), va = va2 * inv_va;
  r.x = Y.y0x; r.y = Y.y0y; r.va = va; r.inv_va = inv_va;
  r.psi = atan2_f(vay, vax);
  r.vadot = (vax * Y.y2x + vay * Y.y2y) * inv_va;
  const double num = Y.y2y * vax - Y.y2x * vay;
  r.psidot = num * inv_va * inv_va;
  r.z = num * inv_va * (1.0 / kG);        // argument of the arctan at :40, i.e. tan(phi_ref)
  r.phi = atan_f(r.z);
  r.u_phi = r.phi;                        // tau_phi * Xdot[phi] + phi with Xdot[phi] never filled (:42-43)
  r.u_v = tau_v * r.vadot + va;
  r.cpsi = vax * inv_va; r.spsi = vay * inv_va;   // cos / sin of arctan2(vay, vax)
}

// LQR gain of DFFFController.get (d2d/guidance.py:78-82): K1 = lqr(A[:3,:3], A[:3,3:], diag(q,q,q3), diag(r1,r2))
// with A from Aircraft.cont_jac (d2d/dynamic.py:32-43).
//
// Rotating the position error into the path frame (T = rot(-psi_ref) (+) 1) leaves Q unchanged (q1 = q2) and
// turns the pair into  A' = v e2 e3^T,  B' = [[0,1],[0,0],[b1,b2]],  b1 = g/v/(1+cos^2 phi),  b2 = g tan(phi)/v^2
// (entries replicated as the reference writes them).  With kappa_j = (sqrt(r1) K_1j, sqrt(r2) K_2j) the Riccati
// equation reads kappa_i . kappa_j = (A'^T P + P A' + Q)_ij, whose (1,1), (2,2), (1,2) entries force
// kappa_1 = sqrt(q) (C, S), kappa_2 = sqrt(q) (S, -C) with C^2 + S^2 = 1.  Writing kappa_3 = (al, be) and using
// P = P^T, the remaining unknowns (theta, al) solve
//     F1 = C al + S be + v (c2 C + e S) = 0,      F2 = al^2 + be^2 - q3 - 2 v c1 sqrt(q) S = 0,
//     be = (c1 sqrt(q) C + e al) / c2,   c1 = sqrt(r1)/b1,  c2 = sqrt(r2),  e = b2 c1,
// a 2x2 Newton iteration (quadratic, warm-started from the previous control step; cold start = the decoupled
// b2 = 0 solution C = 0, S = 1, al = sqrt(q3 + 2 v c1 sqrt(q))).  K' = [[C, S, al]/sqrt(r1) ; [S, -C, be]/sqrt(r2)]
// (times sqrt(q) on the first two columns) and K1 = K' T.  Checked against scipy.linalg.solve_continuous_are
// over v in [0.3, 60], |phi| < 1.4 to 3e-13 (tests/test_care_math.py runs THIS code, compiled for the host by
// csrc/host_check.cu, against SciPy; tests/test_gpu_rollout.py checks the device instance).
// high word of a double (sign, exponent, top 20 mantissa bits): magnitude and sign tests on the integer pipe
__host__ __device__ __forceinline__ int hi_word(double x) {
#ifdef __CUDA_ARCH__
  return __double2hiint(x);
#else
  long long b;
  memcpy(&b, &x, sizeof(b));
  return (int)(b >> 32);
#endif
}

// The Riccati warm start carried from one control step to the next, 9 doubles in the order of d2dx_rollout_out.care_state's
// rows: the solution C, S, al of the previous step (al <= 0 only in a cold state), then the changes of theta (sines of the
// angle steps) at steps n, n-1, n-2 and those of al.  Callers keep it where it suits them and pass an accessor st(k)
// returning a reference to row k.
constexpr int kCareState = D2DX_CARE_STATE_ROWS;
struct CareSol { double C, S, al, be; };   // solution of one step; be = kappa_3's second component
struct ArrayState {                        // the accessor over a plain array
  double* p;
  __host__ __device__ double& operator()(int k) const { return p[k]; }
};

// sqrt(Q), sqrt(R) and their products as care_gain and make_ref use them (folded once on the host, not per step)
struct CareConst { double q3, sr1, sr2, isr1, isr2, sq2, sq_isr1, sq_isr2; };

__host__ __device__ __forceinline__ CareConst care_const(double sq, double q3, double sr1, double sr2) {
  CareConst c;
  c.q3 = q3; c.sr1 = sr1; c.sr2 = sr2; c.isr1 = 1.0 / sr1; c.isr2 = 1.0 / sr2;
  c.sq2 = 2.0 * sq; c.sq_isr1 = sq * c.isr1; c.sq_isr2 = sq * c.isr2;
  return c;
}
__host__ __device__ __forceinline__ CareConst care_const(const d2dx_dfff_gains& g) {
  return care_const(::sqrt(g.q_pos), g.q_psi, ::sqrt(g.r_phi), ::sqrt(g.r_v));
}

struct CareStep { double k1, ba, vc2, ve, k2, q3; };   // per-control-step constants of the two residuals

// residuals F1, F2 at (C, S, al); also returns be
__host__ __device__ __forceinline__ void care_residual(const CareStep& k, double C, double S, double al, double& be, double& F1, double& F2) {
  be = fma(k.k1, C, k.ba * al);
  F1 = fma(C, al, fma(S, be, fma(k.vc2, C, k.ve * S)));
  F2 = fma(al, al, fma(be, be, -fma(k.k2, S, k.q3)));
}

// apply the update (dth, dal): rotate (C, S) by dth (first order + one Newton normalisation step), al += dal
__host__ __device__ __forceinline__ void care_update(double& C, double& S, double& al, double dth, double dal) {
  const double Cn = fma(-S, dth, C), Sn = fma(C, dth, S);
  const double nrm = fma(-0.5, fma(Cn, Cn, Sn * Sn), 1.5);        // 1/sqrt(1 + dth^2) up to O(dth^4)
  C = Cn * nrm; S = Sn * nrm; al += dal;
}

// Full Newton iteration loop (cold starts, trajectory corners, anything the straight-line step did not finish).
struct CareRoot { double C, S, al; bool conv; };
static __host__ __device__ __noinline__ CareRoot care_newton_loop_v(const CareStep k, double C, double S, double al, int max_it) {
  bool conv = false;
  for (int it = 0; it < max_it && !conv; ++it) {
    double be, F1, F2;
    care_residual(k, C, S, al, be, F1, F2);
    const double bt = -k.k1 * S;
    const double J11 = fma(-S, al, fma(C, be, fma(S, bt, fma(k.ve, C, -k.vc2 * S)))), J12 = fma(S, k.ba, C);
    const double J21 = 2.0 * fma(be, bt, -0.5 * k.k2 * C), J22 = 2.0 * fma(be, k.ba, al);
    const double idet = rcp_f(fma(J11, J22, -J12 * J21));
    const double dth = fma(J12, F2, -F1 * J22) * idet, dal = fma(J21, F1, -J11 * F2) * idet;
    const double Cn = C - S * dth, Sn = S + C * dth;
    const double nrm = rsqrt_f(fma(Cn, Cn, Sn * Sn));               // exact normalisation: steps can be large here
    C = Cn * nrm; S = Sn * nrm; al += dal;
    conv = fabs(dth) < 3e-8 && fabs(dal) < 3e-8 * fabs(al);        // quadratic convergence: remaining error ~1e-15
  }
  CareRoot r;
  r.C = C; r.S = S; r.al = al; r.conv = conv;
  return r;
}
__host__ __device__ __forceinline__ bool care_newton_loop(const CareStep& k, double& C, double& S, double& al, int max_it) {
  const CareRoot r = care_newton_loop_v(k, C, S, al, max_it);
  C = r.C; S = r.S; al = r.al;
  return r.conv;
}

// Acceptance bound of the single Newton step: |dth| and |dal| / al below 2^-23 = 1.19e-7, decided on the integer pipe (high
// words; hi(x) < hi(y) implies x < y for positive doubles, and adding 23 << 20 to a high word multiplies by 2^23).  The error
// the step leaves is quadratic in it: <= 1.04 |step|^2 (theta absolute, al relative) around the roots of the C5 population,
// so <= 1.5e-14 -- and the cubic warm start is within 3e-8, so the step stays below the bound.
constexpr int kCareStepTolHi = 0x3E800000;          // hi(2^-23)
constexpr int kCareStepTolExp = 23 << 20;
enum { CARE_FAILED = 0, CARE_LOOP = 1, CARE_FAST = 2 };

// Gain in the path frame.  Warm start = cubic extrapolation of the previous solutions from their last three changes
// (theta rotated by 3 (d[n] - d[n-1]) + d[n-2], al alike), which is O(dt^4) close to the new root while the reference
// moves smoothly (<= 3e-8 on the C5 circles at dt = 0.01); then ONE Newton step in straight-line code, accepted when it
// is below 2^-23.  Otherwise the general loop.  The solution goes to sol and, with the updated history, to st.
// Returns CARE_FAST when the straight-line step was accepted, CARE_LOOP when the loop converged, CARE_FAILED when not
// even the cold start did.
template <class State>
__host__ __device__ __forceinline__ int care_gain(const CareConst& cc, double v, double c1, double e, State&& st, bool cold, CareSol& sol) {
  CareStep k;                                                      // c1 = sqrt(r1)/b1, e = b2 c1
  k.k1 = c1 * cc.sq_isr2; k.ba = e * cc.isr2; k.vc2 = v * cc.sr2; k.ve = v * e; k.k2 = v * c1 * cc.sq2; k.q3 = cc.q3;
  // The warm path runs unconditionally and in straight-line code (a cold state only produces numbers that are thrown away):
  // its instructions share one block with the flatness / arctangent work before it, and ONE branch afterwards takes the cold
  // start, a failed acceptance test and the restart.  The extrapolation needs only the previous step's data, so it can issue
  // before this step's flatness work.
  const double th1 = st(3), th2 = st(4), th3 = st(5), al1 = st(6), al2 = st(7), al3 = st(8);
  st(4) = th1; st(5) = th2; st(7) = al1; st(8) = al2;              // age the history; this step's change goes to 3 and 6
  // extrapolate: rotate (C, S) by the angle whose sine is the extrapolated change p (cos = 1 - p^2/2 up to p^4/8, which the
  // Newton step's normalisation removes), as the changes were measured
  const double p = fma(3.0, th1 - th2, th3), cp = fma(-0.5 * p, p, 1.0);
  double C = fma(st(0), cp, -st(1) * p), S = fma(st(1), cp, st(0) * p), al = st(2) + fma(3.0, al1 - al2, al3);
  double be_, F1, F2;
  care_residual(k, C, S, al, be_, F1, F2);
  const double bt = -k.k1 * S;
  const double J11 = fma(-S, al, fma(C, be_, fma(S, bt, fma(k.ve, C, -k.vc2 * S)))), J12 = fma(S, k.ba, C);
  const double J21 = 2.0 * fma(be_, bt, -0.5 * k.k2 * C), J22 = 2.0 * fma(be_, k.ba, al);
  const double idet = rcp_f(fma(J11, J22, -J12 * J21));
  const double dth = fma(J12, F2, -F1 * J22) * idet, dal = fma(J21, F1, -J11 * F2) * idet;
  care_update(C, S, al, dth, dal);                                 // Newton step
  // accept when the step is tiny AND the root is on the stabilising branch (S > 0, al > 0 there: kappa_2's
  // first component and K_13 are positive for every v, b1 > 0)
  // (sign tests and the fixed threshold on the integer pipe; S, al > 0 <=> sign bit clear, not zero)
  const int hal = hi_word(al);
  int res = (!cold && (hi_word(dth) & 0x7fffffff) < kCareStepTolHi && (hi_word(dal) & 0x7fffffff) + kCareStepTolExp < hal &&
             hi_word(S) > 0 && hal > 0) ? CARE_FAST : CARE_FAILED;
  if (res == CARE_FAILED) {
    if (!cold) {                                                   // corner of the reference, big jump, history still building
      C = st(0); S = st(1); al = st(2);                            // up: iterate from the previous solution, not from the extrapolation
      if (care_newton_loop(k, C, S, al, 40) && S > 0.0 && al > 0.0) res = CARE_LOOP;
    }
    if (res == CARE_FAILED) {                                      // cold start: decoupled (b2 = 0) solution
      C = 0.0; S = 1.0; al = sqrt_f(cc.q3 + k.k2);
      if (care_newton_loop(k, C, S, al, 60)) res = CARE_LOOP;
    }
  }
  // change over this control step (angle from the cross product of the unit vectors); only a small, smooth change is worth
  // extrapolating -- and none after a cold start: the history restarts from zero and the next three steps take the loop
  const double nth = fma(st(0), S, -st(1) * C), nal = al - st(2);
  // (|nth| < 0.02 and |nal| < al / 64 on the integer pipe; a negative al fails the second test)
  const bool keep = !cold && (hi_word(nth) & 0x7fffffff) < 0x3F947AE1 && (hi_word(nal) & 0x7fffffff) + (6 << 20) < hi_word(al);
  st(0) = C; st(1) = S; st(2) = al;
  st(3) = keep ? nth : 0.0; st(6) = keep ? nal : 0.0;
  if (!keep) { st(4) = 0.0; st(5) = 0.0; st(7) = 0.0; st(8) = 0.0; }
  sol.C = C; sol.S = S; sol.al = al; sol.be = fma(k.k1, C, k.ba * al);
  return res;
}

// DFFFController.get (d2d/guidance.py:62-91) split in two.  Everything up to the gain depends on the reference
// trajectory and the wind only -- NOT on the aircraft state -- so the rollout computes it one control step ahead,
// interleaved with the RK4 stages of the current step (two independent dependency chains per thread).
struct RefCtl { double xr, yr, psir, phir, var, uphi, uv, k[6]; };   // reference state, feed-forward input, K1 = K' T (2x3)

template <class State>
__device__ __forceinline__ void make_ref(const FlatOut& Y, const AcPar& a, double tau_v, const CareConst& cc, State&& care,
                                         bool& cold, int& flags, RefCtl& r) {
  FlatState fr;
  flatness(Y, a.wx, a.wy, tau_v, fr);
  // cont_jac at the reference state (d2d/dynamic.py:36-38 as written), with cos^2(atan z) = 1/(1+z^2), tan(atan z) = z:
  //   b1 = g/va/(1+cos^2 phi) = g (1+z^2) / (va (2+z^2)),  b2 = g z / va^2;   c1 = sqrt(r1)/b1,  e = b2 c1
  const double z2 = fr.z * fr.z;
  const double c1 = cc.sr1 * (2.0 + z2) * rcp_f(kG * fr.inv_va * (1.0 + z2));
  const double e = kG * fr.inv_va * fr.inv_va * fr.z * c1;
  CareSol cs;
  if (care_gain(cc, fr.va, c1, e, care, cold, cs) != CARE_FAILED) cold = false;
  else { flags |= 2; cold = true; }
  r.xr = fr.x; r.yr = fr.y; r.psir = fr.psi; r.phir = fr.phi; r.var = fr.va; r.uphi = fr.u_phi; r.uv = fr.u_v;
  // K1 = K' T,  T = rot(-psi_ref) (+) 1,  K' = [[sqrt(q) (C, S), al] / sqrt(r1) ; [sqrt(q) (S, -C), be] / sqrt(r2)]:
  // both rows rotate the same unit vector (C, S)
  const double Cw = fma(cs.C, fr.cpsi, -cs.S * fr.spsi), Sw = fma(cs.C, fr.spsi, cs.S * fr.cpsi);
  r.k[0] = cc.sq_isr1 * Cw; r.k[1] = cc.sq_isr1 * Sw; r.k[2] = cs.al * cc.isr1;
  r.k[3] = cc.sq_isr2 * Sw; r.k[4] = -cc.sq_isr2 * Cw; r.k[5] = cs.be * cc.isr2;
}

// the state-dependent rest: error, wrap, saturations, feedback (d2d/guidance.py:67-70,85-88)
__device__ __forceinline__ void feedback(const RefCtl& r, const double* X, const d2dx_dfff_gains& g, double& u_phi, double& u_v) {
  const double ex = clip_sym(X[0] - r.xr, g.err_sat[0]);
  const double ey = clip_sym(X[1] - r.yr, g.err_sat[1]);
  const double ep = clip_sym(wrap_pi(X[2] - r.psir), g.err_sat[2]);
  u_phi = clip(r.uphi - fma(r.k[0], ex, fma(r.k[1], ey, r.k[2] * ep)), g.u_lo[0], g.u_hi[0]);
  u_v = clip(r.uv - fma(r.k[3], ex, fma(r.k[4], ey, r.k[5] * ep)), g.u_lo[1], g.u_hi[1]);
}

// CircleTraj.get + GVFcontroller.get, d2d/guidance.py:137-146,155-181 (E = [[0,1],[-1,0]], H = 2I)
__device__ __forceinline__ void gvf_control(double px, double py, double psi, double v, double cx, double cy,
                                            double r, double ke, double kd, double& U, double& U1, double& U2) {
  const double dx = px - cx, dy = py - cy;
  const double e = (dx * dx + dy * dy) - r * r;
  const double nx = 2.0 * dx, ny = 2.0 * dy;
  double s, c;
  sincos_b(psi, s, c);
  const double pdx = v * c, pdy = v * s;                 // p_dot
  const double tx = ny, ty = -nx;                        // tau = E n
  const double qx = tx - ke * e * nx, qy = ty - ke * e * ny;   // pd_dot
  const double inrm = rsqrt_f(qx * qx + qy * qy);        // 1/|pd_dot|
  const double qnx = qx * inrm, qny = qy * inrm;         // pd_dot_n
  const double ox = qny, oy = -qnx;                      // E pd_dot_n
  // w = (E - ke e I) H p_dot - ke (n p_dot^T) n
  const double hx = 2.0 * pdx, hy = 2.0 * pdy;
  const double kee = ke * e;
  const double wx_ = (-kee * hx + hy) - ke * (nx * pdx) * nx - ke * (nx * pdy) * ny;
  const double wy_ = (-hx - kee * hy) - ke * (ny * pdx) * nx - ke * (ny * pdy) * ny;
  // U1 = -(m w) . (E pd_dot_n / |pd_dot|),  m = o o^T
  const double ow = ox * wx_ + oy * wy_;
  U1 = -(ox * ow * (ox * inrm) + oy * ow * (oy * inrm));
  U2 = kd * (c * ox + s * oy);
  U = U1 + U2;
}

// Four warp sums at once: two exchange steps leave every lane with ONE of the four quantities (which one: lane bits 4 and 3),
// three butterfly steps finish it -- 6 double shuffles and adds instead of 20.  The totals end in lanes 0 (v0), 8 (v1), 16 (v2)
// and 24 (v3); the summation order is fixed, like warp_sum's.
__device__ __forceinline__ double warp_sum4(double v0, double v1, double v2, double v3, int lane) {
  const bool h16 = lane & 16, h8 = lane & 8;
  double k0 = h16 ? v2 : v0, k1 = h16 ? v3 : v1;              // lanes 0-15 keep (v0, v1), lanes 16-31 keep (v2, v3)
  k0 += __shfl_xor_sync(0xffffffffu, h16 ? v0 : v2, 16);
  k1 += __shfl_xor_sync(0xffffffffu, h16 ? v1 : v3, 16);
  double k = h8 ? k1 : k0;                                    // bit 3 picks the second of the pair
  k += __shfl_xor_sync(0xffffffffu, h8 ? k0 : k1, 8);
  k += __shfl_xor_sync(0xffffffffu, k, 4);
  k += __shfl_xor_sync(0xffffffffu, k, 2);
  k += __shfl_xor_sync(0xffffffffu, k, 1);
  return k;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ void atomic_max_double(double* addr, double val) {   // val >= 0
  atomicMax(reinterpret_cast<unsigned long long*>(addr), static_cast<unsigned long long>(__double_as_longlong(val)));
}

}  // namespace d2dx
