// Second-order solver of the single-aircraft planner NLP (SURVEY 8f #2; replaces prob.solve -> IPOPT, 06_optyplan.py:117-125,
// for one aircraft): control-limited differential dynamic programming on the collocation grid.
//
// The backward-Euler defects of d2d/opty_utils.py:38-50 define the explicit transition
//     psi_i = psi_{i-1} + h g tan(phi_i) / v_i,  x_i = x_{i-1} + h (v_i cos psi_i - w_x),  y_i = y_{i-1} + h (v_i sin psi_i - w_y),
// so the NLP is a discrete optimal-control problem with 3 states and 2 inputs per node.  One iteration = a backward sweep
// that builds, node by node, the exact second-order model of the cost-to-go (first AND second derivatives of the transition:
// a Newton step, not Gauss-Newton -- the planner costs without a bank term have no curvature of their own in phi) and solves
// the 2-variable box-constrained quadratic programme of each node exactly (the input bounds hold at every iterate, no
// substitution), then a forward sweep with feedback and a backtracking line search.  The block-tridiagonal KKT system that
// IPOPT factorises is what the backward sweep eliminates, 3 x 3 blocks at a time.  The terminal conditions enter through an
// augmented Lagrangian (multiplier and penalty updates between sweeps); the state box of x/y_constraint as a quadratic penalty
// of the excess.  Everything is per problem and sequential over the nodes: one THREAD solves one problem, a launch solves a
// population (multi-start, many boundary conditions); the work arrays are interleaved over the problems so that the lanes of a
// warp, which walk the nodes in lock step, touch consecutive doubles.
// __host__ __device__: csrc/host_check.cu runs the same code on the CPU (tests/test_ddp_cpu.py).
#pragma once
#include <stdio.h>

#include "d2dx_device.cuh"

namespace d2dx {

struct DdpProblem {
  int N;
  double h, wx, wy;
  double vsp, kv, kb;              // stage input cost kv (v - vsp)^2 + kb phi^2   (weights already times obj_scale / N / in_div)
  double kobs;                     // obstacle weight times obj_scale / N
  int n_obs, obs_kind;
  double obs[D2DX_MAX_OBSTACLES][3];
  double phi_lo, phi_hi, v_lo, v_hi;
  int has_box;
  double x_lo, x_hi, y_lo, y_hi, w_box;   // w_box = weight * obj_scale / N
};

// fills the solver's problem description from the collocation problem + bounds + box (every aircraft shares them)
__host__ inline int ddp_problem_from(const d2dx_colloc_problem* p, const double* bounds, const double* box, DdpProblem& P, int max_ac = 1) {
  if (!p || p->n_ac < 1 || p->n_ac > max_ac || p->N < 2 || !(p->h > 0) || !bounds) return 1;
  const double sN = p->obj_scale / p->N, nin = sN / (p->in_div >= 1 ? p->in_div : 1);
  P.N = p->N; P.h = p->h; P.wx = p->wind[0]; P.wy = p->wind[1];
  P.vsp = p->vsp; P.kv = p->kvel * nin; P.kb = p->kbank * nin;
  const bool obs = (p->kobs == p->kobs) && p->kobs != 0.0 && p->n_obs > 0;
  P.kobs = obs ? p->kobs * sN : 0.0; P.n_obs = obs ? p->n_obs : 0; P.obs_kind = p->obs_kind;
  for (int o = 0; o < P.n_obs; ++o) { P.obs[o][0] = p->obs[o][0]; P.obs[o][1] = p->obs[o][1]; P.obs[o][2] = p->obs[o][2]; }
  P.phi_lo = bounds[0]; P.phi_hi = bounds[1]; P.v_lo = bounds[2]; P.v_hi = bounds[3];
  P.has_box = box != nullptr;
  if (box) { P.x_lo = box[0]; P.x_hi = box[1]; P.y_lo = box[2]; P.y_hi = box[3]; P.w_box = box[4] * sN; }
  else { P.x_lo = P.y_lo = -1e300; P.x_hi = P.y_hi = 1e300; P.w_box = 0.0; }
  return (P.phi_lo < P.phi_hi && P.v_lo < P.v_hi && P.v_lo > 0.0) ? 0 : 1;
}

struct DdpWork {                   // element (k, node) of an array lives at base[(k * N + node) * stride]
  double *u, *z, *un, *zn, *k, *K;
  long stride;
  int N;
  __host__ __device__ __forceinline__ double& at(double* b, int k, int i) const { return b[((long)k * N + i) * stride]; }
};

__host__ __device__ __forceinline__ double ddp_clip(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

// state cost of a node (obstacles, soft box): value, gradient (gx, gy), Hessian (hxx, hxy, hyy)
__host__ __device__ inline double ddp_state_cost(const DdpProblem& P, double x, double y, double& gx, double& gy, double& hxx, double& hxy,
                                                 double& hyy) {
  double c = 0.0;
  gx = gy = hxx = hxy = hyy = 0.0;
  for (int o = 0; o < P.n_obs; ++o) {
    const double dx = x - P.obs[o][0], dy = y - P.obs[o][1], r = P.obs[o][2];
    double es, cc;
    if (P.obs_kind == 0) { cc = 1.0; es = ::exp(r * r - (dx * dx + dy * dy)); es = es > 1e3 ? 1e3 : es; }   // clip(exp(r^2 - d^2), 0, 1e3), opty_utils.py:108-111
    else { cc = (2.0 / r) * (2.0 / r); es = ::exp(-cc * (dx * dx + dy * dy)); }                               // exp(-(2/r)^2 d^2), :113-117
    c += P.kobs * es;
    const double w1 = -2.0 * cc * es * P.kobs, w2 = 4.0 * cc * cc * es * P.kobs;
    gx += w1 * dx; gy += w1 * dy;
    hxx += w2 * dx * dx + w1; hxy += w2 * dx * dy; hyy += w2 * dy * dy + w1;
  }
  if (P.has_box) {
    const double ex = x < P.x_lo ? x - P.x_lo : (x > P.x_hi ? x - P.x_hi : 0.0);
    const double ey = y < P.y_lo ? y - P.y_lo : (y > P.y_hi ? y - P.y_hi : 0.0);
    c += P.w_box * (ex * ex + ey * ey);
    gx += 2.0 * P.w_box * ex; gy += 2.0 * P.w_box * ey;
    if (ex != 0.0) hxx += 2.0 * P.w_box;
    if (ey != 0.0) hyy += 2.0 * P.w_box;
  }
  return c;
}

__host__ __device__ __forceinline__ double ddp_input_cost(const DdpProblem& P, double phi, double v) {
  const double dv = v - P.vsp;
  return P.kv * dv * dv + P.kb * phi * phi;
}

// one transition (the backward-Euler defect solved for the new state)
__host__ __device__ __forceinline__ void ddp_step(const DdpProblem& P, double x, double y, double psi, double phi, double v, double& xn,
                                                  double& yn, double& pn) {
  pn = psi + P.h * kG * ::tan(phi) / v;
  xn = x + P.h * (v * ::cos(pn) - P.wx);
  yn = y + P.h * (v * ::sin(pn) - P.wy);
}

// exact minimiser of 1/2 d^T Q d + g^T d over the box [lo, hi]^2 (Q positive definite): the nine active sets are tried until
// one satisfies feasibility and the sign conditions.  free[j] tells whether component j ended strictly inside.
__host__ __device__ inline void ddp_box_qp2(double q00, double q01, double q11, double g0, double g1, double lo0, double hi0, double lo1,
                                            double hi1, double* d, bool* free_) {
  const double det = q00 * q11 - q01 * q01;
  const double tol = 1e-12;
  for (int s0 = 0; s0 < 3; ++s0) {
    for (int s1 = 0; s1 < 3; ++s1) {
      double d0, d1;
      if (s0 == 0 && s1 == 0) { d0 = (-g0 * q11 + g1 * q01) / det; d1 = (-g1 * q00 + g0 * q01) / det; }
      else if (s0 == 0) { d1 = s1 == 1 ? lo1 : hi1; d0 = -(g0 + q01 * d1) / q00; }
      else if (s1 == 0) { d0 = s0 == 1 ? lo0 : hi0; d1 = -(g1 + q01 * d0) / q11; }
      else { d0 = s0 == 1 ? lo0 : hi0; d1 = s1 == 1 ? lo1 : hi1; }
      if (s0 == 0 && !(d0 >= lo0 - tol && d0 <= hi0 + tol)) continue;
      if (s1 == 0 && !(d1 >= lo1 - tol && d1 <= hi1 + tol)) continue;
      const double r0 = g0 + q00 * d0 + q01 * d1, r1 = g1 + q01 * d0 + q11 * d1;     // gradient at the candidate
      if (s0 == 1 && r0 < -1e-9 * (fabs(g0) + 1e-300)) continue;
      if (s0 == 2 && r0 > 1e-9 * (fabs(g0) + 1e-300)) continue;
      if (s1 == 1 && r1 < -1e-9 * (fabs(g1) + 1e-300)) continue;
      if (s1 == 2 && r1 > 1e-9 * (fabs(g1) + 1e-300)) continue;
      d[0] = ddp_clip(d0, lo0, hi0); d[1] = ddp_clip(d1, lo1, hi1);
      free_[0] = s0 == 0; free_[1] = s1 == 0;
      return;
    }
  }
  // numerically ambiguous: clamp the unconstrained minimiser, treat clamped components as fixed
  const double u0 = (-g0 * q11 + g1 * q01) / det, u1 = (-g1 * q00 + g0 * q01) / det;
  d[0] = ddp_clip(u0, lo0, hi0); d[1] = ddp_clip(u1, lo1, hi1);
  free_[0] = d[0] == u0; free_[1] = d[1] == u1;
}

struct DdpSweep { double dV1, dV2; bool ok; };

#ifdef __CUDA_ARCH__
__device__ __forceinline__ void ddp_sincos(double x, double& s, double& c) { sincos_any(x, s, c); }   // straight-line fp64 sincos (d2dx_math.cuh)
#else
inline void ddp_sincos(double x, double& s, double& c) { s = ::sin(x); c = ::cos(x); }
#endif

// everything of a node's transition that does not depend on the value function: computed for 32 nodes at once by the lanes of
// the warp that solves the problem (the transcendental functions are the expensive part), consumed one node at a time
struct DdpNodePre { double phi, v, s, c, dph, dvv, dphph, dphv, dv2; };
constexpr int kDdpPre = 9;

__host__ __device__ __forceinline__ void ddp_node_pre(const DdpProblem& P, double phi, double v, double th, DdpNodePre& n) {
  double sp, cp;
  ddp_sincos(th, n.s, n.c);
  ddp_sincos(phi, sp, cp);
  const double tp = sp / cp, sec2 = 1.0 + tp * tp, iv = 1.0 / v, hg = P.h * kG;
  const double del = hg * tp * iv;
  n.phi = phi; n.v = v;
  n.dph = hg * sec2 * iv; n.dvv = -del * iv;
  n.dphph = 2.0 * hg * sec2 * tp * iv; n.dphv = -n.dph * iv; n.dv2 = 2.0 * del * iv * iv;
}

// quadratic model of the cost-to-go as a function of the state: gradient and (symmetric) Hessian
struct DdpValue { double z0, z1, z2, w00, w01, w02, w11, w12, w22; };

// value model at the last node: state cost + lam . c + rho / 2 |c|^2
__host__ __device__ inline void ddp_terminal_value(const DdpProblem& P, double x, double y, double psi, const double* zt, const double* lam,
                                                   double rho, DdpValue& W) {
  double gx, gy, hxx, hxy, hyy;
  ddp_state_cost(P, x, y, gx, gy, hxx, hxy, hyy);
  W.z0 = gx + lam[0] + rho * (x - zt[0]); W.z1 = gy + lam[1] + rho * (y - zt[1]); W.z2 = lam[2] + rho * (psi - zt[2]);
  W.w00 = hxx + rho; W.w01 = hxy; W.w02 = 0.0; W.w11 = hyy + rho; W.w12 = 0.0; W.w22 = rho;
}

// One node of the backward sweep: from the value model W at node i (as a function of z_i, node i's state cost included) to the
// gains k (2), K (2 x 3) of input u_i and the value model at node i-1 (WITHOUT that node's own state cost: the caller adds it).
// Returns false when the regularised Quu is not positive definite.
__host__ __device__ inline bool ddp_backward_node(const DdpProblem& P, const DdpNodePre& n, double mu, int reg_mode, DdpValue& W, double* kk,
                                                  double* K, double& dV1, double& dV2) {
  const double h = P.h, phi = n.phi, v = n.v, s = n.s, c = n.c, dph = n.dph, dvv_ = n.dvv;
  const double w00 = W.w00, w01 = W.w01, w02 = W.w02, w11 = W.w11, w12 = W.w12, w22 = W.w22;
  const double a13 = -h * v * s, a23 = h * v * c;
  const double b11 = a13 * dph, b12 = h * c + a13 * dvv_, b21 = a23 * dph, b22 = h * s + a23 * dvv_, b31 = dph, b32 = dvv_;
  const double p0 = W.z0, p1 = W.z1, p2 = W.z2;
  // first order
  const double qz0 = p0, qz1 = p1, qz2 = a13 * p0 + a23 * p1 + p2;
  const double qu0 = 2.0 * P.kb * phi + b11 * p0 + b21 * p1 + b31 * p2;
  const double qu1 = 2.0 * P.kv * (v - P.vsp) + b12 * p0 + b22 * p1 + b32 * p2;
  // second derivatives of the transition contracted with p
  const double Mth = h * v * (-p0 * s + p1 * c) + p2, Mthth = -h * v * (p0 * c + p1 * s), Mthv = h * (-p0 * s + p1 * c);
  const double Gpp = Mthth, Gpf = Mthth * dph, Gpv = Mthth * dvv_ + Mthv;
  const double Gff = Mthth * dph * dph + Mth * n.dphph, Gfv = Mthth * dph * dvv_ + Mthv * dph + Mth * n.dphv;
  const double Gvv = Mthth * dvv_ * dvv_ + 2.0 * Mthv * dvv_ + Mth * n.dv2;
  // M = Wzz A (columns 0, 1 of Wzz and t = Wzz (a13, a23, 1))
  const double t0 = w00 * a13 + w01 * a23 + w02, t1 = w01 * a13 + w11 * a23 + w12, t2 = w02 * a13 + w12 * a23 + w22;
  const double qzz00 = w00, qzz01 = w01, qzz02 = t0, qzz11 = w11, qzz12 = t1, qzz22 = a13 * t0 + a23 * t1 + t2 + Gpp;
  // Quz = B^T M + G_uz   (rows: phi, v; columns: x, y, psi)
  const double quz00 = b11 * w00 + b21 * w01 + b31 * w02, quz01 = b11 * w01 + b21 * w11 + b31 * w12, quz02 = b11 * t0 + b21 * t1 + b31 * t2 + Gpf;
  const double quz10 = b12 * w00 + b22 * w01 + b32 * w02, quz11 = b12 * w01 + b22 * w11 + b32 * w12, quz12 = b12 * t0 + b22 * t1 + b32 * t2 + Gpv;
  // Quu = l_uu + B^T Wzz B + G_uu
  const double wb00 = w00 * b11 + w01 * b21 + w02 * b31, wb10 = w01 * b11 + w11 * b21 + w12 * b31, wb20 = w02 * b11 + w12 * b21 + w22 * b31;
  const double wb01 = w00 * b12 + w01 * b22 + w02 * b32, wb11 = w01 * b12 + w11 * b22 + w12 * b32, wb21 = w02 * b12 + w12 * b22 + w22 * b32;
  const double quu00 = 2.0 * P.kb + b11 * wb00 + b21 * wb10 + b31 * wb20 + Gff;
  const double quu01 = b11 * wb01 + b21 * wb11 + b31 * wb21 + Gfv;
  const double quu11 = 2.0 * P.kv + b12 * wb01 + b22 * wb11 + b32 * wb21 + Gvv;
  // regularised copy for the step, in variables scaled by the width of their bounds (phi in radians and v in m/s differ by an
  // order of magnitude)
  const double d0 = 1.0 / ((P.phi_hi - P.phi_lo) * (P.phi_hi - P.phi_lo)), d1 = 1.0 / ((P.v_hi - P.v_lo) * (P.v_hi - P.v_lo));
  double r00, r01, r11;
  if (reg_mode == 0) {                             // plain Levenberg-Marquardt: the caller raises mu until every node is definite
    r00 = quu00 + mu * d0; r01 = quu01; r11 = quu11 + mu * d1;
    if (!(r00 > 0.0 && r11 > 0.0 && r00 * r11 - r01 * r01 > 1e-12 * r00 * r11)) return false;
  } else {                                         // eigenvalues replaced by their magnitude (floor: a fraction of the larger one), plus mu
    const double sd = ::sqrt(d0 * d1);
    const double s00 = quu00 / d0, s01 = quu01 / sd, s11 = quu11 / d1;                              // scaled Quu
    const double tr = 0.5 * (s00 + s11), rad = ::sqrt(0.25 * (s00 - s11) * (s00 - s11) + s01 * s01);
    const double l1 = tr + rad, l2 = tr - rad;                                                      // l1 >= l2
    const double fl = 1e-6 * fmax(fabs(l1), fabs(l2)) + 1e-300;
    const double m1 = fmax(fabs(l1), fl) + mu, m2 = fmax(fabs(l2), fl) + mu;
    double ex = s01, ey = l1 - s00;                // unit eigenvector of l1: (s01, l1 - s00) or (l1 - s11, s01), whichever is longer
    if (fabs(l1 - s11) > fabs(ey)) { ex = l1 - s11; ey = s01; }
    const double en = ::sqrt(ex * ex + ey * ey);
    if (en > 0.0) { ex /= en; ey /= en; } else { ex = 1.0; ey = 0.0; }
    const double t00 = m1 * ex * ex + m2 * ey * ey, t01 = (m1 - m2) * ex * ey, t11 = m1 * ey * ey + m2 * ex * ex;
    r00 = t00 * d0; r01 = t01 * sd; r11 = t11 * d1;
    if (!(r00 > 0.0 && r11 > 0.0 && r00 * r11 - r01 * r01 > 0.0)) return false;                     // NaN / overflow only
  }
  bool fr[2];
  ddp_box_qp2(r00, r01, r11, qu0, qu1, P.phi_lo - phi, P.phi_hi - phi, P.v_lo - v, P.v_hi - v, kk, fr);
  // feedback of the free components only: K_F = -R_FF^-1 Quz_F
  double K00 = 0.0, K01 = 0.0, K02 = 0.0, K10 = 0.0, K11 = 0.0, K12 = 0.0;
  if (fr[0] && fr[1]) {
    const double id = 1.0 / (r00 * r11 - r01 * r01);
    K00 = -(r11 * quz00 - r01 * quz10) * id; K01 = -(r11 * quz01 - r01 * quz11) * id; K02 = -(r11 * quz02 - r01 * quz12) * id;
    K10 = -(r00 * quz10 - r01 * quz00) * id; K11 = -(r00 * quz11 - r01 * quz01) * id; K12 = -(r00 * quz12 - r01 * quz02) * id;
  } else if (fr[0]) { K00 = -quz00 / r00; K01 = -quz01 / r00; K02 = -quz02 / r00; }
  else if (fr[1]) { K10 = -quz10 / r11; K11 = -quz11 / r11; K12 = -quz12 / r11; }
  K[0] = K00; K[1] = K01; K[2] = K02; K[3] = K10; K[4] = K11; K[5] = K12;
  dV1 += kk[0] * qu0 + kk[1] * qu1;
  dV2 += 0.5 * (kk[0] * (quu00 * kk[0] + quu01 * kk[1]) + kk[1] * (quu01 * kk[0] + quu11 * kk[1]));
  // value model of the previous node: V = Q along the policy (unregularised Quu)
  const double a0 = quu00 * kk[0] + quu01 * kk[1] + qu0, a1 = quu01 * kk[0] + quu11 * kk[1] + qu1;     // Quu k + Qu
  W.z0 = qz0 + K00 * a0 + K10 * a1 + quz00 * kk[0] + quz10 * kk[1];
  W.z1 = qz1 + K01 * a0 + K11 * a1 + quz01 * kk[0] + quz11 * kk[1];
  W.z2 = qz2 + K02 * a0 + K12 * a1 + quz02 * kk[0] + quz12 * kk[1];
  const double c00 = quu00 * K00 + quu01 * K10, c01 = quu00 * K01 + quu01 * K11, c02 = quu00 * K02 + quu01 * K12;   // Quu K
  const double c10 = quu01 * K00 + quu11 * K10, c11 = quu01 * K01 + quu11 * K11, c12 = quu01 * K02 + quu11 * K12;
  W.w00 = qzz00 + K00 * c00 + K10 * c10 + 2.0 * (K00 * quz00 + K10 * quz10);
  W.w01 = qzz01 + K00 * c01 + K10 * c11 + (K00 * quz01 + K10 * quz11) + (quz00 * K01 + quz10 * K11);
  W.w02 = qzz02 + K00 * c02 + K10 * c12 + (K00 * quz02 + K10 * quz12) + (quz00 * K02 + quz10 * K12);
  W.w11 = qzz11 + K01 * c01 + K11 * c11 + 2.0 * (K01 * quz01 + K11 * quz11);
  W.w12 = qzz12 + K01 * c02 + K11 * c12 + (K01 * quz02 + K11 * quz12) + (quz01 * K02 + quz11 * K12);
  W.w22 = qzz22 + K02 * c02 + K12 * c12 + 2.0 * (K02 * quz02 + K12 * quz12);
  return true;
}

// one node of the forward sweep: new input from the old one, the step and the feedback on the state deviation, then the transition
__host__ __device__ __forceinline__ void ddp_forward_node(const DdpProblem& P, double alpha, double uo0, double uo1, const double* k, const double* K,
                                                          double zo0, double zo1, double zo2, double& x, double& y, double& psi, double& phi,
                                                          double& v) {
  const double dx = x - zo0, dy = y - zo1, dp = psi - zo2;
  phi = ddp_clip(uo0 + alpha * k[0] + K[0] * dx + K[1] * dy + K[2] * dp, P.phi_lo, P.phi_hi);
  v = ddp_clip(uo1 + alpha * k[1] + K[3] * dx + K[4] * dy + K[5] * dp, P.v_lo, P.v_hi);
  double sp, cp, s, c;
  ddp_sincos(phi, sp, cp);
  psi = psi + P.h * kG * (sp / cp) / v;
  ddp_sincos(psi, s, c);
  x = x + P.h * (v * c - P.wx);
  y = y + P.h * (v * s - P.wy);
}

// ---- serial sweeps over one problem's arrays (host build; also the reference of the warp-cooperative device sweeps) ----
struct DdpSerial {
  static constexpr int kMaxCon = 3;
  const DdpProblem& P;
  DdpWork W;
  const double* zt;
  __host__ __device__ DdpSerial(const DdpProblem& p, const DdpWork& w, const double* zt_) : P(p), W(w), zt(zt_) {}

  __host__ __device__ DdpSweep backward(const double* lam, double rho, double mu, int reg_mode) {
    const int N = P.N;
    DdpSweep r = {0.0, 0.0, true};
    DdpValue V;
    ddp_terminal_value(P, W.at(W.z, 0, N - 1), W.at(W.z, 1, N - 1), W.at(W.z, 2, N - 1), zt, lam, rho, V);
    for (int i = N - 1; i >= 1; --i) {
      DdpNodePre n;
      ddp_node_pre(P, W.at(W.u, 0, i), W.at(W.u, 1, i), W.at(W.z, 2, i), n);
      double kk[2], K[6];
      if (!ddp_backward_node(P, n, mu, reg_mode, V, kk, K, r.dV1, r.dV2)) { r.ok = false; return r; }
      W.at(W.k, 0, i) = kk[0]; W.at(W.k, 1, i) = kk[1];
      for (int j = 0; j < 6; ++j) W.at(W.K, j, i) = K[j];
      if (i > 1 && (P.n_obs > 0 || P.has_box)) {
        double gx, gy, hxx, hxy, hyy;
        ddp_state_cost(P, W.at(W.z, 0, i - 1), W.at(W.z, 1, i - 1), gx, gy, hxx, hxy, hyy);
        V.z0 += gx; V.z1 += gy; V.w00 += hxx; V.w01 += hxy; V.w11 += hyy;
      }
    }
    return r;
  }

  // forward sweep with step alpha and feedback: (u, z) -> (un, zn); returns the augmented Lagrangian of the new trajectory
  __host__ __device__ double forward(double alpha, const double* lam, double rho, double& cost, double& cmax) {
    const int N = P.N;
    double x = W.at(W.z, 0, 0), y = W.at(W.z, 1, 0), psi = W.at(W.z, 2, 0);
    W.at(W.zn, 0, 0) = x; W.at(W.zn, 1, 0) = y; W.at(W.zn, 2, 0) = psi;
    W.at(W.un, 0, 0) = W.at(W.u, 0, 0); W.at(W.un, 1, 0) = W.at(W.u, 1, 0);
    cost = ddp_input_cost(P, W.at(W.u, 0, 0), W.at(W.u, 1, 0));
    const bool sc = P.n_obs > 0 || P.has_box;
    double gx, gy, hxx, hxy, hyy;
    if (sc) cost += ddp_state_cost(P, x, y, gx, gy, hxx, hxy, hyy);
    for (int i = 1; i < N; ++i) {
      const double kk[2] = {W.at(W.k, 0, i), W.at(W.k, 1, i)};
      const double K[6] = {W.at(W.K, 0, i), W.at(W.K, 1, i), W.at(W.K, 2, i), W.at(W.K, 3, i), W.at(W.K, 4, i), W.at(W.K, 5, i)};
      double phi, v;
      ddp_forward_node(P, alpha, W.at(W.u, 0, i), W.at(W.u, 1, i), kk, K, W.at(W.z, 0, i - 1), W.at(W.z, 1, i - 1), W.at(W.z, 2, i - 1), x, y, psi,
                       phi, v);
      W.at(W.un, 0, i) = phi; W.at(W.un, 1, i) = v;
      W.at(W.zn, 0, i) = x; W.at(W.zn, 1, i) = y; W.at(W.zn, 2, i) = psi;
      cost += ddp_input_cost(P, phi, v);
      if (sc) cost += ddp_state_cost(P, x, y, gx, gy, hxx, hxy, hyy);
    }
    const double c0 = x - zt[0], c1 = y - zt[1], c2 = psi - zt[2];
    cmax = fmax(fabs(c0), fmax(fabs(c1), fabs(c2)));
    return cost + lam[0] * c0 + lam[1] * c1 + lam[2] * c2 + 0.5 * rho * (c0 * c0 + c1 * c1 + c2 * c2);
  }

  __host__ __device__ void accept() {
    double* t = W.u; W.u = W.un; W.un = t;
    t = W.z; W.z = W.zn; W.zn = t;
  }
  __host__ __device__ int n_con() const { return 3; }
  __host__ __device__ bool enough_solved() const { return false; }
  __host__ __device__ void count_solved() {}
  // terminal error of the current trajectory
  __host__ __device__ void terminal_error(double* c) const {
    const int N = P.N;
    c[0] = W.at(W.z, 0, N - 1) - zt[0]; c[1] = W.at(W.z, 1, N - 1) - zt[1]; c[2] = W.at(W.z, 2, N - 1) - zt[2];
  }
  // start: inputs clipped into the bounds, node 0's input at its own minimiser, gains zero, initial state in place
  __host__ __device__ void prepare(const double* z0) {
    const int N = P.N;
    if (P.kb > 0.0) W.at(W.u, 0, 0) = 0.0;
    if (P.kv > 0.0) W.at(W.u, 1, 0) = P.vsp;
    for (int i = 0; i < N; ++i) {
      W.at(W.u, 0, i) = ddp_clip(W.at(W.u, 0, i), P.phi_lo, P.phi_hi);
      W.at(W.u, 1, i) = ddp_clip(W.at(W.u, 1, i), P.v_lo, P.v_hi);
      W.at(W.k, 0, i) = 0.0; W.at(W.k, 1, i) = 0.0;
      for (int j = 0; j < 6; ++j) W.at(W.K, j, i) = 0.0;
      for (int j = 0; j < 3; ++j) W.at(W.z, j, i) = 0.0;
    }
    W.at(W.z, 0, 0) = z0[0]; W.at(W.z, 1, 0) = z0[1]; W.at(W.z, 2, 0) = z0[2];
  }
};

struct DdpResult { int flag, iterations, outer, swaps; double cost, cmax, lagr, mu, rho; };   // flag 2 solved, 3 stopped unsolved, 4 feasible at the sweep limit; swaps odd: the solution sits in (un, zn)

// The solver: augmented-Lagrangian loop around regularised second-order sweeps.  `S` supplies the sweeps over one problem's
// arrays (DdpSerial on the host, the warp-cooperative DdpWarp in d2dx_ddp.cu); every decision below is a scalar one.
// S::kMaxCon bounds the number of terminal conditions S::n_con() (3 per aircraft).  lam_out (optional): the multipliers of the last
// inner loop, the ones the returned trajectory minimises the augmented Lagrangian for.
template <typename S>
__host__ __device__ inline DdpResult ddp_solve(S& sw_, const double* z0, const d2dx_ddp_options& o, double* lam_out = nullptr) {
  const int nc = sw_.n_con();
  double lam[S::kMaxCon], rho = o.rho0, mu = o.mu0, dmu = 1.0;
  for (int k = 0; k < nc; ++k) lam[k] = 0.0;
  sw_.prepare(z0);
  double cost, cmax, J = sw_.forward(0.0, lam, rho, cost, cmax);     // zero gains: the rollout of the start inputs
  sw_.accept();
  DdpResult res = {3, 0, 0, 1, cost, cmax, J, mu, rho};
  double c_prev = cmax;
  int it = 0;
  bool stop = false;
  for (int outer = 0; outer < o.max_outer && it < o.max_iter && !stop; ++outer) {
    if (lam_out) for (int k = 0; k < nc; ++k) lam_out[k] = lam[k];
    bool converged = false;
    for (int inner = 0; inner < o.max_inner && it < o.max_iter; ++inner, ++it) {
      if (sw_.enough_solved()) { stop = true; break; }     // multi-start: enough other starts of the launch have converged
      DdpSweep sw = sw_.backward(lam, rho, mu, o.reg_mode);
      int tries = 0;
      while (!sw.ok && tries < 12) {               // Quu not positive definite somewhere: more regularisation, sweep again
        dmu = fmax(dmu * o.mu_factor, o.mu_factor); mu = fmax(mu * dmu, o.mu_min);
        sw = sw_.backward(lam, rho, mu, o.reg_mode);
        ++tries;
      }
      if (!sw.ok) { stop = true; break; }
      if (-(sw.dV1 + sw.dV2) <= o.rel_tol * fabs(J) + o.abs_tol && mu <= o.mu_min * 1.0001) { converged = true; break; }   // no predicted decrease left
      double alpha = 1.0, Jn = J, costn = cost, cmaxn = cmax;
      bool accepted = false;
      for (int ls = 0; ls < o.ls_max; ++ls, alpha *= 0.5) {
        Jn = sw_.forward(alpha, lam, rho, costn, cmaxn);
        const double expected = -(alpha * sw.dV1 + alpha * alpha * sw.dV2);      // decrease the quadratic model predicts
        if (Jn == Jn && expected > 0.0 && (J - Jn) >= 1e-4 * expected) { accepted = true; break; }
      }
#if defined(D2DX_DDP_TRACE) && !defined(__CUDA_ARCH__)
      printf("outer %2d inner %2d it %3d  J %.10e cost %.8e cmax %.2e  dV %.2e  alpha %.4f acc %d mu %.1e rho %.0e\n", outer, inner, it, Jn, costn, cmaxn,
             -(sw.dV1 + sw.dV2), alpha, (int)accepted, mu, rho);
#endif
      if (accepted) {
        sw_.accept();
        ++res.swaps;
        const double dJ = J - Jn;
        J = Jn; cost = costn; cmax = cmaxn;
        dmu = fmin(dmu / o.mu_factor, 1.0 / o.mu_factor);
        mu = mu * dmu > o.mu_min ? mu * dmu : o.mu_min;
        if (dJ <= o.rel_tol * fabs(J) + o.abs_tol) { converged = true; ++it; break; }
      } else {
        dmu = fmax(dmu * o.mu_factor, o.mu_factor); mu = fmax(mu * dmu, o.mu_min);
        if (mu > o.mu_max) { converged = true; ++it; break; }        // no step at any regularisation: a (local) minimum of this subproblem
      }
    }
    if (stop) break;
    res.outer = outer + 1;
    if (cmax < o.ctol && converged) { res.flag = 2; sw_.count_solved(); break; }
    // multiplier / penalty update (the rule of the first-order driver: grow rho when the violation did not fall to a quarter)
    double c[S::kMaxCon];
    sw_.terminal_error(c);
    for (int k = 0; k < nc; ++k) lam[k] += rho * c[k];
    if (cmax > 0.25 * c_prev || outer == 0) rho = fmin(rho * o.rho_growth, o.rho_max);
    c_prev = cmax;
    mu = o.mu0; dmu = 1.0;
    J = cost;
    double cc = 0.0;
    for (int k = 0; k < nc; ++k) { J += lam[k] * c[k]; cc += c[k] * c[k]; }
    J += 0.5 * rho * cc;
  }
  if (res.flag != 2 && !stop && cmax < o.ctol) res.flag = 4;       // feasible, but the sweep budget ran out before the cost settled
  res.iterations = it; res.cost = cost; res.cmax = cmax; res.lagr = J; res.mu = mu; res.rho = rho;
  return res;
}

}  // namespace d2dx
