// Second-order solver of the multi-aircraft planner NLP (07_multioptyplan.py:80-88): the control-limited DDP of d2dx_ddp.cuh
// with the n aircraft of a problem in one stage, state z in R^{3n} (x, y, psi of aircraft a at 3a .. 3a+2) and input u in
// R^{2n} (phi, v of aircraft a at 2a, 2a+1).  The transition is block-diagonal (each aircraft flies on its own: ddp_node_pre per
// aircraft); the aircraft are coupled through the collision term of the state cost, so the value model W_zz is a dense
// 3n x 3n matrix and the box QP of a node has 2n variables (projected Newton, Tassa, Mansard & Todorov, ICRA 2014).
//
// A node of the backward sweep is split into steps that each produce rows (or columns) independently of one another:
//   s1 (row r < 3n)   N = W B, M = W A (in place), Qz = A^T Wz
//   s2 (row r < 2n)   Quz = B^T M + G_uz, Quu = l_uu + B^T N + G_uu, Qu
//   s3 (row 3a+2)     Qzz = A^T M (in place; rows 3a, 3a+1 of M already are rows of Qzz)
//   s4 (one)          regularisation test, box QP, Cholesky factor of the free block, expected decrease
//   s5 (column c)     K[:, c] = -R_FF^-1 Quz_F[:, c], C[:, c] = Quu K[:, c] + Quz[:, c]
//   s6 (row r < 3n)   value model of the previous node, plus that node's state cost
// The host sweeps (DdpmSerial) run the steps row after row; the kernel (d2dx_ddp_multi.cu) gives row r to lane r.
// __host__ __device__: csrc/host_check.cu runs the same code on the CPU (tests/test_ddp_multi_cpu.py).
#pragma once
#include "d2dx_ddp.cuh"

namespace d2dx {

constexpr int kDdpmMaxAc = 10;                     // 3n rows of W_zz on the 32 lanes of a warp
constexpr int kDdpmQpIter = 64;                    // projected-Newton iterations of a node's box QP
constexpr int kDdpmQpLs = 40;                      // halvings of its projected line search

struct DdpmProblem {
  DdpProblem a;                                    // transition, input cost, bounds, soft box (every aircraft), obstacles (aircraft 0)
  int n;                                           // aircraft
  double kcol;                                     // collision weight times obj_scale / N; 0: no collision term
  double col_k2;                                   // (kcol_k / rcol)^2
  int col_all;                                     // 1: every pair, 0: the pair (0, 1)
};

__host__ inline int ddpm_problem_from(const d2dx_colloc_problem* p, const double* bounds, const double* box, DdpmProblem& M) {
  if (ddp_problem_from(p, bounds, box, M.a, kDdpmMaxAc)) return 1;
  M.n = p->n_ac;
  const bool col = p->kcol == p->kcol && p->kcol != 0.0 && p->n_ac > 1;
  M.kcol = col ? p->kcol * p->obj_scale / p->N : 0.0;
  M.col_k2 = col ? (p->kcol_k / p->rcol) * (p->kcol_k / p->rcol) : 0.0;
  M.col_all = p->col_all_pairs;
  return col && !(M.col_k2 == M.col_k2 && M.col_k2 < 1e300) ? 1 : 0;
}

__host__ __device__ __forceinline__ bool ddpm_pair(const DdpmProblem& M, int a, int b) {
  return M.kcol != 0.0 && a != b && (M.col_all || (a < 2 && b < 2));
}

// cost of aircraft a's own state terms (soft box; obstacles on aircraft 0, the kind-0 clip flat where it is active, as
// d2dx_shoot_adjoint evaluates them): value, gradient, Hessian (hxx, hxy, hyy)
__host__ __device__ inline double ddpm_own_cost(const DdpmProblem& M, int a, double x, double y, double& gx, double& gy, double& hxx,
                                                double& hxy, double& hyy) {
  const DdpProblem& P = M.a;
  double c = 0.0;
  gx = gy = hxx = hxy = hyy = 0.0;
  for (int o = 0; a == 0 && o < P.n_obs; ++o) {
    const double dx = x - P.obs[o][0], dy = y - P.obs[o][1], r = P.obs[o][2];
    double es, cc;
    if (P.obs_kind == 0) {
      cc = 1.0; es = ::exp(r * r - (dx * dx + dy * dy));
      if (!(es < 1e3)) { c += P.kobs * 1e3; continue; }
    } else { cc = (2.0 / r) * (2.0 / r); es = ::exp(-cc * (dx * dx + dy * dy)); }
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

// state cost of aircraft a at a node (its own terms and the collision terms of the pairs (a, b > a)); z: the node's 3n states
__host__ __device__ inline double ddpm_aircraft_cost(const DdpmProblem& M, int a, const double* z) {
  double gx, gy, hxx, hxy, hyy;
  double c = ddpm_own_cost(M, a, z[3 * a], z[3 * a + 1], gx, gy, hxx, hxy, hyy);
  for (int b = a + 1; b < M.n; ++b) {
    if (!ddpm_pair(M, a, b)) continue;
    const double dx = z[3 * a] - z[3 * b], dy = z[3 * a + 1] - z[3 * b + 1];
    c += M.kcol * ::exp(-M.col_k2 * (dx * dx + dy * dy));
  }
  return c;
}

// adds entry r of the state cost's gradient to g and row r of its Hessian to Wrow (r = 3a + k; nothing for k = 2).  A pair's
// Hessian in (x_a, y_a, x_b, y_b) is [[H, -H], [-H, H]] with H = e (4 k2^2 d d^T - 2 k2 I), e = kcol exp(-k2 |d|^2): indefinite
// near the pair, which the regularisation of Quu absorbs.
__host__ __device__ inline void ddpm_state_row(const DdpmProblem& M, const double* z, int r, double& g, double* Wrow) {
  const int a = r / 3, k = r - 3 * a;
  if (k == 2) return;
  double gx, gy, hxx, hxy, hyy;
  ddpm_own_cost(M, a, z[3 * a], z[3 * a + 1], gx, gy, hxx, hxy, hyy);
  double gr = k == 0 ? gx : gy;
  Wrow[3 * a] += k == 0 ? hxx : hxy;
  Wrow[3 * a + 1] += k == 0 ? hxy : hyy;
  for (int b = 0; b < M.n; ++b) {
    if (!ddpm_pair(M, a, b)) continue;
    const double dx = z[3 * a] - z[3 * b], dy = z[3 * a + 1] - z[3 * b + 1], k2 = M.col_k2;
    const double e = M.kcol * ::exp(-k2 * (dx * dx + dy * dy));
    const double d = k == 0 ? dx : dy;
    gr += -2.0 * k2 * d * e;
    const double h0 = e * (4.0 * k2 * k2 * d * dx - (k == 0 ? 2.0 * k2 : 0.0));
    const double h1 = e * (4.0 * k2 * k2 * d * dy - (k == 1 ? 2.0 * k2 : 0.0));
    Wrow[3 * a] += h0; Wrow[3 * a + 1] += h1;
    Wrow[3 * b] -= h0; Wrow[3 * b + 1] -= h1;
  }
  g += gr;
}

// A and B of one aircraft's transition: a13, a23, then B row-major (3 x 2)
__host__ __device__ __forceinline__ void ddpm_ab(const DdpProblem& P, const double* pre, double* ab) {
  const double h = P.h, v = pre[1], s = pre[2], c = pre[3], dph = pre[4], dvv = pre[5];
  const double a13 = -h * v * s, a23 = h * v * c;
  ab[0] = a13; ab[1] = a23;
  ab[2] = a13 * dph; ab[3] = h * c + a13 * dvv; ab[4] = a23 * dph; ab[5] = h * s + a23 * dvv; ab[6] = dph; ab[7] = dvv;
}

// second derivatives of one aircraft's transition contracted with its costate p (3): Gpp, Gpf, Gpv, Gff, Gfv, Gvv
__host__ __device__ __forceinline__ void ddpm_g(const DdpProblem& P, const double* pre, const double* p, double* G) {
  const double h = P.h, v = pre[1], s = pre[2], c = pre[3], dph = pre[4], dvv = pre[5];
  const double Mth = h * v * (-p[0] * s + p[1] * c) + p[2], Mthth = -h * v * (p[0] * c + p[1] * s), Mthv = h * (-p[0] * s + p[1] * c);
  G[0] = Mthth; G[1] = Mthth * dph; G[2] = Mthth * dvv + Mthv;
  G[3] = Mthth * dph * dph + Mth * pre[6]; G[4] = Mthth * dph * dvv + Mthv * dph + Mth * pre[7];
  G[5] = Mthth * dvv * dvv + 2.0 * Mthv * dvv + Mth * pre[8];
}

// Cholesky factor (lower, into L) of the m x m matrix H[idx[i]][idx[j]]; false when a pivot is not above tol times its diagonal
__host__ __device__ inline bool ddpm_chol(int m, const double* H, int ld, const int* idx, double* L, double tol) {
  for (int j = 0; j < m; ++j) {
    for (int i = j; i < m; ++i) {
      double s = H[idx[i] * ld + idx[j]];
      for (int k = 0; k < j; ++k) s -= L[i * ld + k] * L[j * ld + k];
      if (i == j) {
        if (!(s > tol * H[idx[j] * ld + idx[j]]) || !(s > 0.0)) return false;
        L[j * ld + j] = ::sqrt(s);
      } else {
        L[i * ld + j] = s / L[j * ld + j];
      }
    }
  }
  return true;
}

// x <- L^-T L^-1 x (m entries at x[0], x[xs], x[2 xs], ...)
__host__ __device__ inline void ddpm_chol_solve(int m, const double* L, int ld, double* x, int xs) {
  for (int i = 0; i < m; ++i) {
    double s = x[i * xs];
    for (int k = 0; k < i; ++k) s -= L[i * ld + k] * x[k * xs];
    x[i * xs] = s / L[i * ld + i];
  }
  for (int i = m - 1; i >= 0; --i) {
    double s = x[i * xs];
    for (int k = i + 1; k < m; ++k) s -= L[k * ld + i] * x[k * xs];
    x[i * xs] = s / L[i * ld + i];
  }
}

__host__ __device__ inline double ddpm_qp_value(int m, const double* H, int ld, const double* q, const double* x) {
  double f = 0.0;
  for (int i = 0; i < m; ++i) {
    double hx = 0.0;
    for (int j = 0; j < m; ++j) hx += H[i * ld + j] * x[j];
    f += x[i] * (q[i] + 0.5 * hx);
  }
  return f;
}

// Minimiser of 1/2 x^T H x + q^T x over lo <= x <= hi (m <= 2 kDdpmMaxAc variables, H positive definite with leading dimension ld)
// by projected Newton: the clamped set (at a bound, gradient pushing outwards) is fixed, a Newton step on the free block is
// searched along the projection (Armijo).  On return fr[j] = 1 for the free components, fi[0 .. nf) lists them and L holds the
// Cholesky factor of the free block.  Returns false when a free block is not definite (not for a definite H).
__host__ __device__ inline bool ddpm_box_qp(int m, const double* H, int ld, const double* q, const double* lo, const double* hi, double* x,
                                            int* fr, int* fi, int& nf, double* L) {
  double g[2 * kDdpmMaxAc], d[2 * kDdpmMaxAc], xt[2 * kDdpmMaxAc];
  for (int j = 0; j < m; ++j) x[j] = ddp_clip(0.0, lo[j], hi[j]);
  double f = ddpm_qp_value(m, H, ld, q, x);
  for (int it = 0;; ++it) {
    double gn = 0.0, sc = 0.0;
    nf = 0;
    for (int i = 0; i < m; ++i) {
      double hx = 0.0;
      for (int j = 0; j < m; ++j) hx += H[i * ld + j] * x[j];
      g[i] = q[i] + hx;
      sc = fmax(sc, fmax(fabs(q[i]), fabs(hx)));
      fr[i] = !((x[i] <= lo[i] && g[i] > 0.0) || (x[i] >= hi[i] && g[i] < 0.0));
      if (fr[i]) { fi[nf++] = i; gn = fmax(gn, fabs(g[i])); }
    }
    if (!ddpm_chol(nf, H, ld, fi, L, 0.0)) return false;
    if (nf == 0 || gn <= 1e-13 * sc || it == kDdpmQpIter) return true;
    double gd = 0.0;
    for (int j = 0; j < m; ++j) d[j] = 0.0;
    for (int j = 0; j < nf; ++j) d[j] = -g[fi[j]];
    ddpm_chol_solve(nf, L, ld, d, 1);
    for (int j = nf - 1; j >= 0; --j) { const double t = d[j]; d[j] = 0.0; d[fi[j]] = t; gd += t * g[fi[j]]; }
    bool acc = false;
    double alpha = 1.0, ft = f;
    for (int ls = 0; ls < kDdpmQpLs && gd < 0.0; ++ls, alpha *= 0.5) {
      for (int j = 0; j < m; ++j) xt[j] = ddp_clip(x[j] + alpha * d[j], lo[j], hi[j]);
      ft = ddpm_qp_value(m, H, ld, q, xt);
      if (ft - f <= 0.1 * alpha * gd) { acc = true; break; }
    }
    if (!acc) return true;
    for (int j = 0; j < m; ++j) x[j] = xt[j];
    f = ft;
  }
}

// One node's matrices and vectors (row-major, leading dimensions ldz >= 3n and ldu >= 2n; the warp's shared memory on the device)
struct DdpmNode {
  const DdpmProblem& M;
  int n, ldz, ldu;
  double *W, *Wz, *Nb, *Qz, *Quz, *Quu, *R, *L, *K, *C, *Qu, *kk, *av;
  int *fr, *fi, *nf;
  double *dV;                                      // dV1, dV2 of the sweep
  const double* pre;                               // [n][kDdpPre] of the node, then the 3n states of the previous node
  __host__ __device__ DdpmNode(const DdpmProblem& m_) : M(m_), n(m_.n), ldz((3 * m_.n) | 1), ldu((2 * m_.n) | 1) {}

  // doubles of the matrices above for n aircraft (and ints)
  __host__ __device__ static int doubles(int n) {
    const int lz = (3 * n) | 1, lu = (2 * n) | 1;
    return 3 * n * lz + 3 * n + 3 * n * lu + 3 * n + 2 * n * lz + 3 * 2 * n * lu + 2 * 2 * n * lz + 3 * 2 * n + 2;
  }
  __host__ __device__ static int ints(int n) { return 2 * 2 * n + 2; }
  __host__ __device__ void carve(double* d, int* iw) {
    W = d; d += 3 * n * ldz; Wz = d; d += 3 * n; Nb = d; d += 3 * n * ldu; Qz = d; d += 3 * n;
    Quz = d; d += 2 * n * ldz; Quu = d; d += 2 * n * ldu; R = d; d += 2 * n * ldu; L = d; d += 2 * n * ldu;
    K = d; d += 2 * n * ldz; C = d; d += 2 * n * ldz; Qu = d; d += 2 * n; kk = d; d += 2 * n; av = d; d += 2 * n; dV = d;
    fr = iw; fi = iw + 2 * n; nf = iw + 4 * n;
  }

  // value model at the last node, row r: state cost + lam . c + rho / 2 |c|^2 (z: the last node's states)
  __host__ __device__ void s0(int r, const double* z, const double* zt, const double* lam, double rho) {
    double* w = W + r * ldz;
    for (int c = 0; c < 3 * n; ++c) w[c] = 0.0;
    w[r] = rho;
    Wz[r] = lam[r] + rho * (z[r] - zt[r]);
    ddpm_state_row(M, z, r, Wz[r], w);
  }
  __host__ __device__ void s1(int r) {
    double* w = W + r * ldz;
    double* nb = Nb + r * ldu;
    for (int b = 0; b < n; ++b) {
      double ab[8];
      ddpm_ab(M.a, pre + b * kDdpPre, ab);
      const double w0 = w[3 * b], w1 = w[3 * b + 1], w2 = w[3 * b + 2];
      nb[2 * b] = w0 * ab[2] + w1 * ab[4] + w2 * ab[6];
      nb[2 * b + 1] = w0 * ab[3] + w1 * ab[5] + w2 * ab[7];
      w[3 * b + 2] = w0 * ab[0] + w1 * ab[1] + w2;
    }
    const int a = r / 3;
    if (r - 3 * a < 2) Qz[r] = Wz[r];
    else {
      double ab[8];
      ddpm_ab(M.a, pre + a * kDdpPre, ab);
      Qz[r] = ab[0] * Wz[3 * a] + ab[1] * Wz[3 * a + 1] + Wz[3 * a + 2];
    }
  }
  __host__ __device__ void s2(int r) {
    const int a = r >> 1, j = r & 1;
    const double* pa = pre + a * kDdpPre;
    double ab[8], G[6];
    ddpm_ab(M.a, pa, ab);
    ddpm_g(M.a, pa, Wz + 3 * a, G);
    const double b0 = ab[2 + j], b1 = ab[4 + j], b2 = ab[6 + j];
    const double *m0 = W + 3 * a * ldz, *m1 = m0 + ldz, *m2 = m1 + ldz;
    double* qz = Quz + r * ldz;
    for (int c = 0; c < 3 * n; ++c) qz[c] = b0 * m0[c] + b1 * m1[c] + b2 * m2[c];
    qz[3 * a + 2] += G[1 + j];
    const double *n0 = Nb + 3 * a * ldu, *n1 = n0 + ldu, *n2 = n1 + ldu;
    double* qu = Quu + r * ldu;
    for (int c = 0; c < 2 * n; ++c) qu[c] = b0 * n0[c] + b1 * n1[c] + b2 * n2[c];
    if (j == 0) { qu[2 * a] += 2.0 * M.a.kb + G[3]; qu[2 * a + 1] += G[4]; }
    else { qu[2 * a] += G[4]; qu[2 * a + 1] += 2.0 * M.a.kv + G[5]; }
    const double lu = j == 0 ? 2.0 * M.a.kb * pa[0] : 2.0 * M.a.kv * (pa[1] - M.a.vsp);
    Qu[r] = lu + b0 * Wz[3 * a] + b1 * Wz[3 * a + 1] + b2 * Wz[3 * a + 2];
  }
  __host__ __device__ void s3(int r) {           // r = 3a + 2
    const int a = r / 3;
    double ab[8], G[6];
    ddpm_ab(M.a, pre + a * kDdpPre, ab);
    ddpm_g(M.a, pre + a * kDdpPre, Wz + 3 * a, G);
    const double *m0 = W + 3 * a * ldz, *m1 = m0 + ldz;
    double* m2 = W + r * ldz;
    for (int c = 0; c < 3 * n; ++c) m2[c] = ab[0] * m0[c] + ab[1] * m1[c] + m2[c];
    m2[r] += G[0];
  }
  // regularised Quu (Levenberg-Marquardt in variables scaled by the bound widths), its definiteness, the box QP
  __host__ __device__ bool s4(double mu) {
    const DdpProblem& P = M.a;
    const int m = 2 * n;
    const double d0 = 1.0 / ((P.phi_hi - P.phi_lo) * (P.phi_hi - P.phi_lo)), d1 = 1.0 / ((P.v_hi - P.v_lo) * (P.v_hi - P.v_lo));
    double lo[2 * kDdpmMaxAc], hi[2 * kDdpmMaxAc];
    for (int i = 0; i < m; ++i) {
      for (int j = 0; j < m; ++j) R[i * ldu + j] = Quu[i * ldu + j];
      R[i * ldu + i] += mu * ((i & 1) ? d1 : d0);
      fi[i] = i;
      const double ui = pre[(i >> 1) * kDdpPre + (i & 1)];
      lo[i] = ((i & 1) ? P.v_lo : P.phi_lo) - ui; hi[i] = ((i & 1) ? P.v_hi : P.phi_hi) - ui;
    }
    if (!ddpm_chol(m, R, ldu, fi, L, 1e-12)) return false;
    if (!ddpm_box_qp(m, R, ldu, Qu, lo, hi, kk, fr, fi, *nf, L)) return false;
    double e1 = 0.0, e2 = 0.0;
    for (int i = 0; i < m; ++i) {
      double qk = 0.0;
      for (int j = 0; j < m; ++j) qk += Quu[i * ldu + j] * kk[j];
      e1 += kk[i] * Qu[i]; e2 += kk[i] * qk;
      av[i] = qk + Qu[i];
    }
    dV[0] += e1; dV[1] += 0.5 * e2;
    return true;
  }
  // feedback of the free rows on state c
  __host__ __device__ void s5(int c) {
    const int m = 2 * n, f = *nf;
    for (int i = 0; i < m; ++i) K[i * ldz + c] = 0.0;
    for (int j = 0; j < f; ++j) K[j * ldz + c] = -Quz[fi[j] * ldz + c];
    ddpm_chol_solve(f, L, ldu, K + c, ldz);
    for (int j = f - 1; j >= 0; --j) { const double t = K[j * ldz + c]; K[j * ldz + c] = 0.0; K[fi[j] * ldz + c] = t; }
    for (int i = 0; i < m; ++i) {
      double s = Quz[i * ldz + c];
      for (int j = 0; j < m; ++j) s += Quu[i * ldu + j] * K[j * ldz + c];
      C[i * ldz + c] = s;
    }
  }
  // value model of the previous node (V = Q along the policy, unregularised Quu), plus its state cost when it is not node 0
  __host__ __device__ void s6(int r, bool state_cost) {
    const int m = 2 * n;
    double s = Qz[r];
    for (int i = 0; i < m; ++i) s += K[i * ldz + r] * av[i];
    for (int i = 0; i < m; ++i) s += Quz[i * ldz + r] * kk[i];
    Wz[r] = s;
    double* w = W + r * ldz;
    for (int c = 0; c < 3 * n; ++c) {
      double t = w[c];
      for (int i = 0; i < m; ++i) t += K[i * ldz + r] * C[i * ldz + c] + Quz[i * ldz + r] * K[i * ldz + c];
      w[c] = t;
    }
    if (state_cost) ddpm_state_row(M, pre + n * kDdpPre, r, Wz[r], w);
  }
};

// Work arrays of one problem (contiguous): u, un [N][2n]; z, zn [N][3n]; k [N][2n]; K [N][3n][2n] (column c of node i's gain
// at K + (i 3n + c) 2n)
struct DdpmWork {
  double *u, *z, *un, *zn, *k, *K;
  __host__ __device__ static long doubles(int n, int N) { return (long)N * (12 * n + 6 * n * n); }
  __host__ __device__ void carve(double* b, int n, int N) {
    u = b; b += 2L * n * N; z = b; b += 3L * n * N; un = b; b += 2L * n * N; zn = b; b += 3L * n * N; k = b; b += 2L * n * N; K = b;
  }
};

// the input of row r of node i in the forward sweep (zc: the new states of node i-1)
__host__ __device__ __forceinline__ double ddpm_input(const DdpmProblem& M, const DdpmWork& W, int i, int r, double alpha, const double* zc) {
  const int n = M.n, m = 2 * n;
  double s = W.u[(long)i * m + r] + alpha * W.k[(long)i * m + r];
  const double* Kc = W.K + (long)i * 3 * n * m + r;
  const double* zo = W.z + (long)(i - 1) * 3 * n;
  for (int c = 0; c < 3 * n; ++c) s += Kc[c * m] * (zc[c] - zo[c]);
  return (r & 1) ? ddp_clip(s, M.a.v_lo, M.a.v_hi) : ddp_clip(s, M.a.phi_lo, M.a.phi_hi);
}

// aircraft a's transition (z: its 3 states, in place) and its input cost
__host__ __device__ __forceinline__ double ddpm_transition(const DdpmProblem& M, double phi, double v, double* z) {
  const DdpProblem& P = M.a;
  double sp, cp, s, c;
  ddp_sincos(phi, sp, cp);
  z[2] = z[2] + P.h * kG * (sp / cp) / v;
  ddp_sincos(z[2], s, c);
  z[0] = z[0] + P.h * (v * c - P.wx);
  z[1] = z[1] + P.h * (v * s - P.wy);
  return ddp_input_cost(P, phi, v);
}

// ---- serial sweeps over one problem's arrays (host build; the reference of the warp-cooperative device sweeps) ----
struct DdpmSerial {
  static constexpr int kMaxCon = 3 * kDdpmMaxAc;
  const DdpmProblem& M;
  DdpmWork W;
  const double* zt;                                // [3n] terminal targets
  DdpmNode nd;
  double* pre;                                     // [n kDdpPre + 3n]
  __host__ __device__ DdpmSerial(const DdpmProblem& m, const DdpmWork& w, const double* zt_, double* scratch, int* iscratch, double* pre_)
      : M(m), W(w), zt(zt_), nd(m), pre(pre_) { nd.carve(scratch, iscratch); nd.pre = pre; }
  __host__ __device__ int n_con() const { return 3 * M.n; }
  __host__ __device__ bool enough_solved() const { return false; }
  __host__ __device__ void count_solved() {}

  __host__ __device__ DdpSweep backward(const double* lam, double rho, double mu, int) {
    const int n = M.n, N = M.a.N, m = 2 * n, nz = 3 * n;
    DdpSweep r = {0.0, 0.0, true};
    nd.dV[0] = nd.dV[1] = 0.0;
    for (int q = 0; q < nz; ++q) nd.s0(q, W.z + (long)(N - 1) * nz, zt, lam, rho);
    for (int i = N - 1; i >= 1; --i) {
      for (int a = 0; a < n; ++a) {
        DdpNodePre p;
        ddp_node_pre(M.a, W.u[(long)i * m + 2 * a], W.u[(long)i * m + 2 * a + 1], W.z[(long)i * nz + 3 * a + 2], p);
        double* d = pre + a * kDdpPre;
        d[0] = p.phi; d[1] = p.v; d[2] = p.s; d[3] = p.c; d[4] = p.dph; d[5] = p.dvv; d[6] = p.dphph; d[7] = p.dphv; d[8] = p.dv2;
      }
      for (int c = 0; c < nz; ++c) pre[n * kDdpPre + c] = W.z[(long)(i - 1) * nz + c];
      for (int q = 0; q < nz; ++q) nd.s1(q);
      for (int q = 0; q < m; ++q) nd.s2(q);
      for (int q = 2; q < nz; q += 3) nd.s3(q);
      if (!nd.s4(mu)) { r.ok = false; return r; }
      for (int c = 0; c < nz; ++c) nd.s5(c);
      for (int q = 0; q < nz; ++q) nd.s6(q, i > 1);
      for (int q = 0; q < m; ++q) W.k[(long)i * m + q] = nd.kk[q];
      for (int c = 0; c < nz; ++c)
        for (int q = 0; q < m; ++q) W.K[((long)i * nz + c) * m + q] = nd.K[q * nd.ldz + c];
    }
    r.dV1 = nd.dV[0]; r.dV2 = nd.dV[1];
    return r;
  }

  __host__ __device__ double forward(double alpha, const double* lam, double rho, double& cost, double& cmax) {
    const int n = M.n, N = M.a.N, m = 2 * n, nz = 3 * n;
    double zc[3 * kDdpmMaxAc], us[2 * kDdpmMaxAc];
    for (int c = 0; c < nz; ++c) W.zn[c] = zc[c] = W.z[c];
    for (int q = 0; q < m; ++q) W.un[q] = W.u[q];
    cost = 0.0;
    for (int a = 0; a < n; ++a) cost += ddp_input_cost(M.a, W.u[2 * a], W.u[2 * a + 1]) + ddpm_aircraft_cost(M, a, zc);
    for (int i = 1; i < N; ++i) {
      for (int q = 0; q < m; ++q) us[q] = ddpm_input(M, W, i, q, alpha, zc);
      for (int a = 0; a < n; ++a) cost += ddpm_transition(M, us[2 * a], us[2 * a + 1], zc + 3 * a);
      for (int a = 0; a < n; ++a) cost += ddpm_aircraft_cost(M, a, zc);
      for (int q = 0; q < m; ++q) W.un[(long)i * m + q] = us[q];
      for (int c = 0; c < nz; ++c) W.zn[(long)i * nz + c] = zc[c];
    }
    double J = cost, cc = 0.0;
    cmax = 0.0;
    for (int c = 0; c < nz; ++c) {
      const double e = zc[c] - zt[c];
      cmax = fmax(cmax, fabs(e)); J += lam[c] * e; cc += e * e;
    }
    return J + 0.5 * rho * cc;
  }

  __host__ __device__ void accept() {
    double* t = W.u; W.u = W.un; W.un = t;
    t = W.z; W.z = W.zn; W.zn = t;
  }
  __host__ __device__ void terminal_error(double* c) const {
    const int nz = 3 * M.n;
    for (int q = 0; q < nz; ++q) c[q] = W.z[(long)(M.a.N - 1) * nz + q] - zt[q];
  }
  // start: inputs clipped into the bounds, node 0's inputs at their own minimiser, gains zero, initial states in place
  __host__ __device__ void prepare(const double* z0) {
    const int n = M.n, N = M.a.N, m = 2 * n, nz = 3 * n;
    for (int i = 0; i < N; ++i) {
      for (int q = 0; q < m; ++q) {
        double x = W.u[(long)i * m + q];
        if (i == 0 && (q & 1) == 0 && M.a.kb > 0.0) x = 0.0;
        if (i == 0 && (q & 1) == 1 && M.a.kv > 0.0) x = M.a.vsp;
        W.u[(long)i * m + q] = (q & 1) ? ddp_clip(x, M.a.v_lo, M.a.v_hi) : ddp_clip(x, M.a.phi_lo, M.a.phi_hi);
        W.k[(long)i * m + q] = 0.0;
      }
      for (int c = 0; c < nz * m; ++c) W.K[(long)i * nz * m + c] = 0.0;
      for (int c = 0; c < nz; ++c) W.z[(long)i * nz + c] = i == 0 ? z0[c] : 0.0;
    }
  }
};

}  // namespace d2dx
