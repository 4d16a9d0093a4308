// The 5x5 Riccati reduction of the tracker (Controllers.py:159-186): six unknowns, Newton with the analytic Jacobian and a
// fixed-order 6x6 elimination.  __host__ __device__ so that csrc/host_check.cu can run it on the CPU against SciPy
// (tests/test_care_math.py); derivation in the header comment of d2dx_tracker.cu.
#pragma once
#include "d2dx_device.cuh"

namespace d2dx {

struct Lqr5State { double C, S, p23, p24, p33, p34, p44; };    // al == 0 marks "cold"

struct Lqr5Par { double v, a, b, itp, itv, s1, s2, i1, i2, sq, q3, q4, q5; };

// solves the 6x6 system J d = -F without row exchanges: the equations are taken in the fixed order (1,4), (1,3), (2,4), (3,3), (3,4), (4,4)
// (rows 2, 0, 3, 1, 4, 5), the order in which plain elimination matched LAPACK to 2e-15 on 2700 Newton systems of this
// family (tau_phi 0.01 .. 0.97, v 4 .. 30 m/s, |phi| <= 1.1, condition numbers 11 .. 3900) -- the row exchanges of the
// pivoted version are 13 % of the tracker's instructions.  A pivot below 1e-9 of its row makes the step fail (the caller
// restarts cold and flags the aircraft if that fails too).
__host__ __device__ __forceinline__ bool solve6(double (&J)[6][6], double (&F)[6], double (&d)[6]) {
  constexpr int perm[6] = {2, 0, 3, 1, 4, 5};
  double A[6][7];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
#pragma unroll
    for (int j = 0; j < 6; ++j) A[i][j] = J[perm[i]][j];
    A[i][6] = -F[perm[i]];
  }
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double amax = fabs(A[k][k]);
#pragma unroll
    for (int j = k + 1; j < 6; ++j) amax = fabs(A[k][j]) > amax ? fabs(A[k][j]) : amax;
    ok = ok && (fabs(A[k][k]) > 1e-9 * amax);
    const double ip = rcp_f(A[k][k]);
#pragma unroll
    for (int r = k + 1; r < 6; ++r) {
      const double f = A[r][k] * ip;
#pragma unroll
      for (int j = k + 1; j < 7; ++j) A[r][j] = fma(-f, A[k][j], A[r][j]);
    }
  }
  if (!ok) return false;                                    // also NaN: reported as not converged (flags), like a zero pivot
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double s = A[i][6];
#pragma unroll
    for (int j = i + 1; j < 6; ++j) s = fma(-A[i][j], d[j], s);
    d[i] = s * rcp_f(A[i][i]);
  }
  return true;
}

// Newton on (theta, p23, p24, p33, p34, p44); returns converged
__host__ __device__ inline bool lqr5_newton(const Lqr5Par& P, Lqr5State& u, int max_it) {
  for (int it = 0; it < max_it; ++it) {
    const double C = u.C, S = u.S, sq = P.sq;
    const double x2 = u.p23 * P.i1, y2 = u.p24 * P.i2, x3 = u.p33 * P.i1, y3 = u.p34 * P.i2, x4 = u.p34 * P.i1, y4 = u.p44 * P.i2;
    const double iv = rcp_f(P.v), ia = rcp_f(P.a);
    const double p12 = (x2 * x2 + y2 * y2 - P.q3) * 0.5 * iv;
    const double p01 = sq * (C * x2 + S * y2) * iv;
    const double p02 = sq * (P.s1 * C * P.itp + C * x3 + S * y3) * ia;
    const double p13 = P.s1 * sq * S;
    const double p22 = (u.p23 * P.itp + x2 * x3 + y2 * y3 - P.v * p13) * ia;
    double F[6], J[6][6], d[6];
    F[0] = P.a * p12 - p13 * P.itp - sq * (S * x3 - C * y3);
    F[1] = 2.0 * (P.a * u.p23 - u.p33 * P.itp) - (x3 * x3 + y3 * y3) + P.q4;
    F[2] = p01 + P.b * p12 + P.s2 * sq * C * P.itv - sq * (S * x4 - C * y4);
    F[3] = -P.v * P.s2 * sq * C + p02 + P.b * p22 - u.p24 * P.itv - (x2 * x4 + y2 * y4);
    F[4] = P.a * u.p24 + P.s1 * sq * C + P.b * u.p23 - u.p34 * (P.itp + P.itv) - (x3 * x4 + y3 * y4);
    F[5] = 2.0 * (P.s2 * sq * S + P.b * u.p24 - u.p44 * P.itv) - (x4 * x4 + y4 * y4) + P.q5;
    // d/dtheta
    const double dp01 = sq * (C * y2 - S * x2) * iv, dp02 = sq * (C * y3 - S * x3 - P.s1 * S * P.itp) * ia, dp22 = -P.v * P.s1 * sq * C * ia;
    J[0][0] = -P.s1 * sq * C * P.itp - sq * (C * x3 + S * y3);
    J[1][0] = 0.0;
    J[2][0] = dp01 - P.s2 * sq * S * P.itv - sq * (C * x4 + S * y4);
    J[3][0] = P.v * P.s2 * sq * S + dp02 + P.b * dp22;
    J[4][0] = -P.s1 * sq * S;
    J[5][0] = 2.0 * P.s2 * sq * C;
    // d/dp23
    J[0][1] = P.a * x2 * P.i1 * iv; J[1][1] = 2.0 * P.a; J[2][1] = (sq * C + P.b * x2) * P.i1 * iv;
    J[3][1] = P.b * (P.itp + x3 * P.i1) * ia - x4 * P.i1; J[4][1] = P.b; J[5][1] = 0.0;
    // d/dp24
    J[0][2] = P.a * y2 * P.i2 * iv; J[1][2] = 0.0; J[2][2] = (sq * S + P.b * y2) * P.i2 * iv;
    J[3][2] = P.b * y3 * P.i2 * ia - P.itv - y4 * P.i2; J[4][2] = P.a; J[5][2] = 2.0 * P.b;
    // d/dp33
    J[0][3] = -sq * S * P.i1; J[1][3] = -2.0 * (P.itp + x3 * P.i1); J[2][3] = 0.0;
    J[3][3] = (sq * C + P.b * x2) * P.i1 * ia; J[4][3] = -x4 * P.i1; J[5][3] = 0.0;
    // d/dp34
    J[0][4] = sq * C * P.i2; J[1][4] = -2.0 * y3 * P.i2; J[2][4] = -sq * S * P.i1;
    J[3][4] = (sq * S + P.b * y2) * P.i2 * ia - x2 * P.i1; J[4][4] = -(P.itp + P.itv) - (x3 * P.i1 + y4 * P.i2); J[5][4] = -2.0 * x4 * P.i1;
    // d/dp44
    J[0][5] = 0.0; J[1][5] = 0.0; J[2][5] = sq * C * P.i2; J[3][5] = -y2 * P.i2; J[4][5] = -y3 * P.i2; J[5][5] = -2.0 * (P.itv + y4 * P.i2);
    if (!solve6(J, F, d)) return false;
    const double Cn = C - S * d[0], Sn = S + C * d[0];
    const double nrm = rsqrt_f(Cn * Cn + Sn * Sn);
    u.C = Cn * nrm; u.S = Sn * nrm;
    u.p23 += d[1]; u.p24 += d[2]; u.p33 += d[3]; u.p34 += d[4]; u.p44 += d[5];
    const double scale = fabs(u.p23) + fabs(u.p24) + fabs(u.p33) + fabs(u.p34) + fabs(u.p44);
    const double step = fabs(d[1]) + fabs(d[2]) + fabs(d[3]) + fabs(d[4]) + fabs(d[5]);
    if (fabs(d[0]) < 3e-8 && step < 3e-8 * scale) return true;       // quadratic convergence: error ~1e-15 after this step
  }
  return false;
}

// Warm / cold start logic and the gain rows in the PATH frame: Kp[10] = row-major 2x5 K' = [P_3. / (tau_phi r1) ; P_4. / (tau_v r2)].
// P must carry v, a, b, itp, itv, sq, q3, q4, q5, s1, s2, i1, i2.  Returns false when not even the cold start converged.
__host__ __device__ inline bool lqr5_gain(const Lqr5Par& P, double sr1, double sr2, double tau_phi, double tau_v, double r1, double r2,
                                          Lqr5State& st, double* Kp) {
  bool ok = false;
  if (st.p23 > 0.0) {                                                // warm start from the previous sample
    Lqr5State w = st;
    ok = lqr5_newton(P, w, 12) && w.S > 0.0 && w.p23 > 0.0;
    if (ok) st = w;
  }
  if (!ok) {                                                         // cold: the 3-state gain as the first guess
    const CareConst cc = care_const(P.sq, P.q3, sr1, sr2);
    double s3[kCareState] = {};
    CareSol c3;
    const double c1 = sr1 * rcp_f(P.a), e = P.b * c1;
    care_gain(cc, P.v, c1, e, ArrayState{s3}, true, c3);
    const double al3 = c3.al, be3 = c3.be;
    st.C = c3.C; st.S = c3.S;
    st.p23 = P.s1 * al3; st.p24 = P.s2 * be3;
    st.p33 = tau_phi * (P.a * st.p23 + 0.5 * P.q4);
    st.p44 = tau_v * (P.s2 * P.sq * st.S + P.b * st.p24 + 0.5 * P.q5);
    st.p34 = (P.a * st.p24 + P.s1 * P.sq * st.C + P.b * st.p23) * rcp_f(P.itp + P.itv);
    ok = lqr5_newton(P, st, 40);
  }
  // K' rows: P_3. / (tau_phi r1), P_4. / (tau_v r2)
  const double f1 = 1.0 / (tau_phi * r1), f2 = 1.0 / (tau_v * r2);
  Kp[0] = P.s1 * P.sq * st.C * f1; Kp[1] = P.s1 * P.sq * st.S * f1;
  Kp[5] = P.s2 * P.sq * st.S * f2; Kp[6] = -P.s2 * P.sq * st.C * f2;
  Kp[2] = st.p23 * f1; Kp[3] = st.p33 * f1; Kp[4] = st.p34 * f1;
  Kp[7] = st.p24 * f2; Kp[8] = st.p34 * f2; Kp[9] = st.p44 * f2;
  return ok;
}

}  // namespace d2dx
