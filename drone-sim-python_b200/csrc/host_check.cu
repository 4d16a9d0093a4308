// Host instances of the engine's Riccati reductions and planner solvers (test infrastructure, not part of libd2dx.so): the SAME
// source the kernels inline -- care_gain (d2dx_device.cuh), lqr5_gain (d2dx_lqr5.cuh), the DDP solvers (d2dx_ddp.cuh,
// d2dx_ddp_multi.cuh) -- compiled for the CPU, so that tests/test_care_math.py, test_ddp_cpu.py and test_ddp_multi_cpu.py can
// check them without a GPU.
#include <vector>

#include "d2dx_ddp_multi.cuh"
#include "d2dx_lqr5.cuh"

using namespace d2dx;

extern "C" {

static int care_gain_host(const double* qr4, double v, double phi, int cold, double* state9, double* K0) {
  d2dx_dfff_gains g;
  g.q_pos = qr4[0]; g.q_psi = qr4[1]; g.r_phi = qr4[2]; g.r_v = qr4[3];
  const CareConst cc = care_const(g);
  const double z = tan(phi), z2 = z * z, inv_va = 1.0 / v;
  const double c1 = cc.sr1 * (2.0 + z2) * rcp_f(kG * inv_va * (1.0 + z2));   // as make_ref forms them
  const double e = kG * inv_va * inv_va * z * c1;
  CareSol sol;
  const int res = care_gain(cc, v, c1, e, ArrayState{state9}, cold != 0, sol);
  K0[0] = cc.sq_isr1 * sol.C; K0[1] = cc.sq_isr1 * sol.S; K0[2] = sol.al * cc.isr1;   // make_ref's K1 at psi_ref = 0
  K0[3] = cc.sq_isr2 * sol.S; K0[4] = -cc.sq_isr2 * sol.C; K0[5] = sol.be * cc.isr2;
  return res;
}

// LQR gain of DFFFController.get (d2d/guidance.py:78-82) in the path frame (psi_ref = 0) at reference speed v and bank phi:
// K0[6] = row-major 2x3.  state9 (in/out): C, S, al, then the changes of theta at steps n, n-1, n-2 and those of al
// (d2dx_rollout_out.care_state's rows); cold != 0 ignores it.  Returns 2 when the straight-line step was accepted, 1 when
// the fallback loop converged, 0 when nothing did.
int d2dx_host_care_gain9(const double* qr4 /* q_pos, q_psi, r_phi, r_v */, double v, double phi, int cold, double* state9, double* K0) {
  return care_gain_host(qr4, v, phi, cold, state9, K0);
}

// The same with a 5-double state: C, S, al and the LAST change of theta and al only; the two older changes are taken equal
// to it, which makes the warm start a linear extrapolation.  Returns 1 when converged.
int d2dx_host_care_gain(const double* qr4, double v, double phi, int cold, double* state5, double* K0) {
  double s9[9] = {state5[0], state5[1], state5[2], state5[3], state5[3], state5[3], state5[4], state5[4], state5[4]};
  const int res = care_gain_host(qr4, v, phi, cold, s9, K0);
  state5[0] = s9[0]; state5[1] = s9[1]; state5[2] = s9[2]; state5[3] = s9[3]; state5[4] = s9[6];
  return res != CARE_FAILED ? 1 : 0;
}

// 5-state LQR gain of DiffController.ComputeGain (Controllers.py:159-186) in the path frame: Kp[10] = row-major 2x5.
// state7 (in/out): C, S, p23, p24, p33, p34, p44 (p23 <= 0 = cold).  Returns 1 when converged.
int d2dx_host_lqr5_gain(const double* q5, const double* r2, double v, double phi, double tau_phi, double tau_v, double* state7, double* Kp) {
  const double z = tan(phi), z2 = z * z, inv_va = 1.0 / v;
  Lqr5Par P;
  P.v = v;
  P.a = kG * inv_va * (1.0 + z2) * rcp_f(2.0 + z2);
  P.b = kG * inv_va * inv_va * z;
  P.itp = 1.0 / tau_phi; P.itv = 1.0 / tau_v;
  P.sq = ::sqrt(q5[0]); P.q3 = q5[2]; P.q4 = q5[3]; P.q5 = q5[4];
  const double sr1 = ::sqrt(r2[0]), sr2 = ::sqrt(r2[1]);
  P.s1 = tau_phi * sr1; P.s2 = tau_v * sr2; P.i1 = 1.0 / P.s1; P.i2 = 1.0 / P.s2;
  Lqr5State st = {state7[0], state7[1], state7[2], state7[3], state7[4], state7[5], state7[6]};
  const bool ok = lqr5_gain(P, sr1, sr2, tau_phi, tau_v, r2[0], r2[1], st, Kp);
  state7[0] = st.C; state7[1] = st.S; state7[2] = st.p23; state7[3] = st.p24; state7[4] = st.p33; state7[5] = st.p34; state7[6] = st.p44;
  return ok ? 1 : 0;
}

static d2dx_ddp_options options_or_default(const d2dx_ddp_options* o) {
  d2dx_ddp_options opt;
  if (o) return *o;
  opt.max_iter = 400; opt.max_outer = 30; opt.max_inner = 40; opt.ls_max = 12; opt.ctol = 1e-8; opt.rel_tol = 1e-10; opt.abs_tol = 1e-14;
  opt.rho0 = 10.0; opt.rho_growth = 10.0; opt.rho_max = 1e8; opt.mu0 = 1e-6; opt.mu_min = 1e-8; opt.mu_max = 1e10; opt.mu_factor = 1.6; opt.reg_mode = 0; opt.min_solved = 0;
  return opt;
}

// The planner's second-order solver (d2dx_ddp.cuh) for ONE problem on the CPU: the code of ddp_solve_kernel's thread.
// prob9: N, h, wx, wy, vsp, kv, kb, kobs, obs_kind (weights already normalised as DdpProblem wants them); obs[n_obs][3];
// bounds4; box5 or NULL (x_lo, x_hi, y_lo, y_hi, w_box normalised); z0[3], zt[3]; u[2][N] in/out; xs[3][N] out; info[8] out.
int d2dx_host_ddp_solve(const double* prob9, int n_obs, const double* obs, const double* bounds4, const double* box5, const double* z0,
                        const double* zt, const d2dx_ddp_options* o, double* u, double* xs, double* info) {
  DdpProblem P;
  P.N = (int)prob9[0]; P.h = prob9[1]; P.wx = prob9[2]; P.wy = prob9[3]; P.vsp = prob9[4]; P.kv = prob9[5]; P.kb = prob9[6];
  P.kobs = prob9[7]; P.obs_kind = (int)prob9[8]; P.n_obs = n_obs;
  for (int k = 0; k < n_obs; ++k) { P.obs[k][0] = obs[3 * k]; P.obs[k][1] = obs[3 * k + 1]; P.obs[k][2] = obs[3 * k + 2]; }
  P.phi_lo = bounds4[0]; P.phi_hi = bounds4[1]; P.v_lo = bounds4[2]; P.v_hi = bounds4[3];
  P.has_box = box5 != nullptr;
  if (box5) { P.x_lo = box5[0]; P.x_hi = box5[1]; P.y_lo = box5[2]; P.y_hi = box5[3]; P.w_box = box5[4]; }
  else { P.x_lo = P.y_lo = -1e300; P.x_hi = P.y_hi = 1e300; P.w_box = 0.0; }
  const int N = P.N;
  std::vector<double> work(18 * (size_t)N);
  DdpWork W;
  W.N = N; W.stride = 1;
  W.u = work.data(); W.z = W.u + 2 * N; W.un = W.z + 3 * N; W.zn = W.un + 2 * N; W.k = W.zn + 3 * N; W.K = W.k + 2 * N;
  for (int i = 0; i < 2 * N; ++i) W.u[i] = u[i];
  const d2dx_ddp_options opt = options_or_default(o);
  DdpSerial sweeps(P, W, zt);
  const DdpResult r = ddp_solve(sweeps, z0, opt);
  const double* us = (r.swaps & 1) ? W.un : W.u;
  const double* zs = (r.swaps & 1) ? W.zn : W.z;
  for (int i = 0; i < 2 * N; ++i) u[i] = us[i];
  for (int i = 0; i < 3 * N; ++i) xs[i] = zs[i];
  info[0] = r.flag; info[1] = r.iterations; info[2] = r.outer; info[3] = r.cost; info[4] = r.cmax; info[5] = r.lagr; info[6] = r.mu; info[7] = r.rho;
  return 0;
}

// The coupled multi-aircraft solver (d2dx_ddp_multi.cuh) for ONE problem on the CPU, with the arguments of d2dx_ddp_multi_solve for
// P = 1: p0, p1 [3][n_ac]; u [2][n_ac][N] in/out; xs [3][n_ac][N] out; info[8] out; lam [3][n_ac] out or NULL.  Returns 1 for a
// request d2dx_ddp_multi_solve refuses.
int d2dx_host_ddp_multi_solve(const d2dx_colloc_problem* p, const double* bounds4, const double* box5, const double* p0, const double* p1,
                              const d2dx_ddp_options* o, double* u, double* xs, double* info, double* lam) {
  DdpmProblem M;
  const d2dx_ddp_options opt = options_or_default(o);
  if (ddpm_problem_from(p, bounds4, box5, M) || (opt.reg_mode != 0 && M.n > 1)) return 1;
  const int n = M.n, N = M.a.N;
  std::vector<double> work(DdpmWork::doubles(n, N)), scratch(DdpmNode::doubles(n)), pre(n * kDdpPre + 3 * n);
  std::vector<int> iscratch(DdpmNode::ints(n));
  DdpmWork W;
  W.carve(work.data(), n, N);
  for (int j = 0; j < 2; ++j)
    for (int a = 0; a < n; ++a)
      for (int i = 0; i < N; ++i) W.u[(long)i * 2 * n + 2 * a + j] = u[((long)j * n + a) * N + i];
  double z0[3 * kDdpmMaxAc], zt[3 * kDdpmMaxAc], lm[3 * kDdpmMaxAc];
  for (int k = 0; k < 3; ++k)
    for (int a = 0; a < n; ++a) { z0[3 * a + k] = p0[k * n + a]; zt[3 * a + k] = p1[k * n + a]; }
  DdpmSerial sweeps(M, W, zt, scratch.data(), iscratch.data(), pre.data());
  const DdpResult r = ddp_solve(sweeps, z0, opt, lm);
  const double* us = (r.swaps & 1) ? W.un : W.u;
  const double* zs = (r.swaps & 1) ? W.zn : W.z;
  for (int a = 0; a < n; ++a)
    for (int i = 0; i < N; ++i) {
      for (int j = 0; j < 2; ++j) u[((long)j * n + a) * N + i] = us[(long)i * 2 * n + 2 * a + j];
      for (int k = 0; k < 3; ++k) xs[((long)k * n + a) * N + i] = zs[(long)i * 3 * n + 3 * a + k];
    }
  if (lam)
    for (int k = 0; k < 3; ++k)
      for (int a = 0; a < n; ++a) lam[k * n + a] = lm[3 * a + k];
  info[0] = r.flag; info[1] = r.iterations; info[2] = r.outer; info[3] = r.cost; info[4] = r.cmax; info[5] = r.lagr; info[6] = r.mu; info[7] = r.rho;
  return 0;
}

// The box QP of a node of the coupled solver: minimiser x[n] of 1/2 x^T H x + g^T x over lo <= x <= hi (H[n][n] row-major, positive
// definite, n <= 20), free[n] = 1 where the component is not held at a bound.  Returns 1 when a free block was not definite.
int d2dx_host_box_qp(int n, const double* H, const double* g, const double* lo, const double* hi, double* x, int* free_) {
  if (n < 1 || n > 2 * kDdpmMaxAc) return 1;
  std::vector<double> L((size_t)n * n);
  int fi[2 * kDdpmMaxAc], nf;
  return ddpm_box_qp(n, H, n, g, lo, hi, x, free_, fi, nf, L.data()) ? 0 : 1;
}

}  // extern "C"
