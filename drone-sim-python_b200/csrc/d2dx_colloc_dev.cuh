// Device-side pieces shared by the collocation kernels (d2dx_colloc.cu, d2dx_peer.cu): the per-(aircraft, node)
// residual / Jacobian / input-cost work and the obstacle and collision terms of the planner cost classes.
// Reference: EoM d2d/opty_utils.py:38-50, cost classes d2d/opty_utils.py:55-165, d2d/multiopty_utils.py:29-174.
#pragma once
#include "d2dx_device.cuh"

namespace d2dx {

struct CollocArgs {
  d2dx_colloc_problem p;
  int n_prob, layout;
  uint32_t what;
  const double* free_;
  double *res, *jac, *cost, *grad, *scratch;   // scratch: [kTicketDoubles of int32 tickets][per-block cost partials]
  int TN, APP, ntiles;        // nodes per tile, aircraft per pass, tiles per problem
  int ticket_mode;            // 1: the last block of a problem (atomic ticket) finishes the cost in this kernel;
                              // 0: per-block partials only, colloc_cost_kernel finishes (large batches: no fence in the hot kernel)
  int nparts;                 // cost partials per problem
  int n_free, n_con;          // per problem (fit 32 bits: 5 n_ac N)
  long nnz;
  // host-computed constants (IEEE divisions done once on the host instead of ~40 instructions each per thread)
  double ih;                  // 1 / h
  double sN, norm_in;         // obj_scale / N,  sN / in_div
  double col_kr, nkr2, cw;    // k / r,  -(k/r)^2,  kcol sN (-2) (exact_grad ? (k/r)^2 : 1): weight of es * dx in the gradient
};

inline void colloc_constants(CollocArgs& a) {
  const d2dx_colloc_problem& P = a.p;
  a.ih = 1.0 / P.h;
  a.sN = P.obj_scale / P.N; a.norm_in = a.sN / P.in_div;
  a.col_kr = P.kcol_k / P.rcol; a.nkr2 = -(a.col_kr * a.col_kr);
  a.cw = P.kcol * a.sN * -2.0 * (P.exact_grad ? a.col_kr * a.col_kr : 1.0);
}

constexpr int kTicketDoubles = 32;   // 64 int32 tickets at the head of the caller's scratch buffer

__device__ __forceinline__ bool enabled(double k) { return (k == k) && k != 0.0; }

// CostObstacle on (x, y) (opty_utils.py:99-134, multiopty_utils.py:74-106): adds the unweighted penalty to s_obs and the
// reference-style gradient (no (k/r)^2 unless exact_grad) to (gx, gy)
__device__ __forceinline__ void obstacle_terms(const d2dx_colloc_problem& P, double sN, double x, double y, double& s_obs,
                                               double& gx, double& gy) {
  for (int o = 0; o < P.n_obs; ++o) {
    const double dx = x - P.obs[o][0], dy = y - P.obs[o][1], r = P.obs[o][2];
    double es, f = 1.0;
    if (P.obs_kind == 0) es = clip(exp(r * r - (dx * dx + dy * dy)), 0.0, 1e3);
    else {
      const double kr = 2.0 / r, ux = dx * kr, uy = dy * kr;
      es = fm::exp_neg(-(ux * ux + uy * uy));
      if (P.exact_grad) f = (2.0 / r) * (2.0 / r);
    }
    s_obs += es;
    gx += P.kobs * (sN * -2.0 * dx * es) * f;
    gy += P.kobs * (sN * -2.0 * dy * es) * f;
  }
}

// inputs of one (aircraft, node) beyond its position: heading, bank, speed and the previous node's x, y, psi
struct NodeIn { double psi, phi, v, xp, yp, pp; };
// offsets of the node's x, bank and speed entries inside one problem's free vector (5 n_ac N entries: they fit 32 bits)
struct NodeOff { int ox, ophi, ov; };

__device__ __forceinline__ NodeOff colloc_offsets(const d2dx_colloc_problem& P, int a_l, int i) {
  const int N = P.N, n_ac = P.n_ac, n = 3 * n_ac;
  const int bphi = P.perm_phi ? P.perm_phi[a_l] : a_l;
  const int bv = P.perm_v ? P.perm_v[a_l] : n_ac + a_l;
  NodeOff o;
  o.ox = 3 * a_l * N + i; o.ophi = (n + bphi) * N + i; o.ov = (n + bv) * N + i;
  return o;
}

__device__ __forceinline__ NodeIn colloc_load(const CollocArgs& a, const double* __restrict__ fr, const NodeOff& o, int i) {
  const int N = a.p.N;
  NodeIn in;
  in.psi = fr[o.ox + 2 * N]; in.phi = fr[o.ophi]; in.v = fr[o.ov];
  in.xp = in.yp = in.pp = 0.0;
  if ((a.what & D2DX_EVAL_RESIDUAL) && i >= 1) { in.xp = fr[o.ox - 1]; in.yp = fr[o.ox + N - 1]; in.pp = fr[o.ox + 2 * N - 1]; }
  return in;
}

// element `off` of problem `prob` in an output array with `per` elements per problem.  IDX32: the whole batch of that array has
// fewer than 2^31 elements (the launcher checks), so one 32-bit multiply-add and one widening add replace the 64-bit index chain
template <bool IDX32>
__device__ __forceinline__ double* colloc_out(double* base, int prob, long per, int off) {
  if (IDX32) return base + static_cast<unsigned>(prob * static_cast<int>(per) + off);
  return base + ((size_t)prob * per + off);
}
// One (aircraft a_l, node i < N) of problem `prob`: backward-Euler defects (equation-major, opty layout), the 12 structural
// Jacobian entries (compact or opty-dense), the input cost sums and every gradient entry of the node; (gx, gy) = the
// position gradient the caller accumulated (obstacles, collisions; STORE_XY = false leaves those two entries to the caller).
template <bool STORE_XY = true, bool IDX32 = false>
__device__ __forceinline__ void colloc_node_in(const CollocArgs& a, int prob, int a_l, int i, double x, double y, const NodeIn& in,
                                               const NodeOff& o, double gx, double gy, bool want_cg, double& s_v, double& s_phi) {
  const d2dx_colloc_problem& P = a.p;
  const int N = P.N, n_ac = P.n_ac, n = 3 * n_ac;
  const int ox = o.ox, ophi = o.ophi, ov = o.ov, oy = ox + N, ops = oy + N;
  const double psi = in.psi, phi = in.phi, v = in.v;

  if ((a.what & (D2DX_EVAL_RESIDUAL | D2DX_EVAL_JAC)) && i >= 1) {
    const double ih = a.ih;
    const int nm1 = N - 1;
    double s, c, sp, cp;
    sincos_any(psi, s, c);
    sincos_any(phi, sp, cp);
    const double iv = rcp_f(v);
    const double tn = sp * rcp_f(cp);            // tan(phi)
    const double gtv = kG * tn * iv;             // g tan(phi) / v
    if (a.what & D2DX_EVAL_RESIDUAL) {           // equation-major, node-minor (opty layout)
      double* r = colloc_out<IDX32>(a.res, prob, a.n_con, 3 * a_l * (N - 1) + (i - 1));
      r[0] = (x - in.xp) * ih - v * c + P.wind[0];
      r[nm1] = (y - in.yp) * ih - v * s + P.wind[1];
      r[2 * nm1] = (psi - in.pp) * ih - gtv;
    }
    if (a.what & D2DX_EVAL_JAC) {
      const double j[12] = {ih, v * s, -ih, -c, ih, -v * c, -ih, -s, ih, -ih, -kG * fma(tn, tn, 1.0) * iv, gtv * iv};
      if (a.layout == D2DX_JAC_COMPACT) {        // [n_ac][12][N-1]: coalesced along the node
        double* jo = colloc_out<IDX32>(a.jac, prob, a.nnz, a_l * 12 * (N - 1) + (i - 1));
#pragma unroll
        for (int k = 0; k < 12; ++k) jo[k * nm1] = j[k];
      } else {                                   // opty-dense: [(N-1)][3 n_ac][8 n_ac]
        const int bphi = P.perm_phi ? P.perm_phi[a_l] : a_l, bv = P.perm_v ? P.perm_v[a_l] : n_ac + a_l;
        const int q = 2 * n_ac, W = 2 * n + q;
        double* jo = a.jac + (size_t)prob * a.nnz + ((size_t)(i - 1) * n + 3 * a_l) * W;
        const int cx = 3 * a_l, cp_ = n + 3 * a_l, cphi = 2 * n + bphi, cv = 2 * n + bv;
        if (n_ac == 1) {                         // 24 contiguous values per node, structural zeros included
          jo[0] = j[0]; jo[1] = 0.0; jo[2] = j[1]; jo[3] = j[2]; jo[4] = 0.0; jo[5] = 0.0; jo[6] = 0.0; jo[7] = j[3];
          jo[8] = 0.0; jo[9] = j[4]; jo[10] = j[5]; jo[11] = 0.0; jo[12] = j[6]; jo[13] = 0.0; jo[14] = 0.0; jo[15] = j[7];
          jo[16] = 0.0; jo[17] = 0.0; jo[18] = j[8]; jo[19] = 0.0; jo[20] = 0.0; jo[21] = j[9]; jo[22] = j[10]; jo[23] = j[11];
        } else {                                 // non-zeros only; zeros were laid down by d2dx_colloc_init_dense
          jo[cx] = j[0]; jo[cx + 2] = j[1]; jo[cp_] = j[2]; jo[cv] = j[3];
          jo[W + cx + 1] = j[4]; jo[W + cx + 2] = j[5]; jo[W + cp_ + 1] = j[6]; jo[W + cv] = j[7];
          jo[2 * W + cx + 2] = j[8]; jo[2 * W + cp_ + 2] = j[9]; jo[2 * W + cphi] = j[10]; jo[2 * W + cv] = j[11];
        }
      }
    }
  }
  if (want_cg) {
    const double dv = v - P.vsp;
    s_v += dv * dv; s_phi += phi * phi;
    if (a.what & D2DX_EVAL_GRAD) {
      const double norm_in = a.norm_in;
      double* go = colloc_out<IDX32>(a.grad, prob, a.n_free, 0);
      if (STORE_XY) { go[ox] = gx; go[oy] = gy; }
      go[ops] = 0.0;
      go[ophi] = (P.kbank * 2.0 * phi) * norm_in;
      go[ov] = (P.kvel * 2.0 * dv) * norm_in;
    }
  }
}

template <bool STORE_XY = true, bool IDX32 = false>
__device__ __forceinline__ void colloc_node(const CollocArgs& a, const double* __restrict__ fr, int prob, int a_l, int i,
                                            double x, double y, double gx, double gy, bool want_cg, double& s_v, double& s_phi) {
  const NodeOff o = colloc_offsets(a.p, a_l, i);
  const NodeIn in = colloc_load(a, fr, o, i);
  colloc_node_in<STORE_XY, IDX32>(a, prob, a_l, i, x, y, in, o, gx, gy, want_cg, s_v, s_phi);
}

// cost of one problem from the four summed partials (CostComposit, multiopty_utils.py:156-174 / opty_utils.py:147-165)
__device__ __forceinline__ double colloc_cost_from_sums(const CollocArgs& a, const double* t4, bool use_obs, bool use_col) {
  const d2dx_colloc_problem& P = a.p;
  const double sN = a.sN;
  double c = a.norm_in * (P.kvel * t4[0] + P.kbank * t4[1]);
  if (use_obs) c += P.kobs * (sN * t4[2]);
  if (use_col) c += P.kcol * (sN * t4[3]);
  return c;
}

}  // namespace d2dx
