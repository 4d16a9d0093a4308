// Direct-collocation evaluation: backward-Euler defects of the d2d EoM (d2d/opty_utils.py:38-50), their
// sparse Jacobian, the planner cost and its gradient, over problems x aircraft x nodes.
// Three kernels share the per-(aircraft, node) work of d2dx_colloc_dev.cuh:
//   colloc_kernel<false>   residual + Jacobian + input cost + gradient: the lean HBM-bound path (64 registers);
//   colloc_kernel<true>    + obstacles, the reference's (0,1)-only collision term, ordered all-pairs loops (all-pairs
//                          problems past colloc_pairs_kernel's shared-memory budget or 32-bit output offsets);
//   colloc_pairs_kernel    all-pairs collision of one unsharded problem: one warp = one aircraft x 32 nodes, every unordered
//                          pair evaluated once, its exponential handed to the partner through a write-once shared-memory slot.
// Every global load and store is coalesced along the node index.
#include <type_traits>

#include "d2dx_colloc_dev.cuh"
#include "d2dx_host.h"

namespace d2dx {

constexpr int kCollocThreads = 128;
constexpr int kMaxTickets = 64;
constexpr int kPairWarps = 8;       // warps per block of colloc_pairs_kernel (aircraft w, w + 8, ... per warp)

// finishes the cost of problem `prob`: per-block partials -> scratch; in ticket mode the last block of the problem sums
// them in a fixed order (deterministic) and writes cost[prob].  Called by ONE warp of the block with its four block sums.
__device__ __forceinline__ void cost_finish(const CollocArgs& a, int prob, int part_idx, const double* v4, bool use_obs,
                                            bool use_col, int lane) {
  double* parts = a.scratch + kTicketDoubles + (size_t)prob * a.nparts * 4;
  if (lane == 0) { double* p = parts + part_idx * 4; p[0] = v4[0]; p[1] = v4[1]; p[2] = v4[2]; p[3] = v4[3]; }
  if (!a.ticket_mode) return;
  int32_t* tickets = reinterpret_cast<int32_t*>(a.scratch);
  int last = 0;
  if (lane == 0) {
    __threadfence();
    last = atomicAdd(&tickets[prob], 1) == a.nparts - 1;
  }
  last = __shfl_sync(0xffffffffu, last, 0);
  if (last) {
    __threadfence();
    double t4[4] = {0.0, 0.0, 0.0, 0.0};
    for (int t = lane; t < a.nparts; t += 32)
      for (int k = 0; k < 4; ++k) t4[k] += __ldcg(parts + t * 4 + k);
    for (int k = 0; k < 4; ++k) t4[k] = warp_sum(t4[k]);
    if (lane == 0) {
      a.cost[prob] = colloc_cost_from_sums(a, t4, use_obs, use_col);
      tickets[prob] = 0;
    }
  }
}

// EXTRA = obstacle and / or collision terms present (exp, shared-memory partner loop): obstacles, the (0,1) pair mode and
// all-pairs problems colloc_pairs_kernel does not take.  The plain instantiation is the lean HBM-bound path (residual +
// Jacobian + input cost + gradient) and is held to 64 registers for occupancy.
// One thread = one (aircraft, node); a block covers a tile of TN nodes for APP aircraft per pass.
template <bool EXTRA>
__global__ void __launch_bounds__(kCollocThreads, EXTRA ? 5 : 8) colloc_kernel(const __grid_constant__ CollocArgs a) {
  extern __shared__ double spos[];                 // [n_ac][2][TN] positions of every aircraft on this tile
  __shared__ double sred[kCollocThreads / 32][4];
  const d2dx_colloc_problem& P = a.p;
  const int N = P.N, n_ac = P.n_ac, TN = a.TN;
  const int tid = threadIdx.x;
  const int tile = blockIdx.x % a.ntiles, prob = blockIdx.x / a.ntiles;
  const int il = tid % TN, al = tid / TN;
  const int i = tile * TN + il;
  const double* fr = a.free_ + (size_t)prob * a.n_free;
  const bool want_cg = (a.what & (D2DX_EVAL_COST | D2DX_EVAL_GRAD)) != 0;
  const bool use_col = EXTRA && want_cg && enabled(P.kcol) && n_ac > 1;
  const bool use_obs = EXTRA && want_cg && enabled(P.kobs) && P.n_obs > 0;

  if (use_col) {                                   // stage the tile's positions of ALL aircraft
    for (int idx = tid; idx < n_ac * TN; idx += kCollocThreads) {
      const int g = idx / TN, ii = idx - g * TN, node = tile * TN + ii;
      double x = 0.0, y = 0.0;
      if (node < N) { x = fr[(3 * g) * N + node]; y = fr[(3 * g + 1) * N + node]; }
      spos[(g * 2) * TN + ii] = x; spos[(g * 2 + 1) * TN + ii] = y;
    }
    __syncthreads();
  }

  const double sN = a.sN;                          // _p.obj_scale/_p.num_nodes
  const double col_kr = a.col_kr;                  // (k/r): one multiplication per pair component instead of dx / r * k
  double s_v = 0.0, s_phi = 0.0, s_obs = 0.0, s_col = 0.0;

  for (int a_l = al; a_l < n_ac; a_l += a.APP) {
    if (i >= N) break;
    const int ox = 3 * a_l * N + i;
    const double x = fr[ox], y = fr[ox + N];
    double gx = 0.0, gy = 0.0;
    if (EXTRA && want_cg) {
      if (use_obs && a_l == 0) obstacle_terms(P, sN, x, y, s_obs, gx, gy);   // CostObstacle acts on aircraft 0 only (multiopty_utils.py:74)
      if (use_col) {                               // CostCollision (multiopty_utils.py:120-153), partners from shared memory
        const double cw = a.cw;
        const int b_lo = P.col_all_pairs ? 0 : (a_l == 0 ? 1 : 0);
        const int b_hi = P.col_all_pairs ? n_ac : (a_l == 0 ? 2 : (a_l == 1 ? 1 : 0));
        const double* sp = spos + il;
        for (int b = b_lo; b < b_hi; ++b) {
          if (b == a_l) continue;
          const double dx = x - sp[(b * 2) * TN], dy = y - sp[(b * 2 + 1) * TN];
          const double ux = dx * col_kr, uy = dy * col_kr;
          const double es = fm::exp_neg(-(ux * ux + uy * uy));
          if (a_l < b) s_col += es;                // each pair counted once, at its lower-index member
          const double w = cw * es;
          gx = fma(w, dx, gx); gy = fma(w, dy, gy);
        }
      }
    }
    colloc_node(a, fr, prob, a_l, i, x, y, gx, gy, want_cg, s_v, s_phi);
  }

  // instance constraints (06_optyplan.py:46-49) and their unit Jacobian entries: first tile of each problem
  if (tile == 0) {
    for (int k = tid; k < P.n_inst; k += kCollocThreads) {
      if (a.what & D2DX_EVAL_RESIDUAL)
        a.res[(size_t)prob * a.n_con + 3 * n_ac * (N - 1) + k] = fr[P.inst_var[k] * N + P.inst_node[k]] - P.inst_val[k];
      if (a.what & D2DX_EVAL_JAC) a.jac[(size_t)prob * a.nnz + (a.nnz - P.n_inst) + k] = 1.0;
    }
  }

  if (a.what & D2DX_EVAL_COST) {                   // deterministic: warp shuffles -> block sum in warp order -> per-block partial
    const double v4[4] = {warp_sum(s_v), warp_sum(s_phi), warp_sum(s_obs), warp_sum(s_col)};
    const int lane = tid & 31, w = tid >> 5;
    if (lane == 0) { sred[w][0] = v4[0]; sred[w][1] = v4[1]; sred[w][2] = v4[2]; sred[w][3] = v4[3]; }
    __syncthreads();
    if (w == 0) {
      double b4[4] = {0.0, 0.0, 0.0, 0.0};
      for (int q = 0; q < kCollocThreads / 32; ++q) { b4[0] += sred[q][0]; b4[1] += sred[q][1]; b4[2] += sred[q][2]; b4[3] += sred[q][3]; }
      cost_finish(a, prob, tile, b4, use_obs, use_col, lane);
    }
  }
}

// All-pairs collision mode of one unsharded problem (the generalisation of CostCollision, multiopty_utils.py:120-153, to
// every pair; SURVEY D11).  Block = one 32-node tile of one problem; warp w owns aircraft w, w + 8, ...; lanes = nodes.
//   phase 0  stage x, y of every aircraft (stored twice, at a and a + n, so that partner a +- k needs no modulo);
//   phase A  aircraft a evaluates its pairs (a, a + k), k = 1 .. n/2 (the antipodal round of an even n only from the lower
//            half): own-side gradient in registers, exp value into the write-once slot sE[k-1][a];
//   phase B  aircraft a collects the rounds in which it was the partner (slot sE[k-1][a - k]), then does the node's
//            residual / Jacobian / input-cost work and writes the whole gradient row.
// Two block barriers, no read-modify-write in shared memory, every sum in a fixed order.
// REGS: every warp owns at most two aircraft (n_ac <= 16): their phase-A gradients wait in registers, not in shared memory
// (49 KB per block and 64 registers: four resident blocks = 32 warps per SM instead of 24).
// NAC > 0: the aircraft count is a compile-time constant with NAC = 2 kPairWarps (C4's 16 aircraft): every warp owns aircraft w
// of the lower half and w + NAC / 2 of the upper half, the round counts of both phases are constants, the pair loops unroll
// completely and every shared-memory access of a pair is base + immediate (no pointer or counter arithmetic per pair).
template <bool REGS, int NAC = 0>
__global__ void __launch_bounds__(kPairWarps * 32, REGS ? 4 : 3) colloc_pairs_kernel(const __grid_constant__ CollocArgs a) {
  extern __shared__ double sm[];
  const d2dx_colloc_problem& P = a.p;
  const int N = P.N, n = NAC ? NAC : P.n_ac, half = n / 2;
  const bool even = (n & 1) == 0;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, W = NAC ? kPairWarps : blockDim.x >> 5;
  // grid (tiles, problems); one-dimensional (tile fastest) only beyond 65535 problems: no integer division per thread
  const bool grid2 = gridDim.x == (unsigned)a.ntiles;
  const int tile = grid2 ? blockIdx.x : blockIdx.x % a.ntiles, prob = grid2 ? blockIdx.y : blockIdx.x / a.ntiles;
  const int i = tile * 32 + lane;
  const bool valid = i < N;
  const double* fr = a.free_ + (size_t)prob * a.n_free;
  // positions: [2n rows of aircraft a and a + n][x, y][1 + 32]: column 0 of a row is the node BEFORE the tile (the backward
  // difference of node 0 needs it), so the node work reads its previous node from shared memory, not from DRAM again
  constexpr int R = 33;
  double* spos = sm + 1 + lane;
  double* sE = sm + 2 * n * 2 * R + lane;          // [half][n][32]
  double* sg = sE + half * n * 32;                 // [n][2][32]  own-side position gradient of phase A (!REGS)
  double* sred = sm + (2 * n * 2 * R + half * n * 32 + (REGS ? 0 : n * 64));   // [W][4]
  const bool use_obs = enabled(P.kobs) && P.n_obs > 0;

  // heading, bank and speed of a node are requested ahead of their use -- as L1 prefetches, which hold no registers (keeping the
  // values live across phase B cost 40 B of spills at the 64-register budget and 5 % of the launch time)
  auto prefetch = [&](int a_l) {
    const NodeOff o = colloc_offsets(P, a_l, i);
    asm volatile("prefetch.global.L1 [%0];" ::"l"(fr + o.ox + 2 * N));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(fr + o.ophi));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(fr + o.ov));
  };
  for (int g = w; g < n; g += W) {
    double x = 0.0, y = 0.0;
    if (valid) { x = fr[(3 * g) * N + i]; y = fr[(3 * g + 1) * N + i]; if (REGS) prefetch(g); }
    spos[(g * 2) * R] = x; spos[(g * 2 + 1) * R] = y;
    spos[((g + n) * 2) * R] = x; spos[((g + n) * 2 + 1) * R] = y;
  }
  {                                                // halo column of this warp's rows: lane q -> aircraft w + (q / 2) W, component q % 2
    const int g = w + (lane >> 1) * W, c = lane & 1, ih = tile * 32 - 1;
    if (g < n) {
      const double hv = ih >= 0 ? fr[(3 * g + c) * N + ih] : 0.0;
      sm[(g * 2 + c) * R] = hv; sm[((g + n) * 2 + c) * R] = hv;
    }
  }
  __syncthreads();

  const double sN = a.sN, nkr2 = a.nkr2, cw = a.cw;
  double s_v = 0.0, s_phi = 0.0, s_obs = 0.0, s_col = 0.0;

  // `upper` (a std::bool_constant) tells the NAC instantiation which half a_l is in; the generic one ignores it
  auto phase_a = [&](int a_l, double& gx, double& gy, auto upper) {
    const double* pa = spos + (a_l * 2) * R;
    const double xa = pa[0], ya = pa[R];
    gx = 0.0; gy = 0.0;
    if (use_obs && a_l == 0 && valid) obstacle_terms(P, sN, xa, ya, s_obs, gx, gy);
    if constexpr (NAC > 0) {
      constexpr int kmax = (NAC % 2 == 0 && decltype(upper)::value) ? NAC / 2 - 1 : NAC / 2;
      double* e = sE + a_l * 32;
#pragma unroll
      for (int k = 1; k <= kmax; ++k) {
        const double dx = xa - pa[k * 2 * R], dy = ya - pa[k * 2 * R + R];
        const double es = fm::exp_neg(nkr2 * fma(dx, dx, dy * dy));
        e[(k - 1) * NAC * 32] = es;
        s_col += es;
        const double wgt = cw * es;
        gx = fma(wgt, dx, gx); gy = fma(wgt, dy, gy);
      }
      return;
    }
    const int kmax = (even && a_l >= half) ? half - 1 : half;
    const double* pb = pa + 2 * R;                 // partner a_l + 1
    double* e = sE + a_l * 32;
#pragma unroll 4
    for (int k = 1; k <= kmax; ++k) {
      const double dx = xa - pb[0], dy = ya - pb[R];
      const double es = fm::exp_neg(nkr2 * fma(dx, dx, dy * dy));
      *e = es;
      s_col += es;
      const double wgt = cw * es;
      gx = fma(wgt, dx, gx); gy = fma(wgt, dy, gy);
      pb += 2 * R; e += n * 32;
    }
  };
  auto phase_b = [&](int a_l, double gx, double gy, auto upper) {
    const double* pa = spos + ((a_l + n) * 2) * R;
    const double xa = pa[0], ya = pa[R];
    if constexpr (NAC > 0) {
      constexpr bool up = decltype(upper)::value;
      constexpr int kmax = (NAC % 2 == 0 && !up) ? NAC / 2 - 1 : NAC / 2;
      // slot of round k: sE[(k-1) n + a_l - k], n entries further when a_l - k wraps below 0 -- never for the upper half
      // (a_l >= NAC / 2 >= k), one select per round for the lower half
      const double* pe = sE + (a_l - 1) * 32;
#pragma unroll
      for (int k = 1; k <= kmax; ++k) {
        const double* q = (!up && k > a_l) ? pe + NAC * 32 : pe;
        const double wgt = cw * q[(k - 1) * (NAC - 1) * 32];
        gx = fma(wgt, xa - pa[-k * 2 * R], gx); gy = fma(wgt, ya - pa[-k * 2 * R + R], gy);
      }
    } else {
    const int kmax = (even && a_l < half) ? half - 1 : half;
    const double* pb = pa - 2 * R;                 // partner a_l - 1 (upper copy: no wrap)
    // the slot of round k was written by aircraft a_l - k (mod n): sE[(k-1) n + a_l - k] while a_l - k >= 0, n entries
    // further once it wraps -- two runs with the same constant stride instead of a modulo per pair
    const int k1 = kmax < a_l ? kmax : a_l;
    const int stride = (n - 1) * 32;
    const double* pe = sE + (a_l - 1) * 32;
#pragma unroll 4
    for (int k = 1; k <= k1; ++k, pe += stride, pb -= 2 * R) {
      const double wgt = cw * pe[0];
      gx = fma(wgt, xa - pb[0], gx); gy = fma(wgt, ya - pb[R], gy);
    }
    pe += n * 32;
#pragma unroll 4
    for (int k = k1 + 1; k <= kmax; ++k, pe += stride, pb -= 2 * R) {
      const double wgt = cw * pe[0];
      gx = fma(wgt, xa - pb[0], gx); gy = fma(wgt, ya - pb[R], gy);
    }
    }
    if (valid) {                                   // 32-bit flat output indices: d2dx_colloc_eval checks
      const NodeOff o = colloc_offsets(P, a_l, i);
      const NodeIn in = {fr[o.ox + 2 * N], fr[o.ophi], fr[o.ov], pa[-1], pa[R - 1], i >= 1 ? fr[o.ox + 2 * N - 1] : 0.0};
      colloc_node_in<true, true>(a, prob, a_l, i, xa, ya, in, o, gx, gy, true, s_v, s_phi);
    }
  };

  if (REGS) {
    const bool h0 = w < n, h1 = w + W < n;
    double gx0 = 0.0, gy0 = 0.0, gx1 = 0.0, gy1 = 0.0;
    if (h0) phase_a(w, gx0, gy0, std::false_type{});
    if (h1) phase_a(w + W, gx1, gy1, std::true_type{});
    if (!valid) s_col = 0.0;                       // overhanging lanes of the last tile evaluated zeros
    __syncthreads();
    if (h0) phase_b(w, gx0, gy0, std::false_type{});
    if (h1) phase_b(w + W, gx1, gy1, std::true_type{});
  } else {
    for (int a_l = w; a_l < n; a_l += W) {
      double gx, gy;
      phase_a(a_l, gx, gy, std::false_type{});
      sg[(a_l * 2) * 32] = gx; sg[(a_l * 2 + 1) * 32] = gy;
    }
    if (!valid) s_col = 0.0;
    __syncthreads();
    for (int a_l = w; a_l < n; a_l += W) phase_b(a_l, sg[(a_l * 2) * 32], sg[(a_l * 2 + 1) * 32], std::false_type{});
  }

  if (tile == 0) {                                 // instance constraints: first tile of each problem
    for (int k = threadIdx.x; k < P.n_inst; k += blockDim.x) {
      if (a.what & D2DX_EVAL_RESIDUAL)
        a.res[(size_t)prob * a.n_con + 3 * n * (N - 1) + k] = fr[P.inst_var[k] * N + P.inst_node[k]] - P.inst_val[k];
      if (a.what & D2DX_EVAL_JAC) a.jac[(size_t)prob * a.nnz + (a.nnz - P.n_inst) + k] = 1.0;
    }
  }

  if (a.what & D2DX_EVAL_COST) {
    const double tot = warp_sum4(s_v, s_phi, s_obs, s_col, lane);     // lanes 0 / 8 / 16 / 24 hold the four sums
    if ((lane & 7) == 0) sred[w * 4 + (lane >> 3)] = tot;
    __syncthreads();
    if (w == 0) {
      double b4[4] = {0.0, 0.0, 0.0, 0.0};
      for (int q = 0; q < W; ++q) { b4[0] += sred[q * 4]; b4[1] += sred[q * 4 + 1]; b4[2] += sred[q * 4 + 2]; b4[3] += sred[q * 4 + 3]; }
      cost_finish(a, prob, tile, b4, use_obs, true, lane);
    }
  }
}

static size_t pairs_smem_bytes(int n) {
  const bool regs = n <= 2 * kPairWarps;
  return ((size_t)(2 * n * 2 * 33 + (n / 2) * n * 32 + (regs ? 0 : n * 64)) + kPairWarps * 4) * sizeof(double);
}


// second pass of the cost for large batches: one warp per problem sums the per-block partials in a fixed order
__global__ void __launch_bounds__(128) colloc_cost_kernel(const __grid_constant__ CollocArgs a, int use_obs, int use_col) {
  const int prob = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (prob >= a.n_prob) return;
  const double* all = a.scratch + kTicketDoubles + (size_t)prob * a.nparts * 4;
  double t4[4] = {0.0, 0.0, 0.0, 0.0};
  for (int t = lane; t < a.nparts; t += 32)
    for (int k = 0; k < 4; ++k) t4[k] += all[t * 4 + k];
  for (int k = 0; k < 4; ++k) t4[k] = warp_sum(t4[k]);
  if (lane == 0) a.cost[prob] = colloc_cost_from_sums(a, t4, use_obs, use_col);
}

// COO structure (opty convention, SURVEY appendix B3/B4)
__global__ void colloc_structure_kernel(int n_ac, int N, int layout, int n_inst, const int32_t* __restrict__ perm_phi,
                                        const int32_t* __restrict__ perm_v, const int32_t* __restrict__ inst_var,
                                        const int32_t* __restrict__ inst_node, long nnz, int64_t* __restrict__ rows,
                                        int64_t* __restrict__ cols) {
  const int n = 3 * n_ac, q = 2 * n_ac;
  const long nnz_eom = nnz - n_inst;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < nnz; idx += (long)gridDim.x * blockDim.x) {
    if (idx >= nnz_eom) {
      const int k = (int)(idx - nnz_eom);
      rows[idx] = (int64_t)n * (N - 1) + k;
      cols[idx] = (int64_t)inst_var[k] * N + inst_node[k];
      continue;
    }
    if (layout == D2DX_JAC_OPTY_DENSE) {
      const int W = 2 * n + q;
      const long node = idx / ((long)n * W);
      const int rem = (int)(idx - node * (long)n * W), e = rem / W, c = rem - e * W;
      rows[idx] = (int64_t)e * (N - 1) + node;
      int64_t col;
      if (c < n) col = (int64_t)c * N + node + 1;
      else if (c < 2 * n) col = (int64_t)(c - n) * N + node;
      else col = (int64_t)(n + (c - 2 * n)) * N + node + 1;
      cols[idx] = col;
    } else {
      const long per_ac = 12L * (N - 1);
      const int a_l = (int)(idx / per_ac);
      const int k = (int)((idx - a_l * per_ac) / (N - 1));
      const long node = idx - a_l * per_ac - (long)k * (N - 1);
      const int eq = k / 4;
      const int bphi = perm_phi ? perm_phi[a_l] : a_l, bv = perm_v ? perm_v[a_l] : n_ac + a_l;
      // local column of entry k: eq0 [x_i, psi_i, x_p, v_i]  eq1 [y_i, psi_i, y_p, v_i]  eq2 [psi_i, psi_p, phi_i, v_i]
      const int8_t kind[12] = {0, 2, 3, 7, 1, 2, 4, 7, 2, 5, 6, 7};
      const int kd = kind[k];
      int64_t col;
      if (kd < 3) col = (int64_t)(3 * a_l + kd) * N + node + 1;
      else if (kd < 6) col = (int64_t)(3 * a_l + kd - 3) * N + node;
      else if (kd == 6) col = (int64_t)(n + bphi) * N + node + 1;
      else col = (int64_t)(n + bv) * N + node + 1;
      rows[idx] = (int64_t)(3 * a_l + eq) * (N - 1) + node;
      cols[idx] = col;
    }
  }
}

__global__ void colloc_init_dense_kernel(long nnz, int n_inst, int n_prob, double* __restrict__ jac) {
  const long total = nnz * n_prob;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x)
    jac[idx] = (idx % nnz) >= nnz - n_inst ? 1.0 : 0.0;
}

// CostBank with use_mean = False (d2d/opty_utils.py:68-82): cost = obj_scale max_i phi_i^2; gradient = one entry
// obj_scale 2 phi_i at i = np.argmax(phi^2) (first maximum), zeros elsewhere.  One block per problem.
__global__ void __launch_bounds__(256) bank_max_kernel(int n_free, int off_phi, int N, double obj_scale, const double* __restrict__ free_,
                                                       double* __restrict__ cost, double* __restrict__ grad) {
  __shared__ double sv[8];
  __shared__ int si[8];
  const int prob = blockIdx.x, tid = threadIdx.x;
  const double* fr = free_ + (size_t)prob * n_free;
  double best = -1.0;
  int idx = 0x7fffffff;
  for (int i = tid; i < N; i += 256) {
    const double q = fr[off_phi + i] * fr[off_phi + i];
    if (q > best) { best = q; idx = i; }         // strided scan keeps the first maximum of this thread's subsequence
  }
  auto better = [](double v, int i, double bv, int bi) { return v > bv || (v == bv && i < bi); };
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (better(ov, oi, best, idx)) { best = ov; idx = oi; }
  }
  if ((tid & 31) == 0) { sv[tid >> 5] = best; si[tid >> 5] = idx; }
  __syncthreads();
  if (tid < 32) {
    best = tid < 8 ? sv[tid] : -1.0; idx = tid < 8 ? si[tid] : 0x7fffffff;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
      if (better(ov, oi, best, idx)) { best = ov; idx = oi; }
    }
    if (tid == 0) { sv[0] = best; si[0] = idx; }
  }
  __syncthreads();
  best = sv[0]; idx = si[0];
  if (cost && tid == 0) cost[prob] = obj_scale * best;
  if (grad) {
    double* go = grad + (size_t)prob * n_free;
    for (int k = tid; k < n_free; k += 256) go[k] = (k == off_phi + idx) ? obj_scale * 2.0 * fr[k] : 0.0;
  }
}

int colloc_resident_threads_per_sm() {
  int nb = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, colloc_kernel<false>, kCollocThreads, 0);
  return nb * kCollocThreads;
}

static bool enabled_h(double k) { return (k == k) && k != 0.0; }

static void tile_shape(int n_ac, int& TN, int& APP) {
  TN = 128;
  while (TN > 32 && kCollocThreads / TN < n_ac) TN >>= 1;
  APP = kCollocThreads / TN;
}

static int sizes(const d2dx_colloc_problem* p, int layout, int64_t* s3) {
  const int64_t n_ac = p->n_ac, N = p->N;
  s3[0] = 5 * n_ac * N;
  s3[1] = 3 * n_ac * (N - 1) + p->n_inst;
  s3[2] = (layout == D2DX_JAC_OPTY_DENSE ? (N - 1) * 3 * n_ac * 8 * n_ac : 12 * n_ac * (N - 1)) + p->n_inst;
  return D2DX_OK;
}

static int check_problem(const d2dx_colloc_problem* p, const char* who) {
  D2DX_CHECK_ARG(p, "%s: null problem", who);
  D2DX_CHECK_ARG(p->n_ac >= 1 && p->N >= 2 && p->h > 0, "%s: n_ac=%d N=%d h=%g", who, p->n_ac, p->N, p->h);
  D2DX_CHECK_ARG(p->n_inst >= 0 && (p->n_inst == 0 || (p->inst_var && p->inst_node && p->inst_val)), "%s: instance constraints incomplete", who);
  D2DX_CHECK_ARG(p->n_obs >= 0 && p->n_obs <= D2DX_MAX_OBSTACLES, "%s: n_obs=%d (max %d)", who, p->n_obs, D2DX_MAX_OBSTACLES);
  D2DX_CHECK_ARG(p->in_div >= 1, "%s: in_div=%d", who, p->in_div);
  return D2DX_OK;
}

}  // namespace d2dx

using namespace d2dx;

extern "C" {

int d2dx_colloc_sizes(const d2dx_colloc_problem* p, int32_t layout, int64_t* s3) {
  D2DX_CHECK_ARG(p && s3, "d2dx_colloc_sizes: null argument");
  return sizes(p, layout, s3);
}

int64_t d2dx_colloc_scratch_size(const d2dx_colloc_problem* p, int32_t n_prob) {
  if (!p || n_prob < 1) return 0;
  // 64 int32 tickets (must be zero before the first call; every call leaves them zero) + one partial of 4 doubles per
  // block; the finest tiling any kernel uses is 32 nodes per block
  return kTicketDoubles + (int64_t)n_prob * ((p->N + 31) / 32) * 4;
}

int d2dx_colloc_structure(d2dx_handle* h, const d2dx_colloc_problem* p, int32_t layout, int64_t* rows, int64_t* cols, void* stream) {
  D2DX_NVTX("d2dx_colloc_structure");
  if (int rc = check_problem(p, "d2dx_colloc_structure")) return rc;
  D2DX_CHECK_ARG(h && rows && cols, "d2dx_colloc_structure: null argument");
  int64_t s3[3];
  sizes(p, layout, s3);
  D2DX_CUDA(cudaSetDevice(h->device));
  const int grid = (int)((s3[2] + 255) / 256 < 4096 ? (s3[2] + 255) / 256 : 4096);
  colloc_structure_kernel<<<grid, 256, 0, as_stream(stream)>>>(p->n_ac, p->N, layout, p->n_inst, p->perm_phi, p->perm_v,
                                                                 p->inst_var, p->inst_node, s3[2], rows, cols);
  D2DX_LAUNCH_CHECK("colloc_structure_kernel");
  return D2DX_OK;
}

int d2dx_colloc_init_dense(d2dx_handle* h, const d2dx_colloc_problem* p, int32_t n_prob, double* jac, void* stream) {
  D2DX_NVTX("d2dx_colloc_init_dense");
  if (int rc = check_problem(p, "d2dx_colloc_init_dense")) return rc;
  D2DX_CHECK_ARG(h && jac && n_prob >= 1, "d2dx_colloc_init_dense: bad argument");
  int64_t s3[3];
  sizes(p, D2DX_JAC_OPTY_DENSE, s3);
  D2DX_CUDA(cudaSetDevice(h->device));
  colloc_init_dense_kernel<<<h->sm_count * 8, 256, 0, as_stream(stream)>>>(s3[2], p->n_inst, n_prob, jac);
  D2DX_LAUNCH_CHECK("colloc_init_dense_kernel");
  return D2DX_OK;
}

int d2dx_colloc_eval(d2dx_handle* h, const d2dx_colloc_problem* p, int32_t n_prob, const double* free_, int32_t layout,
                     uint32_t what, double* residual, double* jac, double* cost, double* grad, double* scratch, void* stream) {
  D2DX_NVTX("d2dx_colloc_eval");
  if (int rc = check_problem(p, "d2dx_colloc_eval")) return rc;
  D2DX_CHECK_ARG(h && free_ && n_prob >= 1 && n_prob <= 65536, "d2dx_colloc_eval: n_prob=%d (1..65536 per call)", n_prob);
  D2DX_CHECK_ARG(layout == D2DX_JAC_COMPACT || layout == D2DX_JAC_OPTY_DENSE, "d2dx_colloc_eval: unknown Jacobian layout %d", layout);
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_RESIDUAL) || residual, "d2dx_colloc_eval: residual requested but NULL");
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_JAC) || jac, "d2dx_colloc_eval: jacobian requested but NULL");
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_COST) || (cost && scratch), "d2dx_colloc_eval: cost requested but cost/scratch NULL");
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_GRAD) || grad, "d2dx_colloc_eval: gradient requested but NULL");
  D2DX_CHECK_ARG(5L * p->n_ac * p->N < (1L << 31), "d2dx_colloc_eval: 5 n_ac N = %ld does not fit 32-bit offsets", 5L * p->n_ac * p->N);
  CollocArgs a;
  a.p = *p; a.n_prob = n_prob; a.layout = layout; a.what = what; a.free_ = free_;
  a.res = residual; a.jac = jac; a.cost = cost; a.grad = grad; a.scratch = scratch;
  int64_t s3[3];
  sizes(p, layout, s3);
  a.n_free = (int)s3[0]; a.n_con = (int)s3[1]; a.nnz = s3[2];
  colloc_constants(a);
  D2DX_CUDA(cudaSetDevice(h->device));
  a.ticket_mode = n_prob < kMaxTickets;        // latency-sensitive single evaluations stay one launch
  const bool want_cg = (what & (D2DX_EVAL_COST | D2DX_EVAL_GRAD)) != 0;
  const bool col = want_cg && enabled_h(p->kcol) && p->n_ac > 1;
  const bool obs = want_cg && enabled_h(p->kobs) && p->n_obs > 0;
  cudaStream_t st = as_stream(stream);
  const long per_max = a.nnz > a.n_free ? a.nnz : a.n_free;                    // n_con < n_free
  const bool idx32 = (long)n_prob * per_max < (1L << 31);
  if (col && p->col_all_pairs && idx32 && pairs_smem_bytes(p->n_ac) <= 200 * 1024) {
    a.TN = 32; a.APP = kPairWarps; a.ntiles = (p->N + 31) / 32; a.nparts = a.ntiles;
    const size_t smem = pairs_smem_bytes(p->n_ac);
    const bool regs = p->n_ac <= 2 * kPairWarps;
    auto kern = p->n_ac == 2 * kPairWarps ? colloc_pairs_kernel<true, 2 * kPairWarps> : regs ? colloc_pairs_kernel<true> : colloc_pairs_kernel<false>;
    if (smem > 48 * 1024) D2DX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int warps = p->n_ac < kPairWarps ? p->n_ac : kPairWarps;
    const dim3 grid = n_prob <= 65535 ? dim3((unsigned)a.ntiles, (unsigned)n_prob) : dim3((unsigned)((long)n_prob * a.ntiles));
    kern<<<grid, warps * 32, smem, st>>>(a);
    D2DX_LAUNCH_CHECK("colloc_pairs_kernel");
  } else {
    tile_shape(p->n_ac, a.TN, a.APP);
    a.ntiles = (p->N + a.TN - 1) / a.TN; a.nparts = a.ntiles;
    const unsigned grid = (unsigned)((long)n_prob * a.ntiles);
    if (col || obs) {
      const size_t smem = col ? (size_t)p->n_ac * 2 * a.TN * sizeof(double) : 0;
      if (smem > 48 * 1024) {
        D2DX_CHECK_ARG(smem <= 200 * 1024, "d2dx_colloc_eval: %d aircraft need %zu B of shared memory", p->n_ac, smem);
        D2DX_CUDA(cudaFuncSetAttribute(colloc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      }
      colloc_kernel<true><<<grid, kCollocThreads, smem, st>>>(a);
    } else {
      colloc_kernel<false><<<grid, kCollocThreads, 0, st>>>(a);
    }
    D2DX_LAUNCH_CHECK("colloc_kernel");
  }
  if ((what & D2DX_EVAL_COST) && !a.ticket_mode) {
    colloc_cost_kernel<<<(n_prob + 3) / 4, 128, 0, st>>>(a, obs, col);
    D2DX_LAUNCH_CHECK("colloc_cost_kernel");
  }
  return D2DX_OK;
}

int d2dx_cost_bank_max(d2dx_handle* h, int32_t n_prob, int32_t n_free, int32_t off_phi, int32_t N, double obj_scale, const double* free_,
                       double* cost, double* grad, void* stream) {
  D2DX_NVTX("d2dx_cost_bank_max");
  D2DX_CHECK_ARG(h && free_ && (cost || grad), "d2dx_cost_bank_max: null argument");
  D2DX_CHECK_ARG(n_prob >= 1 && N >= 1 && off_phi >= 0 && off_phi + N <= n_free, "d2dx_cost_bank_max: n_prob=%d off_phi=%d N=%d n_free=%d", n_prob,
                 off_phi, N, n_free);
  D2DX_CUDA(cudaSetDevice(h->device));
  bank_max_kernel<<<n_prob, 256, 0, as_stream(stream)>>>(n_free, off_phi, N, obj_scale, free_, cost, grad);
  D2DX_LAUNCH_CHECK("bank_max_kernel");
  return D2DX_OK;
}

}  // extern "C"
