// Batched second-order solve of multi-aircraft planner problems: one warp = one problem (d2dx_ddp_multi.cuh).  Lane r owns row
// r of the node's 3n x 3n value Hessian (row / column r of the other matrices), so the node algebra of the backward sweep runs
// across the lanes; the box QP of the node runs on lane 0.  Per chunk of 32 nodes the lanes first evaluate the transcendental
// functions of every (node, aircraft) pair and stage them with the previous node's states.  The matrices of a warp live in
// shared memory with odd leading dimensions (conflict-free column access by the lanes).
#include "d2dx_ddp_multi.cuh"
#include "d2dx_host.h"

namespace d2dx {

constexpr int kDdpmWarps = 4;                      // problems (= warps) per block at most
constexpr int kDdpmSmemMax = 200 * 1024;           // bytes of shared memory a block may take

__host__ __device__ inline int ddpm_stage_doubles(int n) { return 32 * (n * kDdpPre + 3 * n); }
__host__ __device__ inline int ddpm_warp_doubles(int n) { return DdpmNode::doubles(n) + ddpm_stage_doubles(n) + 5 * n; }
__host__ __device__ inline int ddpm_warp_ints(int n) { return (DdpmNode::ints(n) + 1) & ~1; }

struct DdpmWarp {
  static constexpr int kMaxCon = 3 * kDdpmMaxAc;
  const DdpmProblem& M;
  DdpmWork W;
  const double* zt;
  DdpmNode nd;
  double *stage, *zc, *us;
  int* flag;
  int lane;
  int* solved;
  int min_solved;
  __device__ DdpmWarp(const DdpmProblem& m, const DdpmWork& w, const double* zt_, double* sm, int* ism, int lane_, int* solved_, int min_solved_)
      : M(m), W(w), zt(zt_), nd(m), lane(lane_), solved(solved_), min_solved(min_solved_) {
    nd.carve(sm, ism);
    stage = sm + DdpmNode::doubles(m.n);
    zc = stage + ddpm_stage_doubles(m.n);
    us = zc + 3 * m.n;
    flag = ism + DdpmNode::ints(m.n) - 1;
  }
  __device__ int n_con() const { return 3 * M.n; }
  __device__ bool enough_solved() const {
    int s = 0;
    if (min_solved > 0 && lane == 0) s = *reinterpret_cast<volatile int*>(solved) >= min_solved;
    return __shfl_sync(0xffffffffu, s, 0) != 0;
  }
  __device__ void count_solved() { if (lane == 0) atomicAdd(solved, 1); }

  __device__ DdpSweep backward(const double* lam, double rho, double mu, int) {
    const int n = M.n, N = M.a.N, m = 2 * n, nz = 3 * n, S = n * kDdpPre + nz;
    DdpSweep r = {0.0, 0.0, true};
    if (lane == 0) nd.dV[0] = nd.dV[1] = 0.0;
    if (lane < nz) nd.s0(lane, W.z + (long)(N - 1) * nz, zt, lam, rho);
    for (int hi = N - 1; hi >= 1 && r.ok; hi -= 32) {         // chunk of nodes hi, hi-1, ..., max(hi-31, 1)
      const int cnt = hi >= 32 ? 32 : hi;
      __syncwarp();
      for (int t = lane; t < cnt * n; t += 32) {
        const int l = t / n, a = t - l * n, i = hi - l;
        DdpNodePre p;
        ddp_node_pre(M.a, W.u[(long)i * m + 2 * a], W.u[(long)i * m + 2 * a + 1], W.z[(long)i * nz + 3 * a + 2], p);
        double* d = stage + l * S + a * kDdpPre;
        d[0] = p.phi; d[1] = p.v; d[2] = p.s; d[3] = p.c; d[4] = p.dph; d[5] = p.dvv; d[6] = p.dphph; d[7] = p.dphv; d[8] = p.dv2;
      }
      for (int t = lane; t < cnt * nz; t += 32) {
        const int l = t / nz, c = t - l * nz;
        stage[l * S + n * kDdpPre + c] = W.z[(long)(hi - l - 1) * nz + c];
      }
      __syncwarp();
      for (int l = 0; l < cnt; ++l) {
        const int i = hi - l;
        nd.pre = stage + l * S;
        if (lane < nz) nd.s1(lane);
        __syncwarp();
        if (lane < m) nd.s2(lane);
        __syncwarp();
        if (lane < nz && lane % 3 == 2) nd.s3(lane);
        if (lane == 0) *flag = nd.s4(mu) ? 1 : 0;
        __syncwarp();
        if (!*flag) { r.ok = false; break; }
        if (lane < nz) {
          nd.s5(lane);
          double* Kg = W.K + ((long)i * nz + lane) * m;
          for (int q = 0; q < m; ++q) Kg[q] = nd.K[q * nd.ldz + lane];
        }
        __syncwarp();
        if (lane < nz) nd.s6(lane, i > 1);
        if (lane < m) W.k[(long)i * m + lane] = nd.kk[lane];
        __syncwarp();
      }
    }
    __syncwarp();
    r.dV1 = nd.dV[0]; r.dV2 = nd.dV[1];
    __syncwarp();
    return r;
  }

  __device__ double forward(double alpha, const double* lam, double rho, double& cost, double& cmax) {
    const int n = M.n, N = M.a.N, m = 2 * n, nz = 3 * n;
    double part = 0.0;
    if (lane < nz) W.zn[lane] = zc[lane] = W.z[lane];
    if (lane < m) W.un[lane] = W.u[lane];
    __syncwarp();
    if (lane < n) part = ddp_input_cost(M.a, W.u[2 * lane], W.u[2 * lane + 1]) + ddpm_aircraft_cost(M, lane, zc);
    for (int i = 1; i < N; ++i) {
      if (lane < m) us[lane] = ddpm_input(M, W, i, lane, alpha, zc);
      __syncwarp();
      if (lane < n) part += ddpm_transition(M, us[2 * lane], us[2 * lane + 1], zc + 3 * lane);
      __syncwarp();
      if (lane < n) part += ddpm_aircraft_cost(M, lane, zc);
      if (lane < m) W.un[(long)i * m + lane] = us[lane];
      if (lane < nz) W.zn[(long)i * nz + lane] = zc[lane];
    }
    __syncwarp();
    cost = warp_sum(part);
    double J = cost, cc = 0.0;
    cmax = 0.0;
    for (int c = 0; c < nz; ++c) {
      const double e = zc[c] - zt[c];
      cmax = fmax(cmax, fabs(e)); J += lam[c] * e; cc += e * e;
    }
    __syncwarp();
    return J + 0.5 * rho * cc;
  }

  __device__ void accept() {
    double* t = W.u; W.u = W.un; W.un = t;
    t = W.z; W.z = W.zn; W.zn = t;
    __syncwarp();
  }
  __device__ void terminal_error(double* c) const {
    const int nz = 3 * M.n;
    for (int q = 0; q < nz; ++q) c[q] = W.z[(long)(M.a.N - 1) * nz + q] - zt[q];
  }
  __device__ void prepare(const double* z0) {
    const int n = M.n, N = M.a.N, m = 2 * n, nz = 3 * n;
    for (int e = lane; e < N * m; e += 32) {
      const int i = e / m, q = e - i * m;
      double x = W.u[e];
      if (i == 0 && (q & 1) == 0 && M.a.kb > 0.0) x = 0.0;
      if (i == 0 && (q & 1) == 1 && M.a.kv > 0.0) x = M.a.vsp;
      W.u[e] = (q & 1) ? ddp_clip(x, M.a.v_lo, M.a.v_hi) : ddp_clip(x, M.a.phi_lo, M.a.phi_hi);
      W.k[e] = 0.0;
    }
    for (long e = lane; e < (long)N * nz * m; e += 32) W.K[e] = 0.0;
    for (int e = lane; e < N * nz; e += 32) W.z[e] = e < nz ? z0[e] : 0.0;
    __syncwarp();
  }
};

struct DdpmArgs {
  DdpmProblem M;
  d2dx_ddp_options o;
  int n_prob, warps;
  const double *p0, *p1;
  double *u, *xs, *info, *lam, *work;
  int* solved;
  int min_solved;
};

__global__ void __launch_bounds__(kDdpmWarps * 32) ddpm_solve_kernel(const __grid_constant__ DdpmArgs a) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int p = blockIdx.x * a.warps + wib;
  if (p >= a.n_prob) return;                        // whole warps leave together
  const int n = a.M.n, N = a.M.a.N, m = 2 * n, nz = 3 * n;
  double* sm = smem + (size_t)wib * ddpm_warp_doubles(n);
  int* ism = reinterpret_cast<int*>(smem + (size_t)a.warps * ddpm_warp_doubles(n)) + wib * ddpm_warp_ints(n);
  DdpmWork W;
  W.carve(a.work + (size_t)p * DdpmWork::doubles(n, N), n, N);
  const double* ui = a.u + (size_t)p * m * N;       // [2][n][N]
  for (int e = lane; e < m * N; e += 32) {
    const int ja = e / N, i = e - ja * N, j = ja / n, ac = ja - j * n;
    W.u[(long)i * m + 2 * ac + j] = ui[e];
  }
  double z0[3 * kDdpmMaxAc], zt[3 * kDdpmMaxAc], lam[3 * kDdpmMaxAc];
  for (int k = 0; k < 3; ++k)
    for (int ac = 0; ac < n; ++ac) { z0[3 * ac + k] = a.p0[(size_t)p * nz + k * n + ac]; zt[3 * ac + k] = a.p1[(size_t)p * nz + k * n + ac]; }
  __syncwarp();
  DdpmWarp sweeps(a.M, W, zt, sm, ism, lane, a.solved, a.min_solved);
  const DdpResult r = ddp_solve(sweeps, z0, a.o, lam);
  __syncwarp();
  const double* us = (r.swaps & 1) ? W.un : W.u;
  const double* zs = (r.swaps & 1) ? W.zn : W.z;
  double* uo = a.u + (size_t)p * m * N;
  double* xo = a.xs + (size_t)p * nz * N;
  for (int e = lane; e < m * N; e += 32) {
    const int ja = e / N, i = e - ja * N, j = ja / n, ac = ja - j * n;
    uo[e] = us[(long)i * m + 2 * ac + j];
  }
  for (int e = lane; e < nz * N; e += 32) {
    const int ka = e / N, i = e - ka * N, k = ka / n, ac = ka - k * n;
    xo[e] = zs[(long)i * nz + 3 * ac + k];
  }
  if (lane == 0) {
    double* io = a.info + (size_t)p * 8;
    io[0] = r.flag; io[1] = r.iterations; io[2] = r.outer; io[3] = r.cost; io[4] = r.cmax; io[5] = r.lagr; io[6] = r.mu; io[7] = r.rho;
    if (a.lam)
      for (int k = 0; k < 3; ++k)
        for (int ac = 0; ac < n; ++ac) a.lam[(size_t)p * nz + k * n + ac] = lam[3 * ac + k];
  }
}

}  // namespace d2dx

using namespace d2dx;

extern "C" {

int64_t d2dx_ddp_multi_work_size(int32_t P, int32_t n_ac, int32_t N) {
  return (P < 1 || N < 2 || n_ac < 1 || n_ac > kDdpmMaxAc) ? 0 : DdpmWork::doubles(n_ac, N) * P + 2;   // + the solved counter
}

int d2dx_ddp_multi_solve(d2dx_handle* h, const d2dx_colloc_problem* p, int32_t n_prob, const double* bounds_host4, const double* state_box_host5,
                         const double* p0, const double* p1, double* u, double* xs, double* info, double* lam_out, double* work,
                         const d2dx_ddp_options* o_host, void* stream) {
  D2DX_NVTX("d2dx_ddp_multi_solve");
  D2DX_CHECK_ARG(h && p && n_prob >= 1 && p0 && p1 && u && xs && info && work, "d2dx_ddp_multi_solve: null argument or n_prob=%d", n_prob);
  DdpmArgs a;
  D2DX_CHECK_ARG(ddpm_problem_from(p, bounds_host4, state_box_host5, a.M) == 0,
                 "d2dx_ddp_multi_solve: needs 1 <= n_ac <= %d, N >= 2, h > 0, bounds phi_lo < phi_hi, 0 < v_lo < v_hi and rcol > 0", kDdpmMaxAc);
  if (o_host) a.o = *o_host; else d2dx_ddp_default_options(&a.o);
  D2DX_CHECK_ARG(a.o.max_iter >= 1 && a.o.max_outer >= 1 && a.o.max_inner >= 1 && a.o.ls_max >= 1 && a.o.mu_factor > 1.0 && a.o.rho0 > 0.0,
                 "d2dx_ddp_multi_solve: bad options");
  D2DX_CHECK_ARG(a.o.reg_mode == 0 || a.M.n == 1, "d2dx_ddp_multi_solve: reg_mode 1 needs n_ac = 1");
  const int n = a.M.n;
  const size_t per_warp = (size_t)ddpm_warp_doubles(n) * sizeof(double) + (size_t)ddpm_warp_ints(n) * sizeof(int);
  a.warps = (int)(kDdpmSmemMax / per_warp) < kDdpmWarps ? (int)(kDdpmSmemMax / per_warp) : kDdpmWarps;
  const size_t smem = per_warp * a.warps;
  a.n_prob = n_prob; a.p0 = p0; a.p1 = p1; a.u = u; a.xs = xs; a.info = info; a.lam = lam_out; a.work = work;
  a.solved = reinterpret_cast<int*>(work + DdpmWork::doubles(n, p->N) * n_prob);
  a.min_solved = a.o.min_solved;
  D2DX_CUDA(cudaSetDevice(h->device));
  D2DX_CUDA(cudaFuncSetAttribute(ddpm_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  D2DX_CUDA(cudaMemsetAsync(a.solved, 0, sizeof(int), as_stream(stream)));
  ddpm_solve_kernel<<<(n_prob + a.warps - 1) / a.warps, a.warps * 32, smem, as_stream(stream)>>>(a);
  D2DX_LAUNCH_CHECK("ddpm_solve_kernel");
  return D2DX_OK;
}

}  // extern "C"
