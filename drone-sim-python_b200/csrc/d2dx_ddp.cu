// Batched second-order planner solve: one thread = one problem (d2dx_ddp.cuh), work arrays interleaved over the problems.
#include "d2dx_ddp.cuh"
#include "d2dx_host.h"

namespace d2dx {

constexpr int kDdpWarps = 4;                       // problems (= warps) per block
constexpr int kDdpSlot = 24;                       // doubles of staging per lane

// Sweeps of ONE problem by ONE warp.  The recursion over the nodes is sequential (lane 0 carries it), but everything around it
// is not: per chunk of 32 nodes the lanes load the trajectory coalesced, evaluate the transcendental functions, the obstacle
// exponentials and the costs of their node in parallel and stage the results in shared memory; lane 0 then runs the node
// algebra from shared memory (about 250 fp64 instructions per node, no memory latency, no libm call in the dependent chain),
// and the lanes write the gains / the new trajectory back coalesced.  Same node functions as the serial host sweeps.
struct DdpWarp {
  static constexpr int kMaxCon = 3;
  const DdpProblem& P;
  DdpWork W;                                        // stride 1: this problem's arrays are contiguous
  const double* zt;
  double* sm;                                       // [32][kDdpSlot] staging of this warp
  int lane;
  int* solved;                                      // launch-wide count of converged problems
  int min_solved;                                   // > 0: stop iterating once that many have converged (multi-start)
  __device__ DdpWarp(const DdpProblem& p, const DdpWork& w, const double* zt_, double* sm_, int lane_, int* solved_, int min_solved_)
      : P(p), W(w), zt(zt_), sm(sm_), lane(lane_), solved(solved_), min_solved(min_solved_) {}
  __device__ bool enough_solved() const {
    int s = 0;
    if (min_solved > 0 && lane == 0) s = *reinterpret_cast<volatile int*>(solved) >= min_solved;
    return __shfl_sync(0xffffffffu, s, 0) != 0;
  }
  __device__ void count_solved() { if (lane == 0) atomicAdd(solved, 1); }
  __device__ int n_con() const { return 3; }

  __device__ DdpSweep backward(const double* lam, double rho, double mu, int reg_mode) {
    const int N = P.N;
    const bool sc = P.n_obs > 0 || P.has_box;
    DdpSweep r = {0.0, 0.0, true};
    DdpValue V;
    ddp_terminal_value(P, W.at(W.z, 0, N - 1), W.at(W.z, 1, N - 1), W.at(W.z, 2, N - 1), zt, lam, rho, V);   // every lane: uniform
    double* my = sm + lane * kDdpSlot;
    for (int hi = N - 1; hi >= 1; hi -= 32) {       // chunk of nodes hi, hi-1, ..., max(hi-31, 1): lane l holds node hi - l
      const int i = hi - lane;
      const int cnt = hi >= 32 ? 32 : hi;
      __syncwarp();
      if (i >= 1) {
        DdpNodePre n;
        ddp_node_pre(P, W.at(W.u, 0, i), W.at(W.u, 1, i), W.at(W.z, 2, i), n);
        my[0] = n.phi; my[1] = n.v; my[2] = n.s; my[3] = n.c; my[4] = n.dph; my[5] = n.dvv; my[6] = n.dphph; my[7] = n.dphv; my[8] = n.dv2;
        if (sc) {
          double gx = 0.0, gy = 0.0, hxx = 0.0, hxy = 0.0, hyy = 0.0;
          if (i > 1) ddp_state_cost(P, W.at(W.z, 0, i - 1), W.at(W.z, 1, i - 1), gx, gy, hxx, hxy, hyy);
          my[9] = gx; my[10] = gy; my[11] = hxx; my[12] = hxy; my[13] = hyy;
        }
      }
      __syncwarp();
      if (lane == 0) {
        for (int l = 0; l < cnt && r.ok; ++l) {
          double* q = sm + l * kDdpSlot;
          DdpNodePre n;
          n.phi = q[0]; n.v = q[1]; n.s = q[2]; n.c = q[3]; n.dph = q[4]; n.dvv = q[5]; n.dphph = q[6]; n.dphv = q[7]; n.dv2 = q[8];
          double kk[2], K[6];
          r.ok = ddp_backward_node(P, n, mu, reg_mode, V, kk, K, r.dV1, r.dV2);
          if (sc) { V.z0 += q[9]; V.z1 += q[10]; V.w00 += q[11]; V.w01 += q[12]; V.w11 += q[13]; }
          q[14] = kk[0]; q[15] = kk[1];
#pragma unroll
          for (int j = 0; j < 6; ++j) q[16 + j] = K[j];
        }
      }
      __syncwarp();
      r.ok = __shfl_sync(0xffffffffu, (int)r.ok, 0) != 0;
      if (!r.ok) break;
      if (i >= 1) {
        W.at(W.k, 0, i) = my[14]; W.at(W.k, 1, i) = my[15];
#pragma unroll
        for (int j = 0; j < 6; ++j) W.at(W.K, j, i) = my[16 + j];
      }
    }
    r.dV1 = __shfl_sync(0xffffffffu, r.dV1, 0); r.dV2 = __shfl_sync(0xffffffffu, r.dV2, 0);
    __syncwarp();
    return r;
  }

  __device__ double forward(double alpha, const double* lam, double rho, double& cost, double& cmax) {
    const int N = P.N;
    const bool sc = P.n_obs > 0 || P.has_box;
    double x = W.at(W.z, 0, 0), y = W.at(W.z, 1, 0), psi = W.at(W.z, 2, 0);      // carried by lane 0
    double part = 0.0;                                                            // this lane's share of the cost
    if (lane == 0) {
      W.at(W.zn, 0, 0) = x; W.at(W.zn, 1, 0) = y; W.at(W.zn, 2, 0) = psi;
      W.at(W.un, 0, 0) = W.at(W.u, 0, 0); W.at(W.un, 1, 0) = W.at(W.u, 1, 0);
      part = ddp_input_cost(P, W.at(W.u, 0, 0), W.at(W.u, 1, 0));
      double gx, gy, hxx, hxy, hyy;
      if (sc) part += ddp_state_cost(P, x, y, gx, gy, hxx, hxy, hyy);
    }
    double* my = sm + lane * kDdpSlot;
    for (int lo = 1; lo < N; lo += 32) {            // chunk of nodes lo .. lo+31: lane l holds node lo + l
      const int i = lo + lane;
      const int cnt = N - lo >= 32 ? 32 : N - lo;
      __syncwarp();
      if (i < N) {
        my[0] = W.at(W.u, 0, i); my[1] = W.at(W.u, 1, i);
        my[2] = W.at(W.k, 0, i); my[3] = W.at(W.k, 1, i);
#pragma unroll
        for (int j = 0; j < 6; ++j) my[4 + j] = W.at(W.K, j, i);
        my[10] = W.at(W.z, 0, i - 1); my[11] = W.at(W.z, 1, i - 1); my[12] = W.at(W.z, 2, i - 1);
      }
      __syncwarp();
      if (lane == 0) {
        for (int l = 0; l < cnt; ++l) {
          double* q = sm + l * kDdpSlot;
          double phi, v;
          ddp_forward_node(P, alpha, q[0], q[1], q + 2, q + 4, q[10], q[11], q[12], x, y, psi, phi, v);
          q[13] = phi; q[14] = v; q[15] = x; q[16] = y; q[17] = psi;
        }
      }
      __syncwarp();
      if (i < N) {
        const double phi = my[13], v = my[14], xn = my[15], yn = my[16];
        W.at(W.un, 0, i) = phi; W.at(W.un, 1, i) = v;
        W.at(W.zn, 0, i) = xn; W.at(W.zn, 1, i) = yn; W.at(W.zn, 2, i) = my[17];
        part += ddp_input_cost(P, phi, v);
        double gx, gy, hxx, hxy, hyy;
        if (sc) part += ddp_state_cost(P, xn, yn, gx, gy, hxx, hxy, hyy);
      }
    }
    __syncwarp();
    cost = warp_sum(part);
    x = __shfl_sync(0xffffffffu, x, 0); y = __shfl_sync(0xffffffffu, y, 0); psi = __shfl_sync(0xffffffffu, psi, 0);
    const double c0 = x - zt[0], c1 = y - zt[1], c2 = psi - zt[2];
    cmax = fmax(fabs(c0), fmax(fabs(c1), fabs(c2)));
    return cost + lam[0] * c0 + lam[1] * c1 + lam[2] * c2 + 0.5 * rho * (c0 * c0 + c1 * c1 + c2 * c2);
  }

  __device__ void accept() {
    double* t = W.u; W.u = W.un; W.un = t;
    t = W.z; W.z = W.zn; W.zn = t;
    __syncwarp();
  }
  __device__ void terminal_error(double* c) const {
    const int N = P.N;
    c[0] = W.at(W.z, 0, N - 1) - zt[0]; c[1] = W.at(W.z, 1, N - 1) - zt[1]; c[2] = W.at(W.z, 2, N - 1) - zt[2];
  }
  __device__ void prepare(const double* z0) {
    const int N = P.N;
    for (int i = lane; i < N; i += 32) {
      double phi = W.at(W.u, 0, i), v = W.at(W.u, 1, i);
      if (i == 0) { if (P.kb > 0.0) phi = 0.0; if (P.kv > 0.0) v = P.vsp; }
      W.at(W.u, 0, i) = ddp_clip(phi, P.phi_lo, P.phi_hi);
      W.at(W.u, 1, i) = ddp_clip(v, P.v_lo, P.v_hi);
      W.at(W.k, 0, i) = 0.0; W.at(W.k, 1, i) = 0.0;
#pragma unroll
      for (int j = 0; j < 6; ++j) W.at(W.K, j, i) = 0.0;
#pragma unroll
      for (int j = 0; j < 3; ++j) W.at(W.z, j, i) = i == 0 ? z0[j] : 0.0;
    }
    __syncwarp();
  }
};

struct DdpArgs {
  DdpProblem P;
  d2dx_ddp_options o;
  int n_prob;
  const double *p0, *p1;
  double *u, *xs, *info, *work;
  int* solved;
  int min_solved;
};

__global__ void __launch_bounds__(kDdpWarps * 32) ddp_solve_kernel(const __grid_constant__ DdpArgs a) {
  __shared__ double stage[kDdpWarps][32 * kDdpSlot];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int p = blockIdx.x * kDdpWarps + wib;
  if (p >= a.n_prob) return;                        // whole warps leave together
  const int N = a.P.N;
  DdpWork W;
  W.N = N; W.stride = 1;
  double* base = a.work + (size_t)p * 18 * N;       // this problem's arrays, contiguous
  W.u = base; W.z = W.u + 2 * N; W.un = W.z + 3 * N; W.zn = W.un + 2 * N; W.k = W.zn + 3 * N; W.K = W.k + 2 * N;
  const double* ui = a.u + (size_t)p * 2 * N;
  for (int i = lane; i < 2 * N; i += 32) W.u[i] = ui[i];
  __syncwarp();
  const double z0[3] = {a.p0[p * 3], a.p0[p * 3 + 1], a.p0[p * 3 + 2]}, zt[3] = {a.p1[p * 3], a.p1[p * 3 + 1], a.p1[p * 3 + 2]};
  DdpWarp sweeps(a.P, W, zt, stage[wib], lane, a.solved, a.min_solved);
  const DdpResult r = ddp_solve(sweeps, z0, a.o);
  __syncwarp();
  const double* us = (r.swaps & 1) ? W.un : W.u;
  const double* zs = (r.swaps & 1) ? W.zn : W.z;
  double* uo = a.u + (size_t)p * 2 * N;
  double* xo = a.xs + (size_t)p * 3 * N;
  for (int i = lane; i < 2 * N; i += 32) uo[i] = us[i];
  for (int i = lane; i < 3 * N; i += 32) xo[i] = zs[i];
  if (lane == 0) {
    double* io = a.info + (size_t)p * 8;
    io[0] = r.flag; io[1] = r.iterations; io[2] = r.outer; io[3] = r.cost; io[4] = r.cmax; io[5] = r.lagr; io[6] = r.mu; io[7] = r.rho;
  }
}

}  // namespace d2dx

using namespace d2dx;

extern "C" {

int d2dx_ddp_default_options(d2dx_ddp_options* o) {
  if (!o) return set_error(D2DX_EINVAL, "d2dx_ddp_default_options: null");
  o->max_iter = 400; o->max_outer = 30; o->max_inner = 40; o->ls_max = 12;
  o->ctol = 1e-8; o->rel_tol = 1e-10; o->abs_tol = 1e-14;
  o->rho0 = 10.0; o->rho_growth = 10.0; o->rho_max = 1e8;
  o->mu0 = 1e-6; o->mu_min = 1e-8; o->mu_max = 1e10; o->mu_factor = 1.6; o->reg_mode = 0; o->min_solved = 0;
  return D2DX_OK;
}

int64_t d2dx_ddp_work_size(int32_t P, int32_t N) { return (P < 1 || N < 2) ? 0 : 18LL * N * P + 2; }   // + the solved counter

int d2dx_ddp_solve(d2dx_handle* h, const d2dx_colloc_problem* p, int32_t n_prob, const double* bounds_host4, const double* state_box_host5,
                   const double* p0, const double* p1, double* u, double* xs, double* info, double* work, const d2dx_ddp_options* o_host,
                   void* stream) {
  D2DX_NVTX("d2dx_ddp_solve");
  D2DX_CHECK_ARG(h && p && n_prob >= 1 && p0 && p1 && u && xs && info && work, "d2dx_ddp_solve: null argument or n_prob=%d", n_prob);
  DdpArgs a;
  D2DX_CHECK_ARG(ddp_problem_from(p, bounds_host4, state_box_host5, a.P) == 0,
                 "d2dx_ddp_solve: needs n_ac = 1, N >= 2, h > 0 and bounds phi_lo < phi_hi, 0 < v_lo < v_hi");
  if (o_host) a.o = *o_host; else d2dx_ddp_default_options(&a.o);
  D2DX_CHECK_ARG(a.o.max_iter >= 1 && a.o.max_outer >= 1 && a.o.max_inner >= 1 && a.o.ls_max >= 1 && a.o.mu_factor > 1.0 && a.o.rho0 > 0.0,
                 "d2dx_ddp_solve: bad options");
  a.n_prob = n_prob; a.p0 = p0; a.p1 = p1; a.u = u; a.xs = xs; a.info = info; a.work = work;
  a.solved = reinterpret_cast<int*>(work + 18LL * p->N * n_prob);
  a.min_solved = a.o.min_solved;
  D2DX_CUDA(cudaSetDevice(h->device));
  D2DX_CUDA(cudaMemsetAsync(a.solved, 0, sizeof(int), as_stream(stream)));
  ddp_solve_kernel<<<(n_prob + kDdpWarps - 1) / kDdpWarps, kDdpWarps * 32, 0, as_stream(stream)>>>(a);
  D2DX_LAUNCH_CHECK("ddp_solve_kernel");
  return D2DX_OK;
}

}  // extern "C"
