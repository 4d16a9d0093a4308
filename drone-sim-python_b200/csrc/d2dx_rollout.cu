// Closed-loop rollout of B aircraft-scenarios under the DFFF controller: one thread = one
// aircraft-scenario, state in fp64 registers, trajectory parameters staged in shared memory,
// SoA logs written with coalesced stores.  Replaces run_simulation (05_test_simulation.py:21-34).
#include "d2dx_device.cuh"
#include "d2dx_host.h"

namespace d2dx {

constexpr int kRolloutThreads = 128;
#ifndef D2DX_ROLLOUT_MIN_BLOCKS
#define D2DX_ROLLOUT_MIN_BLOCKS 4      // <= 128 registers per thread: 16 resident warps per SM
#endif

struct RolloutArgs {
  d2dx_scenarios s;
  d2dx_rollout_out o;
  d2dx_dfff_gains g;
  CareConst cc;               // sqrt(Q), sqrt(R), ... computed on the host: read from the constant bank, not held in registers
  const double* time;
  int i_begin, i_end, nsub, final_control;
};

// 1-D bulk copy global -> shared through the TMA unit (cp.async.bulk), completion on an mbarrier.
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  const uint32_t mb = static_cast<uint32_t>(__cvta_generic_to_shared(bar));
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(dst), "l"(gmem_src), "r"(bytes), "r"(mb) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(static_cast<uint32_t>(__cvta_generic_to_shared(bar))), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
               :: "r"(static_cast<uint32_t>(__cvta_generic_to_shared(bar))), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  const uint32_t mb = static_cast<uint32_t>(__cvta_generic_to_shared(bar));
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}"
      :: "r"(mb), "r"(phase) : "memory");
}

template <int UNIFORM, bool LOGGING, bool LOGREF>
__global__ void __launch_bounds__(kRolloutThreads, D2DX_ROLLOUT_MIN_BLOCKS) rollout_dfff_kernel(const RolloutArgs a) {
  // rows 0..NPAR-1: trajectory parameters; rows NPAR..NPAR+4: wind x, wind y, -1/tau_phi, -1/tau_v, tau_v
  __shared__ __align__(128) double spar[D2DX_SEG_NPAR + 5][kRolloutThreads];
  __shared__ __align__(8) uint64_t bar;
  const int B = a.s.B;
  const int tid = threadIdx.x;
  const int b_raw = blockIdx.x * kRolloutThreads + tid;
  const bool active = b_raw < B;
  const int b = active ? b_raw : B - 1;
  const d2dx_traj_table& tt = a.s.traj;
  const int S = tt.n_seg;

  // ---- stage the trajectory parameters of this block's scenarios in shared memory ----
  int cur_seg = -1, seg_type = UNIFORM;
  if (UNIFORM >= 0) {
    // plain single-segment trajectories with first_seg[b] == b: every parameter row of the tile is one
    // contiguous run of the SoA table -> one TMA bulk copy per row (when the tile is full and 16B aligned)
    const int b0 = blockIdx.x * kRolloutThreads;
    const bool bulk = (b0 + kRolloutThreads <= S) && ((S & 1) == 0) && ((reinterpret_cast<uintptr_t>(tt.seg_par) & 15) == 0);
    constexpr int kRows = (UNIFORM == D2DX_SEG_CIRCLE) ? 6 : (UNIFORM == D2DX_SEG_LINE) ? 5 : D2DX_SEG_NPAR;
    if (bulk) {
      if (tid == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
      __syncthreads();
      if (tid == 0) {
        mbar_expect_tx(&bar, kRows * kRolloutThreads * 8);
        for (int k = 0; k < kRows; ++k)
          tma_load_1d(&spar[k][0], tt.seg_par + (size_t)k * S + b0, kRolloutThreads * 8, &bar);
      }
      mbar_wait(&bar, 0);
    } else {
      for (int k = 0; k < kRows; ++k) spar[k][tid] = tt.seg_par[(size_t)k * S + b];
    }
    cur_seg = b;
  }
  auto P = [&](int k) { return spar[k][tid]; };

  spar[D2DX_SEG_NPAR + 0][tid] = a.s.wind[b]; spar[D2DX_SEG_NPAR + 1][tid] = a.s.wind[B + b];
  spar[D2DX_SEG_NPAR + 2][tid] = -1.0 / a.s.ac[b]; spar[D2DX_SEG_NPAR + 3][tid] = -1.0 / a.s.ac[B + b];
  spar[D2DX_SEG_NPAR + 4][tid] = a.s.ac[B + b];
  // re-read from shared memory at each use: five doubles less to keep in registers across the time loop
  auto load_ac = [&]() {
    AcPar ap;
    ap.wx = spar[D2DX_SEG_NPAR + 0][tid]; ap.wy = spar[D2DX_SEG_NPAR + 1][tid];
    ap.n_inv_tau_phi = spar[D2DX_SEG_NPAR + 2][tid]; ap.n_inv_tau_v = spar[D2DX_SEG_NPAR + 3][tid];
    return ap;
  };
  double X[5];
#pragma unroll
  for (int k = 0; k < 5; ++k) X[k] = a.s.X0[(size_t)k * B + b];

  const CareConst& cc = a.cc;
  // the Riccati warm start (care_gain's state rows) in registers: a shared-memory column per thread measured 2.7 % slower
  double care[kCareState];
#pragma unroll
  for (int k = 0; k < kCareState; ++k) care[k] = a.o.care_state ? a.o.care_state[k * (size_t)B + b] : 0.0;
  bool cold = !(care[2] > 0.0);                                   // no state, or zeros: cold
  int flags = 0;
  double sum_sq = 0.0, max_sq = 0.0;

  int ev = 0, ev_end = 0, ev_next = 0x7fffffff;
  if (a.s.pert_begin) {
    ev = a.s.pert_begin[b]; ev_end = a.s.pert_begin[b + 1];
    while (ev < ev_end && a.s.pert_step[ev] <= a.i_begin) ++ev;
    if (ev < ev_end) ev_next = a.s.pert_step[ev];
  }

  // reference + gain at time t (Trajectory.get, DiffFlatness, cont_jac, LQR): state-independent
  auto reference_at = [&](double t, RefCtl& r) {
    FlatOut Y;
    if (UNIFORM >= 0) {
      segment_eval<false>(UNIFORM, P, t, Y);
    } else {
      double te;
      const int seg = composite_locate(tt, b, t, te);
      if (seg != cur_seg) {            // (re)load this thread's parameter column
        cur_seg = seg; seg_type = tt.seg_type[seg];
        for (int k = 0; k < D2DX_SEG_NPAR; ++k) spar[k][tid] = tt.seg_par[(size_t)k * S + seg];
      }
      segment_eval<false>(seg_type, P, te, Y, &tt);
    }
    make_ref(Y, load_ac(), spar[D2DX_SEG_NPAR + 4][tid], cc, ArrayState{care}, cold, flags, r);
  };

  const int log_every = a.o.log_every > 0 ? a.o.log_every : 1;
  const int n_samples = a.i_end - a.i_begin + (a.final_control ? 1 : 0);
  double t = a.time[a.i_begin];
  // samples until the next logged one (a countdown instead of an integer modulo per step)
  int log_in = (log_every - a.i_begin % log_every) % log_every;
  for (int n = 0; n < n_samples; ++n) {
    const int i = a.i_begin + n;
    // ---- DFFFController.get: reference + gain (state-independent), then the state feedback ----
    RefCtl ref;
    reference_at(t, ref);
    double u_phi, u_v;
    feedback(ref, X, a.g, u_phi, u_v);
    const double ex = X[0] - ref.xr, ey = X[1] - ref.yr, d2 = ex * ex + ey * ey;
    sum_sq += d2; max_sq = __double_as_longlong(d2) > __double_as_longlong(max_sq) ? d2 : max_sq;   // both >= 0: the integer order is the fp64 order
    const bool log_now = LOGGING && log_in == 0;
    log_in = log_now ? log_every - 1 : log_in - 1;
    if (log_now && active) {
      const size_t row = (size_t)(i / log_every);
      if (a.o.X_log) {
#pragma unroll
        for (int k = 0; k < 5; ++k) a.o.X_log[(row * 5 + k) * B + b] = X[k];
      }
      if (a.o.U_log) { a.o.U_log[(row * 2) * B + b] = u_phi; a.o.U_log[(row * 2 + 1) * B + b] = u_v; }
      if (LOGREF && a.o.Xr_log) {
        double* q = a.o.Xr_log + row * 5 * B + b;
        q[0] = ref.xr; q[(size_t)B] = ref.yr; q[2 * (size_t)B] = ref.psir; q[3 * (size_t)B] = ref.phir; q[4 * (size_t)B] = ref.var;
      }
      if (LOGREF && a.o.K_log) {
#pragma unroll
        for (int k = 0; k < 6; ++k) a.o.K_log[(row * 6 + k) * B + b] = ref.k[k];
      }
    }
    if (i == a.i_end) break;           // trailing controller evaluation of 05_test_simulation.py:33
    // ---- Aircraft.disc_dyn (fixed-step RK4), then perturbation ----
    // (computing the next reference here, one step ahead and interleaved with the RK4 stages, was tried in round 1:
    //  the extra live state pushed the kernel over 128 registers and it ran 7 % slower)
    const double t1 = a.time[i + 1];
    if (a.nsub == 1) rk4_step<true>(load_ac(), X, u_phi, u_v, t1 - t, 1);        // uniform branch on a kernel argument
    else rk4_step(load_ac(), X, u_phi, u_v, t1 - t, a.nsub);
    t = t1;
    if (i + 1 == ev_next) {            // perturbation event (05_test_simulation.py:32)
#pragma unroll
      for (int k = 0; k < 5; ++k) X[k] += a.s.pert_dx[(size_t)k * a.s.n_events + ev];
      ++ev;
      ev_next = ev < ev_end ? a.s.pert_step[ev] : 0x7fffffff;
    }
  }
  if (!isfinite(X[0] + X[1] + X[2] + X[3] + X[4])) flags |= 1;

  if (active) {
#pragma unroll
    for (int k = 0; k < 5; ++k) a.o.X_final[(size_t)k * B + b] = X[k];
    if (a.o.sum_sq_err) a.o.sum_sq_err[b] += sum_sq;
    if (a.o.max_err) a.o.max_err[b] = fmax(a.o.max_err[b], sqrt(max_sq));
    if (a.o.flags) a.o.flags[b] |= flags;
    if (a.o.care_state) {
#pragma unroll
      for (int k = 0; k < kCareState; ++k) a.o.care_state[k * (size_t)B + b] = (k == 2 && cold) ? 0.0 : care[k];
    }
  }
  if (a.o.pop_stats) {                 // population reductions: warp shuffles, one atomic per warp
    const double ws = warp_sum(active ? sum_sq : 0.0);
    const double wm = warp_max(active ? sqrt(max_sq) : 0.0);
    if ((tid & 31) == 0) { atomicAdd(a.o.pop_stats, ws); atomic_max_double(a.o.pop_stats + 1, wm); }
  }
}

template <int UNIFORM>
static int launch_rollout(const RolloutArgs& a, bool logging, cudaStream_t st) {
  const int grid = (a.s.B + kRolloutThreads - 1) / kRolloutThreads;
  const bool logref = a.o.Xr_log || a.o.K_log;
  if (logref) rollout_dfff_kernel<UNIFORM, true, true><<<grid, kRolloutThreads, 0, st>>>(a);
  else if (logging) rollout_dfff_kernel<UNIFORM, true, false><<<grid, kRolloutThreads, 0, st>>>(a);
  else rollout_dfff_kernel<UNIFORM, false, false><<<grid, kRolloutThreads, 0, st>>>(a);
  D2DX_LAUNCH_CHECK("rollout_dfff_kernel");
  return D2DX_OK;
}

int rollout_resident_threads_per_sm() {
  int nb = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rollout_dfff_kernel<D2DX_SEG_CIRCLE, false, false>, kRolloutThreads, 0);
  return nb * kRolloutThreads;
}

}  // namespace d2dx

using namespace d2dx;

extern "C" int d2dx_rollout_dfff(d2dx_handle* h, const d2dx_scenarios* s, const double* time, int32_t i_begin,
                                 int32_t i_end, int32_t nsub, int32_t final_control,
                                 const d2dx_dfff_gains* gains_host, const d2dx_rollout_out* out, void* stream) {
  D2DX_NVTX("d2dx_rollout_dfff");
  D2DX_CHECK_ARG(h && s && time && out, "d2dx_rollout_dfff: null argument");
  D2DX_CHECK_ARG(s->B > 0 && s->traj.n_traj == s->B, "d2dx_rollout_dfff: B=%d, traj.n_traj=%d", s->B, s->traj.n_traj);
  D2DX_CHECK_ARG(s->X0 && s->wind && s->ac && out->X_final, "d2dx_rollout_dfff: X0, wind, ac, X_final are required");
  D2DX_CHECK_ARG(i_begin >= 0 && i_end >= i_begin && nsub >= 1, "d2dx_rollout_dfff: bad range [%d,%d] or nsub=%d", i_begin, i_end, nsub);
  D2DX_CHECK_ARG(s->traj.n_seg > 0 && s->traj.seg_par && s->traj.seg_type && s->traj.first_seg && s->traj.traj_dur,
                 "d2dx_rollout_dfff: incomplete trajectory table");
  RolloutArgs a;
  a.s = *s; a.o = *out; a.time = time;
  a.i_begin = i_begin; a.i_end = i_end; a.nsub = nsub; a.final_control = final_control;
  if (gains_host) a.g = *gains_host; else d2dx_dfff_default_gains(&a.g);
  D2DX_CHECK_ARG(a.g.err_sat[0] >= 0 && a.g.err_sat[1] >= 0 && a.g.err_sat[2] >= 0, "gains: err_sat must be >= 0 (symmetric saturation)");
  a.cc = care_const(a.g);
  D2DX_CHECK_ARG(a.g.q_pos > 0 && a.g.q_psi > 0 && a.g.r_phi > 0 && a.g.r_v > 0, "d2dx_rollout_dfff: Q, R must be positive");
  D2DX_CUDA(cudaSetDevice(h->device));
  const bool logging = out->X_log || out->U_log || out->Xr_log || out->K_log;
  cudaStream_t st = as_stream(stream);
  D2DX_CHECK_ARG(s->traj.uniform_type == 0 || s->traj.n_seg == s->traj.n_traj,
                 "d2dx_rollout_dfff: uniform_type=%d promises one plain segment per trajectory but n_seg=%d != n_traj=%d",
                 s->traj.uniform_type, s->traj.n_seg, s->traj.n_traj);
  switch (s->traj.uniform_type - 1) {
    case D2DX_SEG_CIRCLE: return launch_rollout<D2DX_SEG_CIRCLE>(a, logging, st);
    case D2DX_SEG_POLY: return launch_rollout<D2DX_SEG_POLY>(a, logging, st);
    case D2DX_SEG_LINE: return launch_rollout<D2DX_SEG_LINE>(a, logging, st);
    default: return launch_rollout<-1>(a, logging, st);
  }
}
