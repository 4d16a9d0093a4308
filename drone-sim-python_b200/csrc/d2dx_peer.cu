// Aircraft-sharded collocation evaluation in ONE kernel per rank, exchanging over NVLink peer memory (SURVEY 8e: C4, one
// problem -- or a batch of problems -- split by aircraft over the GPUs of one box).
//
// Every rank owns an exchange buffer (cudaMalloc) that all other ranks map (CUDA IPC between processes, plain pointers
// inside one process).  One evaluation =
//   phase 0  each block stores its tiles of the OWNED aircraft's x, y straight from free_local into every peer's position
//            table -- for ALL its tiles before anything else;
//   phase 1  residual / Jacobian / input cost / gradient of psi, phi, v of the owned aircraft (needs no remote data: this is
//            what hides the NVLink latency);
//   phase 2  read the same tile of every peer from the own table (spinning until it has arrived), stage all positions in
//            shared memory;
//   phase 3  collision terms of the owned aircraft against every other aircraft, gradient of x, y;
//   phase 4  the block of a problem's last tile sums this rank's per-tile partials, writes the four sums to every rank and
//            adds up the sums of all ranks: every rank ends with the same, deterministic total cost.
// The exchange carries its own arrival flags ("LL" protocol, as in NCCL's low-latency path): every double travels as two
// 8-byte words {half of the bits, evaluation number}; an 8-byte store arrives whole, so a receiver that reads both
// evaluation numbers it expects holds valid data -- no memory fence (MEMBAR.SYS cost ~4 us per use in the fence + flag
// version, profiles/r2_sharded_c4.md), no separate flag, one NVLink traversal of latency.  Twice the bytes, of a 128 kB
// exchange.  There is no collective call and no host synchronisation; the evaluation number lives on the
// device, so the launch can be captured in a CUDA graph and replayed.  Phase 4 doubles as the barrier that keeps
// evaluation e + 1 from overwriting tables a slower rank still reads in evaluation e.
// A peer that never answers costs `spin_cycles` per wait and is reported by d2dx_peer_status (never a hang).
#include <string.h>

#include "d2dx_colloc_dev.cuh"
#include "d2dx_host.h"

struct d2dx_peer {
  int device, world, rank, max_prob, n_total, N, ntiles;
  unsigned char* local;                       // this rank's exchange buffer
  unsigned char* base[D2DX_PEER_MAX_WORLD];   // every rank's buffer as mapped here (base[rank] == local)
  bool ipc_opened[D2DX_PEER_MAX_WORLD];
  bool connected;
  size_t bytes, off_cpart, off_lpart, off_pos;
  int resident_blocks;
};

namespace d2dx {

constexpr int kPeerWarps = 8;

struct PeerCtrl {
  uint32_t epoch, done_blocks, timeouts, pad;
  unsigned long long stamp[8];   // %globaltimer [ns] of the last evaluation, block 0 / the last block of problem 0:
                                 // 0 start, 1 tiles published, 2 local work done, 3 peers' positions arrived, 4 pair terms done,
                                 // 5 own cost sums sent, 6 all ranks' sums arrived (cost written), 7 block 0 leaves
};

struct PeerArgs {
  CollocArgs c;                  // c.p = the local shard as a problem of n_own aircraft; outputs shard-local
  int n_total, a_lo;             // owned aircraft are global [a_lo, a_lo + c.p.n_ac) of n_total
  int world, rank, max_prob, ntiles;
  unsigned char* base[D2DX_PEER_MAX_WORLD];
  size_t off_cpart, off_lpart, off_pos;
  long long spin_cycles;
};

// LL words: {low 32 bits | evaluation number << 32}, {high 32 bits | evaluation number << 32}, stored and loaded as one
// 16-byte access (each 8-byte half is delivered whole)
__device__ __forceinline__ void ll_store(unsigned long long* slot, double v, uint32_t epoch) {
  const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(v));
  const unsigned long long e = static_cast<unsigned long long>(epoch) << 32;
  const unsigned long long w0 = (bits & 0xffffffffull) | e, w1 = (bits >> 32) | e;
  asm volatile("st.relaxed.sys.global.v2.b64 [%0], {%1, %2};" :: "l"(slot), "l"(w0), "l"(w1) : "memory");
}
// true when both halves carry `epoch`
__device__ __forceinline__ bool ll_try_load(const unsigned long long* slot, uint32_t epoch, double& v) {
  unsigned long long w0, w1;
  asm volatile("ld.relaxed.sys.global.v2.b64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(slot) : "memory");
  v = __longlong_as_double(static_cast<long long>((w0 & 0xffffffffull) | (w1 << 32)));
  return static_cast<uint32_t>(w0 >> 32) == epoch && static_cast<uint32_t>(w1 >> 32) == epoch;
}
// spins until the value of this evaluation has arrived; false on timeout (v then undefined)
__device__ __forceinline__ bool ll_load(const unsigned long long* slot, uint32_t epoch, long long spin_cycles, double& v) {
  if (ll_try_load(slot, epoch, v)) return true;
  const long long t0 = clock64();
  while (!ll_try_load(slot, epoch, v)) {
    if (clock64() - t0 > spin_cycles) return false;
  }
  return true;
}
__device__ __forceinline__ unsigned long long now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

__global__ void __launch_bounds__(kPeerWarps * 32, 3) colloc_peer_kernel(const __grid_constant__ PeerArgs g) {
  extern __shared__ double sm[];                   // [n_total][2][32] positions, then [W][4] reduction scratch
  const CollocArgs& a = g.c;
  const d2dx_colloc_problem& P = a.p;
  const int N = P.N, n_own = P.n_ac, n_total = g.n_total;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, W = blockDim.x >> 5;
  double* spos = sm + lane;
  double* sred = sm + n_total * 64;
  unsigned char* mine = g.base[g.rank];
  PeerCtrl* ctrl = reinterpret_cast<PeerCtrl*>(mine);
  const uint32_t epoch = *reinterpret_cast<volatile uint32_t*>(&ctrl->epoch) + 1u;
  if (blockIdx.x == 0 && threadIdx.x == 0) ctrl->stamp[0] = now_ns();
  const bool want_cg = (a.what & (D2DX_EVAL_COST | D2DX_EVAL_GRAD)) != 0;
  const bool use_col = want_cg && enabled(P.kcol) && n_total > 1;
  const bool use_obs = want_cg && enabled(P.kobs) && P.n_obs > 0;
  const int n_items = a.n_prob * g.ntiles;
  const unsigned long long* pos_in = reinterpret_cast<const unsigned long long*>(mine + g.off_pos);
  const unsigned long long* cpart_in = reinterpret_cast<const unsigned long long*>(mine + g.off_cpart);
  unsigned long long* lpart = reinterpret_cast<unsigned long long*>(mine + g.off_lpart);

  // ---- sweep A: publish the owned positions of EVERY tile this block will process before anything else: by the time the
  // block comes to a tile's collision terms the peers' stores for it have long landed (the NVLink latency of a batch is
  // paid once, not per tile) ----
  if (use_col && g.world > 1) {
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int prob = item / g.ntiles, tile = item - prob * g.ntiles;
      const int i = tile * 32 + lane;
      if (i < N) {
        const double* fr = a.free_ + (size_t)prob * a.n_free;
        for (int a_l = w; a_l < n_own; a_l += W) {
          const double x = fr[(3 * a_l) * N + i], y = fr[(3 * a_l + 1) * N + i];
          const size_t o = ((((size_t)prob * n_total + g.a_lo + a_l) * 2) * N + i) * 2;      // two words per value
          for (int r = 0; r < g.world; ++r) {
            if (r == g.rank) continue;
            unsigned long long* dst = reinterpret_cast<unsigned long long*>(g.base[r] + g.off_pos);
            ll_store(dst + o, x, epoch); ll_store(dst + o + 2 * (size_t)N, y, epoch);
          }
        }
      }
    }
  }
  const bool stamper = blockIdx.x == 0 && threadIdx.x == 0;
  if (stamper) ctrl->stamp[1] = now_ns();

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {   // same order on every rank: see the deadlock note in DESIGN
    const int prob = item / g.ntiles, tile = item - prob * g.ntiles;
    const int i = tile * 32 + lane;
    const bool valid = i < N;
    const double* fr = a.free_ + (size_t)prob * a.n_free;
    __syncthreads();                               // shared memory of the previous item is free

    if (use_col) {                                 // the owned positions of this tile into shared memory
      for (int a_l = w; a_l < n_own; a_l += W) {
        const int gl = g.a_lo + a_l;
        double x = 0.0, y = 0.0;
        if (valid) { x = fr[(3 * a_l) * N + i]; y = fr[(3 * a_l + 1) * N + i]; }
        spos[(gl * 2) * 32] = x; spos[(gl * 2 + 1) * 32] = y;
      }
    }

    // ---- phase 1: everything that needs no remote data ----
    double s_v = 0.0, s_phi = 0.0, s_obs = 0.0, s_col = 0.0;
    if (valid) {
      for (int a_l = w; a_l < n_own; a_l += W) {
        const int ox = 3 * a_l * N + i;
        colloc_node<false>(a, fr, prob, a_l, i, fr[ox], fr[ox + N], 0.0, 0.0, want_cg, s_v, s_phi);
      }
    }

    if (stamper && item == 0) ctrl->stamp[2] = now_ns();
    // ---- phase 2: the peers' positions of this tile ----
    if (use_col) {
      bool arrived = true;
      for (int gl = w; gl < n_total; gl += W) {
        if (gl >= g.a_lo && gl < g.a_lo + n_own) continue;
        double x = 0.0, y = 0.0;
        if (valid) {
          const size_t o = ((((size_t)prob * n_total + gl) * 2) * N + i) * 2;
          arrived = ll_load(pos_in + o, epoch, g.spin_cycles, x) && arrived;
          arrived = ll_load(pos_in + o + 2 * (size_t)N, epoch, g.spin_cycles, y) && arrived;
        }
        spos[(gl * 2) * 32] = x; spos[(gl * 2 + 1) * 32] = y;
      }
      if (!arrived) atomicAdd(&ctrl->timeouts, 1u);
      __syncthreads();
    }
    if (stamper && item == 0) ctrl->stamp[3] = now_ns();

    // ---- phase 3: obstacle and collision terms of the owned aircraft, gradient of x, y ----
    if (want_cg && valid) {
      for (int a_l = w; a_l < n_own; a_l += W) {
        const int gl = g.a_lo + a_l;
        const int ox = 3 * a_l * N + i;
        const double x = fr[ox], y = fr[ox + N];
        double gx = 0.0, gy = 0.0;
        if (use_obs && gl == 0) obstacle_terms(P, a.sN, x, y, s_obs, gx, gy);
        if (use_col) {
          const int b_lo = P.col_all_pairs ? 0 : (gl == 0 ? 1 : 0);
          const int b_hi = P.col_all_pairs ? n_total : (gl == 0 ? 2 : (gl == 1 ? 1 : 0));
          const double* pb = spos + (b_lo * 2) * 32;
#pragma unroll 4
          for (int b = b_lo; b < b_hi; ++b, pb += 64) {
            if (b == gl) continue;
            const double dx = x - pb[0], dy = y - pb[32];
            const double es = fm::exp_neg(a.nkr2 * fma(dx, dx, dy * dy));
            if (gl < b) s_col += es;               // each pair counted once, at the owner of its lower-index aircraft
            const double wgt = a.cw * es;
            gx = fma(wgt, dx, gx); gy = fma(wgt, dy, gy);
          }
        }
        if (a.what & D2DX_EVAL_GRAD) {
          double* go = a.grad + (size_t)prob * a.n_free;
          go[ox] = gx; go[ox + N] = gy;
        }
      }
    }

    if (stamper && item == 0) ctrl->stamp[4] = now_ns();
    // instance constraints of the owned aircraft: first tile of each problem
    if (tile == 0) {
      for (int k = threadIdx.x; k < P.n_inst; k += blockDim.x) {
        if (a.what & D2DX_EVAL_RESIDUAL)
          a.res[(size_t)prob * a.n_con + 3 * n_own * (N - 1) + k] = fr[P.inst_var[k] * N + P.inst_node[k]] - P.inst_val[k];
        if (a.what & D2DX_EVAL_JAC) a.jac[(size_t)prob * a.nnz + (a.nnz - P.n_inst) + k] = 1.0;
      }
    }

    // ---- phase 4: cost partials; the last block of the problem exchanges them (also the end-of-evaluation barrier) ----
    const double v4[4] = {warp_sum(s_v), warp_sum(s_phi), warp_sum(s_obs), warp_sum(s_col)};
    if (lane == 0) { sred[w * 4 + 0] = v4[0]; sred[w * 4 + 1] = v4[1]; sred[w * 4 + 2] = v4[2]; sred[w * 4 + 3] = v4[3]; }
    __syncthreads();
    if (w == 0) {
      double b4[4] = {0.0, 0.0, 0.0, 0.0};
      for (int q = 0; q < W; ++q) { b4[0] += sred[q * 4]; b4[1] += sred[q * 4 + 1]; b4[2] += sred[q * 4 + 2]; b4[3] += sred[q * 4 + 3]; }
      // the block's four sums go to its LOCAL slot, again as self-validating words: the block of the problem's LAST tile
      // (every other tile of the problem has a lower item index: in progress or done, on any rank) collects them without
      // atomics or fences, in a fixed order
      unsigned long long* parts = lpart + ((size_t)prob * g.ntiles * 4) * 2;
      if (lane < 4) ll_store(parts + (tile * 4 + lane) * 2, lane == 0 ? b4[0] : (lane == 1 ? b4[1] : (lane == 2 ? b4[2] : b4[3])), epoch);
      if (tile == g.ntiles - 1) {
        double t4[4] = {0.0, 0.0, 0.0, 0.0};
        bool arrived = true;
        for (int t = lane; t < g.ntiles; t += 32) {
          double v[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) arrived = ll_load(parts + (t * 4 + k) * 2, epoch, g.spin_cycles, v[k]) && arrived;
#pragma unroll
          for (int k = 0; k < 4; ++k) t4[k] += v[k];
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) t4[k] = warp_sum(t4[k]);
        // this rank's four sums -> every rank (lane k sends sum k; own buffer included), then lane r collects rank r's
        if (lane < 4) {
          const double mine_k = lane == 0 ? t4[0] : (lane == 1 ? t4[1] : (lane == 2 ? t4[2] : t4[3]));
          for (int r = 0; r < g.world; ++r)
            ll_store(reinterpret_cast<unsigned long long*>(g.base[r] + g.off_cpart) + (((size_t)g.rank * g.max_prob + prob) * 4 + lane) * 2, mine_k, epoch);
        }
        if (lane == 0 && prob == 0) ctrl->stamp[5] = now_ns();
        double r4[4] = {0.0, 0.0, 0.0, 0.0};
        if (lane < g.world) {
          const unsigned long long* cp = cpart_in + (((size_t)lane * g.max_prob + prob) * 4) * 2;
#pragma unroll
          for (int k = 0; k < 4; ++k) arrived = ll_load(cp + 2 * k, epoch, g.spin_cycles, r4[k]) && arrived;
        }
        if (!arrived) atomicAdd(&ctrl->timeouts, 1u);
        double s4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) s4[k] = warp_sum(r4[k]);     // the same lanes hold the same values on every rank: identical totals
        if (lane == 0 && (a.what & D2DX_EVAL_COST)) a.cost[prob] = colloc_cost_from_sums(a, s4, use_obs, use_col);
        if (lane == 0 && prob == 0) ctrl->stamp[6] = now_ns();
      }
    }
  }

  // the last block to leave advances the evaluation number (all blocks read it long ago)
  __syncthreads();
  if (stamper) ctrl->stamp[7] = now_ns();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&ctrl->done_blocks, 1u) == gridDim.x - 1) {
      ctrl->done_blocks = 0;
      __threadfence();
      *reinterpret_cast<volatile uint32_t*>(&ctrl->epoch) = epoch;
    }
  }
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace d2dx

using namespace d2dx;

extern "C" {

int d2dx_peer_create(d2dx_handle* h, int32_t world, int32_t rank, int32_t max_prob, int32_t n_ac_total, int32_t N, d2dx_peer** out) {
  D2DX_CHECK_ARG(h && out, "d2dx_peer_create: null argument");
  D2DX_CHECK_ARG(world >= 1 && world <= D2DX_PEER_MAX_WORLD && rank >= 0 && rank < world, "d2dx_peer_create: rank %d of %d (max %d)", rank, world,
                 D2DX_PEER_MAX_WORLD);
  D2DX_CHECK_ARG(max_prob >= 1 && n_ac_total >= 1 && N >= 2, "d2dx_peer_create: max_prob=%d n_ac_total=%d N=%d", max_prob, n_ac_total, N);
  D2DX_CHECK_ARG((size_t)n_ac_total * 64 * sizeof(double) + kPeerWarps * 4 * sizeof(double) <= 200 * 1024,
                 "d2dx_peer_create: %d aircraft do not fit the shared-memory position tile", n_ac_total);
  D2DX_CUDA(cudaSetDevice(h->device));
  d2dx_peer* p = new d2dx_peer;
  memset(p, 0, sizeof(*p));
  p->device = h->device; p->world = world; p->rank = rank; p->max_prob = max_prob; p->n_total = n_ac_total; p->N = N;
  p->ntiles = (N + 31) / 32;
  size_t o = align_up(sizeof(PeerCtrl), 256);
  p->off_cpart = o; o = align_up(o + 2 * sizeof(double) * (size_t)world * max_prob * 4, 256);        // LL: two words per value
  p->off_lpart = o; o = align_up(o + 2 * sizeof(double) * (size_t)max_prob * p->ntiles * 4, 256);
  p->off_pos = o; o = align_up(o + 2 * sizeof(double) * (size_t)max_prob * n_ac_total * 2 * N, 256);  // LL: two words per value
  p->bytes = o;
  void* buf = nullptr;
  cudaError_t e = cudaMalloc(&buf, p->bytes);
  if (e != cudaSuccess) { delete p; return set_error(D2DX_ECUDA, "d2dx_peer_create: cudaMalloc(%zu): %s", o, cudaGetErrorString(e)); }
  e = cudaMemset(buf, 0, p->bytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { cudaFree(buf); delete p; return set_error(D2DX_ECUDA, "d2dx_peer_create: cudaMemset: %s", cudaGetErrorString(e)); }
  p->local = static_cast<unsigned char*>(buf);
  p->base[rank] = p->local;
  p->connected = world == 1;
  int nb = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, colloc_peer_kernel, kPeerWarps * 32, 0);
  p->resident_blocks = (nb > 0 ? nb : 1) * h->sm_count;
  *out = p;
  return D2DX_OK;
}

int d2dx_peer_ipc_handle(d2dx_peer* p, void* handle_host64) {
  D2DX_CHECK_ARG(p && handle_host64, "d2dx_peer_ipc_handle: null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == D2DX_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
  D2DX_CUDA(cudaSetDevice(p->device));
  cudaIpcMemHandle_t hd;
  D2DX_CUDA(cudaIpcGetMemHandle(&hd, p->local));
  memcpy(handle_host64, &hd, sizeof(hd));
  return D2DX_OK;
}

int d2dx_peer_connect_ipc(d2dx_peer* p, const void* handles_host) {
  D2DX_CHECK_ARG(p && handles_host, "d2dx_peer_connect_ipc: null argument");
  D2DX_CUDA(cudaSetDevice(p->device));
  const unsigned char* hs = static_cast<const unsigned char*>(handles_host);
  for (int r = 0; r < p->world; ++r) {
    if (r == p->rank) continue;
    cudaIpcMemHandle_t hd;
    memcpy(&hd, hs + (size_t)r * D2DX_IPC_HANDLE_BYTES, sizeof(hd));
    void* ptr = nullptr;
    D2DX_CUDA(cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    p->base[r] = static_cast<unsigned char*>(ptr);
    p->ipc_opened[r] = true;
  }
  p->connected = true;
  return D2DX_OK;
}

int d2dx_peer_connect_local(d2dx_peer* p, d2dx_peer* const* peers_host) {
  D2DX_CHECK_ARG(p && peers_host, "d2dx_peer_connect_local: null argument");
  for (int r = 0; r < p->world; ++r) {
    D2DX_CHECK_ARG(peers_host[r] && peers_host[r]->rank == r && peers_host[r]->world == p->world && peers_host[r]->bytes == p->bytes,
                   "d2dx_peer_connect_local: entry %d is not rank %d of the same exchange", r, r);
    if (peers_host[r]->device != p->device) {
      D2DX_CUDA(cudaSetDevice(p->device));
      cudaError_t e = cudaDeviceEnablePeerAccess(peers_host[r]->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
        return set_error(D2DX_ECUDA, "d2dx_peer_connect_local: no peer access %d -> %d: %s", p->device, peers_host[r]->device, cudaGetErrorString(e));
      cudaGetLastError();
    }
    p->base[r] = peers_host[r]->local;
  }
  p->connected = true;
  return D2DX_OK;
}

int d2dx_peer_status(d2dx_peer* p, int32_t* status_host4) {
  D2DX_CHECK_ARG(p && status_host4, "d2dx_peer_status: null argument");
  D2DX_CUDA(cudaSetDevice(p->device));
  PeerCtrl c;
  D2DX_CUDA(cudaMemcpy(&c, p->local, sizeof(c), cudaMemcpyDeviceToHost));
  status_host4[0] = (int32_t)c.timeouts; status_host4[1] = (int32_t)c.epoch; status_host4[2] = p->resident_blocks;
  status_host4[3] = (int32_t)(p->bytes >> 10);
  return D2DX_OK;
}

int d2dx_peer_timeline(d2dx_peer* p, uint64_t* stamps_host8) {
  D2DX_CHECK_ARG(p && stamps_host8, "d2dx_peer_timeline: null argument");
  D2DX_CUDA(cudaSetDevice(p->device));
  PeerCtrl c;
  D2DX_CUDA(cudaMemcpy(&c, p->local, sizeof(c), cudaMemcpyDeviceToHost));
  for (int k = 0; k < 8; ++k) stamps_host8[k] = c.stamp[k];
  return D2DX_OK;
}

int d2dx_peer_destroy(d2dx_peer* p) {
  if (!p) return D2DX_OK;
  cudaSetDevice(p->device);
  for (int r = 0; r < p->world; ++r)
    if (p->ipc_opened[r] && p->base[r]) cudaIpcCloseMemHandle(p->base[r]);
  if (p->local) cudaFree(p->local);
  delete p;
  return D2DX_OK;
}

int d2dx_colloc_eval_peer(d2dx_handle* h, d2dx_peer* peer, const d2dx_colloc_problem* p, int32_t n_prob, int32_t a_lo,
                          const double* free_local, uint32_t what, double* residual, double* jac, double* cost, double* grad,
                          void* stream) {
  D2DX_NVTX("d2dx_colloc_eval_peer");
  D2DX_CHECK_ARG(h && peer && p && free_local, "d2dx_colloc_eval_peer: null argument");
  D2DX_CHECK_ARG(peer->connected, "d2dx_colloc_eval_peer: the exchange is not connected (d2dx_peer_connect_ipc / _local)");
  D2DX_CHECK_ARG(p->N == peer->N && n_prob >= 1 && n_prob <= peer->max_prob, "d2dx_colloc_eval_peer: N=%d (exchange %d), n_prob=%d (max %d)", p->N,
                 peer->N, n_prob, peer->max_prob);
  D2DX_CHECK_ARG(p->n_ac >= 1 && a_lo >= 0 && a_lo + p->n_ac <= peer->n_total, "d2dx_colloc_eval_peer: shard [%d,+%d) of %d", a_lo, p->n_ac,
                 peer->n_total);
  D2DX_CHECK_ARG(p->h > 0 && p->in_div >= 1 && p->n_obs >= 0 && p->n_obs <= D2DX_MAX_OBSTACLES, "d2dx_colloc_eval_peer: bad problem description");
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_RESIDUAL) || residual, "d2dx_colloc_eval_peer: residual requested but NULL");
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_JAC) || jac, "d2dx_colloc_eval_peer: jacobian requested but NULL");
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_COST) || cost, "d2dx_colloc_eval_peer: cost requested but NULL");
  D2DX_CHECK_ARG(!(what & D2DX_EVAL_GRAD) || grad, "d2dx_colloc_eval_peer: gradient requested but NULL");
  PeerArgs g;
  memset(&g, 0, sizeof(g));
  CollocArgs& a = g.c;
  a.p = *p; a.n_prob = n_prob; a.layout = D2DX_JAC_COMPACT; a.what = what; a.free_ = free_local;
  a.res = residual; a.jac = jac; a.cost = cost; a.grad = grad; a.scratch = nullptr;
  a.TN = 32; a.APP = kPeerWarps; a.ntiles = peer->ntiles; a.nparts = peer->ntiles; a.ticket_mode = 1;
  a.n_free = 5 * p->n_ac * p->N; a.n_con = 3 * p->n_ac * (p->N - 1) + p->n_inst; a.nnz = 12L * p->n_ac * (p->N - 1) + p->n_inst;
  colloc_constants(a);
  g.n_total = peer->n_total; g.a_lo = a_lo;
  g.world = peer->world; g.rank = peer->rank; g.max_prob = peer->max_prob; g.ntiles = peer->ntiles;
  for (int r = 0; r < peer->world; ++r) g.base[r] = peer->base[r];
  g.off_cpart = peer->off_cpart; g.off_lpart = peer->off_lpart; g.off_pos = peer->off_pos;
  g.spin_cycles = 2000000000LL;                  // ~1 s at 1.9 GHz
  D2DX_CUDA(cudaSetDevice(h->device));
  const size_t smem = ((size_t)peer->n_total * 64 + kPeerWarps * 4) * sizeof(double);
  if (smem > 48 * 1024) D2DX_CUDA(cudaFuncSetAttribute(colloc_peer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int items = n_prob * peer->ntiles;
  const int warps = p->n_ac < kPeerWarps ? p->n_ac : kPeerWarps;
  int nb = 0;                                    // co-resident blocks of THIS launch shape: every waiting block must be resident
  D2DX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, colloc_peer_kernel, warps * 32, smem));
  const int resident = (nb > 0 ? nb : 1) * h->sm_count;
  const int grid = items < resident ? items : resident;
  colloc_peer_kernel<<<grid, warps * 32, smem, as_stream(stream)>>>(g);
  D2DX_LAUNCH_CHECK("colloc_peer_kernel");
  return D2DX_OK;
}

}  // extern "C"
