// Handle / error plumbing and the batched single-call entry points of the d2d model
// (Trajectory.get, Aircraft.cont_dyn / disc_dyn / cont_jac, DiffFlatness, DFFFController.get).
#include <math.h>
#include <string.h>

#include "d2dx_device.cuh"
#include "d2dx_host.h"

namespace d2dx {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int rollout_resident_threads_per_sm();
int formation_resident_threads_per_sm();
int colloc_resident_threads_per_sm();

constexpr int kThreads = 128;
inline int grid_for(long n) { return (int)((n + kThreads - 1) / kThreads); }

// Trajectory.get for every (time sample, trajectory)
__global__ void __launch_bounds__(kThreads) traj_eval_kernel(const d2dx_traj_table tt, int nT, const double* __restrict__ time,
                                                              double* __restrict__ Y) {
  const int B = tt.n_traj, S = tt.n_seg;
  const long idx = (long)blockIdx.x * kThreads + threadIdx.x;
  if (idx >= (long)B * nT) return;
  const int b = (int)(idx % B), it = (int)(idx / B);
  double te;
  const int seg = composite_locate(tt, b, time[it], te);
  auto P = [&](int k) { return tt.seg_par[(size_t)k * S + seg]; };
  FlatOut o;
  segment_eval<true>(tt.seg_type[seg], P, te, o, &tt);
  double* y = Y + (size_t)it * 8 * B + b;
  y[0] = o.y0x; y[(size_t)B] = o.y0y; y[2 * (size_t)B] = o.y1x; y[3 * (size_t)B] = o.y1y;
  y[4 * (size_t)B] = o.y2x; y[5 * (size_t)B] = o.y2y; y[6 * (size_t)B] = o.y3x; y[7 * (size_t)B] = o.y3y;
}

__device__ __forceinline__ AcPar load_ac(const double* W, const double* ac, int n, int i) {
  AcPar a;
  a.wx = W[i]; a.wy = W[n + i];
  a.n_inv_tau_phi = -1.0 / ac[i]; a.n_inv_tau_v = -1.0 / ac[n + i];
  return a;
}

__global__ void __launch_bounds__(kThreads) cont_dyn_kernel(int n, const double* __restrict__ X, const double* __restrict__ U,
                                                             const double* __restrict__ W, const double* __restrict__ ac,
                                                             double* __restrict__ Xdot) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  const AcPar a = load_ac(W, ac, n, i);
  double d[5];
  cont_dyn(a, X[2 * (size_t)n + i], X[3 * (size_t)n + i], X[4 * (size_t)n + i], U[i], U[n + i], d[0], d[1], d[2], d[3], d[4]);
  for (int k = 0; k < 5; ++k) Xdot[(size_t)k * n + i] = d[k];
}

__global__ void __launch_bounds__(kThreads) disc_dyn_kernel(int n, const double* __restrict__ X, const double* __restrict__ U,
                                                             const double* __restrict__ W, const double* __restrict__ ac,
                                                             double dt, int nsub, double* __restrict__ Xn) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  const AcPar a = load_ac(W, ac, n, i);
  double x[5];
  for (int k = 0; k < 5; ++k) x[k] = X[(size_t)k * n + i];
  rk4_step(a, x, U[i], U[n + i], dt, nsub);
  for (int k = 0; k < 5; ++k) Xn[(size_t)k * n + i] = x[k];
}

__global__ void __launch_bounds__(kThreads) norm_mpi_pi_kernel(int n, const double* __restrict__ v, double* __restrict__ out) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i < n) out[i] = wrap_pi(v[i]);
}

// Aircraft.cont_jac, d2d/dynamic.py:32-43 (both "as written" entries kept)
__global__ void __launch_bounds__(kThreads) cont_jac_kernel(int n, const double* __restrict__ Xr, const double* __restrict__ ac,
                                                             double* __restrict__ A, double* __restrict__ Bm) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  const double psi = Xr[2 * (size_t)n + i], phi = Xr[3 * (size_t)n + i], va = Xr[4 * (size_t)n + i];
  double s, c;
  sincos(psi, &s, &c);
  const double cphi = cos(phi), cphi2 = cphi * cphi, tphi = tan(phi);
  double a[25] = {0};
  a[0 * 5 + 2] = -va * s; a[0 * 5 + 4] = c;
  a[1 * 5 + 2] = va * c;  a[1 * 5 + 4] = s;
  a[2 * 5 + 3] = kG / va / (1.0 + cphi2); a[2 * 5 + 4] = kG / (va * va) * tphi;
  a[3 * 5 + 3] = -1.0 / ac[i];
  a[4 * 5 + 4] = -1.0 / ac[n + i];
  for (int k = 0; k < 25; ++k) A[(size_t)k * n + i] = a[k];
  double bm[10] = {0};
  bm[3 * 2 + 0] = 1.0 / ac[i]; bm[4 * 2 + 1] = 1.0 / ac[n + i];
  for (int k = 0; k < 10; ++k) Bm[(size_t)k * n + i] = bm[k];
}

__global__ void __launch_bounds__(kThreads) flatness_kernel(int n, const double* __restrict__ Ys, const double* __restrict__ W,
                                                             const double* __restrict__ ac, double* __restrict__ Xr,
                                                             double* __restrict__ Ur, double* __restrict__ Xd) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  FlatOut Y;
  Y.y0x = Ys[i]; Y.y0y = Ys[(size_t)n + i]; Y.y1x = Ys[2 * (size_t)n + i]; Y.y1y = Ys[3 * (size_t)n + i];
  Y.y2x = Ys[4 * (size_t)n + i]; Y.y2y = Ys[5 * (size_t)n + i]; Y.y3x = Y.y3y = 0.0;
  FlatState r;
  flatness(Y, W[i], W[n + i], ac[n + i], r);
  Xr[i] = r.x; Xr[(size_t)n + i] = r.y; Xr[2 * (size_t)n + i] = r.psi; Xr[3 * (size_t)n + i] = r.phi; Xr[4 * (size_t)n + i] = r.va;
  Ur[i] = r.u_phi; Ur[(size_t)n + i] = r.u_v;
  if (Xd) {
    Xd[i] = 0.0; Xd[(size_t)n + i] = 0.0; Xd[2 * (size_t)n + i] = r.psidot; Xd[3 * (size_t)n + i] = 0.0; Xd[4 * (size_t)n + i] = r.vadot;
  }
}

__global__ void __launch_bounds__(kThreads) dfff_control_kernel(const d2dx_traj_table tt, const double* __restrict__ X, double t,
                                                                 const double* __restrict__ W, const double* __restrict__ ac,
                                                                 const d2dx_dfff_gains g, double* __restrict__ U,
                                                                 double* __restrict__ Xr, double* __restrict__ K,
                                                                 double* __restrict__ care_state) {
  const int B = tt.n_traj, S = tt.n_seg;
  const int b = blockIdx.x * kThreads + threadIdx.x;
  if (b >= B) return;
  double te;
  const int seg = composite_locate(tt, b, t, te);
  auto P = [&](int k) { return tt.seg_par[(size_t)k * S + seg]; };
  FlatOut Y;
  segment_eval<false>(tt.seg_type[seg], P, te, Y, &tt);
  const AcPar a = load_ac(W, ac, B, b);
  double x[5];
  for (int k = 0; k < 5; ++k) x[k] = X[(size_t)k * B + b];
  const CareConst cc = care_const(g);
  double cs[kCareState] = {};
  if (care_state)
    for (int k = 0; k < kCareState; ++k) cs[k] = care_state[k * (size_t)B + b];
  bool cold = !(cs[2] > 0.0);
  int flags = 0;
  RefCtl rc;
  double u_phi, u_v;
  make_ref(Y, a, ac[B + b], cc, ArrayState{cs}, cold, flags, rc);
  feedback(rc, x, g, u_phi, u_v);
  U[b] = u_phi; U[(size_t)B + b] = u_v;
  if (Xr) { Xr[b] = rc.xr; Xr[(size_t)B + b] = rc.yr; Xr[2 * (size_t)B + b] = rc.psir; Xr[3 * (size_t)B + b] = rc.phir; Xr[4 * (size_t)B + b] = rc.var; }
  if (K) for (int k = 0; k < 6; ++k) K[(size_t)k * B + b] = rc.k[k];
  if (care_state) {
    for (int k = 0; k < kCareState; ++k) care_state[k * (size_t)B + b] = (k == 2 && cold) ? 0.0 : cs[k];
  }
}

// FP64 pipe probe: 16 independent DFMA chains per thread
__global__ void dfma_burn_kernel(int iters, double* sink) {
  double a[16];
  const double x = 1.0 + 1e-9 * threadIdx.x, y = 1e-12 * (blockIdx.x + 1);
#pragma unroll
  for (int k = 0; k < 16; ++k) a[k] = k * 0.5;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = fma(a[k], x, y);
  }
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < 16; ++k) s += a[k];
  if (s == 123.456) *sink = s;
}

__global__ void math_probe_kernel(int n, const double* __restrict__ x, const double* __restrict__ y, double* __restrict__ out) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  double s, c;
  fm::sincos(x[i], s, c);
  out[i] = s; out[(size_t)n + i] = c; out[2 * (size_t)n + i] = fm::atan2(y[i], x[i]); out[3 * (size_t)n + i] = fm::atan(x[i]);
  out[4 * (size_t)n + i] = fm::div(y[i], x[i]); out[5 * (size_t)n + i] = fm::sqrt(fabs(x[i])); out[6 * (size_t)n + i] = fm::rsqrt(fabs(x[i]));
  out[7 * (size_t)n + i] = fm::rcp(x[i]);
  out[8 * (size_t)n + i] = fma(-x[i], fm::rcp_seed(x[i]), 1.0);                 // residuals of the two MUFU seeds
  const double ax = fabs(x[i]), ys = fm::rsqrt_seed(ax);
  out[9 * (size_t)n + i] = fma(-ax * ys, ys, 1.0);
  out[10 * (size_t)n + i] = wrap_pi(x[i]);
  fm::sincos_small(x[i], s, c);
  out[11 * (size_t)n + i] = s; out[12 * (size_t)n + i] = c;
}

}  // namespace d2dx

using namespace d2dx;

extern "C" {

int d2dx_math_probe(d2dx_handle* h, int32_t n, const double* x, const double* y, double* out, void* stream) {
  D2DX_NVTX("d2dx_math_probe");
  D2DX_CHECK_ARG(h && n > 0 && x && y && out, "d2dx_math_probe: bad argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  math_probe_kernel<<<grid_for(n), kThreads, 0, as_stream(stream)>>>(n, x, y, out);
  D2DX_LAUNCH_CHECK("math_probe_kernel");
  return D2DX_OK;
}

int d2dx_dfma_burn(d2dx_handle* h, int32_t blocks, int32_t threads, int32_t iters, double* sink, void* stream) {
  D2DX_NVTX("d2dx_dfma_burn");
  D2DX_CHECK_ARG(h && blocks > 0 && threads > 0 && threads <= 1024 && iters > 0 && sink, "d2dx_dfma_burn: bad argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  dfma_burn_kernel<<<blocks, threads, 0, as_stream(stream)>>>(iters, sink);
  D2DX_LAUNCH_CHECK("dfma_burn_kernel");
  return D2DX_OK;
}

int d2dx_version(void) { return D2DX_VERSION; }
const char* d2dx_last_error(void) { return g_err; }

int d2dx_create(int device, d2dx_handle** out) {
  D2DX_CHECK_ARG(out, "d2dx_create: null out pointer");
  int n = 0;
  D2DX_CUDA(cudaGetDeviceCount(&n));
  D2DX_CHECK_ARG(device >= 0 && device < n, "d2dx_create: device %d out of range (%d CUDA devices)", device, n);
  D2DX_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  D2DX_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return set_error(D2DX_EUNSUPPORTED, "d2dx is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
  d2dx_handle* h = new d2dx_handle;
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  *out = h;
  return D2DX_OK;
}

int d2dx_destroy(d2dx_handle* h) {
  if (!h) return D2DX_OK;
  cudaSetDevice(h->device);
  delete h;
  return D2DX_OK;
}

int d2dx_device_info(d2dx_handle* h, int32_t* w) {
  D2DX_CHECK_ARG(h && w, "d2dx_device_info: null argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  w[0] = h->sm_count;
  w[1] = rollout_resident_threads_per_sm();
  w[2] = formation_resident_threads_per_sm();
  w[3] = colloc_resident_threads_per_sm();
  return D2DX_OK;
}

int d2dx_dfff_default_gains(d2dx_dfff_gains* g) {
  if (!g) return set_error(D2DX_EINVAL, "d2dx_dfff_default_gains: null");
  g->q_pos = 1.0; g->q_psi = 0.1; g->r_phi = 8.0; g->r_v = 1.0;                 // d2d/guidance.py:79
  g->err_sat[0] = 20.0; g->err_sat[1] = 20.0; g->err_sat[2] = kPi / 3; g->err_sat[3] = kPi / 4; g->err_sat[4] = 1.0;   // :69
  const double phisat = 45.0 * (kPi / 180.0);                                  // np.deg2rad(45), :87
  g->u_lo[0] = -phisat; g->u_lo[1] = 4.0; g->u_hi[0] = phisat; g->u_hi[1] = 20.0;
  return D2DX_OK;
}

static int check_table(const d2dx_traj_table* tt, const char* who) {
  D2DX_CHECK_ARG(tt && tt->n_traj > 0 && tt->n_seg > 0, "%s: empty trajectory table", who);
  D2DX_CHECK_ARG(tt->first_seg && tt->n_segs && tt->traj_t0 && tt->traj_dur && tt->seg_type && tt->seg_end && tt->seg_par,
                 "%s: incomplete trajectory table", who);
  return D2DX_OK;
}

int d2dx_traj_eval(d2dx_handle* h, const d2dx_traj_table* tt, int32_t nT, const double* time, double* Y, void* stream) {
  D2DX_NVTX("d2dx_traj_eval");
  D2DX_CHECK_ARG(h && time && Y && nT > 0, "d2dx_traj_eval: bad argument");
  if (int rc = check_table(tt, "d2dx_traj_eval")) return rc;
  D2DX_CUDA(cudaSetDevice(h->device));
  traj_eval_kernel<<<grid_for((long)tt->n_traj * nT), kThreads, 0, as_stream(stream)>>>(*tt, nT, time, Y);
  D2DX_LAUNCH_CHECK("traj_eval_kernel");
  return D2DX_OK;
}

int d2dx_norm_mpi_pi(d2dx_handle* h, int32_t n, const double* v, double* out, void* stream) {
  D2DX_NVTX("d2dx_norm_mpi_pi");
  D2DX_CHECK_ARG(h && n > 0 && v && out, "d2dx_norm_mpi_pi: bad argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  norm_mpi_pi_kernel<<<grid_for(n), kThreads, 0, as_stream(stream)>>>(n, v, out);
  D2DX_LAUNCH_CHECK("norm_mpi_pi_kernel");
  return D2DX_OK;
}

int d2dx_cont_dyn(d2dx_handle* h, int32_t n, const double* X, const double* U, const double* W, const double* ac,
                  double* Xdot, void* stream) {
  D2DX_NVTX("d2dx_cont_dyn");
  D2DX_CHECK_ARG(h && n > 0 && X && U && W && ac && Xdot, "d2dx_cont_dyn: bad argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  cont_dyn_kernel<<<grid_for(n), kThreads, 0, as_stream(stream)>>>(n, X, U, W, ac, Xdot);
  D2DX_LAUNCH_CHECK("cont_dyn_kernel");
  return D2DX_OK;
}

int d2dx_disc_dyn(d2dx_handle* h, int32_t n, const double* X, const double* U, const double* W, const double* ac,
                  double dt, int32_t nsub, double* Xnext, void* stream) {
  D2DX_NVTX("d2dx_disc_dyn");
  D2DX_CHECK_ARG(h && n > 0 && X && U && W && ac && Xnext && nsub >= 1, "d2dx_disc_dyn: bad argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  disc_dyn_kernel<<<grid_for(n), kThreads, 0, as_stream(stream)>>>(n, X, U, W, ac, dt, nsub, Xnext);
  D2DX_LAUNCH_CHECK("disc_dyn_kernel");
  return D2DX_OK;
}

int d2dx_cont_jac(d2dx_handle* h, int32_t n, const double* Xr, const double* ac, double* A, double* Bm, void* stream) {
  D2DX_NVTX("d2dx_cont_jac");
  D2DX_CHECK_ARG(h && n > 0 && Xr && ac && A && Bm, "d2dx_cont_jac: bad argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  cont_jac_kernel<<<grid_for(n), kThreads, 0, as_stream(stream)>>>(n, Xr, ac, A, Bm);
  D2DX_LAUNCH_CHECK("cont_jac_kernel");
  return D2DX_OK;
}

int d2dx_flatness(d2dx_handle* h, int32_t n, const double* Ys, const double* W, const double* ac, double* Xr, double* Ur,
                  double* Xrdot, void* stream) {
  D2DX_NVTX("d2dx_flatness");
  D2DX_CHECK_ARG(h && n > 0 && Ys && W && ac && Xr && Ur, "d2dx_flatness: bad argument");
  D2DX_CUDA(cudaSetDevice(h->device));
  flatness_kernel<<<grid_for(n), kThreads, 0, as_stream(stream)>>>(n, Ys, W, ac, Xr, Ur, Xrdot);
  D2DX_LAUNCH_CHECK("flatness_kernel");
  return D2DX_OK;
}

int d2dx_dfff_control(d2dx_handle* h, const d2dx_traj_table* tt, const double* X, double t, const double* W,
                      const double* ac, const d2dx_dfff_gains* gains_host, double* U, double* Xr, double* K,
                      double* care_state, void* stream) {
  D2DX_NVTX("d2dx_dfff_control");
  D2DX_CHECK_ARG(h && X && W && ac && U, "d2dx_dfff_control: bad argument");
  if (int rc = check_table(tt, "d2dx_dfff_control")) return rc;
  d2dx_dfff_gains g;
  if (gains_host) g = *gains_host; else d2dx_dfff_default_gains(&g);
  D2DX_CHECK_ARG(g.err_sat[0] >= 0 && g.err_sat[1] >= 0 && g.err_sat[2] >= 0, "gains: err_sat must be >= 0 (symmetric saturation)");
  D2DX_CUDA(cudaSetDevice(h->device));
  dfff_control_kernel<<<grid_for(tt->n_traj), kThreads, 0, as_stream(stream)>>>(*tt, X, t, W, ac, g, U, Xr, K, care_state);
  D2DX_LAUNCH_CHECK("dfff_control_kernel");
  return D2DX_OK;
}

}  // extern "C"
