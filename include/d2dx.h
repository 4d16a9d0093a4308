/* d2dx -- C ABI of the B200-native d2d trajectory-evaluation engine.
 *
 * The reference (rajashree-srikanth/drone-sim-python) is pure Python and has no FFI of its own: the
 * drop-in boundary is the duck-typed `d2d` call surface (SURVEY.md section 8b).  Every entry point
 * below names the reference interface it replaces (file:line relative to the reference's `src/`).
 * A ctypes binding of exactly these symbols is what a maintainer adds on the reference side
 * (INTEGRATION.md); the package `d2d_b200` ships that binding together with `d2d`-compatible classes.
 *
 * Conventions
 *   - plain C: pointers and sizes only; no torch / C++ types cross the boundary;
 *   - every `double*`, `int32_t*`, `int64_t*` is a DEVICE pointer owned by the caller unless the
 *     parameter is documented as "host";
 *   - arrays are structure-of-arrays with the batch index fastest: `X[5][B]` means element
 *     (state k, scenario b) lives at `X[k*B + b]`;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream),
 *     allocates nothing and keeps no hidden state;
 *   - return value 0 = OK, otherwise a D2DX_E* code with text in d2dx_last_error() (thread-local);
 *   - all arithmetic is IEEE fp64.
 */
#ifndef D2DX_H
#define D2DX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D2DX_VERSION 106

enum { D2DX_OK = 0, D2DX_EINVAL = 1, D2DX_ECUDA = 2, D2DX_EUNSUPPORTED = 3 };

typedef struct d2dx_handle d2dx_handle;

/* -------- life cycle -------- */
int d2dx_version(void);
const char* d2dx_last_error(void);
/* binds a handle to CUDA device `device` (no allocation beyond a few bytes of scratch) */
int d2dx_create(int device, d2dx_handle** out);
int d2dx_destroy(d2dx_handle* h);
/* properties: what[0]=SM count, [1]=max resident threads of the DFFF rollout kernel per SM,
 * [2]=same for the formation kernel, [3]=same for the collocation kernel (host int array[4]) */
int d2dx_device_info(d2dx_handle* h, int32_t* what_host4);

/* -------- trajectory table --------
 * One trajectory per aircraft-scenario, made of >= 1 segments.
 * Replaces the Trajectory class family: TrajectoryLine d2d/trajectory.py:125-141, TrajectoryCircle
 * :143-160, MinSnapPoly/PolynomialOne :47-82,166-187, CompositeTraj :190-208, SpaceIndexedTraj
 * :220-241 (line geometry + polynomial dynamics, as TrajSiDemo d2d/trajectory_factory.py:177-185),
 * TrajSlalom d2d/trajectory_factory.py:121-145. */
enum {
  D2DX_SEG_LINE = 0,    /* par: 0 t0 | 1 p1x 2 p1y | 3 (un*v)x 4 (un*v)y                         */
  D2DX_SEG_CIRCLE = 1,  /* par: 0 t0 | 1 cx 2 cy | 3 r | 4 omega=v/r | 5 alpha0                   */
  D2DX_SEG_SLALOM = 2,  /* par: 0 t0 | 1 p1x 2 p1y | 3 (un*v)x 4 (un*v)y | 5 phase                */
  D2DX_SEG_POLY = 3,    /* par: 0 t0 | 1..8 x coefs[0][0..7] | 9..16 y coefs[0][0..7]             */
  D2DX_SEG_SI_LINE = 4, /* SpaceIndexedTraj, line geometry: 0 unused | 1 p1x 2 p1y 3 (un*v)x 4 (un*v)y (geometry, t0=0)
                           dynamics lambda(t): slot 16 = 0 -> polynomial 5..12 coefs[0][0..7] in (t - slot 14) (PolynomialOne,
                           AffineOne, CstOne with slot 14 = 0; one linear piece of FooOne, d2d/trajectory_factory.py:225-234,
                           with slot 14 = its knot); slot 16 = 1 -> SinOne (d2d/trajectory.py:26-38): 5 c | 6 a | 7 om | 8 t0 */
  D2DX_SEG_TABLE = 5,   /* par: 0 t0(unused) | 1 first row in the tab_* arrays | 2 number of rows:
                           TrajTabulated, d2d/trajectory_factory.py:149-171 (zero-order lookup of a
                           planner solution: row = first sample time >= t, row 0 past the end)       */
  D2DX_SEG_SI_CIRCLE = 6 /* SpaceIndexedTraj, circle geometry (as TrajSiSpline's, d2d/trajectory_factory.py:246): 0 t0 of the
                           geometry | 1 cx 2 cy | 3 r | 4 omega | 13 alpha0; dynamics as D2DX_SEG_SI_LINE               */
};
#define D2DX_SEG_NPAR 17

typedef struct {
  int32_t n_traj;            /* = B                                                              */
  int32_t n_seg;             /* total number of segments S                                       */
  const int32_t* first_seg;  /* [B]  index of the trajectory's first segment                     */
  const int32_t* n_segs;     /* [B]  number of segments (>= 1)                                   */
  const double* traj_t0;     /* [B]  CompositeTraj.t0                                            */
  const double* traj_dur;    /* [B]  CompositeTraj.duration (np.sum of step durations);
                                     <= 0 marks a plain (non-composite) trajectory: no fmod      */
  const int32_t* seg_type;   /* [S]                                                              */
  const double* seg_end;     /* [S]  CompositeTraj.steps_end (np.cumsum)                         */
  const double* seg_par;     /* [D2DX_SEG_NPAR][S]                                               */
  int32_t uniform_type;      /* 0 (what a zero-initialised table gets): mixed -- the generic kernel reads the whole table;
                                1 + D2DX_SEG_*: EVERY trajectory is ONE plain segment of that type, n_seg == n_traj and
                                first_seg[b] == b -- selects a specialised kernel that reads seg_par only (n_segs,
                                traj_t0, traj_dur, seg_type, seg_end are not consulted).  seg_par should be 16-byte
                                aligned (rows then move as TMA bulk copies; plain loads otherwise)               */
  /* sample tables of D2DX_SEG_TABLE segments (all NULL when there is none): time, x, y and the
   * ground velocity v cos(psi) + wx, v sin(psi) + wy of each stored sample                        */
  int32_t n_tab;
  const double* tab_time;    /* [n_tab] */
  const double* tab_x;       /* [n_tab] */
  const double* tab_y;       /* [n_tab] */
  const double* tab_vx;      /* [n_tab] */
  const double* tab_vy;      /* [n_tab] */
} d2dx_traj_table;

/* Trajectory.get(t) for every trajectory and every t: Y[nT][8][B], row 2*k+c = k-th derivative of
 * component c (d2d/trajectory.py:88-122).  `time` is a device array [nT]. */
int d2dx_traj_eval(d2dx_handle* h, const d2dx_traj_table* tt, int32_t nT, const double* time,
                   double* Y, void* stream);

/* -------- single calls of the d2d model (batched over n) -------- */
/* Aircraft.cont_dyn, d2d/dynamic.py:14-23.  X[5][n], U[2][n], W[2][n], ac[2][n]=(tau_phi,tau_v) */
int d2dx_cont_dyn(d2dx_handle* h, int32_t n, const double* X, const double* U, const double* W,
                  const double* ac, double* Xdot, void* stream);
/* Aircraft.disc_dyn, d2d/dynamic.py:25-28, with fixed-step RK4 (nsub sub-steps, ZOH) for LSODA */
int d2dx_disc_dyn(d2dx_handle* h, int32_t n, const double* X, const double* U, const double* W,
                  const double* ac, double dt, int32_t nsub, double* Xnext, void* stream);
/* Aircraft.cont_jac, d2d/dynamic.py:32-43.  A[25][n] (row-major 5x5), Bm[10][n] (row-major 5x2) */
int d2dx_cont_jac(d2dx_handle* h, int32_t n, const double* Xr, const double* ac, double* A,
                  double* Bm, void* stream);
/* DiffFlatness.state_and_input_from_output, d2d/guidance.py:23-47.  Ys[8][n] as in d2dx_traj_eval */
int d2dx_flatness(d2dx_handle* h, int32_t n, const double* Ys, const double* W, const double* ac,
                  double* Xr, double* Ur, double* Xrdot, void* stream);

/* norm_mpi_pi, d2d/utils.py:7 / d2d/guidance.py:10: out[i] = (v[i] + pi) % (2 pi) - pi with NumPy's floored modulo */
int d2dx_norm_mpi_pi(d2dx_handle* h, int32_t n, const double* v, double* out, void* stream);

/* controller constants of DFFFController.get, d2d/guidance.py:69,79,87-88 */
typedef struct {
  double q_pos, q_psi;       /* Q = diag(q_pos, q_pos, q_psi)   reference: 1, 0.1                */
  double r_phi, r_v;         /* R = diag(r_phi, r_v)            reference: 8, 1                  */
  double err_sat[5];         /* reference: 20, 20, pi/3, pi/4, 1                                 */
  double u_lo[2], u_hi[2];   /* reference: (-45deg, 4), (45deg, 20)                              */
} d2dx_dfff_gains;
int d2dx_dfff_default_gains(d2dx_dfff_gains* g_host);

/* Rows of the Riccati warm start (care_state): the previous solution (C, S, alpha; alpha = 0 when cold), then the changes of
 * theta and of alpha over the last three control steps, from which the next solution is extrapolated. */
#define D2DX_CARE_STATE_ROWS 9

/* DFFFController.get(X, t), d2d/guidance.py:62-91, for B aircraft at one time `t`.
 * Outputs U[2][B]; optional Xr[5][B], K[6][B] (row-major 2x3 = K[:, :3]; K[:, 3:] is zero).
 * care_state[D2DX_CARE_STATE_ROWS][B] (optional, in/out, zero-initialised) warm-starts the Riccati solve. */
int d2dx_dfff_control(d2dx_handle* h, const d2dx_traj_table* tt, const double* X, double t,
                      const double* W, const double* ac, const d2dx_dfff_gains* gains_host,
                      double* U, double* Xr, double* K, double* care_state, void* stream);

/* -------- closed-loop rollout, DFFF controller --------
 * Replaces run_simulation, 05_test_simulation.py:21-34, for B aircraft-scenarios at once. */
typedef struct {
  int32_t B;
  const double* X0;          /* [5][B]                                                           */
  const double* wind;        /* [2][B]  WindField.sample, d2d/guidance.py:12-16 (constant field) */
  const double* ac;          /* [2][B]  tau_phi, tau_v  (d2d/dynamic.py:11-12)                   */
  d2dx_traj_table traj;
  /* perturbation events `X[i] += perts[i]` (05_test_simulation.py:32), CSR by scenario, sorted by
   * step inside a scenario; all NULL = none */
  const int32_t* pert_begin; /* [B+1]                                                            */
  const int32_t* pert_step;  /* [n_events] sample index i the perturbation is added to           */
  const double* pert_dx;     /* [5][n_events]                                                    */
  int32_t n_events;
} d2dx_scenarios;

typedef struct {
  int32_t log_every;         /* sample i is logged at row i/log_every when i % log_every == 0    */
  double* X_log;             /* [n_rows][5][B] or NULL                                           */
  double* U_log;             /* [n_rows][2][B] or NULL                                           */
  double* Xr_log;            /* [n_rows][5][B] or NULL   (DFFFController.Xref, guidance.py:66)   */
  double* K_log;             /* [n_rows][6][B] or NULL   (DFFFController.K, guidance.py:83)      */
  double* X_final;           /* [5][B]  state at sample i_end                                    */
  double* sum_sq_err;        /* [B] or NULL  += sum_i |X[i,:2]-Xr[i,:2]|^2 over this call        */
  double* max_err;           /* [B] or NULL  = max(previous, max_i |X[i,:2]-Xr[i,:2]|)           */
  int32_t* flags;            /* [B] or NULL  |= 1 non-finite state seen, 2 Riccati not converged */
  double* care_state;        /* [D2DX_CARE_STATE_ROWS][B] or NULL  Riccati warm start carried between calls (zeros = cold) */
  double* pop_stats;         /* [2] or NULL  += sum over scenarios of sum_sq_err; max of max_err */
} d2dx_rollout_out;

/* Advances every scenario from sample i_begin to sample i_end of `time` (device array [T], the
 * reference's np.arange grid): for i in (i_begin, i_end]: U[i-1]=ctl(X[i-1],time[i-1]);
 * X[i]=rk4(X[i-1],U[i-1],dt=time[i]-time[i-1]); X[i]+=perts[i].  X0 is the state at i_begin.  With
 * final_control != 0 the extra U[i_end]=ctl(X[i_end],time[i_end]) of 05_test_simulation.py:33 is made. */
int d2dx_rollout_dfff(d2dx_handle* h, const d2dx_scenarios* s, const double* time, int32_t i_begin,
                      int32_t i_end, int32_t nsub, int32_t final_control,
                      const d2dx_dfff_gains* gains_host, const d2dx_rollout_out* out, void* stream);

/* -------- 5-state LQR tracker on sampled references (SURVEY 8f #1) --------
 * Replaces Controllers.DiffFlatness.ComputeFlatness (Controllers.py:62-108), DiffController.ComputeGain (:159-186) and
 * the loop of implement_controller (10_opt_traj_tracking.py:72-89): full-state LQR with Q = diag(q), R = diag(r) on the
 * complete linearisation of d2d/dynamic.py:32-43, references given by samples of the flat output and its derivatives. */
typedef struct {
  double q[5];               /* reference: 1, 1, 0.1, 0.01, 0.01   (q[0] must equal q[1])                 */
  double r[2];               /* reference: 8, 1                                                           */
  double err_sat[5];         /* reference: 20, 20, pi/3, pi/4, 1                                          */
  double u_lo[2], u_hi[2];   /* reference: (-60 deg, 4), (60 deg, 20)                                     */
} d2dx_tracker_gains;
int d2dx_tracker_default_gains(d2dx_tracker_gains* g_host);
/* ComputeFlatness for n references: Ys[8][n] (rows as d2dx_traj_eval: Y, Yd, Ydd, Yddd) -> Xr[5][n], Ur[2][n] */
int d2dx_flatness5(d2dx_handle* h, int32_t n, const double* Ys, const double* W, const double* ac, double* Xr,
                   double* Ur, void* stream);
/* ComputeGain for n aircraft: X[5][n], Ys[8][n] -> U[2][n]; optional Xr[5][n], dX[5][n], K[10][n] (row-major 2x5);
 * lqr_state[7][n] (optional, in/out, zero-initialised) warm-starts the Riccati solve */
int d2dx_tracker_control(d2dx_handle* h, int32_t n, const double* X, const double* Ys, const double* W,
                         const double* ac, const d2dx_tracker_gains* gains_host, double* U, double* Xr, double* dX,
                         double* K, double* lqr_state, void* stream);
typedef struct {
  int32_t M, T;              /* aircraft, reference samples                                                */
  const double* ref;         /* [T][6][M]  x, y, xd, yd, xdd, ydd of each sample (third derivative = 0,
                                          10_opt_traj_tracking.py:77)                                    */
  const double* X0;          /* [5][M]                                                                    */
  const double* wind;        /* [2][M]                                                                    */
  const double* ac;          /* [2][M]  tau_phi, tau_v                                                    */
  double dt;                 /* sample spacing (time_opt[1] - time_opt[0], :42)                           */
} d2dx_tracker;
typedef struct {
  double* X_log;             /* [T][5][M] or NULL   row i = state at sample i                             */
  double* U_log;             /* [T][2][M] or NULL   row i-1 = input applied from sample i-1 to i          */
  double* Xr_log;            /* [T][5][M] or NULL   row i-1 (X_ref_array)                                  */
  double* dX_log;            /* [T][5][M] or NULL   row i-1 (dX_array)                                     */
  double* K_log;             /* [T][10][M] or NULL  row i-1                                                */
  double* X_final;           /* [5][M]                                                                    */
  int32_t* flags;            /* [M] or NULL  |= 1 non-finite state, 2 Riccati not converged               */
  double* lqr_state;         /* [7][M] or NULL  warm start carried between calls                          */
} d2dx_tracker_out;
/* for i in (i_begin, i_end]: (Xr, dX, U) = ComputeGain(X[i-1], sample i); X[i] = rk4(X[i-1], U, dt, nsub) */
int d2dx_rollout_tracker(d2dx_handle* h, const d2dx_tracker* in, int32_t i_begin, int32_t i_end, int32_t nsub,
                         const d2dx_tracker_gains* gains_host, const d2dx_tracker_out* out, void* stream);

/* -------- circular formation (DCF + GVF) -------- */
/* DCFController.get, d2d/guidance.py:103-126, for F formations of n_ac aircraft.
 * p[2][F*n_ac], c[2][F*n_ac] (aircraft f*n_ac+j), Binc[n_ac][n_e] (host, row-major, shared by all
 * formations), z_des[n_e] (host).  Outputs Ur[F*n_ac], e_deg[F*n_e] (degrees). */
int d2dx_dcf(d2dx_handle* h, int32_t F, int32_t n_ac, int32_t n_e, const double* Binc_host,
             const double* z_des_host, double kr, const double* p, const double* c, double* Ur,
             double* e_deg, void* stream);
/* CircleTraj.get, d2d/guidance.py:137-146: X[5][n], c[2][n], r[n] -> out[3][n] = (e, n_x, n_y); H is the constant 2 I */
int d2dx_circle_implicit(d2dx_handle* h, int32_t n, const double* X, const double* c, const double* r, double* out,
                         void* stream);
/* CircleTraj.get + GVFcontroller.get, d2d/guidance.py:137-146,155-181: X[5][n], c[2][n], r[n] ->
 * out[3][n] = (U, U1, U2) */
int d2dx_gvf(d2dx_handle* h, int32_t n, const double* X, const double* c, const double* r, double ke,
             double kd, double* out, void* stream);

typedef struct {
  int32_t F, n_ac, n_e;
  const double* X0;          /* [5][F*n_ac]                                                      */
  const double* c;           /* [2][F*n_ac]  circle centre of each aircraft                      */
  const double* r;           /* [F*n_ac]     nominal radius R                                    */
  const double* ac;          /* [2][F*n_ac]  tau_phi, tau_v                                      */
  const double* Binc_host;   /* host [n_ac][n_e] incidence matrix (08_CircularFormation_Full.py:49-60) */
  const double* z_des_host;  /* host [n_e]                                                       */
  double ke, kd, kr, v_c;    /* 08_CircularFormation_Full.py:39-41,90                            */
} d2dx_formations;

typedef struct {
  int32_t log_every;
  double* X_log;             /* [n_rows][5][F*n_ac] or NULL                                      */
  double* U_log;             /* [n_rows][F*n_ac] or NULL   roll set-point arctan(U/9.81)         */
  double* Rr_log;            /* [n_rows][F*n_ac] or NULL   commanded radius (row i holds step i's) */
  double* eth_log;           /* [n_rows][F*n_e] or NULL    phase errors in degrees               */
  double* X_final;           /* [5][F*n_ac]                                                      */
  int32_t* flags;            /* [F*n_ac] or NULL                                                 */
} d2dx_formation_out;

/* Loop of CircularFormationGVF, 08_CircularFormation_Full.py:73-94 (c per aircraft as in
 * 09_CircularFormation_diffcentre.py:33,87): samples i_begin..i_end of a uniform grid of step dt. */
int d2dx_rollout_formation(d2dx_handle* h, const d2dx_formations* f, double dt, int32_t i_begin,
                           int32_t i_end, int32_t nsub, const d2dx_formation_out* out, void* stream);

/* -------- direct collocation: residual, Jacobian, cost, gradient --------
 * Replaces what IPOPT calls back through opty.direct_collocation.Problem (06_optyplan.py:62-71,
 * 07_multioptyplan.py:69-78): constraints(free), jacobian(free), obj(free), obj_grad(free), with the
 * EoM of d2d/opty_utils.py:38-50 and the cost classes of d2d/opty_utils.py:55-165 and
 * d2d/multiopty_utils.py:29-174. */
enum { D2DX_JAC_COMPACT = 0, D2DX_JAC_OPTY_DENSE = 1 };
enum { D2DX_EVAL_RESIDUAL = 1, D2DX_EVAL_JAC = 2, D2DX_EVAL_COST = 4, D2DX_EVAL_GRAD = 8 };
#define D2DX_MAX_OBSTACLES 16

typedef struct {
  int32_t n_ac, N;           /* aircraft, collocation nodes                                      */
  double h;                  /* node interval                                                    */
  double wind[2];            /* constant wind of the planner (`+ w` in the EoM, opty_utils.py:42-43) */
  /* input block order inside `free`: aircraft a's phi block is input block perm_phi[a], its v block
   * is perm_v[a] (device int32 [n_ac] each, or NULL = the planner's numeric order,
   * 07_multioptyplan.py:45-47).  opty itself sorts by name (SURVEY D9). */
  const int32_t* perm_phi;
  const int32_t* perm_v;
  /* instance constraints free[var*N+node]-value (06_optyplan.py:46-49): device arrays [n_inst] */
  int32_t n_inst;
  const int32_t* inst_var;
  const int32_t* inst_node;
  const double* inst_val;
  /* cost = obj_scale * ( (kvel*sum (v-vsp)^2 + kbank*sum phi^2) / (N*in_div)
   *                      + kobs/N * sum_obstacles sum_i es + kcol/N * sum_pairs sum_i es ) */
  double obj_scale, vsp, kvel, kbank;
  int32_t in_div;            /* 1 single-aircraft classes, n_ac multi-aircraft classes           */
  double kobs;               /* NaN or 0 disables (multiopty_utils.py:166)                       */
  int32_t obs_kind, n_obs;   /* kind 0: clip(exp(r^2-d^2),0,1e3); kind 1: exp(-(2/r)^2 d^2)      */
  double obs[D2DX_MAX_OBSTACLES][3];  /* cx, cy, r  -- applied to aircraft 0 (multiopty_utils.py:74) */
  double kcol, rcol, kcol_k; /* CostCollision (multiopty_utils.py:120-153); NaN or 0 disables    */
  int32_t col_all_pairs;     /* 0: aircraft (0,1) only as the reference; 1: all pairs            */
  int32_t exact_grad;        /* 0: reference gradients (omit (k/r)^2, SURVEY D11); 1: exact      */
} d2dx_colloc_problem;

/* sizes: n_free=5*n_ac*N, n_con=3*n_ac*(N-1)+n_inst,
 * nnz: compact 12*n_ac*(N-1)+n_inst, opty-dense (N-1)*3n_ac*8n_ac+n_inst  (host int64[3]) */
int d2dx_colloc_sizes(const d2dx_colloc_problem* p_host, int32_t layout, int64_t* sizes_host3);
/* COO structure of the Jacobian values (device int64 rows[nnz], cols[nnz]) */
int d2dx_colloc_structure(d2dx_handle* h, const d2dx_colloc_problem* p_host, int32_t layout,
                          int64_t* rows, int64_t* cols, void* stream);
/* one-time initialisation of an opty-dense value buffer (structural zeros + instance ones) for
 * n_prob problems; d2dx_colloc_eval then only rewrites the non-zeros */
int d2dx_colloc_init_dense(d2dx_handle* h, const d2dx_colloc_problem* p_host, int32_t n_prob,
                           double* jac, void* stream);
/* Evaluates n_prob problems sharing one description: free[n_prob][n_free] ->
 * residual[n_prob][n_con], jac[n_prob][nnz], cost[n_prob], grad[n_prob][n_free] (any may be NULL if
 * its flag is clear).  scratch: device doubles, at least d2dx_colloc_scratch_size(...) elements. */
/* scratch must be ZERO before its first use (it starts with the tickets of the single-launch cost reduction; every call
 * leaves them zero again) and must not be shared by evaluations in flight on different streams. */
int64_t d2dx_colloc_scratch_size(const d2dx_colloc_problem* p_host, int32_t n_prob);
int d2dx_colloc_eval(d2dx_handle* h, const d2dx_colloc_problem* p_host, int32_t n_prob,
                     const double* free_, int32_t layout, uint32_t what, double* residual,
                     double* jac, double* cost, double* grad, double* scratch, void* stream);
/* CostBank with use_mean = False (d2d/opty_utils.py:68-82): cost[p] = obj_scale * max_i phi_i^2 over the N values
 * free[p][off_phi .. off_phi+N); grad[p][n_free] = zeros except obj_scale * 2 phi at the first maximum (np.argmax).
 * cost or grad may be NULL. */
int d2dx_cost_bank_max(d2dx_handle* h, int32_t n_prob, int32_t n_free, int32_t off_phi, int32_t N, double obj_scale,
                       const double* free_, double* cost, double* grad, void* stream);
/* -------- aircraft-sharded evaluation over NVLink peer memory: ONE kernel per rank, no collective call (SURVEY 8e) --------
 * The exchange step the north star names ("all-gather aircraft positions for the cross-shard avoidance terms, reduce
 * costs") done by the evaluation kernel itself: each rank stores its aircraft's x, y straight from free_local into every
 * peer's position table (peer memory), computes everything local while the stores travel, reads the peers' tiles from its
 * own table (every value travels with the evaluation number in the same 8-byte words, so arrival needs neither a fence nor
 * a flag), adds the collision terms, and the block of a problem's last tile exchanges the four cost sums the same way, so
 * that every rank ends with the identical total cost[n_prob].  Serves the callbacks of 07_multioptyplan.py:69-78 when one
 * problem is spread over the GPUs of a box.
 *
 * d2dx_peer_create allocates this rank's exchange buffer (the only allocation; capacity: max_prob problems of n_ac_total
 * aircraft x N nodes).  Between processes the ranks swap d2dx_peer_ipc_handle blobs (64 bytes each, e.g. with
 * torch.distributed.all_gather_object) and call d2dx_peer_connect_ipc; inside one process d2dx_peer_connect_local takes
 * the other ranks' objects.  Every rank must then make the same sequence of d2dx_colloc_eval_peer calls (same n_prob,
 * same `what`); a call is asynchronous on `stream`, may be captured in a CUDA graph, and never blocks forever: a peer
 * that does not answer within ~1 s per wait is counted in status[0] of d2dx_peer_status ([1] = evaluations completed,
 * [2] = resident blocks the kernel is sized for, [3] = exchange buffer KiB) and the outputs of that call are undefined. */
typedef struct d2dx_peer d2dx_peer;
#define D2DX_PEER_MAX_WORLD 16
#define D2DX_IPC_HANDLE_BYTES 64
int d2dx_peer_create(d2dx_handle* h, int32_t world, int32_t rank, int32_t max_prob, int32_t n_ac_total, int32_t N,
                     d2dx_peer** out);
int d2dx_peer_ipc_handle(d2dx_peer* p, void* handle_host64);
int d2dx_peer_connect_ipc(d2dx_peer* p, const void* handles_host /* [world][64], rank order */);
int d2dx_peer_connect_local(d2dx_peer* p, d2dx_peer* const* peers_host /* [world], rank order */);
int d2dx_peer_status(d2dx_peer* p, int32_t* status_host4);
/* %globaltimer stamps [ns] of the last evaluation on this rank (block 0 and the block that finished problem 0): 0 kernel
 * start, 1 tiles published, 2 local work done, 3 peers' positions arrived, 4 pair terms done, 5 own cost sums sent,
 * 6 every rank's sums arrived, 7 block 0 leaves -- where the latency of a sharded evaluation goes */
int d2dx_peer_timeline(d2dx_peer* p, uint64_t* stamps_host8);
int d2dx_peer_destroy(d2dx_peer* p);
/* `p_local_host` describes THIS rank's shard as a problem of n_ac = number of owned aircraft (in_div must be the TOTAL
 * aircraft count); the owned aircraft are global aircraft [a_lo, a_lo + n_ac) of the exchange's n_ac_total.  free_local,
 * residual, jac (compact layout) and grad use the shard-local layout, for n_prob problems stacked on a leading axis;
 * cost[n_prob] receives the TOTAL cost of each problem (all ranks' shares, summed in rank order). */
int d2dx_colloc_eval_peer(d2dx_handle* h, d2dx_peer* peer, const d2dx_colloc_problem* p_local_host, int32_t n_prob,
                          int32_t a_lo, const double* free_local, uint32_t what, double* residual, double* jac,
                          double* cost, double* grad, void* stream);

/* -------- single-shooting evaluation of the planner NLP (SURVEY 8f #2) --------
 * On the backward-Euler grid the defects of d2dx_colloc_eval determine the states from the inputs:
 *   psi_i = psi_{i-1} + h g tan(phi_i)/v_i,  x_i = x_{i-1} + h (v_i cos psi_i - w_x),  y_i = y_{i-1} + h (v_i sin psi_i - w_y),
 * so a solver can iterate on the inputs only.  For P problems at once (problem-major, node index fastest):
 *   u[P][2][n_ac][N]      inputs phi, v at every node (node 0 enters the cost only)
 *   p0[P][3][n_ac], p1[P][3][n_ac]   initial state and terminal target (x, y, psi) of each aircraft
 *   lam[P][3][n_ac], rho[P]          augmented-Lagrangian multipliers / penalty of the terminal constraints
 * d2dx_shoot_forward fills xs[P][3][n_ac][N] (x, y, psi) and c[P][3][n_ac] = state(N-1) - p1.
 * d2dx_shoot_adjoint (after forward, same arguments) returns per-aircraft shares (sum over n_ac = the totals)
 *   cost[P][n_ac]  of the planner cost of d2dx_colloc_problem (exact value),
 *   lagr[P][n_ac]  of cost + sum lam.c + rho/2 |c|^2,   and grad[P][2][n_ac][N] = d lagr / d u   (exact derivatives).
 * `p_host` supplies n_ac, N, h, wind and the cost description (instance constraints, permutations and exact_grad are
 * ignored: the terminal targets come from p1, gradients are always exact).
 * Box constraints by substitution: with `bounds` = {phi_lo, phi_hi, v_lo, v_hi} (HOST array; NULL = none) `u` holds
 * angles theta with phi = mid + half sin(theta) (likewise v); forward writes the physical inputs to u_phys (same shape
 * as u), adjoint reads them and returns the gradient with respect to theta.
 * Soft state box: with `state_box` = {x_lo, x_hi, y_lo, y_hi, weight} (HOST array; NULL = none) the cost gains
 * weight * obj_scale / N * sum over aircraft and nodes of the squared excess of x_i, y_i over the box (the planners'
 * x/y_constraint, which IPOPT treats as variable bounds). */
int d2dx_shoot_forward(d2dx_handle* h, const d2dx_colloc_problem* p_host, int32_t P, const double* u, const double* bounds,
                       const double* p0, const double* p1, double* u_phys, double* xs, double* c, void* stream);
int d2dx_shoot_adjoint(d2dx_handle* h, const d2dx_colloc_problem* p_host, int32_t P, const double* u, const double* bounds,
                       const double* state_box, const double* u_phys, const double* xs, const double* c, const double* lam,
                       const double* rho, double* cost, double* lagr, double* grad, void* stream);

/* -------- batched augmented-Lagrangian L-BFGS driver (the solver behind Planner.run; replaces prob.solve -> IPOPT,
 * 06_optyplan.py:117-125, 07_multioptyplan.py:80-88) --------
 * P independent problems  min f(x) s.t. c(x) = 0, x in R^n, n_con constraints each.  The caller evaluates the augmented
 * Lagrangian L = f + lam.c + rho/2 |c|^2, its gradient and c at `x_trial`; one tick consumes that evaluation and writes
 * the next point to evaluate into x_trial (L-BFGS direction, Armijo backtracking, multiplier/penalty updates and the
 * termination tests are per problem, on the device).  [evaluate, tick] has no host decision inside and can be captured
 * in a CUDA graph; *n_running (device) holds the number of problems still iterating after each tick. */
typedef struct {
  int32_t m;            /* history pairs (1..32) */
  int32_t max_inner;    /* accepted steps per multiplier update */
  int32_t max_outer;    /* multiplier updates */
  int32_t ls_max;       /* halvings per line search */
  int32_t window;       /* inner loop stops when L fell by < ftol max(1,|L|) over `window` accepted steps ... */
  double gtol;          /* ... or |grad|_inf <= gtol */
  double ftol;
  double ctol;          /* a problem is solved when max|c| < ctol after an inner loop */
  double rho0, rho_max; /* penalty: starts at rho0, x3 (up to rho_max) when max|c| did not fall to a quarter */
  int32_t keep_history; /* 1: keep the L-BFGS pairs across multiplier updates that leave rho unchanged; 0: restart every time */
} d2dx_lbfgs_options;
/* offsets (in doubles) into the state buffer: [0] total size, [1] x[P][n], [2] g[P][n], [3] scalars[P][offsets[6]]
 * (0 L, 4 previous max|c|, 5 max|c|, 6 cost), [4] c at x [P][n_con], [5] int32 meta[P][offsets[7]]
 * (0 flag: 0/1 iterating, 2 solved, 3 stopped unsolved; 5 evaluations; 6 multiplier updates; 10 accepted steps). */
int d2dx_lbfgs_layout(int32_t P, int32_t n, int32_t n_con, const d2dx_lbfgs_options* o, int64_t offsets[8]);
int d2dx_lbfgs_init(d2dx_handle* h, int32_t P, int32_t n, int32_t n_con, const d2dx_lbfgs_options* o, double* state,
                    double* lam, double* rho, void* stream);
/* f_parts[P][n_parts]: shares of L summed in index order; cost_parts (nullable): shares of f, reported in scalars[6]. */
int d2dx_al_lbfgs_tick(d2dx_handle* h, int32_t P, int32_t n, int32_t n_con, const d2dx_lbfgs_options* o, double* state,
                       double* x_trial, const double* f_parts, const double* cost_parts, int32_t n_parts, const double* grad,
                       const double* c, double* lam, double* rho, int32_t* n_running, void* stream);

/* -------- second-order solve of the single-aircraft planner NLP (replaces prob.solve -> IPOPT, 06_optyplan.py:117-125) --------
 * Control-limited differential dynamic programming on the collocation grid (exact second-order model of the backward-Euler
 * transition, the 2-variable box QP of every node solved exactly: phi / v bounds hold at every iterate), terminal conditions by
 * an augmented Lagrangian, state box as a quadratic penalty of the excess.  One THREAD solves one problem; P problems (multi-start,
 * many boundary conditions) per launch.  p_host: n_ac must be 1; N, h, wind and the cost description are used.
 *   bounds_host4    {phi_lo, phi_hi, v_lo, v_hi} (host)          state_box_host5  {x_lo, x_hi, y_lo, y_hi, weight} or NULL (host)
 *   p0[P][3], p1[P][3]  initial state and terminal target (x, y, psi)
 *   u[P][2][N]      in: start (phi, v per node), out: solution     xs[P][3][N]  out: states of the solution
 *   info[P][8]      out: flag (2 solved, 3 stopped unsolved, 4 terminal conditions met but the sweep limit reached before the cost
 *                   settled), iterations, multiplier updates, cost, max |terminal error|,
 *                   augmented Lagrangian, final regularisation, final penalty
 *   work            device doubles, at least d2dx_ddp_work_size(P, N) */
typedef struct {
  int32_t max_iter;      /* sweeps (backward + line search) per problem in total */
  int32_t max_outer;     /* multiplier updates */
  int32_t max_inner;     /* sweeps per multiplier update */
  int32_t ls_max;        /* halvings per line search */
  double ctol;           /* solved when max |terminal error| < ctol at a converged inner loop */
  double rel_tol, abs_tol;   /* inner loop converged when the (predicted or achieved) decrease <= rel_tol |L| + abs_tol */
  double rho0, rho_growth, rho_max;
  double mu0, mu_min, mu_max, mu_factor;   /* Levenberg-Marquardt regularisation of Quu and its adaptation */
  int32_t reg_mode;      /* 0: plain mu (raised until every node's Quu is definite); 1: eigenvalues of Quu replaced by their magnitude, plus mu */
  int32_t min_solved;    /* > 0: problems still iterating stop (flag 3) once this many problems of the launch have converged --
                            multi-start, where the stragglers are the starts in an infeasible local minimum; 0: every problem runs out */
} d2dx_ddp_options;
int d2dx_ddp_default_options(d2dx_ddp_options* o_host);
int64_t d2dx_ddp_work_size(int32_t P, int32_t N);
int d2dx_ddp_solve(d2dx_handle* h, const d2dx_colloc_problem* p_host, int32_t P, const double* bounds_host4,
                   const double* state_box_host5, const double* p0, const double* p1, double* u, double* xs, double* info,
                   double* work, const d2dx_ddp_options* o_host, void* stream);

/* -------- second-order solve of the multi-aircraft planner NLP (replaces prob.solve -> IPOPT, 07_multioptyplan.py:80-88) --------
 * The control-limited DDP of d2dx_ddp_solve with the n_ac aircraft of a problem in one stage: 3 n_ac states, 2 n_ac inputs, the
 * transition block-diagonal per aircraft, the aircraft coupled through the collision term (its exact Hessian in the value model);
 * the 2 n_ac-variable box QP of every node by projected Newton; 3 n_ac terminal conditions by an augmented Lagrangian.  One WARP
 * solves one problem.  p_host: 1 <= n_ac <= 10; the cost terms are those of d2dx_shoot_adjoint (soft box on every aircraft,
 * obstacles on aircraft 0, collision on the pair (0, 1) or every pair).  Layouts as the shooting kernels:
 *   p0[P][3][n_ac], p1[P][3][n_ac]     initial states and terminal targets (x, y, psi)
 *   u[P][2][n_ac][N]                   in: start (phi, v), out: solution      xs[P][3][n_ac][N]  out: states of the solution
 *   info[P][8]                         as d2dx_ddp_solve
 *   lam_out[P][3][n_ac] or NULL        multipliers of the last inner loop (the returned inputs minimise the Lagrangian for them)
 *   work                               device doubles, at least d2dx_ddp_multi_work_size(P, n_ac, N)
 * Options as d2dx_ddp_solve; reg_mode 1 is refused for n_ac > 1 (D2DX_EINVAL), as are n_ac outside 1 .. 10 and bad bounds. */
int64_t d2dx_ddp_multi_work_size(int32_t P, int32_t n_ac, int32_t N);
int d2dx_ddp_multi_solve(d2dx_handle* h, const d2dx_colloc_problem* p_host, int32_t P, const double* bounds_host4,
                         const double* state_box_host5, const double* p0, const double* p1, double* u, double* xs, double* info,
                         double* lam_out, double* work, const d2dx_ddp_options* o_host, void* stream);

/* -------- pure-pursuit guidance on a sampled path (PurePursuitControler, d2d/guidance.py:204-245; SURVEY 8f #4) --------
 * nearest sample of the path to the aircraft (first minimum of the Euclidean distance, as np.argmin), carrot `lookahead`
 * samples further (wrapping at the end), phi_c = clip(-K wrap(psi - atan2(carrot - position)), +-sat_phi), v_c = v_sp.
 * Upstream: path = traj.get(t)[0] for t in arange(0, traj.duration, 0.01), lookahead = 100, K = 1, sat 45 deg, v_sp 10. */
typedef struct {
  int32_t n_pts;
  const double* px;      /* [n_pts] device */
  const double* py;
  int32_t lookahead;
  double K, sat_phi, v_sp;
} d2dx_pursuit;
/* X[5][B] -> U[2][B] (and the index of the nearest sample, nullable) */
int d2dx_pursuit_control(d2dx_handle* h, const d2dx_pursuit* p, int32_t B, const double* X, double* U, int32_t* idx_closest,
                         void* stream);
/* closed loop (run_simulation, 05_test_simulation.py:21-34, with this controller): steps i_begin .. i_end-1 of `dt` (RK4,
 * nsub sub-steps, heading wrapped per step); X_log[T][5][B] rows i_begin..i_end, U_log[T][2][B] / idx_log[T][B] rows
 * i_begin..i_end-1 (all nullable); X_final[5][B]. */
int d2dx_rollout_pursuit(d2dx_handle* h, const d2dx_pursuit* p, int32_t B, const double* X0, const double* wind, const double* ac,
                         double dt, int32_t i_begin, int32_t i_end, int32_t nsub, double* X_log, double* U_log, int32_t* idx_log,
                         double* X_final, void* stream);

/* -------- diagnostics -------- */
/* FP64 roofline probe: every thread runs `iters` rounds of 16 independent DFMA chains (32*iters flop per
 * thread); the caller times it with CUDA events.  sink: device double[1] (keeps the chains alive). */
int d2dx_dfma_burn(d2dx_handle* h, int32_t blocks, int32_t threads, int32_t iters, double* sink, void* stream);
/* the engine's straight-line fp64 elementary functions on n argument pairs (x[n], y[n] device):
 * out[13][n] = sin x, cos x, atan2(y, x), atan x, y / x, sqrt|x|, 1/sqrt|x|, 1/x, and the residuals 1 - x y0, 1 - |x| y0^2 of the
 * hardware reciprocal / reciprocal-square-root seeds the last four start from, norm_mpi_pi(x) (bit-exact against NumPy's
 * (x + pi) % (2 pi) - pi), and the small-angle sin x, cos x of the RK4 stage headings (|x| < 2^-5)   (accuracy tests) */
int d2dx_math_probe(d2dx_handle* h, int32_t n, const double* x, const double* y, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* D2DX_H */
