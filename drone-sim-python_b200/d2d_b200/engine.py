"""Thin device-level wrapper of the C ABI: torch is used for device buffers, streams and nothing else."""
import ctypes as C
import os
import threading

import numpy as np
import torch

from . import _lib
from ._lib import check, lib

F64 = torch.float64


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class PackedTrajectories:
    """Host-side (NumPy) trajectory table in the layout of d2dx_traj_table."""

    def __init__(self, first_seg, n_segs, traj_t0, traj_dur, seg_type, seg_end, seg_par, uniform_type=-1, tables=None):
        self.first_seg = np.ascontiguousarray(first_seg, np.int32)
        self.n_segs = np.ascontiguousarray(n_segs, np.int32)
        self.traj_t0 = np.ascontiguousarray(traj_t0, np.float64)
        self.traj_dur = np.ascontiguousarray(traj_dur, np.float64)
        self.seg_type = np.ascontiguousarray(seg_type, np.int32)
        self.seg_end = np.ascontiguousarray(seg_end, np.float64)
        self.seg_par = np.ascontiguousarray(seg_par, np.float64)
        self.uniform_type = int(uniform_type)
        # (5, n_tab) rows time, x, y, vx, vy of the D2DX_SEG_TABLE segments, or None
        self.tables = None if tables is None else np.ascontiguousarray(tables, np.float64)
        assert self.seg_par.shape == (_lib.SEG_NPAR, len(self.seg_type))

    @property
    def n_traj(self): return len(self.first_seg)

    @property
    def n_seg(self): return len(self.seg_type)

    def bytes(self):
        return sum(a.nbytes for a in (self.first_seg, self.n_segs, self.traj_t0, self.traj_dur, self.seg_type,
                                      self.seg_end, self.seg_par))


class DeviceTable:
    """A PackedTrajectories resident in HBM plus the C struct that points at it."""

    def __init__(self, eng, packed, non_blocking=False):
        self.packed = packed
        self.t = {k: eng.to_device(getattr(packed, k), non_blocking) for k in
                  ("first_seg", "n_segs", "traj_t0", "traj_dur", "seg_type", "seg_end", "seg_par")}
        self.c = _lib.TrajTable(packed.n_traj, packed.n_seg, *[_ptr(self.t[k]) for k in
                                ("first_seg", "n_segs", "traj_t0", "traj_dur", "seg_type", "seg_end", "seg_par")],
                                packed.uniform_type + 1)      # ABI: 0 = mixed, 1 + type = uniform
        if packed.tables is not None:
            self.tab = eng.to_device(packed.tables, non_blocking)
            n = packed.tables.shape[1]
            base, es = self.tab.data_ptr(), 8 * n
            self.c.n_tab = n
            self.c.tab_time, self.c.tab_x, self.c.tab_y, self.c.tab_vx, self.c.tab_vy = (base + k * es for k in range(5))


class Engine:
    """One engine per process and device (`cuda:LOCAL_RANK` by default)."""

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("d2d_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        torch.cuda.set_device(self.device)
        h = C.c_void_p()
        check(lib.d2dx_create(self.device_index, C.byref(h)), "d2dx_create")
        self.h = h
        info = (C.c_int32 * 4)()
        check(lib.d2dx_device_info(self.h, info), "d2dx_device_info")
        self.sm_count, self.rollout_threads_per_sm, self.formation_threads_per_sm, self.colloc_threads_per_sm = list(info)
        self.launches = 0                      # kernels launched through this engine (bench `gpu_launches`)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                lib.d2dx_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---- buffers -------------------------------------------------------------------------------
    def to_device(self, a, non_blocking=False):
        if isinstance(a, torch.Tensor):
            return a.to(self.device, non_blocking=non_blocking).contiguous()
        a = np.ascontiguousarray(a)
        if not a.flags.writeable:
            a = a.copy()
        t = torch.from_numpy(a)
        return t.to(self.device, non_blocking=non_blocking)

    def empty(self, *shape, dtype=F64):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    def zeros(self, *shape, dtype=F64):
        return torch.zeros(*shape, dtype=dtype, device=self.device)

    def stream_ptr(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def table(self, packed, non_blocking=False):
        return DeviceTable(self, packed, non_blocking)

    # ---- single calls ----------------------------------------------------------------------------
    def traj_eval(self, table, time_dev):
        nT, B = time_dev.numel(), table.packed.n_traj
        Y = self.empty(nT, 8, B)
        check(lib.d2dx_traj_eval(self.h, C.byref(table.c), nT, _ptr(time_dev), _ptr(Y), self.stream_ptr()), "d2dx_traj_eval")
        self.launches += 1
        return Y

    def cont_dyn(self, X, U, W, ac):
        n = X.shape[1]; out = self.empty(5, n)
        check(lib.d2dx_cont_dyn(self.h, n, _ptr(X), _ptr(U), _ptr(W), _ptr(ac), _ptr(out), self.stream_ptr()), "d2dx_cont_dyn")
        self.launches += 1
        return out

    def disc_dyn(self, X, U, W, ac, dt, nsub=1):
        n = X.shape[1]; out = self.empty(5, n)
        check(lib.d2dx_disc_dyn(self.h, n, _ptr(X), _ptr(U), _ptr(W), _ptr(ac), float(dt), int(nsub), _ptr(out), self.stream_ptr()), "d2dx_disc_dyn")
        self.launches += 1
        return out

    def cont_jac(self, Xr, ac):
        n = Xr.shape[1]; A = self.empty(25, n); Bm = self.empty(10, n)
        check(lib.d2dx_cont_jac(self.h, n, _ptr(Xr), _ptr(ac), _ptr(A), _ptr(Bm), self.stream_ptr()), "d2dx_cont_jac")
        self.launches += 1
        return A, Bm

    def flatness(self, Ys, W, ac):
        n = Ys.shape[1]; Xr = self.empty(5, n); Ur = self.empty(2, n); Xd = self.empty(5, n)
        check(lib.d2dx_flatness(self.h, n, _ptr(Ys), _ptr(W), _ptr(ac), _ptr(Xr), _ptr(Ur), _ptr(Xd), self.stream_ptr()), "d2dx_flatness")
        self.launches += 1
        return Xr, Ur, Xd

    def default_gains(self):
        g = _lib.DfffGains()
        check(lib.d2dx_dfff_default_gains(C.byref(g)), "d2dx_dfff_default_gains")
        return g

    def dfff_control(self, table, X, t, W, ac, gains=None, care_state=None):
        B = X.shape[1]; U = self.empty(2, B); Xr = self.empty(5, B); K = self.empty(6, B)
        check(lib.d2dx_dfff_control(self.h, C.byref(table.c), _ptr(X), float(t), _ptr(W), _ptr(ac),
                                    C.byref(gains) if gains is not None else None, _ptr(U), _ptr(Xr), _ptr(K),
                                    _ptr(care_state), self.stream_ptr()), "d2dx_dfff_control")
        self.launches += 1
        return U, Xr, K

    # ---- rollouts ----------------------------------------------------------------------------------
    def rollout_dfff(self, table, X0, wind, ac, time_dev, i_begin, i_end, nsub=1, final_control=False, gains=None,
                     log_every=1, X_log=None, U_log=None, Xr_log=None, K_log=None, X_final=None, sum_sq_err=None,
                     max_err=None, flags=None, care_state=None, pop_stats=None, perts=None):
        B = X0.shape[1]
        if X_final is None:
            X_final = self.empty(5, B)
        s = _lib.Scenarios()
        s.B = B; s.X0 = _ptr(X0); s.wind = _ptr(wind); s.ac = _ptr(ac); s.traj = table.c
        if perts is not None:
            s.pert_begin, s.pert_step, s.pert_dx = _ptr(perts[0]), _ptr(perts[1]), _ptr(perts[2])
            s.n_events = int(perts[1].numel())
        o = _lib.RolloutOut(int(log_every), _ptr(X_log), _ptr(U_log), _ptr(Xr_log), _ptr(K_log), _ptr(X_final),
                            _ptr(sum_sq_err), _ptr(max_err), _ptr(flags), _ptr(care_state), _ptr(pop_stats))
        check(lib.d2dx_rollout_dfff(self.h, C.byref(s), _ptr(time_dev), int(i_begin), int(i_end), int(nsub),
                                    int(bool(final_control)), C.byref(gains) if gains is not None else None,
                                    C.byref(o), self.stream_ptr()), "d2dx_rollout_dfff")
        self.launches += 1
        return X_final

    def dcf(self, Binc, z_des, kr, p, c):
        """p, c: device [2][F*n_ac]; Binc host (n_ac, n_e); z_des host (n_e,)."""
        Binc = np.ascontiguousarray(Binc, np.float64); z_des = np.ascontiguousarray(z_des, np.float64).reshape(-1)
        n_ac, n_e = Binc.shape
        M = p.shape[1]; F = M // n_ac
        Ur = self.empty(M); e = self.empty(F * max(n_e, 1))
        check(lib.d2dx_dcf(self.h, F, n_ac, n_e, Binc.ctypes.data_as(C.POINTER(C.c_double)),
                           z_des.ctypes.data_as(C.POINTER(C.c_double)), float(kr), _ptr(p), _ptr(c), _ptr(Ur), _ptr(e),
                           self.stream_ptr()), "d2dx_dcf")
        self.launches += 1
        return Ur, e[:F * n_e]

    def norm_mpi_pi(self, v):
        out = torch.empty_like(v)
        check(lib.d2dx_norm_mpi_pi(self.h, v.numel(), _ptr(v), _ptr(out), self.stream_ptr()), "d2dx_norm_mpi_pi")
        self.launches += 1
        return out

    def circle_implicit(self, X, c, r):
        n = X.shape[1]; out = self.empty(3, n)
        check(lib.d2dx_circle_implicit(self.h, n, _ptr(X), _ptr(c), _ptr(r), _ptr(out), self.stream_ptr()), "d2dx_circle_implicit")
        self.launches += 1
        return out

    def gvf(self, X, c, r, ke, kd):
        n = X.shape[1]; out = self.empty(3, n)
        check(lib.d2dx_gvf(self.h, n, _ptr(X), _ptr(c), _ptr(r), float(ke), float(kd), _ptr(out), self.stream_ptr()), "d2dx_gvf")
        self.launches += 1
        return out

    def rollout_formation(self, n_ac, Binc, z_des, X0, c, r, ac, ke, kd, kr, v_c, dt, i_begin, i_end, nsub,
                          log_every=1, X_log=None, U_log=None, Rr_log=None, eth_log=None, X_final=None, flags=None):
        Binc = np.ascontiguousarray(Binc, np.float64); z_des = np.ascontiguousarray(z_des, np.float64).reshape(-1)
        n_e = Binc.shape[1] if Binc.ndim == 2 else 0
        M = X0.shape[1]; F = M // n_ac
        if X_final is None:
            X_final = self.empty(5, M)
        f = _lib.Formations(F, n_ac, n_e, _ptr(X0), _ptr(c), _ptr(r), _ptr(ac),
                            Binc.ctypes.data_as(C.POINTER(C.c_double)), z_des.ctypes.data_as(C.POINTER(C.c_double)),
                            float(ke), float(kd), float(kr), float(v_c))
        o = _lib.FormationOut(int(log_every), _ptr(X_log), _ptr(U_log), _ptr(Rr_log), _ptr(eth_log), _ptr(X_final), _ptr(flags))
        check(lib.d2dx_rollout_formation(self.h, C.byref(f), float(dt), int(i_begin), int(i_end), int(nsub), C.byref(o),
                                         self.stream_ptr()), "d2dx_rollout_formation")
        self.launches += 1
        return X_final

    # ---- 5-state LQR tracker ---------------------------------------------------------------------
    def flatness5(self, Ys, W, ac):
        n = Ys.shape[1]; Xr = self.empty(5, n); Ur = self.empty(2, n)
        check(lib.d2dx_flatness5(self.h, n, _ptr(Ys), _ptr(W), _ptr(ac), _ptr(Xr), _ptr(Ur), self.stream_ptr()), "d2dx_flatness5")
        self.launches += 1
        return Xr, Ur

    def tracker_control(self, X, Ys, W, ac, gains=None, lqr_state=None):
        n = X.shape[1]; U = self.empty(2, n); Xr = self.empty(5, n); dX = self.empty(5, n); K = self.empty(10, n)
        check(lib.d2dx_tracker_control(self.h, n, _ptr(X), _ptr(Ys), _ptr(W), _ptr(ac), C.byref(gains) if gains is not None else None,
                                       _ptr(U), _ptr(Xr), _ptr(dX), _ptr(K), _ptr(lqr_state), self.stream_ptr()), "d2dx_tracker_control")
        self.launches += 1
        return U, Xr, dX, K

    def rollout_tracker(self, ref, X0, wind, ac, dt, i_begin, i_end, nsub, gains=None, X_log=None, U_log=None, Xr_log=None,
                        dX_log=None, K_log=None, X_final=None, flags=None, lqr_state=None):
        T, _, M = ref.shape
        if X_final is None:
            X_final = self.empty(5, M)
        t = _lib.Tracker(M, T, _ptr(ref), _ptr(X0), _ptr(wind), _ptr(ac), float(dt))
        o = _lib.TrackerOut(_ptr(X_log), _ptr(U_log), _ptr(Xr_log), _ptr(dX_log), _ptr(K_log), _ptr(X_final), _ptr(flags), _ptr(lqr_state))
        check(lib.d2dx_rollout_tracker(self.h, C.byref(t), int(i_begin), int(i_end), int(nsub),
                                       C.byref(gains) if gains is not None else None, C.byref(o), self.stream_ptr()), "d2dx_rollout_tracker")
        self.launches += 1
        return X_final

    # ---- collocation -------------------------------------------------------------------------------
    def colloc_sizes(self, prob, layout=_lib.JAC_COMPACT):
        s = (C.c_int64 * 3)()
        check(lib.d2dx_colloc_sizes(C.byref(prob), layout, s), "d2dx_colloc_sizes")
        return tuple(int(v) for v in s)

    def colloc_scratch(self, prob, n_prob):
        return self.zeros(max(int(lib.d2dx_colloc_scratch_size(C.byref(prob), n_prob)), 1))

    def colloc_structure(self, prob, layout=_lib.JAC_COMPACT):
        nnz = self.colloc_sizes(prob, layout)[2]
        rows = self.empty(nnz, dtype=torch.int64); cols = self.empty(nnz, dtype=torch.int64)
        check(lib.d2dx_colloc_structure(self.h, C.byref(prob), layout, _ptr(rows), _ptr(cols), self.stream_ptr()), "d2dx_colloc_structure")
        self.launches += 1
        return rows, cols

    def colloc_init_dense(self, prob, n_prob, jac):
        check(lib.d2dx_colloc_init_dense(self.h, C.byref(prob), n_prob, _ptr(jac), self.stream_ptr()), "d2dx_colloc_init_dense")
        self.launches += 1

    def colloc_eval(self, prob, n_prob, free, layout, what, residual, jac, cost, grad, scratch):
        check(lib.d2dx_colloc_eval(self.h, C.byref(prob), n_prob, _ptr(free), layout, what, _ptr(residual), _ptr(jac),
                                   _ptr(cost), _ptr(grad), _ptr(scratch), self.stream_ptr()), "d2dx_colloc_eval")
        self.launches += 1

    def cost_bank_max(self, free, off_phi, N, obj_scale, want_cost=True, want_grad=True):
        """free: device (n_prob, n_free) -> (cost (n_prob,), grad (n_prob, n_free)) of CostBank's max mode"""
        n_prob, n_free = free.shape
        cost = self.empty(n_prob) if want_cost else None
        grad = self.empty(n_prob, n_free) if want_grad else None
        check(lib.d2dx_cost_bank_max(self.h, n_prob, n_free, int(off_phi), int(N), float(obj_scale), _ptr(free), _ptr(cost), _ptr(grad),
                                     self.stream_ptr()), "d2dx_cost_bank_max")
        self.launches += 1
        return cost, grad


    # ---- peer exchange (aircraft-sharded collocation over NVLink peer memory) -------------------------------
    def peer_create(self, world, rank, max_prob, n_ac_total, N):
        return PeerExchange(self, world, rank, max_prob, n_ac_total, N)

    def colloc_eval_peer(self, peer, prob_local, n_prob, a_lo, free_local, what, residual, jac, cost, grad):
        check(lib.d2dx_colloc_eval_peer(self.h, peer.p, C.byref(prob_local), n_prob, a_lo, _ptr(free_local), what, _ptr(residual),
                                        _ptr(jac), _ptr(cost), _ptr(grad), self.stream_ptr()), "d2dx_colloc_eval_peer")
        self.launches += 1

    # ---- single shooting (planner NLP solve) ------------------------------------------------------------
    def shoot_forward(self, prob, P, u, bounds, p0, p1, u_phys, xs, c):
        b = (C.c_double * 4)(*bounds) if bounds is not None else None
        check(lib.d2dx_shoot_forward(self.h, C.byref(prob), P, _ptr(u), b, _ptr(p0), _ptr(p1), _ptr(u_phys), _ptr(xs), _ptr(c),
                                     self.stream_ptr()), "d2dx_shoot_forward")

    def shoot_adjoint(self, prob, P, u, bounds, u_phys, xs, c, lam, rho, cost, lagr, grad, state_box=None):
        b = (C.c_double * 4)(*bounds) if bounds is not None else None
        sb = (C.c_double * 5)(*state_box) if state_box is not None else None
        check(lib.d2dx_shoot_adjoint(self.h, C.byref(prob), P, _ptr(u), b, sb, _ptr(u_phys), _ptr(xs), _ptr(c), _ptr(lam), _ptr(rho),
                                     _ptr(cost), _ptr(lagr), _ptr(grad), self.stream_ptr()), "d2dx_shoot_adjoint")

    def lbfgs_layout(self, P, n, n_con, opts):
        off = (C.c_int64 * 8)()
        check(lib.d2dx_lbfgs_layout(P, n, n_con, C.byref(opts), off), "d2dx_lbfgs_layout")
        return list(off)

    def lbfgs_init(self, P, n, n_con, opts, state, lam, rho):
        check(lib.d2dx_lbfgs_init(self.h, P, n, n_con, C.byref(opts), _ptr(state), _ptr(lam), _ptr(rho), self.stream_ptr()), "d2dx_lbfgs_init")

    def al_lbfgs_tick(self, P, n, n_con, opts, state, x_trial, f_parts, cost_parts, n_parts, grad, c, lam, rho, n_running):
        check(lib.d2dx_al_lbfgs_tick(self.h, P, n, n_con, C.byref(opts), _ptr(state), _ptr(x_trial), _ptr(f_parts), _ptr(cost_parts),
                                     n_parts, _ptr(grad), _ptr(c), _ptr(lam), _ptr(rho), _ptr(n_running), self.stream_ptr()),
              "d2dx_al_lbfgs_tick")

    # ---- second-order planner solve (control-limited DDP, one thread per problem) ------------------------------
    def ddp_options(self, **kw):
        o = _lib.DdpOptions()
        check(lib.d2dx_ddp_default_options(C.byref(o)), "d2dx_ddp_default_options")
        for k, v in kw.items():
            setattr(o, k, v)
        return o

    def ddp_solve(self, prob, P, bounds, state_box, p0, p1, u, xs, info, opts=None):
        """u (P,2,N) in/out, xs (P,3,N) out, info (P,8) out, p0 / p1 (P,3): device tensors; bounds / state_box host tuples."""
        b = (C.c_double * 4)(*bounds)
        sb = (C.c_double * 5)(*state_box) if state_box is not None else None
        work = self.empty(int(lib.d2dx_ddp_work_size(P, prob.N)))
        check(lib.d2dx_ddp_solve(self.h, C.byref(prob), P, b, sb, _ptr(p0), _ptr(p1), _ptr(u), _ptr(xs), _ptr(info), _ptr(work),
                                 C.byref(opts) if opts is not None else None, self.stream_ptr()), "d2dx_ddp_solve")
        self.launches += 1

    def ddp_multi_solve(self, prob, P, bounds, state_box, p0, p1, u, xs, info, lam=None, opts=None):
        """coupled multi-aircraft solve (one warp per problem): u (P,2,n_ac,N) in/out, xs (P,3,n_ac,N) out, info (P,8) out,
        lam (P,3,n_ac) out or None, p0 / p1 (P,3,n_ac): device tensors; bounds / state_box host tuples."""
        b = (C.c_double * 4)(*bounds)
        sb = (C.c_double * 5)(*state_box) if state_box is not None else None
        work = self.empty(int(lib.d2dx_ddp_multi_work_size(P, prob.n_ac, prob.N)))
        check(lib.d2dx_ddp_multi_solve(self.h, C.byref(prob), P, b, sb, _ptr(p0), _ptr(p1), _ptr(u), _ptr(xs), _ptr(info),
                                       _ptr(lam), _ptr(work), C.byref(opts) if opts is not None else None,
                                       self.stream_ptr()), "d2dx_ddp_multi_solve")
        self.launches += 1

    # ---- pure pursuit ------------------------------------------------------------------------------------
    def pursuit(self, pts, lookahead=100, K=1., sat_phi=np.deg2rad(45.), v_sp=10.):
        """device copy of a sampled path (n_pts, 2) + the controller constants -> (struct, keep-alive tensors)"""
        px = self.to_device(np.ascontiguousarray(np.asarray(pts, np.float64)[:, 0]))
        py = self.to_device(np.ascontiguousarray(np.asarray(pts, np.float64)[:, 1]))
        return _lib.Pursuit(len(pts), px.data_ptr(), py.data_ptr(), int(lookahead), float(K), float(sat_phi), float(v_sp)), (px, py)

    def pursuit_control(self, pp, X):
        B = X.shape[1]
        U, idx = self.empty(2, B), self.zeros(B, dtype=torch.int32)
        check(lib.d2dx_pursuit_control(self.h, C.byref(pp), B, _ptr(X), _ptr(U), _ptr(idx), self.stream_ptr()), "d2dx_pursuit_control")
        return U, idx

    def rollout_pursuit(self, pp, X0, wind, ac, dt, i_begin, i_end, nsub=1, X_log=None, U_log=None, idx_log=None):
        B = X0.shape[1]
        Xf = self.empty(5, B)
        check(lib.d2dx_rollout_pursuit(self.h, C.byref(pp), B, _ptr(X0), _ptr(wind), _ptr(ac), float(dt), i_begin, i_end, nsub,
                                       _ptr(X_log), _ptr(U_log), _ptr(idx_log), _ptr(Xf), self.stream_ptr()), "d2dx_rollout_pursuit")
        return Xf

    def math_probe(self, x, y):
        """Engine elementary functions on device arrays x, y -> [13][n] (sin, cos, atan2(y,x), atan x, y/x, sqrt|x|, rsqrt|x|, 1/x, the residuals
        of the hardware reciprocal and reciprocal-square-root seeds, norm_mpi_pi(x), and the small-angle sin x, cos x for |x| < 2^-5)."""
        n = x.numel(); out = self.empty(13, n)
        check(lib.d2dx_math_probe(self.h, n, _ptr(x), _ptr(y), _ptr(out), self.stream_ptr()), "d2dx_math_probe")
        self.launches += 1
        return out

    def measure_fp64_peak(self, iters=20000, reps=5, details=False):
        """TFLOP/s of a pure DFMA kernel (16 independent chains per thread, 8 x 256 threads per SM), best of reps.
        details=True also returns the probe's parameters so that the division can be redone from the bench line."""
        sink = self.zeros(1)
        blocks, threads = self.sm_count * 8, 256
        best, best_ms = 0., None
        for _ in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            check(lib.d2dx_dfma_burn(self.h, blocks, threads, iters, _ptr(sink), self.stream_ptr()), "d2dx_dfma_burn")
            e1.record(); e1.synchronize()
            ms = e0.elapsed_time(e1)
            tf = blocks * threads * iters * 32.0 / (ms * 1e-3) / 1e12
            if tf > best:
                best, best_ms = tf, ms
        if details:
            return best, {"blocks": blocks, "threads": threads, "iters": iters, "flop_per_thread_iter": 32, "ms": best_ms,
                          "formula": "blocks*threads*iters*32 / ms"}
        return best


class PeerExchange:
    """One rank's exchange buffer of the fused aircraft-sharded evaluation (d2dx_peer_*, include/d2dx.h)."""

    def __init__(self, eng, world, rank, max_prob, n_ac_total, N):
        self.eng, self.world, self.rank = eng, int(world), int(rank)
        p = C.c_void_p()
        check(lib.d2dx_peer_create(eng.h, self.world, self.rank, int(max_prob), int(n_ac_total), int(N), C.byref(p)), "d2dx_peer_create")
        self.p = p

    def ipc_handle(self):
        buf = C.create_string_buffer(_lib.IPC_HANDLE_BYTES)
        check(lib.d2dx_peer_ipc_handle(self.p, buf), "d2dx_peer_ipc_handle")
        return buf.raw

    def connect_ipc(self, handles):
        """handles: list of `world` 64-byte blobs in rank order (all_gather_object of ipc_handle())."""
        blob = b"".join(bytes(h_) for h_ in handles)
        assert len(blob) == self.world * _lib.IPC_HANDLE_BYTES
        check(lib.d2dx_peer_connect_ipc(self.p, blob), "d2dx_peer_connect_ipc")

    def connect_local(self, peers):
        """peers: the `world` PeerExchange objects of one process, rank order."""
        arr = (C.c_void_p * self.world)(*[q.p for q in peers])
        check(lib.d2dx_peer_connect_local(self.p, arr), "d2dx_peer_connect_local")

    def status(self):
        s = (C.c_int32 * 4)()
        check(lib.d2dx_peer_status(self.p, s), "d2dx_peer_status")
        return {"timeouts": s[0], "evaluations": s[1], "resident_blocks": s[2], "buffer_kib": s[3]}

    def timeline(self):
        """ns since kernel start of the last evaluation's phases on this rank (d2dx_peer_timeline)"""
        s = (C.c_uint64 * 8)()
        check(lib.d2dx_peer_timeline(self.p, s), "d2dx_peer_timeline")
        names = ("published", "local_done", "positions_arrived", "pairs_done", "cost_sent", "cost_arrived", "block0_leaves")
        return {n: (int(s[k + 1]) - int(s[0])) if s[k + 1] else None for k, n in enumerate(names)}

    def close(self):
        if getattr(self, "p", None):
            lib.d2dx_peer_destroy(self.p)
            self.p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default = None
_lock = threading.Lock()


def get_engine():
    """Process-wide default engine on cuda:LOCAL_RANK (created on first use)."""
    global _default
    with _lock:
        if _default is None:
            _default = Engine()
        return _default
