"""ctypes driver of the host build of the planner's second-order solvers (csrc/host_check.cu -> tests/native/libd2dx_hostcheck.so):
used by tests/test_ddp_cpu.py, tests/test_ddp_multi_cpu.py and for development without a GPU."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tests", "native", "libd2dx_hostcheck.so")


class DdpOptions(C.Structure):
    _fields_ = [("max_iter", C.c_int32), ("max_outer", C.c_int32), ("max_inner", C.c_int32), ("ls_max", C.c_int32), ("ctol", C.c_double),
                ("rel_tol", C.c_double), ("abs_tol", C.c_double), ("rho0", C.c_double), ("rho_growth", C.c_double), ("rho_max", C.c_double),
                ("mu0", C.c_double), ("mu_min", C.c_double), ("mu_max", C.c_double), ("mu_factor", C.c_double), ("reg_mode", C.c_int32), ("min_solved", C.c_int32)]


def default_options(**kw):
    o = DdpOptions(400, 30, 40, 12, 1e-8, 1e-10, 1e-14, 10., 10., 1e8, 1e-6, 1e-8, 1e10, 1.6, 0, 0)
    for k, v in kw.items():
        setattr(o, k, v)
    return o


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(LIB)
        dp = C.POINTER(C.c_double)
        _lib.d2dx_host_ddp_solve.argtypes = [dp, C.c_int, dp, dp, dp, dp, dp, C.POINTER(DdpOptions), dp, dp, dp]
        _lib.d2dx_host_ddp_multi_solve.argtypes = [C.c_void_p, dp, dp, dp, dp, C.POINTER(DdpOptions), dp, dp, dp, dp]
        _lib.d2dx_host_box_qp.argtypes = [C.c_int, dp, dp, dp, dp, dp, C.POINTER(C.c_int)]
    return _lib


def solve(N, h, wind, vsp, kvel, kbank, bounds, z0, zt, phi0, v0, obstacles=(), kobs=0., obs_kind=0, box=None, obj_scale=1., in_div=1, opts=None):
    """one problem; weights are the planner's (kvel, kbank, kobs), normalised here like d2dx_ddp.cu does.  Returns u (2,N), xs (3,N), info dict"""
    dp = C.POINTER(C.c_double)
    sN = obj_scale / N
    prob = np.array([N, h, wind[0], wind[1], vsp, kvel * sN / in_div, kbank * sN / in_div, kobs * sN if len(obstacles) else 0., obs_kind], float)
    obs = np.ascontiguousarray(np.asarray(obstacles, float).reshape(-1, 3)) if len(obstacles) else np.zeros((1, 3))
    b = np.asarray(bounds, float)
    bx = None if box is None else np.array([box[0], box[1], box[2], box[3], box[4] * sN], float)
    u = np.ascontiguousarray(np.stack([np.broadcast_to(phi0, (N,)), np.broadcast_to(v0, (N,))]).astype(float))
    xs, info = np.zeros((3, N)), np.zeros(8)
    z0, zt = np.asarray(z0, float), np.asarray(zt, float)
    o = opts or default_options()
    P = lambda a: a.ctypes.data_as(dp)
    lib().d2dx_host_ddp_solve(P(prob), len(obstacles), P(obs), P(b), None if bx is None else P(bx), P(z0), P(zt), C.byref(o), P(u), P(xs), P(info))
    keys = ("flag", "iterations", "outer", "cost", "cmax", "lagr", "mu", "rho")
    return u, xs, dict(zip(keys, info))


def colloc_problem(n_ac, N, h, wind=(0., 0.), vsp=10., kvel=0., kbank=0., obstacles=(), kobs=0., obs_kind=0, kcol=0., rcol=3., kcol_k=2.,
                   all_pairs=False, obj_scale=1., in_div=None):
    """d2dx_colloc_problem of the multi-aircraft classes (in_div = n_ac unless given); the struct of d2d_b200._lib."""
    from d2d_b200 import _lib as L
    p = L.CollocProblem()
    p.n_ac, p.N, p.h = n_ac, N, h
    p.wind[0], p.wind[1] = wind
    p.obj_scale, p.vsp, p.kvel, p.kbank, p.in_div = obj_scale, vsp, kvel, kbank, n_ac if in_div is None else in_div
    p.kobs, p.obs_kind, p.n_obs = kobs, obs_kind, len(obstacles)
    for k, o in enumerate(obstacles):
        p.obs[k][0], p.obs[k][1], p.obs[k][2] = o
    p.kcol, p.rcol, p.kcol_k, p.col_all_pairs = kcol, rcol, kcol_k, int(all_pairs)
    return p


def solve_multi(prob, bounds, p0, p1, phi0, v0, box=None, opts=None):
    """one coupled problem (d2dx_host_ddp_multi_solve): prob a d2dx_colloc_problem, p0 / p1 (3, n_ac), phi0 / v0 broadcastable to
    (n_ac, N), box (x_lo, x_hi, y_lo, y_hi, weight) or None.  Returns u (2, n_ac, N), xs (3, n_ac, N), info dict (with lam (3, n_ac))"""
    dp = C.POINTER(C.c_double)
    n, N = prob.n_ac, prob.N
    u = np.ascontiguousarray(np.stack([np.broadcast_to(np.asarray(phi0, float).reshape(-1, 1) if np.ndim(phi0) < 2 else phi0, (n, N)),
                                       np.broadcast_to(np.asarray(v0, float).reshape(-1, 1) if np.ndim(v0) < 2 else v0, (n, N))]).astype(float))
    xs, info, lam = np.zeros((3, n, N)), np.zeros(8), np.zeros((3, n))
    P = lambda a: np.ascontiguousarray(a, dtype=float).ctypes.data_as(dp)
    b, z0, zt = np.asarray(bounds, float), np.ascontiguousarray(np.asarray(p0, float).reshape(3, n)), np.ascontiguousarray(np.asarray(p1, float).reshape(3, n))
    bx = None if box is None else np.asarray(box, float)
    o = opts or default_options()
    rc = lib().d2dx_host_ddp_multi_solve(C.byref(prob), P(b), None if bx is None else P(bx), P(z0), P(zt), C.byref(o), P(u), P(xs), P(info),
                                         P(lam))
    if rc:
        raise ValueError("d2dx_host_ddp_multi_solve refused the problem")
    keys = ("flag", "iterations", "outer", "cost", "cmax", "lagr", "mu", "rho")
    return u, xs, {**dict(zip(keys, info)), "lam": lam}


def box_qp(H, g, lo, hi):
    """d2dx_host_box_qp: minimiser of 1/2 x^T H x + g^T x over [lo, hi] and the free flags"""
    dp = C.POINTER(C.c_double)
    n = len(g)
    H, g, lo, hi = (np.ascontiguousarray(a, dtype=float) for a in (H, g, lo, hi))
    x, fr = np.zeros(n), np.zeros(n, np.int32)
    P = lambda a: a.ctypes.data_as(dp)
    if lib().d2dx_host_box_qp(n, P(H), P(g), P(lo), P(hi), P(x), fr.ctypes.data_as(C.POINTER(C.c_int))):
        raise ValueError("d2dx_host_box_qp: a free block was not definite")
    return x, fr.astype(bool)


if __name__ == "__main__":
    import time
    # exp_0: turn around, 10 s at 10 Hz; and the C3 grid (20 s at 50 Hz)
    for N, h, T in ((101, 0.1, 10.), (1001, 0.02, 20.)):
        for phi0 in (0.1, -0.1, 0.3):
            t0 = time.perf_counter()
            u, xs, info = solve(N, h, (0., 0.), 12., 1., 0., (-np.deg2rad(30), np.deg2rad(30), 9., 14.), (0., 0., 0.), (0., 30., np.pi), phi0, 12.)
            print(N, phi0, {k: (f"{v:.3e}" if isinstance(v, float) and abs(v) < 1e-2 else v) for k, v in info.items()}, f"{time.perf_counter() - t0:.3f}s")
