"""ctypes binding of libd2dx.so -- exactly the symbols declared in include/d2dx.h.

There is no CPU fallback: importing this module fails loudly when the shared library is
missing, and `Engine()` fails loudly when no CUDA device is present."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("D2DX_LIB") or os.path.join(_HERE, "libd2dx.so")     # D2DX_LIB: A/B builds of the same ABI

SEG_LINE, SEG_CIRCLE, SEG_SLALOM, SEG_POLY, SEG_SI_LINE, SEG_TABLE, SEG_SI_CIRCLE = range(7)
SEG_NPAR = 17
JAC_COMPACT, JAC_OPTY_DENSE = 0, 1
EVAL_RESIDUAL, EVAL_JAC, EVAL_COST, EVAL_GRAD = 1, 2, 4, 8
EVAL_ALL = 15
MAX_OBSTACLES = 16
PEER_MAX_WORLD, IPC_HANDLE_BYTES = 16, 64
CARE_STATE_ROWS = 9    # D2DX_CARE_STATE_ROWS: rows of the Riccati warm start (care_state)

c_dp = C.c_void_p      # device pointers travel as integers


class TrajTable(C.Structure):
    _fields_ = [("n_traj", C.c_int32), ("n_seg", C.c_int32),
                ("first_seg", c_dp), ("n_segs", c_dp), ("traj_t0", c_dp), ("traj_dur", c_dp),
                ("seg_type", c_dp), ("seg_end", c_dp), ("seg_par", c_dp), ("uniform_type", C.c_int32),
                ("n_tab", C.c_int32), ("tab_time", c_dp), ("tab_x", c_dp), ("tab_y", c_dp), ("tab_vx", c_dp), ("tab_vy", c_dp)]


class DfffGains(C.Structure):
    _fields_ = [("q_pos", C.c_double), ("q_psi", C.c_double), ("r_phi", C.c_double), ("r_v", C.c_double),
                ("err_sat", C.c_double * 5), ("u_lo", C.c_double * 2), ("u_hi", C.c_double * 2)]


class Scenarios(C.Structure):
    _fields_ = [("B", C.c_int32), ("X0", c_dp), ("wind", c_dp), ("ac", c_dp), ("traj", TrajTable),
                ("pert_begin", c_dp), ("pert_step", c_dp), ("pert_dx", c_dp), ("n_events", C.c_int32)]


class RolloutOut(C.Structure):
    _fields_ = [("log_every", C.c_int32), ("X_log", c_dp), ("U_log", c_dp), ("Xr_log", c_dp), ("K_log", c_dp),
                ("X_final", c_dp), ("sum_sq_err", c_dp), ("max_err", c_dp), ("flags", c_dp),
                ("care_state", c_dp), ("pop_stats", c_dp)]


class TrackerGains(C.Structure):
    _fields_ = [("q", C.c_double * 5), ("r", C.c_double * 2), ("err_sat", C.c_double * 5),
                ("u_lo", C.c_double * 2), ("u_hi", C.c_double * 2)]


class Tracker(C.Structure):
    _fields_ = [("M", C.c_int32), ("T", C.c_int32), ("ref", c_dp), ("X0", c_dp), ("wind", c_dp), ("ac", c_dp), ("dt", C.c_double)]


class TrackerOut(C.Structure):
    _fields_ = [("X_log", c_dp), ("U_log", c_dp), ("Xr_log", c_dp), ("dX_log", c_dp), ("K_log", c_dp), ("X_final", c_dp),
                ("flags", c_dp), ("lqr_state", c_dp)]


class Formations(C.Structure):
    _fields_ = [("F", C.c_int32), ("n_ac", C.c_int32), ("n_e", C.c_int32),
                ("X0", c_dp), ("c", c_dp), ("r", c_dp), ("ac", c_dp),
                ("Binc_host", C.POINTER(C.c_double)), ("z_des_host", C.POINTER(C.c_double)),
                ("ke", C.c_double), ("kd", C.c_double), ("kr", C.c_double), ("v_c", C.c_double)]


class FormationOut(C.Structure):
    _fields_ = [("log_every", C.c_int32), ("X_log", c_dp), ("U_log", c_dp), ("Rr_log", c_dp), ("eth_log", c_dp),
                ("X_final", c_dp), ("flags", c_dp)]


class CollocProblem(C.Structure):
    _fields_ = [("n_ac", C.c_int32), ("N", C.c_int32), ("h", C.c_double), ("wind", C.c_double * 2),
                ("perm_phi", c_dp), ("perm_v", c_dp),
                ("n_inst", C.c_int32), ("inst_var", c_dp), ("inst_node", c_dp), ("inst_val", c_dp),
                ("obj_scale", C.c_double), ("vsp", C.c_double), ("kvel", C.c_double), ("kbank", C.c_double),
                ("in_div", C.c_int32), ("kobs", C.c_double), ("obs_kind", C.c_int32), ("n_obs", C.c_int32),
                ("obs", (C.c_double * 3) * MAX_OBSTACLES),
                ("kcol", C.c_double), ("rcol", C.c_double), ("kcol_k", C.c_double),
                ("col_all_pairs", C.c_int32), ("exact_grad", C.c_int32)]


class D2dxError(RuntimeError):
    pass


class Pursuit(C.Structure):
    """d2dx_pursuit (include/d2dx.h)."""
    _fields_ = [("n_pts", C.c_int32), ("px", C.c_void_p), ("py", C.c_void_p), ("lookahead", C.c_int32),
                ("K", C.c_double), ("sat_phi", C.c_double), ("v_sp", C.c_double)]


class DdpOptions(C.Structure):
    """d2dx_ddp_options (include/d2dx.h)."""
    _fields_ = [("max_iter", C.c_int32), ("max_outer", C.c_int32), ("max_inner", C.c_int32), ("ls_max", C.c_int32), ("ctol", C.c_double),
                ("rel_tol", C.c_double), ("abs_tol", C.c_double), ("rho0", C.c_double), ("rho_growth", C.c_double), ("rho_max", C.c_double),
                ("mu0", C.c_double), ("mu_min", C.c_double), ("mu_max", C.c_double), ("mu_factor", C.c_double), ("reg_mode", C.c_int32), ("min_solved", C.c_int32)]


class LbfgsOptions(C.Structure):
    """d2dx_lbfgs_options (include/d2dx.h)."""
    _fields_ = [("m", C.c_int32), ("max_inner", C.c_int32), ("max_outer", C.c_int32), ("ls_max", C.c_int32), ("window", C.c_int32),
                ("gtol", C.c_double), ("ftol", C.c_double), ("ctol", C.c_double), ("rho0", C.c_double), ("rho_max", C.c_double),
                ("keep_history", C.c_int32)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (or `make -C drone-sim-python_b200/csrc`). "
            "d2d_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    H = C.c_void_p
    P = C.POINTER
    i32, i64, u32, dbl = C.c_int32, C.c_int64, C.c_uint32, C.c_double
    sig = {
        "d2dx_version": (C.c_int, []),
        "d2dx_last_error": (C.c_char_p, []),
        "d2dx_create": (C.c_int, [C.c_int, P(H)]),
        "d2dx_destroy": (C.c_int, [H]),
        "d2dx_device_info": (C.c_int, [H, P(i32)]),
        "d2dx_traj_eval": (C.c_int, [H, P(TrajTable), i32, c_dp, c_dp, c_dp]),
        "d2dx_cont_dyn": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_disc_dyn": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp, dbl, i32, c_dp, c_dp]),
        "d2dx_cont_jac": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_flatness": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_dfff_default_gains": (C.c_int, [P(DfffGains)]),
        "d2dx_dfff_control": (C.c_int, [H, P(TrajTable), c_dp, dbl, c_dp, c_dp, P(DfffGains), c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_rollout_dfff": (C.c_int, [H, P(Scenarios), c_dp, i32, i32, i32, i32, P(DfffGains), P(RolloutOut), c_dp]),
        "d2dx_tracker_default_gains": (C.c_int, [P(TrackerGains)]),
        "d2dx_flatness5": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_tracker_control": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp, P(TrackerGains), c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_rollout_tracker": (C.c_int, [H, P(Tracker), i32, i32, i32, P(TrackerGains), P(TrackerOut), c_dp]),
        "d2dx_dcf": (C.c_int, [H, i32, i32, i32, P(dbl), P(dbl), dbl, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_norm_mpi_pi": (C.c_int, [H, i32, c_dp, c_dp, c_dp]),
        "d2dx_circle_implicit": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_gvf": (C.c_int, [H, i32, c_dp, c_dp, c_dp, dbl, dbl, c_dp, c_dp]),
        "d2dx_rollout_formation": (C.c_int, [H, P(Formations), dbl, i32, i32, i32, P(FormationOut), c_dp]),
        "d2dx_colloc_sizes": (C.c_int, [P(CollocProblem), i32, P(i64)]),
        "d2dx_colloc_structure": (C.c_int, [H, P(CollocProblem), i32, c_dp, c_dp, c_dp]),
        "d2dx_colloc_init_dense": (C.c_int, [H, P(CollocProblem), i32, c_dp, c_dp]),
        "d2dx_colloc_scratch_size": (i64, [P(CollocProblem), i32]),
        "d2dx_colloc_eval": (C.c_int, [H, P(CollocProblem), i32, c_dp, i32, u32, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_cost_bank_max": (C.c_int, [H, i32, i32, i32, i32, dbl, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_peer_create": (C.c_int, [H, i32, i32, i32, i32, i32, P(H)]),
        "d2dx_peer_ipc_handle": (C.c_int, [H, C.c_char_p]),
        "d2dx_peer_connect_ipc": (C.c_int, [H, C.c_char_p]),
        "d2dx_peer_connect_local": (C.c_int, [H, P(H)]),
        "d2dx_peer_status": (C.c_int, [H, P(i32)]),
        "d2dx_peer_timeline": (C.c_int, [H, P(C.c_uint64)]),
        "d2dx_peer_destroy": (C.c_int, [H]),
        "d2dx_colloc_eval_peer": (C.c_int, [H, H, P(CollocProblem), i32, i32, c_dp, u32, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_shoot_forward": (C.c_int, [H, P(CollocProblem), i32, c_dp, P(dbl), c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_shoot_adjoint": (C.c_int, [H, P(CollocProblem), i32, c_dp, P(dbl), P(dbl), c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_lbfgs_layout": (C.c_int, [i32, i32, i32, P(LbfgsOptions), P(i64)]),
        "d2dx_lbfgs_init": (C.c_int, [H, i32, i32, i32, P(LbfgsOptions), c_dp, c_dp, c_dp, c_dp]),
        "d2dx_al_lbfgs_tick": (C.c_int, [H, i32, i32, i32, P(LbfgsOptions), c_dp, c_dp, c_dp, c_dp, i32, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_ddp_default_options": (C.c_int, [P(DdpOptions)]),
        "d2dx_ddp_work_size": (i64, [i32, i32]),
        "d2dx_ddp_solve": (C.c_int, [H, P(CollocProblem), i32, P(dbl), P(dbl), c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, P(DdpOptions), c_dp]),
        "d2dx_ddp_multi_work_size": (i64, [i32, i32, i32]),
        "d2dx_ddp_multi_solve": (C.c_int, [H, P(CollocProblem), i32, P(dbl), P(dbl), c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, P(DdpOptions), c_dp]),
        "d2dx_pursuit_control": (C.c_int, [H, P(Pursuit), i32, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_rollout_pursuit": (C.c_int, [H, P(Pursuit), i32, c_dp, c_dp, c_dp, dbl, i32, i32, i32, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "d2dx_dfma_burn": (C.c_int, [H, i32, i32, i32, c_dp, c_dp]),
        "d2dx_math_probe": (C.c_int, [H, i32, c_dp, c_dp, c_dp, c_dp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)        # AttributeError here = header and library out of sync
        fn.restype, fn.argtypes = res, args
    return lib, sig


lib, SIGNATURES = _load()
EXPORTED = tuple(SIGNATURES)


def check(rc, what=""):
    if rc != 0:
        raise D2dxError(f"{what}: d2dx error {rc}: {lib.d2dx_last_error().decode()}")
