"""Three-phase mission of 11_full_sim_case1.py / 12_full_sim_case2.py (SURVEY 8f #4, orchestration only) on the engine:
phase 1  GVF circular formation with per-aircraft centres until a stop criterion     (rollout_formation_kernel)
phase 2  multi-aircraft plan from the reached states to the formation entry states    (planner solve, shooting.py)
         followed by 5-state LQR tracking of the plan                                 (rollout_tracker_kernel)
phase 3  tracking of a pre-computed formation trajectory, repeated until t_sim_end     (rollout_tracker_kernel)
Function names and return tuples follow the scripts; plotting and animation are left out."""
import numpy as np

from . import multiopty_utils as d2mou
from . import opty_utils as d2ou
from .controllers import track
from .planner import MultiPlanner
from .simulation import chain_incidence, formation_rollout

ConstructBMatrix = chain_incidence                                   # 11_full_sim_case1.py:82-92


class trap_4:
    """Planner scenario of phase 2 (multi_opt_planner.py:170-242: exp_0 -> exp_5 -> trap_4, attributes flattened)."""
    name, desc = "trap_4", "trapezoidal formation with 4 aircraft"
    t0, t1, hz = 0., 10., 10
    wind = d2ou.WindField()
    initial_guess = "tri"
    tol, max_iter = 1e-5, 5000
    vref, dpsi = 12, 0
    x_constraint, y_constraint = (-150, 150), (-150, 150)
    phi_constraint = (-np.deg2rad(40.), np.deg2rad(40.))
    v_constraint = (9., 15.)
    obstacles = []
    ncases = 1
    cost, obj_scale = d2mou.CostComposit(kvel=70., kbank=1., kobs=float("nan"), kcol=10., vsp=12, obss=[], obs_kind=0, rcol=10), 1.e0

    @staticmethod
    def set_case(idx): pass

    @staticmethod
    def label(idx): return ""


def first_stop_index(X, X0f=None, e_theta=None, tol=(3., 3., np.deg2rad(0.5))):
    """Loop index i at which the scripts break, or None.  case 1 (11_full_sim_case1.py:140-175): at the TOP of iteration i,
    when every aircraft was within `tol` of X0f[:3] after the previous step (row i-1 >= 1); rows [:i] are kept.
    case 2 (12_full_sim_case2.py:156-164): INSIDE iteration i, when all e_theta of that iteration (row i) are <= 0.5 (signed,
    as written); rows [:i+1] are kept.  X (T, n_ac, 5), e_theta (T, n_ac-1) in the scripts' row conventions."""
    if e_theta is not None:
        hit = np.nonzero((e_theta[1:] <= 0.5).all(axis=1))[0]
        return int(hit[0]) + 1 if len(hit) else None
    ok = (np.abs(X[:, :, :3] - np.asarray(X0f, float)[None, :, :3]) <= np.asarray(tol)).all(axis=(1, 2))
    hit = np.nonzero(ok[1:])[0]
    return int(hit[0]) + 2 if len(hit) else None


def CircularFormationGVF(c, r, v, n_ac, X0f, t_start=0, t_step=0.05, t_end=1000, stop="states", chunk=4000, nsub=5,
                         X1=(20, 30, -np.pi / 2, 0, 10), ke=0.0004, kd=25, kr=20, z_des=None):
    """Phase 1 (11_full_sim_case1.py:94-177): returns X_array, U_array, U1_array, U2_array, Ur_array, e_theta_array,
    time, t_f, truncated where the script's loop breaks.  The formation is advanced `chunk` steps per launch and the
    stop criterion is evaluated on the logged states between launches (the model is time-invariant, so restarting from
    the last state is exact).  U1/U2 (debug split of the GVF output) are zeros, as in simulation.CircularFormationGVF."""
    time = np.arange(t_start, t_end, t_step)
    c = np.asarray(c, float).reshape(n_ac, 2)
    z_des = np.zeros(n_ac - 1) if z_des is None else np.asarray(z_des, float)
    X0 = np.tile(np.asarray(X1, float), (n_ac, 1))
    Xs, Us, Rs, Es = [X0[None]], [], [np.zeros((1, n_ac))], [np.zeros((1, n_ac - 1))]
    done, i_stop = 1, None
    while done < len(time) and i_stop is None:
        T = min(chunk, len(time) - done) + 1
        o = formation_rollout(c, r, n_ac, T, t_step, ke, kd, kr, z_des, X0, v_c=v, nsub=nsub)
        Xs.append(o["X"][0, 1:]); Us.append(o["U"][0, :-1]); Rs.append(o["Rr"][0, 1:]); Es.append(o["e_theta"][0, 1:])
        X0 = o["X_final"][0]
        done += T - 1
        i_stop = first_stop_index(np.concatenate(Xs), X0f) if stop == "states" else first_stop_index(None, e_theta=np.concatenate(Es))
        if i_stop is not None and i_stop > len(time) - 1:                # the loop ends before it could see the criterion
            i_stop = None
    X_all, R_all, E_all = np.concatenate(Xs), np.concatenate(Rs), np.concatenate(Es)
    U_all = np.zeros((len(X_all), n_ac, 2))
    U_all[:-1, :, 0], U_all[:-1, :, 1] = np.concatenate(Us), float(v)   # row i-1 = input of step i-1 -> i
    if i_stop is None:
        keep, t_f = len(X_all), t_end
    else:
        keep, t_f = (i_stop if stop == "states" else i_stop + 1), time[i_stop - 1]
        U_all[keep - 1:] = 0.                                            # not yet written when the script breaks
    Z = np.zeros((keep, n_ac))
    return X_all[:keep], U_all[:keep], Z, Z.copy(), R_all[:keep], E_all[:keep], time[:keep], t_f


def implement_controller(n_ac, time, x_ref, y_ref, v, w, X0s, nsub=10):
    """implement_controller(n_ac, time, x_ref, y_ref, v, w, X0s) of 11_full_sim_case1.py:241-291 ->
    X_array, U_array, X_ref_array, Yd_ref_array, Ydd_ref_array, dX_array."""
    X, U, Xr, Yd, Ydd, dX, _ = track(np.asarray(time, float), np.asarray(x_ref, float), np.asarray(y_ref, float), w,
                                     np.asarray(X0s, dtype=np.float64), nsub=nsub)
    return X, U, Xr, Yd, Ydd, dX


def trajectory_optimization(scen, n_starts=1, method="auto"):
    """Phase 2.1 (11_full_sim_case1.py:180-194) without the plots: returns the solved planner.  `method` goes to
    MultiPlanner.run ("ddp": the coupled second-order solver)."""
    _p = None
    for _case in range(scen.ncases):
        scen.set_case(_case)
        _p = MultiPlanner(scen, initialize=True)
        _p.configure(tol=scen.tol, max_iter=scen.max_iter)
        _p.run(initial_guess=_p.get_initial_guess(scen.initial_guess), n_starts=n_starts, method=method)
        _p.interpret_solution()
    return _p


def ExtractTrajData(df, n_ac):                                           # 11_full_sim_case1.py:206-217
    time_track = np.array(df["time"])
    x_ref, y_ref, psi_ref = (np.stack([np.array(df[f"{k}_{i + 1}"]) for i in range(n_ac)], axis=1) for k in ("x", "y", "psi"))
    return time_track, x_ref, y_ref, psi_ref


def ExtendTraj_symm(n_ac, x_ref, y_ref, psi_ref, time):
    """11_full_sim_case1.py:219-239: completes a trajectory that is symmetric about the y axis with the halves flown by
    the other aircraft (aircraft i continues on the half that starts where i ends).  As upstream, the appended half of
    `psi_ref` is filled from y (psi is not used by the tracker)."""
    time = np.append(time, time + time[-1])
    x0, xf, y0, yf = x_ref[0, :], x_ref[-1, :], y_ref[0, :], y_ref[-1, :]
    ax = [int(np.nonzero((x0 == xf[i]) & (y0 == yf[i]))[0][0]) for i in range(n_ac)]
    x_sym, y_sym = x_ref[:, ax], y_ref[:, ax]
    return time, np.append(x_ref, x_sym, axis=0), np.append(y_ref, y_sym, axis=0), np.append(psi_ref, y_sym, axis=0)


def full_sim(df, n_ac=4, v=15, w=(0, 0), r=60, c=((0, -20), (25, -20), (25, -100), (0, -100)),
             X1_f=((0, 40, 0, 0, 12), (25, 40, 0, 0, 12), (25, -40, 0, 0, 12), (0, -40, 0, 0, 12)),
             X2_f=((75, 40, 0, 0, 12), (100, 40, 0, 0, 12), (100, -40, 0, 0, 12), (75, -40, 0, 0, 12)),
             t_opt=6, t_sim_end=200, t_step=0.05, t_end_1=1000, stop="states", scen=trap_4, n_starts=1,
             method="auto"):
    """main() of 11_full_sim_case1.py:405-499 (stop="states") / 12_full_sim_case2.py (stop="e_theta") without plots.
    `df`: the phase-3 formation trajectory (columns time, x_i, y_i, psi_i; `inf_traj_10s.csv` upstream).
    `method`: the planner's solver in phase 2 (MultiPlanner.run).
    Returns a dict: X, U, time (all phases appended as upstream), the per-phase pieces and the solved planner."""
    X1, U1, _, _, Ur, e_theta, time_1, t1_f = CircularFormationGVF(np.asarray(c, float), r, v, n_ac, X1_f, 0, t_step, t_end_1, stop=stop)
    X_array, U_array, time = X1, U1, time_1
    # phase 2: plan from the reached states, then track the plan
    X2_i = tuple(map(tuple, X1[-1]))
    scen.t1, scen.p0s, scen.p1s = t_opt, X2_i, X2_f
    _p = trajectory_optimization(scen, n_starts=n_starts, method=method)
    x_ref_2, y_ref_2, time_opt = np.array(_p.sol_x).T, np.array(_p.sol_y).T, np.array(_p.sol_time)
    X2, U2, Xr2, Yd2, Ydd2, dX2 = implement_controller(n_ac, time_opt, x_ref_2, y_ref_2, v, list(w), X2_i)
    X_array, U_array = np.append(X_array, X2, axis=0), np.append(U_array, U2, axis=0)
    time = np.append(time, time_opt + t1_f, axis=0)
    # phase 3: the pre-computed formation trajectory, repeated
    X3_i = tuple(map(tuple, X2[-1]))
    time_3, x_ref_3, y_ref_3, psi_ref_3 = ExtractTrajData(df, n_ac)
    time_3, x_ref_3, y_ref_3, _ = ExtendTraj_symm(n_ac, x_ref_3, y_ref_3, psi_ref_3, time_3)
    X3_all, laps = [], 0
    while time[-1] <= t_sim_end:
        X3, U3, *_ = implement_controller(n_ac, time_3, x_ref_3, y_ref_3, v, list(w), X3_i)   # every lap restarts from X3_i, as upstream
        X_array, U_array = np.append(X_array, X3, axis=0), np.append(U_array, U3, axis=0)
        X3_all.append(X3)
        time = np.append(time, time_3 + time[-1], axis=0)
        laps += 1
    return {"X": X_array, "U": U_array, "time": time, "phase1": (X1, U1, Ur, e_theta, time_1, t1_f), "planner": _p,
            "phase2": (X2, U2, Xr2, time_opt), "phase3": (np.concatenate(X3_all) if X3_all else None, time_3, x_ref_3, y_ref_3), "laps": laps}
