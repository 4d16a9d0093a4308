"""Closed-loop simulation on the engine: `run_simulation` / `test_simulation` of 05_test_simulation.py and
`CircularFormationGVF` of 08_CircularFormation_Full.py / 09_CircularFormation_diffcentre.py, plus the batched
forms (`rollout`, `formation_rollout`) that the single-scenario functions are thin views of.

Host arrays in, host arrays out: each call copies its inputs to HBM, launches the fused rollout kernel and
copies the requested logs back."""
import numpy as np
import torch

from . import trajectory as ddt
from .dynamic import Aircraft
from .engine import get_engine
from .guidance import DFFFController, PurePursuitControler, WindField


def _perts_csr(eng, perts_list, T):
    """Dense per-scenario perturbation arrays (T,5) -> sparse CSR events on the device (or None)."""
    begin, steps, dxs = [0], [], []
    for p in perts_list:
        if p is not None:
            p = np.asarray(p, dtype=np.float64)
            rows = np.nonzero(np.any(p != 0., axis=1))[0]
            rows = rows[rows >= 1]                           # perts[0] is never applied (05_test_simulation.py:28-32)
            steps += list(rows); dxs += [p[r] for r in rows]
        begin.append(len(steps))
    if not steps:
        return None
    return (eng.to_device(np.asarray(begin, np.int32)), eng.to_device(np.asarray(steps, np.int32)),
            eng.to_device(np.ascontiguousarray(np.asarray(dxs, np.float64).T)))


class RolloutResult:
    """X (B,T_log,5), U (B,T_log,2), optional Xref (B,T_log,5), K (B,T_log,2,5), X_final (B,5),
    sum_sq_err (B,), max_err (B,), flags (B,)."""
    pass


def _family(tr):
    """Kernel family of a trajectory: the segment type when a specialised rollout kernel exists for it, else -1."""
    from . import _lib
    if tr.is_composite():
        return -1
    segs = tr.segments()
    return segs[0][0] if len(segs) == 1 and segs[0][0] in (_lib.SEG_CIRCLE, _lib.SEG_POLY, _lib.SEG_LINE) else -1


def _rollout_by_family(time, trajs, wind, X0, perts, tau_phi, tau_v, fams, **kw):
    """Mixed populations: one launch per trajectory family (warps stay homogeneous and the specialised kernels apply,
    SURVEY section 7 "sort scenarios by type"), results scattered back to the caller's order."""
    B = len(trajs)
    wind = np.broadcast_to(np.asarray(wind, dtype=np.float64).reshape(-1, 2), (B, 2))
    tp = np.broadcast_to(np.asarray(tau_phi, dtype=np.float64), (B,))
    tv = np.broadcast_to(np.asarray(tau_v, dtype=np.float64), (B,))
    parts = []
    for fam in sorted(set(fams)):
        idx = np.nonzero(np.asarray(fams) == fam)[0]
        sub = rollout(time, [trajs[i] for i in idx], wind[idx], X0[idx], perts=None if perts is None else [perts[i] for i in idx],
                      tau_phi=tp[idx], tau_v=tv[idx], group_by_family=False, **kw)
        parts.append((idx, sub))
    res = RolloutResult()
    first = parts[0][1]
    res.time_log = first.time_log
    for name in ("X_final", "sum_sq_err", "max_err", "flags", "X", "U", "Xref", "K"):
        if hasattr(first, name):
            ref = getattr(first, name)
            out = np.zeros((B,) + ref.shape[1:], dtype=ref.dtype)
            for idx, sub in parts:
                out[idx] = getattr(sub, name)
            setattr(res, name, out)
    res.pop_sum_sq_err = float(sum(sub.pop_sum_sq_err for _, sub in parts))
    res.pop_max_err = float(max(sub.pop_max_err for _, sub in parts))
    return res


def rollout(time, trajs, wind, X0, perts=None, tau_phi=0.01, tau_v=1., nsub=1, log_every=1, log_ref=False,
            final_control=True, gains=None, engine=None, chunk_steps=None, return_log=True, group_by_family=True):
    """Batched run_simulation (05_test_simulation.py:21-34) for B aircraft-scenarios.

    time   (T,) sample grid shared by all scenarios (np.arange as the reference builds it)
    trajs  list of B Trajectory objects, or a CircleBatch / MinSnapBatch
    wind   (2,) or (B,2);  X0 (B,5);  perts None or list of B arrays (T,5) / None
    tau_phi, tau_v scalars or (B,) arrays;  nsub RK4 sub-steps per control step
    """
    eng = engine or get_engine()
    time = np.ascontiguousarray(time, dtype=np.float64)
    T = len(time)
    X0 = np.asarray(X0, dtype=np.float64).reshape(-1, 5)
    B = len(X0)
    if group_by_family and isinstance(trajs, (list, tuple)) and B >= 256 and len(trajs) == B:
        fams = [_family(tr) for tr in trajs]
        if len(set(fams)) > 1:
            return _rollout_by_family(time, trajs, wind, X0, perts, tau_phi, tau_v, fams, nsub=nsub, log_every=log_every, log_ref=log_ref,
                                      final_control=final_control, gains=gains, engine=eng, chunk_steps=chunk_steps, return_log=return_log)
    packed = ddt.pack(trajs)
    if packed.n_traj != B:
        raise ValueError(f"{packed.n_traj} trajectories for {B} initial states")
    tab = eng.table(packed)
    wind = np.broadcast_to(np.asarray(wind, dtype=np.float64).reshape(-1, 2), (B, 2))
    ac = np.stack([np.broadcast_to(np.asarray(tau_phi, dtype=np.float64), (B,)), np.broadcast_to(np.asarray(tau_v, dtype=np.float64), (B,))])
    X0d, Wd, acd, td = eng.to_device(np.ascontiguousarray(X0.T)), eng.to_device(np.ascontiguousarray(wind.T)), eng.to_device(ac), eng.to_device(time)
    pd = _perts_csr(eng, perts, T) if perts is not None else None
    n_rows = (T - 1) // log_every + 1
    X_log = eng.empty(n_rows, 5, B) if return_log else None
    U_log = eng.empty(n_rows, 2, B) if return_log else None
    Xr_log = eng.empty(n_rows, 5, B) if (log_ref and return_log) else None
    K_log = eng.empty(n_rows, 6, B) if (log_ref and return_log) else None
    sum_sq, max_err = eng.zeros(B), eng.zeros(B)
    flags = eng.zeros(B, dtype=torch.int32)
    from . import _lib
    care = eng.zeros(_lib.CARE_STATE_ROWS, B)
    pop = eng.zeros(2)
    X_final = eng.empty(5, B)
    chunk = chunk_steps or (T - 1)
    i, Xc = 0, X0d
    while True:
        j = min(i + chunk, T - 1)
        last = j == T - 1
        eng.rollout_dfff(tab, Xc, Wd, acd, td, i, j, nsub=nsub, final_control=(final_control and last), gains=gains,
                         log_every=log_every, X_log=X_log, U_log=U_log, Xr_log=Xr_log, K_log=K_log, X_final=X_final,
                         sum_sq_err=sum_sq, max_err=max_err, flags=flags, care_state=care, pop_stats=pop, perts=pd)
        if last:
            break
        i, Xc = j, X_final
    if return_log and not final_control and (T - 1) % log_every == 0:
        # without the trailing controller evaluation (05_test_simulation.py:33) the kernel never visits sample T-1: its state
        # row comes from X_final, its input / reference / gain rows do not exist and read zero
        X_log[n_rows - 1] = X_final
        for t_ in (U_log, Xr_log, K_log):
            if t_ is not None:
                t_[n_rows - 1].zero_()
    res = RolloutResult()
    res.time_log = time[::log_every]
    res.X_final = X_final.cpu().numpy().T
    res.sum_sq_err, res.max_err, res.flags = sum_sq.cpu().numpy(), max_err.cpu().numpy(), flags.cpu().numpy()
    res.pop_sum_sq_err, res.pop_max_err = (float(v) for v in pop.cpu().numpy())
    if return_log:
        res.X = X_log.permute(2, 0, 1).contiguous().cpu().numpy()
        res.U = U_log.permute(2, 0, 1).contiguous().cpu().numpy()
        if log_ref:
            res.Xref = Xr_log.permute(2, 0, 1).contiguous().cpu().numpy()
            K3 = K_log.permute(2, 0, 1).contiguous().cpu().numpy().reshape(B, n_rows, 2, 3)
            res.K = np.concatenate([K3, np.zeros((B, n_rows, 2, 2))], axis=3)
    return res


def run_simulation(time, aircraft, windfield, ctl, X0, perts):
    """Drop-in for run_simulation(time, aircraft, windfield, ctl, X0, perts) -> X (T,5), U (T,2), Yref (T,4,2)
    (05_test_simulation.py:21-34).  `ctl` must be a DFFFController; its Xref / K logs are filled as upstream."""
    time = np.asarray(time, dtype=np.float64)
    if isinstance(ctl, PurePursuitControler):
        if np.any(np.asarray(perts)):
            raise ValueError("the pure-pursuit rollout takes no state perturbations")
        W = windfield.sample(time[0], None)
        X, U, idx = pursuit_rollout(ctl, time, np.asarray(X0, dtype=np.float64).reshape(1, 5), W, aircraft.tau_phi, aircraft.tau_v,
                                    nsub=getattr(aircraft, "nsub", 1))
        n = len(ctl.pts_2d)
        ctl.ref_pos += list(ctl.pts_2d[idx[:, 0]])
        ctl.carrot += list(ctl.pts_2d[(idx[:, 0] + 100) % n])
        return X[:, 0], U[:, 0], ctl.traj.get_many(time)
    if not isinstance(ctl, DFFFController):
        raise TypeError("run_simulation takes a DFFFController or a PurePursuitControler")
    W = windfield.sample(time[0], None)
    res = rollout(time, [ctl.traj], W, np.asarray(X0, dtype=np.float64).reshape(1, 5), perts=[perts],
                  tau_phi=aircraft.tau_phi, tau_v=aircraft.tau_v, nsub=getattr(aircraft, "nsub", 1), log_ref=True)
    ctl.Xref += list(res.Xref[0])
    ctl.K += list(res.K[0])
    Yref = ctl.traj.get_many(time)
    return res.X[0], res.U[0], Yref


def pursuit_rollout(ctl, time, X0, wind, tau_phi=0.01, tau_v=1., nsub=1):
    """B aircraft chasing the path of one PurePursuitControler in one launch: X0 (B,5), wind (2,) or (B,2).
    Returns X (T,B,5), U (T,B,2) (last row = control at the final state, 05_test_simulation.py:33), idx (T,B)."""
    eng = get_engine()
    time = np.asarray(time, dtype=np.float64)
    X0 = np.asarray(X0, dtype=np.float64).reshape(-1, 5)
    B, T = len(X0), len(time)
    wind = np.broadcast_to(np.asarray(wind, dtype=np.float64).reshape(-1, 2), (B, 2))
    ac = np.stack([np.full(B, tau_phi, dtype=np.float64), np.full(B, tau_v, dtype=np.float64)])
    X_log, U_log, idx_log = eng.empty(T, 5, B), eng.empty(T, 2, B), eng.zeros(T, B, dtype=torch.int32)
    pp = ctl.device_path()
    Xf = eng.rollout_pursuit(pp, eng.to_device(np.ascontiguousarray(X0.T)), eng.to_device(np.ascontiguousarray(wind.T)),
                             eng.to_device(ac), time[1] - time[0], 0, T - 1, nsub, X_log=X_log, U_log=U_log, idx_log=idx_log)
    U_last, idx_last = eng.pursuit_control(pp, Xf)
    U_log[T - 1], idx_log[T - 1] = U_last, idx_last
    return X_log.permute(0, 2, 1).cpu().numpy(), U_log.permute(0, 2, 1).cpu().numpy(), idx_log.cpu().numpy()


def test_simulation(scen, **_ignored):
    """Every aircraft of a scenario in ONE launch (the loop of 05_test_simulation.py:37-53).
    Returns Xs, Us, Yrefs lists like the upstream loop accumulates."""
    n = len(scen.trajs)
    W = scen.windfield.sample(scen.time[0], None)
    if getattr(scen, "ppctl", False):                        # 05_test_simulation.py:40-41: one pure-pursuit controller per trajectory
        Xs, Us = [], []
        for tr, ac, X0 in zip(scen.trajs, scen.aircrafts, scen.X0s):
            X, U, _ = pursuit_rollout(PurePursuitControler(tr), scen.time, np.asarray(X0, dtype=np.float64).reshape(1, 5), W, ac.tau_phi, ac.tau_v)
            Xs.append(X[:, 0]); Us.append(U[:, 0])
        return Xs, Us, [tr.get_many(scen.time) for tr in scen.trajs]
    res = rollout(scen.time, scen.trajs, W, np.asarray([np.asarray(x, dtype=np.float64) for x in scen.X0s[:n]]),
                  perts=list(scen.perts), tau_phi=[a.tau_phi for a in scen.aircrafts], tau_v=[a.tau_v for a in scen.aircrafts])
    Yrefs = [tr.get_many(scen.time) for tr in scen.trajs]
    return list(res.X), list(res.U), Yrefs


def chain_incidence(n_ac):
    """Incidence matrix of the line graph 0-1-...-(n_ac-1) (08_CircularFormation_Full.py:49-60)."""
    B = np.zeros((n_ac, max(n_ac - 1, 0)))
    for j in range(n_ac - 1):
        B[j, j], B[j + 1, j] = -1, 1
    return B


def formation_rollout(c, r, n_ac, time_len, dt, ke, kd, kr, z_des, X0, v_c=15., nsub=5, tau_phi=0.01, tau_v=1.,
                      B=None, log_every=1, engine=None, return_log=True):
    """F formations of n_ac aircraft in one launch.  c (F,n_ac,2), r scalar or (F,n_ac), X0 (F,n_ac,5).
    Returns dict with X (F,T,n_ac,5), U (F,T,n_ac), Rr (F,T,n_ac), e_theta (F,T,n_e) in the reference's row
    conventions (08_CircularFormation_Full.py:77-78,86: row i of Rr / e_theta belongs to step i-1 -> i)."""
    eng = engine or get_engine()
    c = np.asarray(c, dtype=np.float64).reshape(-1, n_ac, 2)
    F = len(c)
    M = F * n_ac
    X0 = np.broadcast_to(np.asarray(X0, dtype=np.float64), (F, n_ac, 5)).reshape(M, 5)
    r = np.broadcast_to(np.asarray(r, dtype=np.float64), (F, n_ac)).reshape(M)
    Binc = chain_incidence(n_ac) if B is None else np.asarray(B, dtype=np.float64)
    n_e = Binc.shape[1]
    ac = np.stack([np.full(M, tau_phi, dtype=np.float64), np.full(M, tau_v, dtype=np.float64)])
    T = int(time_len)
    n_rows = (T - 1) // log_every + 1
    X_log = eng.empty(n_rows, 5, M) if return_log else None
    U_log = eng.zeros(n_rows, M) if return_log else None
    Rr_log = eng.zeros(n_rows, M) if return_log else None
    eth_log = eng.zeros(n_rows, F * max(n_e, 1)) if return_log else None
    flags = eng.zeros(M, dtype=torch.int32)
    Xf = eng.rollout_formation(n_ac, Binc, z_des, eng.to_device(np.ascontiguousarray(X0.T)),
                               eng.to_device(np.ascontiguousarray(c.reshape(M, 2).T)), eng.to_device(r), eng.to_device(ac),
                               ke, kd, kr, v_c, dt, 0, T - 1, nsub, log_every=log_every, X_log=X_log, U_log=U_log,
                               Rr_log=Rr_log, eth_log=eth_log, flags=flags)
    out = {"X_final": Xf.cpu().numpy().T.reshape(F, n_ac, 5), "flags": flags.cpu().numpy().reshape(F, n_ac)}
    if return_log:
        out["X"] = X_log.cpu().numpy().reshape(n_rows, 5, F, n_ac).transpose(2, 0, 3, 1)
        out["U"] = U_log.cpu().numpy().reshape(n_rows, F, n_ac).transpose(1, 0, 2)
        if log_every == 1:                                   # reference row convention: row i holds step (i-1)'s value
            Rr = Rr_log.cpu().numpy().reshape(n_rows, F, n_ac).transpose(1, 0, 2)
            eth = eth_log.cpu().numpy()[:, :F * n_e].reshape(n_rows, F, n_e).transpose(1, 0, 2)
            out["Rr"] = np.concatenate([np.zeros((F, 1, n_ac)), Rr[:, :-1]], axis=1)
            out["e_theta"] = np.concatenate([np.zeros((F, 1, n_e)), eth[:, :-1]], axis=1)
    return out


def CircularFormationGVF(c, r, n_ac, t_end, ke=0.0004, kd=15, kr=20, z_des=None, t_step=0.05, nsub=5, tau_phi=0.01):
    """Drop-in for CircularFormationGVF(c, r, n_ac, t_end) (08_CircularFormation_Full.py:21-97) ->
    X_array, U_array, time, U1_array, U2_array, Ur_array, e_theta_array.  `c` may be one centre (2,) or one per
    aircraft (n_ac,2) as in script 09.  U1/U2 (debug split of the GVF output) are not logged by the rollout
    kernel and are returned as zeros; use GVFcontroller.get for them."""
    time = np.arange(0, t_end, t_step)
    c = np.asarray(c, dtype=np.float64)
    c_ = np.ones((n_ac, 2)) * c if c.ndim == 1 else c
    z_des = np.ones(n_ac - 1) * (np.pi * 2 / n_ac) if z_des is None else np.asarray(z_des, dtype=np.float64)
    X1 = np.array([20, 30, -np.pi / 2, 0, 10])               # 08_CircularFormation_Full.py:44
    o = formation_rollout(c_[None], r, n_ac, len(time), t_step, ke, kd, kr, z_des, X1, nsub=nsub, tau_phi=tau_phi)
    zeros = np.zeros((len(time), n_ac))
    return o["X"][0], o["U"][0], time, zeros, zeros.copy(), o["Rr"][0], o["e_theta"][0]


class MonteCarloRollout:
    """Monte-Carlo sweep of B independent plain-circle (or min-snap) scenarios (SURVEY 8d, config C5) with
    persistent pinned host buffers and device buffers.

    `run()` is the host-facing call: asynchronous H2D of the inputs from pinned memory, the rollout in
    `n_chunks` launches, and D2H of the decimated logs of chunk k on a copy stream while chunk k+1 computes;
    it returns NumPy views of the pinned result buffers.  `run_device()` is the same sweep with the inputs
    already resident in HBM and nothing copied back."""

    def __init__(self, B, time, seg_type, nsub=1, log_every=100, n_chunks=10, log_u=True, host_log=True, engine=None, host_log_u=True):
        from . import _lib
        from .engine import PackedTrajectories
        self.eng = eng = engine or get_engine()
        self.B, self.nsub, self.log_every = int(B), int(nsub), int(log_every)
        self.time = np.ascontiguousarray(time, dtype=np.float64)
        self.T = len(self.time)
        self.n_rows = (self.T - 1) // self.log_every + 1
        self.seg_type = int(seg_type)
        self.n_par_rows = {_lib.SEG_CIRCLE: 6, _lib.SEG_LINE: 5}.get(self.seg_type, _lib.SEG_NPAR)
        pin = lambda *shape, dtype=torch.float64: torch.empty(*shape, dtype=dtype).pin_memory()
        B = self.B
        # pinned host inputs / outputs
        self.h_X0, self.h_wind, self.h_ac, self.h_par = pin(5, B), pin(2, B), pin(2, B), pin(self.n_par_rows, B)
        self.h_Xf, self.h_ss, self.h_mx, self.h_flags = pin(5, B), pin(B), pin(B), pin(B, dtype=torch.int32)
        self.h_pop = pin(2)
        self.host_log, self.log_u = host_log, log_u
        self.h_Xlog = pin(self.n_rows, 5, B) if host_log else None
        self.h_Ulog = pin(self.n_rows, 2, B) if (host_log and log_u and host_log_u) else None      # host_log_u=False: only the STATE log travels
        # device buffers
        self.d_X0, self.d_wind, self.d_ac = eng.empty(5, B), eng.empty(2, B), eng.empty(2, B)
        par = eng.zeros(_lib.SEG_NPAR, B)
        ar = np.arange(B, dtype=np.int32)
        self.table = eng.table(PackedTrajectories(ar, np.ones(B, np.int32), np.zeros(B), np.zeros(B),
                                                  np.full(B, self.seg_type, np.int32), np.zeros(B), np.zeros((_lib.SEG_NPAR, B)),
                                                  self.seg_type))
        self.d_par = self.table.t["seg_par"]
        del par
        self.d_time = eng.to_device(self.time)
        self.d_Xlog = eng.empty(self.n_rows, 5, B)
        self.d_Ulog = eng.empty(self.n_rows, 2, B) if log_u else None
        self.d_Xf, self.d_Xa, self.d_Xb = eng.empty(5, B), eng.empty(5, B), eng.empty(5, B)
        self.d_ss, self.d_mx, self.d_flags = eng.zeros(B), eng.zeros(B), eng.zeros(B, dtype=torch.int32)
        self.d_care, self.d_pop = eng.zeros(_lib.CARE_STATE_ROWS, B), eng.zeros(2)
        # chunk boundaries aligned to the log stride
        steps = self.T - 1
        per = max(self.log_every, ((steps + n_chunks - 1) // n_chunks + self.log_every - 1) // self.log_every * self.log_every)
        self.bounds = list(range(0, steps, per)) + [steps]
        self.copy_stream = torch.cuda.Stream(device=eng.device)
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in (self.h_X0, self.h_wind, self.h_ac, self.h_par))
        self.d2h_bytes = sum(t.numel() * t.element_size() for t in (self.h_Xf, self.h_ss, self.h_mx, self.h_flags, self.h_pop)) + \
            sum(t.numel() * t.element_size() for t in (self.h_Xlog, self.h_Ulog) if t is not None)
        self.launches_per_run = len(self.bounds) - 1

    def set_inputs(self, par_rows, wind, X0, tau_phi=0.01, tau_v=1.):
        """par_rows (n_par_rows,B) segment parameters; wind (B,2); X0 (B,5).  Fills the pinned input buffers."""
        self.h_par.numpy()[...] = par_rows
        self.h_wind.numpy()[...] = np.asarray(wind, dtype=np.float64).T
        self.h_X0.numpy()[...] = np.asarray(X0, dtype=np.float64).T
        self.h_ac.numpy()[0], self.h_ac.numpy()[1] = tau_phi, tau_v

    def upload(self):
        self.d_X0.copy_(self.h_X0, non_blocking=True); self.d_wind.copy_(self.h_wind, non_blocking=True)
        self.d_ac.copy_(self.h_ac, non_blocking=True); self.d_par[:self.n_par_rows].copy_(self.h_par, non_blocking=True)

    def _sweep(self, copy_logs):
        eng = self.eng
        self.d_ss.zero_(); self.d_mx.zero_(); self.d_flags.zero_(); self.d_care.zero_(); self.d_pop.zero_()
        cur = torch.cuda.current_stream(eng.device)
        Xin, ping = self.d_X0, [self.d_Xa, self.d_Xb]
        for k in range(len(self.bounds) - 1):
            i, j = self.bounds[k], self.bounds[k + 1]
            last = j == self.T - 1
            Xout = self.d_Xf if last else ping[k % 2]
            eng.rollout_dfff(self.table, Xin, self.d_wind, self.d_ac, self.d_time, i, j, nsub=self.nsub, final_control=last,
                             log_every=self.log_every, X_log=self.d_Xlog, U_log=self.d_Ulog, X_final=Xout, sum_sq_err=self.d_ss,
                             max_err=self.d_mx, flags=self.d_flags, care_state=self.d_care, pop_stats=self.d_pop)
            Xin = Xout
            if copy_logs and self.host_log:
                r0 = (i + self.log_every - 1) // self.log_every
                r1 = (j // self.log_every + 1) if last else (j + self.log_every - 1) // self.log_every
                if r1 > r0:
                    ev = torch.cuda.Event(); ev.record(cur)
                    with torch.cuda.stream(self.copy_stream):
                        self.copy_stream.wait_event(ev)
                        self.h_Xlog[r0:r1].copy_(self.d_Xlog[r0:r1], non_blocking=True)
                        if self.h_Ulog is not None:
                            self.h_Ulog[r0:r1].copy_(self.d_Ulog[r0:r1], non_blocking=True)

    def run_device(self):
        """Inputs resident in HBM, results left in HBM (d_Xf, d_ss, d_mx, d_flags, d_Xlog, d_Ulog, d_pop)."""
        self._sweep(copy_logs=False)

    def run(self):
        """Host buffers in, host buffers out; returns when everything has landed in pinned memory."""
        self.upload()
        self._sweep(copy_logs=True)
        self.h_Xf.copy_(self.d_Xf, non_blocking=True); self.h_ss.copy_(self.d_ss, non_blocking=True)
        self.h_mx.copy_(self.d_mx, non_blocking=True); self.h_flags.copy_(self.d_flags, non_blocking=True)
        self.h_pop.copy_(self.d_pop, non_blocking=True)
        torch.cuda.current_stream(self.eng.device).synchronize()
        self.copy_stream.synchronize()
        out = {"X_final": self.h_Xf.numpy().T, "sum_sq_err": self.h_ss.numpy(), "max_err": self.h_mx.numpy(),
               "flags": self.h_flags.numpy(), "pop_sum_sq_err": float(self.h_pop[0]), "pop_max_err": float(self.h_pop[1])}
        if self.host_log:
            out["X_log"] = self.h_Xlog.numpy()
            if self.h_Ulog is not None:
                out["U_log"] = self.h_Ulog.numpy()
        return out
