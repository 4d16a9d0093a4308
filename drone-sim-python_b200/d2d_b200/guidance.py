"""Guidance laws -- the `d2d.guidance` call surface (d2d/guidance.py:10-181), evaluated by the engine.

Single calls (`DFFFController.get`, `DCFController.get`, `GVFcontroller.get`, ...) keep the reference's
signatures and return types; each is one kernel launch on a batch of size 1 (or n).  Closed-loop simulations
should use `d2d_b200.simulation`, which fuses controller and integrator in one rollout kernel."""
import numpy as np

from . import trajectory as ddt
from .dynamic import Aircraft
from .engine import get_engine


def norm_mpi_pi(v):
    """Wrap to [-pi, pi) with floored modulo (d2d/guidance.py:10), evaluated by the engine (bit-identical to NumPy's `%`)."""
    eng = get_engine()
    a = np.asarray(v, dtype=np.float64)
    out = eng.norm_mpi_pi(eng.to_device(np.ascontiguousarray(a.reshape(-1)))).cpu().numpy().reshape(a.shape)
    return float(out) if a.ndim == 0 else out


class WindField:
    """Constant wind (d2d/guidance.py:12-19)."""

    def __init__(self, w=[0., 0.]):
        self.w = w

    def sample(self, t, loc):
        return self.w

    def summarize(self):
        return f"{self.w} m/s"


class DiffFlatness:
    """Flat output -> state and input (d2d/guidance.py:22-47).  Called without an instance, as the reference does."""

    def state_and_input_from_output(Ys, W, ac):
        eng = get_engine()
        Ys = np.asarray(Ys, dtype=np.float64)
        single = Ys.ndim == 2
        Yb = Ys.reshape(-1, 4, 2)
        n = len(Yb)
        Yd = eng.to_device(np.ascontiguousarray(Yb.reshape(n, 8).T))
        Wd = eng.to_device(np.ascontiguousarray(np.broadcast_to(np.asarray(W, dtype=np.float64).reshape(-1, 2), (n, 2)).T))
        acd = eng.to_device(np.ascontiguousarray(np.broadcast_to(np.array([[ac.tau_phi], [ac.tau_v]]), (2, n))))
        Xr, Ur, Xd = (a.cpu().numpy().T for a in eng.flatness(Yd, Wd, acd))
        return (Xr[0], Ur[0], Xd[0]) if single else (Xr, Ur, Xd)


class DFFFController:
    """Differential-flatness feed-forward + LQR feedback (d2d/guidance.py:52-91).  `get(X, t)` returns the
    saturated input U and appends the reference state and the gain to `Xref` / `K` like the reference."""

    def __init__(self, traj, ac, wind):
        self.traj, self.ac, self.wind = traj, ac, wind
        self.dt = 0.01
        self.time = np.arange(0, traj.duration, self.dt)
        self.carrot, self.ref_pos = [0, 0], [0, 0]
        self.Xref, self.K = [], []
        self._table = None
        self._care = None

    def get(self, X, t):
        eng = get_engine()
        if self._table is None:
            self._table = eng.table(ddt.pack([self.traj]))
            from . import _lib
            self._care = eng.zeros(_lib.CARE_STATE_ROWS, 1)
        W = np.asarray(self.wind.sample(t, None), dtype=np.float64).reshape(2, 1)
        acd = eng.to_device(np.array([[self.ac.tau_phi], [self.ac.tau_v]]))
        Xd = eng.to_device(np.asarray(X, dtype=np.float64).reshape(5, 1))
        U, Xr, K = eng.dfff_control(self._table, Xd, t, eng.to_device(W), acd, care_state=self._care)
        self.Xref.append(Xr.cpu().numpy()[:, 0])
        K5 = np.zeros((2, 5))
        K5[:, :3] = K.cpu().numpy()[:, 0].reshape(2, 3)
        self.K.append(K5)
        return U.cpu().numpy()[:, 0]


class DCFController:
    """Distributed circular-formation controller (d2d/guidance.py:99-126)."""

    def get(self, n_ac, B, c, p, z_des, kr):
        eng = get_engine()
        z_des = np.asarray(z_des, dtype=np.float64)
        B = np.asarray(B, dtype=np.float64).reshape(n_ac, -1)
        c = np.asarray(c, dtype=np.float64)
        if c.shape != (n_ac, 2):
            raise ValueError(f"operands could not be broadcast together: p is (2,{n_ac}), c.T is {c.T.shape} "
                             "(c must be (n_ac, 2), cf. d2d/guidance.py:106)")
        pd = eng.to_device(np.ascontiguousarray(np.asarray(p, dtype=np.float64).reshape(2, n_ac)))
        cd = eng.to_device(np.ascontiguousarray(c.T))
        Ur, e = eng.dcf(B, z_des.reshape(-1), kr, pd, cd)
        return Ur.cpu().numpy().reshape(n_ac, 1), e.cpu().numpy().reshape(-1, 1)


class CircleTraj:
    """Implicit circle e = |p - c|^2 - r^2, its gradient n and Hessian H = 2I (d2d/guidance.py:133-146)."""

    def __init__(self, c=np.array([0, 0])):
        self.c = c

    def get(self, X, r=1):
        eng = get_engine()
        Xd = eng.to_device(np.asarray(X, dtype=np.float64).reshape(5, 1))
        cd = eng.to_device(np.asarray(self.c, dtype=np.float64).reshape(2, 1))
        rd = eng.to_device(np.asarray(r, dtype=np.float64).reshape(1))
        e, nx, ny = eng.circle_implicit(Xd, cd, rd).cpu().numpy()[:, 0]
        return np.asarray(e), np.asarray([nx, ny]), np.asarray([[2, 0], [0, 2]])


class GVFcontroller:
    """Guidance vector field heading controller (d2d/guidance.py:148-181)."""

    def __init__(self, traj, ac, wind):
        self.traj, self.ac, self.wind = traj, ac, wind

    def get(self, X, ke, kd, e, n, H):
        """(e, n) as returned by CircleTraj.get(X, r): they fix the circle for this state, c = p - n/2 and
        r^2 = |n/2|^2 - e, which is what the device function takes.  H is the constant 2I of the circle."""
        eng = get_engine()
        X = np.asarray(X, dtype=np.float64).reshape(5)
        n = np.asarray(n, dtype=np.float64).reshape(2)
        c = X[:2] - n / 2
        r = np.sqrt(max(float(np.sum(np.square(n / 2))) - float(np.asarray(e).reshape(-1)[0]), 0.))
        out = eng.gvf(eng.to_device(X.reshape(5, 1)), eng.to_device(c.reshape(2, 1)), eng.to_device(np.array([r])), ke, kd)
        U, U1, U2 = out.cpu().numpy()[:, 0]
        return U, U1, U2


class VelControler:
    """Timing PI loop of d2d/guidance.py:188-202 (host arithmetic; unused upstream: control_vel is False)."""

    def __init__(self):
        self.Kp, self.Ki = 2., 0.001
        self.sat_err, self.sat_vel, self.ref_vel, self.sum_err = 10., 4, 10., 0.

    def get(self, tself, tref):
        timing_error = np.clip(tself - tref, -self.sat_err, self.sat_err)
        self.sum_err += timing_error
        return self.ref_vel - np.clip(self.Kp * timing_error + self.Ki * self.sum_err, -self.sat_vel, self.sat_vel)


class PurePursuitControler:
    """Pure pursuit on the trajectory sampled every 0.01 s (d2d/guidance.py:204-245): carrot 100 samples (10 m at 10 m/s)
    ahead of the nearest sample, phi_sp = clip(-wrap(psi - bearing to the carrot), +-45 deg), v_sp = 10.  `get(X, t)` and
    the closed loop (simulation.run_simulation / simulation.pursuit_rollout) run on the engine."""

    def __init__(self, traj):
        self.traj = traj
        self.time = np.arange(0, traj.duration, 0.01)
        self.pts_2d = np.asarray(traj.get_many(self.time))[:, 0, :]
        self.sat_phi = np.deg2rad(45.)
        self.ref_pos, self.carrot = [], []
        self.vel_ctl = VelControler()
        self.control_vel = False
        self._pp = None

    def device_path(self):
        if self._pp is None:
            self._pp = get_engine().pursuit(self.pts_2d, lookahead=int(10 / 10 / 0.01), K=1., sat_phi=self.sat_phi, v_sp=10.)
        return self._pp[0]

    def get(self, X, t):
        eng = get_engine()
        U, idx = eng.pursuit_control(self.device_path(), eng.to_device(np.asarray(X, dtype=np.float64).reshape(5, 1)))
        i = int(idx.item())
        ic = i + 100
        self.ref_pos.append(self.pts_2d[i])
        self.carrot.append(self.pts_2d[ic - len(self.pts_2d) if ic >= len(self.pts_2d) else ic])
        U = U.cpu().numpy()[:, 0]
        if self.control_vel:
            U[1] = self.vel_ctl.get(self.time[i], t)
        return U
