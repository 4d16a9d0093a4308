"""Planner front-ends -- the `Planner` classes of 06_optyplan.py:25-145 (single aircraft) and
07_multioptyplan.py:28-121 (aircraft set), with `self.prob` backed by the collocation kernel instead of
opty's generated code.  `prob` exposes what IPOPT calls (`obj`, `obj_grad`, `con`, `con_jac`,
`jacobianstructure`, `num_free`); `run()` solves the NLP on the GPU by single shooting (d2d_b200/shooting.py)
instead of IPOPT."""
import numpy as np

from . import shooting

from . import multiopty_utils as d2mou
from . import opty_utils as d2ou
from .collocation import CollocationProblem


def _node_of(t, t0, h, N):
    """opty attaches an instance constraint to the grid node nearest to its time (SURVEY 8a B4)."""
    return int(min(max(round((t - t0) / h), 0), N - 1))


def inputs_from_path(x, y, h, phi_b, v_b, smooth_s=1.0, g=9.81):
    """Inputs that roughly fly a guessed path (x, y per node): airspeed from the node spacing, bank from the heading rate
    (phi = atan(v psi_dot / g)) after a moving average of `smooth_s` seconds, both clipped inside the bounds.  A shooting
    solve cannot use a state guess directly; this turns the planners' `tri` / straight-line guesses into an input guess
    that bends the same way."""
    x, y = np.asarray(x, float), np.asarray(y, float)
    dx, dy = np.gradient(x), np.gradient(y)
    v = np.clip(np.hypot(dx, dy) / h, v_b[0] + 0.05 * (v_b[1] - v_b[0]), v_b[1] - 0.05 * (v_b[1] - v_b[0]))
    psi = np.unwrap(np.arctan2(dy, dx))
    w = max(int(round(smooth_s / h)) | 1, 1)
    psid = np.gradient(psi) / h
    if w > 1 and len(psid) > w:
        psid = np.convolve(np.pad(psid, w // 2, mode="edge"), np.ones(w) / w, mode="valid")
    phi = np.arctan(v * psid / g)
    return np.clip(phi, 0.9 * phi_b[0], 0.9 * phi_b[1]), v


class _PlannerBase:
    def configure(self, tol=1e-8, max_iter=3000):
        self.tol, self.max_iter = tol, max_iter

    def run(self, initial_guess=None, n_starts=1, seed=0, verbose=False, state_weight=1000., min_solved=None, **_):
        """`self.solution, info = prob.solve(initial_guess)` of 06_optyplan.py:117-125 / 07_multioptyplan.py:80-88,
        solved by single shooting + augmented Lagrangian (shooting.solve).  Only the input part of `initial_guess`
        seeds the solve (the states follow from the inputs).  n_starts > 1 adds randomly perturbed starts solved in the
        same launches; the feasible one of least cost is kept (`min_solved=k` returns as soon as k starts have converged).  State bounds (x/y_constraint) enter as a soft box
        (`state_weight` x squared excess, averaged over the nodes); `self.info["state_bounds_ok"]` tells whether the result
        respects them strictly."""
        guess = self.get_initial_guess() if initial_guess is None else np.asarray(initial_guess, dtype=float)
        n, N = self._n_ac, self.num_nodes
        phi_b, v_b = self._bounds["phi"], self._bounds["v"]
        if phi_b is None or v_b is None:
            raise ValueError("run() needs phi_constraint and v_constraint (lo, hi) on the experiment / scenario")
        phi = np.stack([guess[sl] for sl in self._phi_slices()])
        v = np.stack([guess[sl] for sl in self._v_slices()])
        if _.get("guess_from_path", False):                       # opt-in: bend the input guess like the guessed path (measured: no gain on upstream's experiments)
            for a, (sx, sy) in enumerate(zip(self._x_slices(), self._y_slices())):
                if np.ptp(guess[sx]) + np.ptp(guess[sy]) > 1e-9 and not np.any(phi[a]):
                    phi[a], v[a] = inputs_from_path(guess[sx], guess[sy], self.time_step, phi_b, v_b)
        phi, v = phi[None], v[None]
        if n_starts > 1:
            rng = np.random.default_rng(seed)
            k = np.concatenate([[0.], np.ones(n_starts - 1)])[:, None, None]      # start 0 is the caller's guess
            phi = phi + k * rng.normal(0., 0.25 * (phi_b[1] - phi_b[0]), (n_starts, n, 1))
            v = v + k * rng.normal(0., 0.25 * (v_b[1] - v_b[0]), (n_starts, n, 1))
        p0, p1 = self._boundary_states()
        box = None
        if "x" in self._bounds or "y" in self._bounds:
            bx, by = self._bounds.get("x", (-np.inf, np.inf)), self._bounds.get("y", (-np.inf, np.inf))
            box = (max(bx[0], -1e300), min(bx[1], 1e300), max(by[0], -1e300), min(by[1], 1e300), state_weight)
        tol = getattr(self, "tol", 1e-8)
        method = _.get("method", "lbfgs" if _.get("driver") == "host" else "auto")
        frees = info = None
        if n == 1 and method in ("auto", "ddp"):
            # second-order solve (control-limited DDP, one GPU thread per start): the caller's start, a deterministic family of
            # constant-bank starts (both turn directions) and random ones; milliseconds, so it always gets at least nine starts
            n_ddp = max(n_starts, 9)
            fam = np.array([0., 0.3, -0.3, 0.7, -0.7, 0.1, -0.1, 0.95, -0.95]) * max(abs(phi_b[0]), abs(phi_b[1]))
            rng = np.random.default_rng(seed)
            phi_s = np.concatenate([phi[:, 0], np.repeat(fam[:, None], N, 1), rng.uniform(phi_b[0], phi_b[1], (n_ddp, 1)) * np.ones((1, N))])[:n_ddp]
            v_s = np.concatenate([v[:, 0], np.full((len(fam), N), float(np.clip(getattr(self, "_vref", v[0, 0].mean()), *v_b))),
                                  rng.uniform(v_b[0], v_b[1], (n_ddp, 1)) * np.ones((1, N))])[:n_ddp]
            nlp = shooting.ShootingNLP(self.prob, p0, p1, phi_b, v_b, P=n_ddp, state_box=box)
            # asked for one solution (n_starts = 1): stop as soon as three starts have converged; asked for many: run them all out
            k_enough = (min_solved if min_solved is not None else (3 if n_starts == 1 else 0))
            frees, info = shooting.solve_ddp(nlp, phi_s, v_s, ctol=min(tol, 1e-6), verbose=verbose, min_solved=k_enough)
            info["nfev"] = info["iterations"]
            if method == "auto" and not np.isin(info["flag"], (2, 4)).any():
                frees = info = None                                   # no start converged: hand the problem to the first-order driver
        elif method == "ddp":
            # coupled second-order solve (one GPU warp per start): the caller's start, its mirror image (the other turn directions)
            # and the perturbed starts drawn above, n_starts in all (at least the first two)
            k = max(n_starts, 2)
            phi_s, v_s = np.concatenate([phi[:1], -phi[:1], phi[1:]])[:k], np.concatenate([v[:1], v[:1], v[1:]])[:k]
            nlp = shooting.ShootingNLP(self.prob, p0, p1, phi_b, v_b, P=len(phi_s), state_box=box)
            k_enough = (min_solved if min_solved is not None else (3 if n_starts == 1 else 0))
            frees, info = shooting.solve_ddp(nlp, phi_s, v_s, ctol=min(tol, 1e-6), verbose=verbose, min_solved=k_enough)
            info["nfev"] = info["iterations"]
        if frees is None:
            nlp = shooting.ShootingNLP(self.prob, p0, p1, phi_b, v_b, P=n_starts, state_box=box)
            driver = shooting.solve_host if _.get("driver") == "host" else shooting.solve
            kw = {} if driver is shooting.solve_host else {"min_solved": min_solved}
            theta, info = driver(nlp, nlp.theta_of(np.clip(phi, *phi_b), np.clip(v, *v_b)), ctol=min(tol, 1e-6),
                                 max_inner=min(getattr(self, "max_iter", 3000), 500), verbose=verbose, **kw)
            info["method"] = "lbfgs"
            frees = nlp.free_vectors()
        if self.prob.c.perm_phi:                                                  # opty input order: place the input blocks by rank
            frees = self._to_opty_order(frees)
        feas = info["c_max"] < 100 * min(tol, 1e-6)
        if info.get("method") == "ddp" and np.isin(info["flag"], (2, 4)).any():
            feas = np.isin(info["flag"], (2, 4))                                  # starts cut short by the early exit are not candidates
        best = int(np.argmin(np.where(feas, info["cost"], np.inf))) if feas.any() else int(np.argmin(info["c_max"]))
        self.solution = frees[best].copy()
        info.update(best=best, feasible=bool(feas[best]), solutions=frees)
        ok = True
        for key, sls in (("x", self._x_slices()), ("y", self._y_slices())):
            if key in self._bounds:
                lo, hi = self._bounds[key]
                ok = ok and all(self.solution[sl].min() >= lo - 1e-9 and self.solution[sl].max() <= hi + 1e-9 for sl in sls)
        info["state_bounds_ok"] = ok
        self.info = info
        self.interpret_solution()
        return info

    def evaluate(self, free):
        """residual, Jacobian values, cost, gradient at `free` in one fused launch."""
        return self.prob.evaluate(free)


class Planner(_PlannerBase):
    """Single-aircraft planner (06_optyplan.py:25-145).  `exp` carries t0, t1, hz, p0, p1, wind, cost, obj_scale,
    phi/v/x/y constraints, vref (d2d/optyplan_scenarios.py)."""

    def __init__(self, exp, initialize=True, jac_layout="dense"):
        self.exp, self.obj_scale = exp, exp.obj_scale
        self.num_nodes, self.time_step, self.duration = d2ou.planner_timing(exp.t0, exp.t1, exp.hz)
        self.wind, self.aircraft = exp.wind, d2ou.Aircraft()
        N = self.num_nodes
        self._slice_x, self._slice_y, self._slice_psi, self._slice_phi, self._slice_v = \
            [slice(k * N, (k + 1) * N, 1) for k in range(5)]                        # :35-39
        n0 = _node_of(exp.t0, exp.t0, self.time_step, N)
        n1 = _node_of(exp.t1, exp.t0, self.time_step, N)
        self._instance_constraints = [(k, n0, exp.p0[k]) for k in range(3)] + [(k, n1, exp.p1[k]) for k in range(3)]   # :46-49
        self._bounds = {"phi": exp.phi_constraint, "v": exp.v_constraint}           # :53-57 (variable bounds for the NLP solver)
        if exp.x_constraint is not None: self._bounds["x"] = exp.x_constraint
        if exp.y_constraint is not None: self._bounds["y"] = exp.y_constraint
        self.obstacles = getattr(exp, "obstacles", ())
        if initialize:
            w = exp.wind.sample_num(0., 0., 0.)
            self.prob = CollocationProblem(1, N, self.time_step, wind=w, inst=self._instance_constraints,
                                           cost=exp.cost.spec(), obj_scale=self.obj_scale, layout=jac_layout, multi=False)

    _n_ac = 1
    def _phi_slices(self): return [self._slice_phi]
    def _v_slices(self): return [self._slice_v]
    def _x_slices(self): return [self._slice_x]
    def _y_slices(self): return [self._slice_y]
    def _boundary_states(self):
        return np.array(self.exp.p0[:3], float).reshape(3, 1), np.array(self.exp.p1[:3], float).reshape(3, 1)

    def get_initial_guess(self, kind="tri", seed=None):                             # :79-115
        N = self.num_nodes
        guess = np.zeros(5 * N)
        p0, p1 = np.array(self.exp.p0[:2], dtype=float), np.array(self.exp.p1[:2], dtype=float)
        if kind == "rnd":
            rng = np.random.default_rng(seed)
            cx = self.exp.x_constraint or [-100, 100]
            cy = self.exp.y_constraint or [-100, 100]
            guess[self._slice_x] = rng.uniform(cx[0], cx[1], N)
            guess[self._slice_y] = rng.uniform(cy[0], cy[1], N)
            guess[self._slice_psi] = rng.uniform(-np.pi, np.pi, N)
        elif kind == "tri":
            x, y, psi, phi, v = d2ou.triangle(p0, p1, self.exp.vref, self.duration, N, go_left=-1.)
            guess[self._slice_x], guess[self._slice_y], guess[self._slice_psi] = x, y, psi
            guess[self._slice_phi], guess[self._slice_v] = phi, v
        else:
            guess[self._slice_x] = np.linspace(p0[0], p1[0], N)
            guess[self._slice_y] = np.linspace(p0[1], p1[1], N)
        return guess

    def interpret_solution(self):                                                   # :127-133
        self.sol_time = np.linspace(0.0, self.duration, num=self.num_nodes)
        s = self.solution
        self.sol_x, self.sol_y, self.sol_psi = s[self._slice_x], s[self._slice_y], s[self._slice_psi]
        self.sol_phi, self.sol_v = s[self._slice_phi], s[self._slice_v]

    def save_solution(self, filename):                                              # :135-139 (same .npz keys)
        wind = np.array([self.wind.sample_num(_t, _x, _y) for _t, _x, _y in zip(self.sol_time, self.sol_x, self.sol_y)])
        np.savez(filename, sol_time=self.sol_time, sol_x=self.sol_x, sol_y=self.sol_y, sol_psi=self.sol_psi,
                 sol_phi=self.sol_phi, sol_v=self.sol_v, wind=wind)

    def load_solution(self, filename):                                              # :141-145
        d = np.load(filename)
        self.sol_time, self.sol_x, self.sol_y, self.sol_psi, self.sol_phi, self.sol_v = \
            [d[k] for k in ("sol_time", "sol_x", "sol_y", "sol_psi", "sol_phi", "sol_v")]
        self.solution = np.concatenate([self.sol_x, self.sol_y, self.sol_psi, self.sol_phi, self.sol_v])


class MultiPlanner(_PlannerBase):
    """Aircraft-set planner (07_multioptyplan.py:28-121).  `scen` carries t0, t1, hz, p0s, p1s, wind, cost,
    obj_scale, constraints, vref."""

    def __init__(self, scen, initialize=True, jac_layout="compact", input_order="numeric"):
        self.scen, self.obj_scale, self.wind = scen, scen.obj_scale, scen.wind
        self.acs = d2mou.AircraftSet(n=len(scen.p0s))
        self.num_nodes, self.time_step, self.duration = d2ou.planner_timing(scen.t0, scen.t1, scen.hz)
        N, n = self.num_nodes, self.acs.nb_aicraft
        self._slice_x = [slice((0 + 3 * i) * N, (1 + 3 * i) * N, 1) for i in range(n)]          # :41-47
        self._slice_y = [slice((1 + 3 * i) * N, (2 + 3 * i) * N, 1) for i in range(n)]
        self._slice_psi = [slice((2 + 3 * i) * N, (3 + 3 * i) * N, 1) for i in range(n)]
        o = 3 * n * N
        self._slice_phi = [slice(o + i * N, o + (i + 1) * N, 1) for i in range(n)]
        o += n * N
        self._slice_v = [slice(o + i * N, o + (i + 1) * N, 1) for i in range(n)]
        n0 = _node_of(scen.t0, scen.t0, self.time_step, N)
        n1 = _node_of(scen.t1, scen.t0, self.time_step, N)
        self._instance_constraints = [(3 * i + k, n0, p[k]) for i, p in enumerate(scen.p0s) for k in range(3)] + \
                                     [(3 * i + k, n1, p[k]) for i, p in enumerate(scen.p1s) for k in range(3)]   # :53-56
        self._bounds = {"phi": getattr(scen, "phi_constraint", None), "v": getattr(scen, "v_constraint", None)}   # :58-64
        if getattr(scen, "x_constraint", None) is not None: self._bounds["x"] = scen.x_constraint
        if getattr(scen, "y_constraint", None) is not None: self._bounds["y"] = scen.y_constraint
        if initialize:
            w = scen.wind.sample_num(0., 0., 0.)
            self.prob = CollocationProblem(n, N, self.time_step, wind=w, inst=self._instance_constraints,
                                           cost=scen.cost.spec(), obj_scale=self.obj_scale, layout=jac_layout,
                                           input_order=input_order, multi=True)

    @property
    def _n_ac(self): return self.acs.nb_aicraft
    def _phi_slices(self): return self._slice_phi
    def _v_slices(self): return self._slice_v
    def _x_slices(self): return self._slice_x
    def _y_slices(self): return self._slice_y
    def _boundary_states(self):
        return np.array([p[:3] for p in self.scen.p0s], float).T, np.array([p[:3] for p in self.scen.p1s], float).T

    def _to_opty_order(self, frees):
        """numeric input blocks [phi_0..phi_{n-1} | v_0..v_{n-1}] -> opty's name-sorted block order (SURVEY D9)."""
        n, N = self.acs.nb_aicraft, self.num_nodes
        names = [f"phi{i}" for i in range(n)] + [f"v{i}" for i in range(n)]
        rank = {nm: k for k, nm in enumerate(sorted(names))}
        out = frees.copy()
        o = 3 * n * N
        for j, nm in enumerate(names):
            out[:, o + rank[nm] * N:o + (rank[nm] + 1) * N] = frees[:, o + j * N:o + (j + 1) * N]
        return out

    def get_initial_guess(self, what="tri", seed=None):                             # :94-112
        N, n = self.num_nodes, self.acs.nb_aicraft
        guess = np.zeros(5 * n * N)
        if what == "rnd":
            rng = np.random.default_rng(seed)
            for i in range(n):
                guess[self._slice_x[i]] = rng.uniform(-100, 100, N)
                guess[self._slice_y[i]] = rng.uniform(-100, 100, N)      # upstream draws y from the x range too (:99-102)
                guess[self._slice_psi[i]] = rng.uniform(-np.pi, np.pi, N)
                guess[self._slice_phi[i]] = rng.uniform(self.scen.phi_constraint[0], self.scen.phi_constraint[1], N)
                guess[self._slice_v[i]] = rng.uniform(self.scen.v_constraint[0], self.scen.v_constraint[1], N)
        else:
            for i, (p0, p1) in enumerate(zip(self.scen.p0s, self.scen.p1s)):
                x, y, psi, phi, v = d2ou.triangle(np.array(p0)[:2], np.array(p1)[:2], self.scen.vref, self.duration, N, go_left=-1.)
                guess[self._slice_x[i]], guess[self._slice_y[i]], guess[self._slice_psi[i]] = x, y, psi
                guess[self._slice_phi[i]], guess[self._slice_v[i]] = phi, v
        return guess

    def interpret_solution(self):                                                   # :115-121
        s = self.solution
        self.sol_time = np.linspace(0.0, self.duration, num=self.num_nodes)
        self.sol_x, self.sol_y = [s[k] for k in self._slice_x], [s[k] for k in self._slice_y]
        self.sol_psi, self.sol_v, self.sol_phi = [s[k] for k in self._slice_psi], [s[k] for k in self._slice_v], [s[k] for k in self._slice_phi]


    def load_csv(self, filename):
        """Reads a solution exported by save_csv / by 07_multioptyplan.py:476-489 into `self.solution`."""
        import pandas as pd
        df = pd.read_csv(filename)
        N, n = self.num_nodes, self.acs.nb_aicraft
        if len(df) != N:
            raise ValueError(f"{filename}: {len(df)} rows for a {N}-node problem")
        sol = np.zeros(5 * n * N)
        for i in range(n):
            sol[self._slice_x[i]], sol[self._slice_y[i]], sol[self._slice_psi[i]] = df[f"x_{i + 1}"], df[f"y_{i + 1}"], df[f"psi_{i + 1}"]
            sol[self._slice_phi[i]], sol[self._slice_v[i]] = df[f"phi_{i + 1}"], df[f"v_{i + 1}"]
        self.solution = sol
        self.interpret_solution()

    def save_csv(self, filename):
        """time, x_i, y_i, psi_i, phi_i, v_i (1-based i) per node -- the export of 07_multioptyplan.py:476-489, the
        input format of the tracker (10_opt_traj_tracking.py:30-38)."""
        import pandas as pd
        self.interpret_solution()
        cols = {"time": self.sol_time}
        for i in range(self.acs.nb_aicraft):
            cols[f"x_{i + 1}"], cols[f"y_{i + 1}"], cols[f"psi_{i + 1}"] = self.sol_x[i], self.sol_y[i], self.sol_psi[i]
            cols[f"phi_{i + 1}"], cols[f"v_{i + 1}"] = self.sol_phi[i], self.sol_v[i]
        pd.DataFrame(cols).to_csv(filename, index=False)


def compute_or_load(_p, force_recompute=False, filename="/tmp/optyplan.npz", tol=1e-5, max_iter=1500, initial_guess=None):
    """Cache front end of 06_optyplan.py:152-164: loads a cached solution when there is one, else solves (`_p.run`)
    and saves."""
    import os
    if force_recompute or not os.path.exists(filename):
        _p.configure(tol, max_iter)
        _p.run(_p.get_initial_guess() if initial_guess is None else initial_guess)
        _p.save_solution(filename)
    else:
        _p.load_solution(filename)


class exp_0:
    """Single-aircraft experiment 0 (d2d/optyplan_scenarios.py:9-28); other experiments subclass and override."""
    ncases = 1
    tol, max_iter = 1e-5, 1500
    vref = 12.
    cost = d2ou.CostAirVel(vref)
    obj_scale = 1.
    wind = d2ou.WindField(w=[0., 0.])
    obstacles = ()
    t0, p0 = 0., (0., 0., 0., 0., 10.)
    t1, p1 = 10., (0., 30., np.pi, 0., 10.)
    x_constraint, y_constraint = None, None
    phi_constraint = (-np.deg2rad(30.), np.deg2rad(30.))
    v_constraint = (9., 14.)
    hz = 10.
    name, desc = "exp0", "Turn around - 12m/s objective"
