"""NLP driver for the planners (SURVEY 8f #2): what `prob.solve(initial_guess)` (opty -> IPOPT) does in
06_optyplan.py:117-125 and 07_multioptyplan.py:80-88, re-posed for the GPU.

The backward-Euler defects of the collocation constraints fix the states once the inputs are chosen, so the solver
iterates on the inputs only (single shooting on the collocation grid): the 3 n_ac (N-1) defect constraints hold by
construction, the initial states are data, and only the 3 n_ac terminal conditions remain -- handled by an augmented
Lagrangian.  The input bounds are removed by the substitution phi = mid + half sin(theta).  Each Lagrangian/gradient
evaluation is two kernel launches (`d2dx_shoot_forward`, `d2dx_shoot_adjoint`) for P problems at once (multi-start or
a population of boundary conditions); the quasi-Newton update around them is batched limited-memory BFGS on device
tensors (vector algebra only).  The result satisfies the reference's constraints (`CollocationProblem.con`) to the
requested tolerance; like any local method it returns a local optimum that can differ from IPOPT's."""
import numpy as np
import torch



class ShootingNLP:
    """P simultaneous problems sharing one description (`prob`: a CollocationProblem, which supplies n_ac, N, h, wind
    and the cost).  p0, p1: (3, n_ac) or (P, 3, n_ac) initial states / terminal targets (x, y, psi).
    Device arrays are problem-major (include/d2dx.h): theta/u_phys/grad (P, 2, n_ac, N), xs (P, 3, n_ac, N)."""

    def __init__(self, prob, p0, p1, phi_bounds, v_bounds, P=1, engine=None, state_box=None):
        self.eng = e = engine or prob.eng
        self.prob, self.c_prob = prob, prob.c
        self.n_ac, self.N, self.P = prob.n_ac, prob.N, int(P)
        self.bounds = (float(phi_bounds[0]), float(phi_bounds[1]), float(v_bounds[0]), float(v_bounds[1]))
        self.mid = np.array([0.5 * (self.bounds[0] + self.bounds[1]), 0.5 * (self.bounds[2] + self.bounds[3])])
        self.half = np.array([0.5 * (self.bounds[1] - self.bounds[0]), 0.5 * (self.bounds[3] - self.bounds[2])])
        bc = lambda a: e.to_device(np.ascontiguousarray(np.broadcast_to(
            np.asarray(a, np.float64).reshape(-1, 3, self.n_ac), (self.P, 3, self.n_ac))))
        self.p0, self.p1 = bc(p0), bc(p1)
        n_ac, N = self.n_ac, self.N
        self.n, self.n_con = 2 * n_ac * N, 3 * n_ac
        self.u_phys, self.xs = e.empty(self.P, 2, n_ac, N), e.empty(self.P, 3, n_ac, N)
        self.c = e.empty(self.P, 3, n_ac)
        self.lam, self.rho = e.zeros(self.P, 3, n_ac), e.zeros(self.P) + 10.
        self.cost_ac, self.lagr_ac, self.grad = e.empty(self.P, n_ac), e.empty(self.P, n_ac), e.empty(self.P, 2, n_ac, N)
        self.nfev = 0
        self.state_box = None if state_box is None else tuple(float(v) for v in state_box)      # x_lo, x_hi, y_lo, y_hi, weight

    # ---- variables ------------------------------------------------------------------------------------
    def theta_of(self, phi, v):
        """host (n_ac, N) or (P, n_ac, N) physical inputs -> device theta (P, n); values are clipped just inside the bounds."""
        u = np.stack([np.asarray(phi, np.float64).reshape(-1, self.n_ac, self.N), np.asarray(v, np.float64).reshape(-1, self.n_ac, self.N)], 1)
        s = (u - self.mid[None, :, None, None]) / self.half[None, :, None, None]
        th = np.arcsin(np.clip(s, -0.999, 0.999))
        return self.eng.to_device(np.ascontiguousarray(np.broadcast_to(th, (self.P, 2, self.n_ac, self.N)))).reshape(self.P, self.n)

    def launch(self, theta):
        """the two kernels of one evaluation at theta (P, n); results stay in the buffers (graph-capturable)."""
        e = self.eng
        e.shoot_forward(self.c_prob, self.P, theta, self.bounds, self.p0, self.p1, self.u_phys, self.xs, self.c)
        e.shoot_adjoint(self.c_prob, self.P, theta, self.bounds, self.u_phys, self.xs, self.c, self.lam, self.rho,
                        self.cost_ac, self.lagr_ac, self.grad, state_box=self.state_box)
        self.nfev += 1

    def evaluate(self, theta):
        """theta: device (P, n).  Returns fresh (lagrangian (P,), gradient (P, n))."""
        self.launch(theta)
        return self.lagr_ac.sum(1), self.grad.reshape(self.P, self.n).clone()

    @property
    def cost(self): return self.cost_ac.sum(1)

    def free_vectors(self):
        """(P, num_free) host array in the planner's layout [x,y,psi per aircraft | phi per aircraft | v per aircraft]
        from the last evaluation."""
        xs = self.xs.permute(0, 2, 1, 3).reshape(self.P, -1)                      # [P][ac][k][N]
        return torch.cat([xs, self.u_phys.reshape(self.P, -1)], dim=1).cpu().numpy()


def lbfgs(fun, x, m=20, maxit=500, gtol=1e-10, ftol=1e-10, window=10, ls_max=30):
    """Batched limited-memory BFGS with Armijo backtracking: column p of x (n, P) is an independent problem.
    fun(x) -> (f (P,), g (n, P)) fresh tensors.  A problem stops when |g|_inf <= gtol, when f fell by less than
    ftol max(1, |f|) over the last `window` iterations, or when its line search fails twice in a row.
    Returns x, f, g, iterations."""
    n, P = x.shape
    kw = dict(dtype=x.dtype, device=x.device)
    f, g = fun(x)
    S, Y, rh = torch.zeros(m, n, P, **kw), torch.zeros(m, n, P, **kw), torch.zeros(m, P, **kw)
    gamma, have = torch.ones(P, **kw), torch.zeros(P, dtype=torch.bool, device=x.device)
    done = torch.zeros(P, dtype=torch.bool, device=x.device)
    head = cnt = it = 0
    f_hist = []
    for it in range(maxit):
        gn = g.abs().amax(0)
        done = done | (gn <= gtol)
        f_hist.append(f)
        if len(f_hist) > window:
            f_old = f_hist.pop(0)
            done = done | ((f_old - f) <= ftol * f.abs().clamp_min(1.0))
        if bool(done.all()):
            break
        q, al = g.clone(), []
        order = [(head - 1 - j) % m for j in range(min(cnt, m))]                # newest -> oldest
        for j in order:
            a = rh[j] * (S[j] * q).sum(0)
            al.append(a)
            q -= a * Y[j]
        r = q * gamma
        for j, a in zip(reversed(order), reversed(al)):
            r += S[j] * (a - rh[j] * (Y[j] * r).sum(0))
        d = -r
        bad = ~((g * d).sum(0) < -1e-14 * gn * gn)                               # not a descent direction -> steepest descent
        scale0 = 1.0 / g.abs().sum(0).clamp_min(1e-300)
        d = torch.where(bad | ~have, -g * torch.where(have, gamma, scale0), d)
        alpha, acc = torch.ones(P, **kw), done.clone()
        xn, fn, gnew = x.clone(), f.clone(), g.clone()
        for _ in range(ls_max):
            xt = x + alpha * d
            ft, gt = fun(xt)
            ok = (ft <= f + 1e-4 * alpha * (g * d).sum(0) + 1e-15 * f.abs()) & ~acc & torch.isfinite(ft)
            xn, fn, gnew = torch.where(ok, xt, xn), torch.where(ok, ft, fn), torch.where(ok, gt, gnew)
            acc = acc | ok
            if bool(acc.all()):
                break
            alpha = torch.where(acc, alpha, alpha * 0.5)
        failed = ~acc
        s, y = xn - x, gnew - g
        sy, ss, yy = (s * y).sum(0), (s * s).sum(0), (y * y).sum(0)
        good = (sy > 1e-10 * torch.sqrt(ss * yy)) & acc & ~done
        S[head], Y[head] = s * good, y * good
        rh[head] = torch.where(good, 1.0 / sy.clamp_min(1e-300), torch.zeros_like(sy))
        gamma, have = torch.where(good, sy / yy.clamp_min(1e-300), gamma), have | good
        head, cnt = (head + 1) % m, cnt + 1
        if bool(failed.any()):                                                   # drop the history of the problems that stalled
            S[:, :, failed], Y[:, :, failed], rh[:, failed] = 0, 0, 0
            done = done | (failed & (bad | ~have))
            have = have & ~failed
        x, f, g = xn, fn, gnew
    return x, f, g, it


def solve_host(nlp, theta, ctol=1e-8, gtol=1e-10, ftol=1e-10, max_outer=30, max_inner=500, rho0=10., rho_max=1e6, m=20, verbose=False):
    """Augmented-Lagrangian loop around the torch `lbfgs` (lock-step line searches, host decisions every iteration) --
    the cross-check of `solve`; same update rules."""
    nlp.lam.zero_()
    nlp.rho.fill_(rho0)
    total, c_prev = 0, None

    def fun(xT):
        f, g = nlp.evaluate(xT.t().contiguous())
        return f, g.t().contiguous()
    for outer in range(max_outer):
        xT, f, g, it = lbfgs(fun, theta.t().contiguous(), m=m, maxit=max_inner, gtol=gtol, ftol=ftol)
        theta = xT.t().contiguous()
        total += it
        nlp.launch(theta)                                                        # buffers at the returned point
        cmax = nlp.c.abs().amax(dim=(1, 2))
        if verbose:
            print(f"outer {outer}: inner its {it}, cost {nlp.cost.min().item():.6e}..{nlp.cost.max().item():.6e}, "
                  f"|c| {cmax.max().item():.2e}, rho {nlp.rho.max().item():.0f}")
        if bool((cmax < ctol).all()):
            break
        nlp.lam += nlp.rho[:, None, None] * nlp.c
        slow = (cmax > ctol) & ((cmax > 0.25 * c_prev) if c_prev is not None else torch.ones_like(cmax, dtype=torch.bool))
        nlp.rho.copy_(torch.where(slow, (nlp.rho * 3).clamp_max(rho_max), nlp.rho))
        c_prev = cmax
    return theta, {"outer": outer + 1, "iterations": total, "nfev": nlp.nfev, "c_max": cmax.cpu().numpy(),
                   "cost": nlp.cost.cpu().numpy()}


def solve(nlp, theta, ctol=1e-8, gtol=1e-10, ftol=1e-10, max_outer=30, max_inner=500, rho0=10., rho_max=1e6, m=20,
          window=10, ls_max=30, ticks_per_check=64, max_ticks=None, use_graph=True, min_solved=None, keep_history=False,
          verbose=False):
    """Device-resident solve: every tick = [d2dx_shoot_forward, d2dx_shoot_adjoint, d2dx_al_lbfgs_tick]; `ticks_per_check`
    ticks are captured in one CUDA graph and replayed until no problem is iterating (one host read per replay).
    Problems advance independently (own line search, multipliers, termination); `min_solved` stops the replays as soon as
    that many problems have converged (multi-start: the stragglers are usually the infeasible starts).  Returns theta (P, n) at the solutions
    and an info dict; `nlp.free_vectors()` then gives the planner-layout solutions."""
    from . import _lib
    e, P, n, n_con = nlp.eng, nlp.P, nlp.n, nlp.n_con
    o = _lib.LbfgsOptions(m=m, max_inner=max_inner, max_outer=max_outer, ls_max=ls_max, window=window, gtol=gtol, ftol=ftol,
                          ctol=ctol, rho0=rho0, rho_max=rho_max, keep_history=int(keep_history))
    off = e.lbfgs_layout(P, n, n_con, o)
    state = e.empty(off[0])
    n_running = e.zeros(1, dtype=torch.int32)
    xt = theta.reshape(P, n).clone()
    e.lbfgs_init(P, n, n_con, o, state, nlp.lam, nlp.rho)

    def tick():
        nlp.launch(xt)
        e.al_lbfgs_tick(P, n, n_con, o, state, xt, nlp.lagr_ac, nlp.cost_ac, nlp.n_ac, nlp.grad, nlp.c, nlp.lam, nlp.rho, n_running)

    def ticks():
        for _ in range(ticks_per_check):
            tick()
    tick()                                                                       # warm-up outside the capture (lazy module load)
    torch.cuda.synchronize(e.device)
    replay = ticks
    if use_graph:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=torch.cuda.Stream(device=e.device)):
            ticks()
        replay = g.replay
    max_ticks = max_ticks or int(1.5 * max_outer * max_inner)
    done_ticks = 1
    meta = state[off[5]:off[5] + P * off[7] // 2].view(torch.int32).view(P, off[7])
    while done_ticks < max_ticks:
        replay()
        done_ticks += ticks_per_check
        running = int(n_running.item())
        if verbose:
            print(f"ticks {done_ticks}: {running} of {P} problems iterating")
        if running == 0 or (min_solved is not None and int((meta[:, 0] == 2).sum().item()) >= min_solved):
            break
    theta = state[off[1]:off[1] + P * n].view(P, n).clone()
    nlp.launch(theta)                                                            # buffers (states, physical inputs, c) at the solutions
    meta_h = meta.cpu().numpy()
    return theta, {"outer": int(meta_h[:, 6].max()), "iterations": int(meta_h[:, 10].max()), "nfev": int(meta_h[:, 5].max()),
                   "ticks": done_ticks, "flag": meta_h[:, 0].copy(), "iterations_each": meta_h[:, 10].copy(),
                   "c_max": nlp.c.abs().amax(dim=(1, 2)).cpu().numpy(), "cost": nlp.cost.cpu().numpy()}


def solve_ddp(nlp, phi0, v0, ctol=1e-8, retries=4, opts=None, verbose=False, min_solved=0):
    """Second-order solve of P problems: control-limited DDP on the collocation grid.  One aircraft per problem: d2dx_ddp_solve
    (one GPU thread per problem); several (n_ac <= 10): d2dx_ddp_multi_solve (the aircraft coupled through the collision term,
    one warp per problem).  phi0, v0: host (P, n_ac, N) start inputs or anything that broadcasts to it ((P, N) when n_ac = 1).
    Problems that end unsolved climb a retry ladder.  One aircraft: the same start with the other regularisation
    (eigenvalue-modified Newton: better on tightly saturated problems, plain Levenberg-Marquardt: better elsewhere), then the
    mirrored bank profile (the other turn direction -- the usual reason for an infeasible local minimum) with either, and last
    the original start with four times the sweep budget (the clipped exponential obstacles of exp_4 converge in ~500 sweeps,
    beyond the default 400).  Several aircraft (plain regularisation only): every bank profile mirrored, then the original start
    with four times the sweep budget.  `min_solved=k` (multi-start of ONE problem): the launch ends as soon as k starts
    have converged and the ladder is only climbed when none has.  Returns (frees (P, num_free) in the planner layout, info);
    with several aircraft info["lam"] (P, 3, n_ac) holds the terminal multipliers of each returned solution."""
    e, P, N, n = nlp.eng, nlp.P, nlp.N, nlp.n_ac
    kw = dict(ctol=ctol, min_solved=int(min_solved)) if opts is None else {f: getattr(opts, f) for f, _ in opts._fields_}
    lo, hi, vlo, vhi = nlp.bounds

    def starts(a):
        a = np.asarray(a, np.float64)
        return np.broadcast_to(a.reshape(-1, 1, N) if n == 1 and a.ndim else a, (P, n, N))
    u0 = np.clip(np.stack([starts(phi0), starts(v0)], 1), np.array([lo, vlo])[None, :, None, None], np.array([hi, vhi])[None, :, None, None])
    u = e.to_device(np.ascontiguousarray(u0))
    xs, info, lam = e.empty(P, 3, n, N), e.zeros(P, 8), e.zeros(P, 3, n)
    p0, p1 = nlp.p0.contiguous(), nlp.p1.contiguous()

    def run(cnt, p0_, p1_, u_, xs_, info_, lam_, o):
        if n == 1:
            e.ddp_solve(nlp.c_prob, cnt, nlp.bounds, nlp.state_box, p0_, p1_, u_, xs_, info_, o)
        else:
            e.ddp_multi_solve(nlp.c_prob, cnt, nlp.bounds, nlp.state_box, p0_, p1_, u_, xs_, info_, lam_, o)
    mode0 = int(kw.get("reg_mode", 0))
    run(P, p0, p1, u, xs, info, lam, e.ddp_options(**{**kw, "reg_mode": mode0}))
    ih = info.cpu().numpy()
    total_its = ih[:, 1].copy()
    base = e.ddp_options(**kw)
    if n == 1:
        ladder = [(1.0, 1 - mode0, 1), (-1.0, mode0, 1), (-1.0, 1 - mode0, 1), (1.0, mode0, 4)][:retries]
    else:
        ladder = [(-1.0, mode0, 1), (1.0, mode0, 4)][:retries]
    for r, (sign, mode, scale) in enumerate(ladder):
        bad = np.nonzero(ih[:, 0] != 2)[0]
        if len(bad) == 0 or (min_solved > 0 and len(bad) < P):
            break
        seed = u0[bad].copy()
        seed[:, 0] *= sign
        if sign < 0 and not np.any(seed[:, 0]):
            seed[:, 0] = 0.3 * hi
        idx = torch.from_numpy(bad).to(e.device)
        ub, xb, ib, lb = e.to_device(np.ascontiguousarray(seed)), e.empty(len(bad), 3, n, N), e.zeros(len(bad), 8), e.zeros(len(bad), 3, n)
        run(len(bad), p0[idx].contiguous(), p1[idx].contiguous(), ub, xb, ib, lb,
            e.ddp_options(**{**kw, "reg_mode": mode, "max_iter": int(base.max_iter) * scale, "max_outer": int(base.max_outer) * (2 if scale > 1 else 1)}))
        ibh = ib.cpu().numpy()
        better = torch.from_numpy((ibh[:, 0] == 2) | (ibh[:, 4] < ih[bad, 4])).to(e.device)
        sel = idx[better]
        u[sel], xs[sel], info[sel], lam[sel] = ub[better], xb[better], ib[better], lb[better]
        total_its[bad] += ibh[:, 1]
        ih = info.cpu().numpy()
        if verbose:
            print(f"retry {r} (bank sign {sign:+.0f}, regularisation {mode}, sweep budget x{scale}): {len(bad)} problems re-seeded, {(ibh[:, 0] == 2).sum()} of them solved")
    frees = torch.cat([xs.permute(0, 2, 1, 3).reshape(P, 3 * n * N), u.reshape(P, 2 * n * N)], dim=1).cpu().numpy()
    nlp.xs.copy_(xs); nlp.u_phys.copy_(u)
    out = {"flag": ih[:, 0].astype(int), "iterations_each": total_its.astype(int), "iterations": int(total_its.max()), "outer": int(ih[:, 2].max()),
           "cost": ih[:, 3].copy(), "c_max": ih[:, 4].copy(), "method": "ddp"}
    if n > 1:
        out["lam"], out["rho"] = lam.cpu().numpy(), ih[:, 7].copy()
    return frees, out
