"""Coupled multi-aircraft second-order solve on the GPU (d2dx_ddp_multi_solve: one warp per problem) through the engine, the
planner front end and the mission: the kernel against the host build of the same solver, upstream's multi-aircraft experiments,
a population of four-aircraft problems in one launch, the argument checks and phase 2 of the mission."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "scripts"))

pytestmark = pytest.mark.gpu

X1_F = ((0, 40, 0, 0, 12), (25, 40, 0, 0, 12), (25, -40, 0, 0, 12), (0, -40, 0, 0, 12))      # mission.full_sim's phase-2 boundary states
X2_F = ((75, 40, 0, 0, 12), (100, 40, 0, 0, 12), (100, -40, 0, 0, 12), (75, -40, 0, 0, 12))


def _planner(exp, case=0):
    from d2d_b200 import planner as pl
    exp.set_case(case)
    p = pl.MultiPlanner(exp)
    p.configure(tol=exp.tol, max_iter=exp.max_iter)
    return p


def _trap4():
    from d2d_b200 import mission
    s = mission.trap_4
    s.t1, s.p0s, s.p1s = 6, X1_F, X2_F
    return s


def _separation(p):
    n = p.acs.nb_aicraft
    return min([np.hypot(p.sol_x[a] - p.sol_x[b], p.sol_y[a] - p.sol_y[b]).min() for a in range(n) for b in range(a)] or [np.inf])


@pytest.mark.parametrize("name", ["exp_5", "gvf_trial_3ac"])
def test_kernel_matches_host_build(name):
    """same problem, same start: the warp-cooperative kernel and the serial host sweeps agree (different summation orders)"""
    import ddp_host as dh
    from d2d_b200 import multiopty_scenarios as S
    exp = getattr(S, name)
    p = _planner(exp, 1 if name == "exp_5" else 0)
    n, N = p.acs.nb_aicraft, p.num_nodes
    guess = p.get_initial_guess("tri")
    phi = np.stack([guess[sl] for sl in p._phi_slices()])
    v = np.stack([guess[sl] for sl in p._v_slices()])
    p0, p1 = p._boundary_states()
    box = (*exp.x_constraint, *exp.y_constraint, 1000.) if exp.x_constraint is not None else None
    bounds = (*exp.phi_constraint, *exp.v_constraint)
    u_h, xs_h, info_h = dh.solve_multi(p.prob.c, bounds, p0, p1, np.clip(phi, *exp.phi_constraint), np.clip(v, *exp.v_constraint), box=box)
    e = p.prob.eng
    u = e.to_device(np.ascontiguousarray(np.stack([np.clip(phi, *exp.phi_constraint), np.clip(v, *exp.v_constraint)])[None]))
    xs, info, lam = e.empty(1, 3, n, N), e.zeros(1, 8), e.zeros(1, 3, n)
    e.ddp_multi_solve(p.prob.c, 1, bounds, box, e.to_device(p0[None].copy()), e.to_device(p1[None].copy()), u, xs, info, lam)
    ih = info.cpu().numpy()[0]
    S.exp_5.set_case(0)
    assert ih[0] == info_h["flag"] == 2
    assert abs(ih[3] - info_h["cost"]) < 1e-9 * abs(info_h["cost"])
    np.testing.assert_allclose(u.cpu().numpy()[0], u_h, rtol=0, atol=1e-7)
    np.testing.assert_allclose(lam.cpu().numpy()[0], info_h["lam"], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("name,case", [("exp_1_0", 0), ("exp_2", 0), ("exp_4", 0), ("exp_5", 0), ("exp_5", 1), ("exp_5_1", 0),
                                       ("gvf_trial_3ac", 0), ("trap_4", 0)])
def test_upstream_experiments_with_ddp(name, case):
    """07_multioptyplan.py's experiments and the mission's phase-2 problem through MultiPlanner.run(method="ddp")"""
    from d2d_b200 import multiopty_scenarios as S
    exp = _trap4() if name == "trap_4" else getattr(S, name)
    p = _planner(exp, case)
    info = p.run(initial_guess=p.get_initial_guess("tri"), n_starts=4, method="ddp")
    sep = _separation(p)
    S.exp_5.set_case(0)
    assert info["method"] == "ddp" and info["feasible"]
    assert np.abs(p.prob.con(p.solution)).max() < 10 * exp.tol
    c = p.prob.obj(p.solution)
    if exp.x_constraint is not None:                              # the reported cost includes the soft state box (weight 1000)
        ex = [np.maximum(np.asarray(s) - hi, 0.) + np.minimum(np.asarray(s) - lo, 0.) for sl, (lo, hi) in
              ((p.sol_x, exp.x_constraint), (p.sol_y, exp.y_constraint)) for s in sl]
        c += 1000. * exp.obj_scale / p.num_nodes * sum(np.sum(e * e) for e in ex)
    assert abs(c - info["cost"][info["best"]]) <= 1e-10 * abs(c)
    for a in range(p.acs.nb_aicraft):
        assert p.sol_phi[a].min() >= exp.phi_constraint[0] and p.sol_phi[a].max() <= exp.phi_constraint[1]
        assert p.sol_v[a].min() >= exp.v_constraint[0] and p.sol_v[a].max() <= exp.v_constraint[1]
        np.testing.assert_allclose([p.sol_x[a][-1], p.sol_y[a][-1], p.sol_psi[a][-1]], exp.p1s[a][:3], atol=1e-4)
    if name == "exp_5":
        assert (sep < 1.0) if case == 0 else (sep > 4.0)


def test_population_of_four_aircraft_problems():
    """1024 trap_4 problems with random targets: at least 97 % solved by the first launch (98.1 % measured on a B200), at least 99 %
    after the retry ladder, sampled solutions feasible"""
    from d2d_b200 import shooting
    from d2d_b200.collocation import CollocationProblem
    s = _trap4()
    p = _planner(s)
    n, N, P = 4, p.num_nodes, 1024
    rng = np.random.default_rng(7)
    p0, p1 = p._boundary_states()
    p1s = p1[None] + np.stack([rng.uniform(-8, 8, (P, n)), rng.uniform(-8, 8, (P, n)), rng.uniform(-0.3, 0.3, (P, n))], 1)
    nlp = shooting.ShootingNLP(p.prob, p0, p1s, s.phi_constraint, s.v_constraint, P=P, state_box=(-150, 150, -150, 150, 1000.))
    _, info1 = shooting.solve_ddp(nlp, 0., 12., ctol=1e-8, retries=0)
    frees, info = shooting.solve_ddp(nlp, 0., 12., ctol=1e-8)
    assert (info1["flag"] == 2).mean() >= 0.97 and (info["flag"] == 2).mean() >= 0.99, ((info1["flag"] == 2).mean(), (info["flag"] == 2).mean())
    for k in np.nonzero(info["flag"] == 2)[0][:3]:
        inst = [(3 * a + j, 0, p0[j, a]) for a in range(n) for j in range(3)] + [(3 * a + j, N - 1, p1s[k, j, a]) for a in range(n) for j in range(3)]
        q = CollocationProblem(n, N, p.time_step, inst=inst, cost=s.cost.spec(), multi=True)
        assert np.abs(q.con(frees[k])).max() < 1e-7


def test_abi_refusals():
    """n_ac = 11 and the eigenvalue regularisation with several aircraft are refused (D2DX_EINVAL)"""
    from d2d_b200 import _lib
    from d2d_b200.collocation import CollocationProblem, CostSpec
    from d2d_b200.engine import get_engine
    e = get_engine()
    for n_ac, mode in ((11, 0), (2, 1)):
        prob = CollocationProblem(n_ac, 21, 0.1, cost=CostSpec(vsp=12., kvel=1.))
        u, xs, info = e.zeros(1, 2, n_ac, 21) + 12., e.zeros(1, 3, n_ac, 21), e.zeros(1, 8)
        p0 = e.zeros(1, 3, n_ac)
        with pytest.raises(_lib.D2dxError, match="error 1:"):
            e.ddp_multi_solve(prob.c, 1, (-0.5, 0.5, 9., 15.), None, p0, p0, u, xs, info, None, e.ddp_options(reg_mode=mode))


def test_mission_phase2_with_ddp():
    """mission.full_sim(method="ddp"): all three phases run and phase 2's plan is feasible and ends at X2_f"""
    import pandas as pd
    from d2d_b200 import mission
    g = np.load(os.path.join(HERE, "golden", "tracker.npz"))
    cols = {"time": g["inf/time"]}
    for i in range(4):
        cols[f"x_{i + 1}"], cols[f"y_{i + 1}"], cols[f"psi_{i + 1}"] = g["inf/x_ref"][:, i], g["inf/y_ref"][:, i], 0 * g["inf/time"]
    out = mission.full_sim(pd.DataFrame(cols), t_sim_end=150, method="ddp")
    p = out["planner"]
    assert p.info["method"] == "ddp" and p.info["feasible"]
    assert np.abs(p.prob.con(p.solution)).max() < 1e-4
    for a in range(4):
        np.testing.assert_allclose([p.sol_x[a][-1], p.sol_y[a][-1]], X2_F[a][:2], atol=1e-4)
    assert out["laps"] >= 1 and np.isfinite(out["X"]).all()
