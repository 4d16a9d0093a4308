"""The coupled multi-aircraft second-order solver (csrc/d2dx_ddp_multi.cuh) on the CPU: csrc/host_check.cu compiles the code of the
GPU warp for the host.  Checked: the projected-Newton box QP of a node, the reduction to the single-aircraft solver for one
aircraft, the decoupling of aircraft without a coupling term, and the head-on pair of exp_5 with the collision cost (feasible,
separated, first-order optimal for the returned multipliers)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import ddp_host as dh  # noqa: E402
from oracle import d2d_oracle as orc  # noqa: E402

B30 = (-np.deg2rad(30.), np.deg2rad(30.), 9., 14.)
B40 = (-np.deg2rad(40.), np.deg2rad(40.), 9., 15.)


def _box_qp2(H, g, lo, hi):
    """exact minimiser of a 2-variable box QP by the active-set enumeration of ddp_box_qp2 (d2dx_ddp.cuh)"""
    best = None
    for s0 in (None, lo[0], hi[0]):
        for s1 in (None, lo[1], hi[1]):
            x = np.array([0. if s0 is None else s0, 0. if s1 is None else s1])
            free = [s0 is None, s1 is None]
            if all(free):
                x = np.linalg.solve(H, -g)
            elif free[0]:
                x[0] = -(g[0] + H[0, 1] * x[1]) / H[0, 0]
            elif free[1]:
                x[1] = -(g[1] + H[0, 1] * x[0]) / H[1, 1]
            if np.any(x < lo - 1e-12) or np.any(x > hi + 1e-12):
                continue
            f = 0.5 * x @ H @ x + g @ x
            if best is None or f < best[0]:
                best = (f, x)
    return best[1]


@pytest.mark.parametrize("n", [2, 5, 12, 20])
def test_box_qp_kkt(n):
    """random SPD problems with bounds that cut through the unconstrained minimiser: x in the box, the KKT sign conditions,
    and for n = 2 the exact 2-variable minimiser"""
    rng = np.random.default_rng(n)
    for trial in range(20):
        A = rng.normal(size=(n, n))
        H = A @ A.T + 0.05 * np.eye(n)
        g = rng.normal(size=n) * 3.
        lo, hi = -rng.uniform(0.05, 1., n), rng.uniform(0.05, 1., n)
        x, free = dh.box_qp(H, g, lo, hi)
        gr = g + H @ x
        scale = np.abs(g).max() + np.abs(H @ x).max()
        assert np.all(x >= lo) and np.all(x <= hi)
        assert np.all(gr[x == lo] >= 0.) and np.all(gr[x == hi] <= 0.)
        assert np.all(np.abs(gr[free]) < 1e-10 * scale)
        assert np.all((x == lo) | (x == hi) | free)
        if n == 2:
            np.testing.assert_allclose(x, _box_qp2(H, g, lo, hi), rtol=0, atol=1e-12)
        if trial == 0 and n > 2:
            assert 0 < free.sum() < n                         # mixed active bounds


def test_one_aircraft_reduces_to_the_single_solver():
    """exp_0 (N = 101) through the coupled solver: the optimum 0.752912, and the single-aircraft solver's answer from the same start"""
    N, h = 101, 0.1
    prob = dh.colloc_problem(1, N, h, vsp=12., kvel=1.)
    u, xs, info = dh.solve_multi(prob, B30, [[0.], [0.], [0.]], [[0.], [30.], [np.pi]], 0.1, 12.)
    u1, xs1, info1 = dh.solve(N, h, (0., 0.), 12., 1., 0., B30, (0., 0., 0.), (0., 30., np.pi), 0.1, 12.)
    assert info["flag"] == 2 and info1["flag"] == 2
    assert abs(info["cost"] - 0.752912) < 2e-6
    assert abs(info["cost"] - info1["cost"]) < 1e-9 * info1["cost"]
    np.testing.assert_allclose(u[:, 0], u1, atol=1e-7)


def test_decoupled_aircraft_solve_independently():
    """two aircraft, different boundary conditions, no coupling term: the sum of the two single-aircraft solves (in_div = 2).  Tight
    tolerances on both sides, so that the two stopping points agree; the inputs are only weakly determined where the bank cost is
    the only curvature, hence 5e-6 on them."""
    N, h = 101, 0.1
    p0 = np.array([[0., 20.], [0., -10.], [0., 0.5]])
    p1 = np.array([[0., 130.], [30., 5.], [np.pi, 0.2]])
    opts = dict(rel_tol=1e-14, ctol=1e-11, abs_tol=0.)
    prob = dh.colloc_problem(2, N, h, vsp=12., kvel=1., kbank=0.5)
    u, xs, info = dh.solve_multi(prob, B30, p0, p1, 0.1, 12., opts=dh.default_options(**opts))
    assert info["flag"] == 2
    total = 0.
    for a in range(2):
        ua, _, ia = dh.solve(N, h, (0., 0.), 12., 1., 0.5, B30, p0[:, a].copy(), p1[:, a].copy(), 0.1, 12., in_div=2,
                             opts=dh.default_options(**opts))
        assert ia["flag"] == 2
        total += ia["cost"]
        np.testing.assert_allclose(u[:, a], ua, atol=5e-6)
    assert abs(info["cost"] - total) < 1e-9 * total


def _exp5(case):
    """exp_5 (2 aircraft face to face, 07_multioptyplan.py:345-366) on a 10 Hz grid; case 1 adds the collision cost (rcol 10)"""
    N, h = int(4.2 * 10) + 1, 0.1
    spec = dict(vsp=12., kvel=70., kbank=1., obj_scale=1.)
    if case == 1:
        spec.update(kcol=10., rcol=10., kcol_k=2., pairs="01")
    prob = dh.colloc_problem(2, N, h, vsp=12., kvel=70., kbank=1., kcol=spec.get("kcol", 0.), rcol=10., kcol_k=2.)
    p0 = np.array([[0., 50.], [0., 0.], [0., np.pi]])
    p1 = np.array([[50., 0.], [0., 0.], [0., np.pi]])
    return prob, spec, p0, p1, N, h


def _separation(xs):
    return np.hypot(xs[0, 0] - xs[0, 1], xs[1, 0] - xs[1, 1]).min()


def test_collision_coupling_exp5():
    """exp_5 case 1: solved, feasible under the reference's constraints, inputs in the bounds, the pair kept apart (case 0, without
    the collision term, flies through), and a first-order point of the augmented Lagrangian for the returned multipliers"""
    prob, spec, p0, p1, N, h = _exp5(1)
    u, xs, info = dh.solve_multi(prob, B40, p0, p1, [[0.05], [-0.05]], 12.)
    assert info["flag"] == 2
    free = np.concatenate([np.concatenate([xs[0, a], xs[1, a], xs[2, a]]) for a in range(2)] + [u[0, 0], u[0, 1], u[1, 0], u[1, 1]])
    inst = [(3 * a + k, 0, p0[k, a]) for a in range(2) for k in range(3)] + [(3 * a + k, N - 1, p1[k, a]) for a in range(2) for k in range(3)]
    assert np.abs(orc.colloc_residual(free, N, 2, h, (0., 0.), inst)).max() < 1e-7
    assert u[0].min() >= B40[0] and u[0].max() <= B40[1] and u[1].min() >= B40[2] and u[1].max() <= B40[3]
    cost_o, _ = orc.cost_and_grad(free, N, 2, spec, multi=True)
    assert abs(cost_o - info["cost"]) < 1e-10 * abs(cost_o)
    assert _separation(xs) > 4.
    prob0, _, _, _, _, _ = _exp5(0)
    u0, xs0, info0 = dh.solve_multi(prob0, B40, p0, p1, [[0.05], [-0.05]], 12.)
    assert info0["flag"] == 2 and _separation(xs0) < 1.

    lam, rho = info["lam"], info["rho"]
    L = lambda ph, v: orc.shoot_lagrangian(ph, v, p0, p1, h, (0., 0.), spec, lam, rho, multi=True)[2]
    g = np.zeros_like(u)
    for j in range(2):
        eps = 1e-6 if j == 0 else 1e-5
        for a in range(2):
            for i in range(N):
                up, um = u.copy(), u.copy()
                up[j, a, i] += eps; um[j, a, i] -= eps
                g[j, a, i] = (L(up[0], up[1]) - L(um[0], um[1])) / (2 * eps)
    lo, hi = np.array([B40[0], B40[2]])[:, None, None], np.array([B40[1], B40[3]])[:, None, None]
    proj = np.where(u <= lo, np.minimum(g, 0.), np.where(u >= hi, np.maximum(g, 0.), g))
    assert np.abs(proj).max() < 1e-7, np.abs(proj).max()             # measured 2.9e-9 (central differences, steps 1e-6 / 1e-5)
