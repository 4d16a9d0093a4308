"""Collocation kernel (through the C ABI) vs golden vectors derived from the reference's sympy EoM and cost
classes.  Tolerance: north_star's 1e-10 relative on residuals and Jacobian entries."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-10


def _inst(g, tag):
    return [(int(k), int(n), v) for (k, n, v) in g[f"{tag}/inst"]]


@pytest.mark.parametrize("tag", ["c3", "c3w"])
def test_c3_single_aircraft(golden, tag):
    from d2d_b200.collocation import CollocationProblem, CostSpec
    g = golden["colloc"]
    N, h = 1001, 0.02
    free, inst = g["c3/free"], _inst(g, "c3")
    for layout in ("compact", "dense"):
        prob = CollocationProblem(1, N, h, wind=g[f"{tag}/wind"], inst=inst, cost=CostSpec(vsp=12., kvel=1.), layout=layout)
        assert prob.num_free == 5 * N and prob.num_constraints == 3 * (N - 1) + 6
        res, jac, cost, grad = prob.evaluate(free)
        np.testing.assert_allclose(res, g[f"{tag}/residual"], rtol=RTOL, atol=1e-11)
        rows, cols = prob.jacobianstructure()
        if layout == "dense":
            np.testing.assert_allclose(jac[:-6], g[f"{tag}/jac_dense"].reshape(-1), rtol=RTOL, atol=0)
            np.testing.assert_array_equal(rows[:-6], g["c3/rows"].reshape(-1))
            np.testing.assert_array_equal(cols[:-6], g["c3/cols"].reshape(-1))
        else:
            D = np.zeros((3 * (N - 1) + 6, 5 * N)); D[rows, cols] = jac
            D2 = np.zeros_like(D); np.add.at(D2, (g["c3/rows"].reshape(-1), g["c3/cols"].reshape(-1)), g[f"{tag}/jac_dense"].reshape(-1))
            np.testing.assert_allclose(D[:-6], D2[:-6], rtol=RTOL, atol=0)
        np.testing.assert_array_equal(jac[-6:], np.ones(6))
        assert list(rows[-6:]) == list(range(3 * (N - 1), 3 * (N - 1) + 6))
        assert list(cols[-6:]) == [0, N, 2 * N, N - 1, 2 * N - 1, 3 * N - 1]
        np.testing.assert_allclose(cost, g["cost1/airvel/noisy/cost"], rtol=RTOL)
        np.testing.assert_allclose(grad, g["cost1/airvel/noisy/grad"], rtol=RTOL, atol=1e-300)
    # the cached IPOPT solution of the reference satisfies the constraints
    prob = CollocationProblem(1, N, h, inst=inst)
    assert np.abs(prob.con(g["c3/sol"])).max() < 1e-6


SINGLE = {
    "airvel": dict(vsp=12., kvel=1.), "bank": dict(kbank=1.), "input": dict(vsp=12., kvel=1., kbank=50.),
    "obs0": dict(kobs=1., obstacles=[(30, 0, 15.)], obs_kind=0), "obs1": dict(kobs=1., obstacles=[(5, 15, 10.)], obs_kind=1),
    "composit": dict(vsp=15., kvel=.5, kbank=1., kobs=.5, obstacles=[(5, 15, 10)], obs_kind=0),
    "composit1": dict(vsp=12., kvel=.7, kbank=1.5, kobs=2., obstacles=[(5, 15, 10), (-3., 20., 6.)], obs_kind=1),
}


@pytest.mark.parametrize("name", sorted(SINGLE))
def test_single_aircraft_costs(golden, name):
    from d2d_b200.collocation import CollocationProblem, CostSpec
    g = golden["colloc"]
    prob = CollocationProblem(1, 1001, 0.02, cost=CostSpec(**SINGLE[name]))
    for tag, free in (("sol", g["c3/sol"]), ("noisy", g["c3/free"])):
        np.testing.assert_allclose(prob.obj(free), g[f"cost1/{name}/{tag}/cost"], rtol=RTOL)
        np.testing.assert_allclose(prob.obj_grad(free), g[f"cost1/{name}/{tag}/grad"], rtol=RTOL, atol=1e-300)


MULTI = {
    "input": dict(vsp=12., kvel=70., kbank=1.), "airvel": dict(vsp=12., kvel=1.), "bank": dict(kbank=1.),
    "obs0": dict(kobs=1., obstacles=[(60., 5., 12.)], obs_kind=0), "obs1": dict(kobs=1., obstacles=[(60., 5., 12.)], obs_kind=1),
    "collision": dict(kcol=1., rcol=10.),
    "composit": dict(vsp=12., kvel=70., kbank=1., kobs=0.5, kcol=10., obstacles=[(60., 5., 12.), (-20., 30., 8.)], obs_kind=1, rcol=10.),
    "composit_nocol": dict(vsp=12., kvel=2., kbank=1.),
}


@pytest.mark.parametrize("tag,n_ac,N,h", [("m3", 3, 20, 0.1), ("c4", 16, 500, 0.02)])
def test_multi_aircraft(golden, tag, n_ac, N, h):
    from d2d_b200.collocation import CollocationProblem, CostSpec
    g = golden["colloc"]
    free, inst = g[f"{tag}/free"], _inst(g, tag)
    prob = CollocationProblem(n_ac, N, h, wind=g[f"{tag}/wind"], inst=inst, cost=CostSpec(**MULTI["composit"]))
    res, jac, cost, grad = prob.evaluate(free)
    np.testing.assert_allclose(res, g[f"{tag}/residual"], rtol=RTOL, atol=1e-10)
    rows, cols = prob.jacobianstructure()
    n, q = 3 * n_ac, 2 * n_ac
    D = {}
    # golden non-zeros: (N-1, nnz/node) at (eq, dense col) -> scatter both into dicts keyed by (row, col)
    ee, cc = g[f"{tag}/nz_eq"], g[f"{tag}/nz_col"]
    i = np.arange(N - 1)
    ref = {}
    for k, (e, c) in enumerate(zip(ee, cc)):
        if c < n: col = c * N + i + 1
        elif c < 2 * n: col = (c - n) * N + i
        else: col = (n + (c - 2 * n)) * N + i + 1
        for ii in (0, 1, N - 2):
            ref[(e * (N - 1) + ii, int(col[ii]))] = g[f"{tag}/jac_nz"][ii, k]
    got = {(int(r), int(c)): v for r, c, v in zip(rows, cols, jac)}
    for key, v in ref.items():
        assert abs(got[key] - v) <= RTOL * abs(v), key
    # full compare through a dense scatter on the small case
    if tag == "m3":
        Dg = np.zeros((prob.num_constraints, prob.num_free)); Dg[rows, cols] = jac
        pd = CollocationProblem(n_ac, N, h, wind=g[f"{tag}/wind"], inst=inst, layout="dense")
        jd = pd.con_jac(free); rd, cd = pd.jacobianstructure()
        np.testing.assert_allclose(jd[:-len(inst)], g["m3/jac_dense"].reshape(-1), rtol=RTOL, atol=0)
        Dd = np.zeros_like(Dg); np.add.at(Dd, (rd, cd), jd)
        np.testing.assert_array_equal(Dg, Dd)
    np.testing.assert_allclose(cost, g[f"{tag}/cost/composit/cost"], rtol=RTOL)
    np.testing.assert_allclose(grad, g[f"{tag}/cost/composit/grad"], rtol=RTOL, atol=1e-14)
    for name, spec in MULTI.items():
        p2 = CollocationProblem(n_ac, N, h, cost=CostSpec(**spec))
        np.testing.assert_allclose(p2.obj(free), g[f"{tag}/cost/{name}/cost"], rtol=RTOL, err_msg=name)
        gr, ref_g = p2.obj_grad(free), g[f"{tag}/cost/{name}/grad"]
        if len(ref_g) != len(gr): gr = gr[::7]
        np.testing.assert_allclose(gr, ref_g, rtol=RTOL, atol=1e-14, err_msg=name)


def test_all_pairs_collision_and_batch_against_oracle():
    """All-pairs generalisation (SURVEY D11) and a batch of problems in one launch, vs the oracle."""
    from oracle import d2d_oracle as orc
    from d2d_b200.collocation import CollocationProblem, CostSpec
    rng = np.random.default_rng(11)
    n_ac, N, h, n_prob = 7, 150, 0.05, 9
    free = rng.normal(0, 8., (n_prob, 5 * n_ac * N)); free[:, 4 * n_ac * N:] = 12 + rng.normal(0, 1, (n_prob, n_ac * N))
    for exact in (False, True):
        spec = dict(vsp=12., kvel=3., kbank=2., kcol=10., rcol=10., pairs="all", exact_grad=exact, kobs=1.5, obstacles=[(1., 2., 6.)], obs_kind=1)
        prob = CollocationProblem(n_ac, N, h, wind=(1., 2.), cost=CostSpec(vsp=12., kvel=3., kbank=2., kcol=10., rcol=10., all_pairs=True,
                                  exact_grad=exact, kobs=1.5, obstacles=[(1., 2., 6.)], obs_kind=1))
        res, jac, cost, grad = prob.evaluate(free)
        for p in range(n_prob):
            np.testing.assert_allclose(res[p], orc.colloc_residual(free[p], N, n_ac, h, (1., 2.), []), rtol=RTOL, atol=1e-10)
            np.testing.assert_allclose(jac[p], orc.colloc_jac_compact(free[p], N, n_ac, h).reshape(-1), rtol=RTOL)
            co, go = orc.cost_and_grad(free[p], N, n_ac, spec, multi=True)
            np.testing.assert_allclose(cost[p], co, rtol=RTOL)
            np.testing.assert_allclose(grad[p], go, rtol=RTOL, atol=1e-13)
    rows, cols = prob.jacobianstructure()
    ro, co_ = orc.colloc_structure(N, n_ac, [], "compact")
    np.testing.assert_array_equal(rows, ro); np.testing.assert_array_equal(cols, co_)


def test_opty_name_sorted_input_order(golden):
    """12 aircraft: opty orders phi10, phi11 before phi2 (SURVEY D9); the permuted problem evaluated on the
    permuted free vector equals the numeric-order problem."""
    from d2d_b200.collocation import CollocationProblem, CostSpec
    names = [str(s) for s in golden["colloc"]["sorted_inputs_12"]]
    n_ac, N, h = 12, 40, 0.1
    rng = np.random.default_rng(2)
    free = rng.normal(0, 5., 5 * n_ac * N); free[4 * n_ac * N:] += 12
    cs = CostSpec(vsp=12., kvel=1., kbank=1.)
    a = CollocationProblem(n_ac, N, h, cost=cs)
    b = CollocationProblem(n_ac, N, h, cost=cs, input_order="opty")
    numeric = [f"phi{i}(t)" for i in range(n_ac)] + [f"v{i}(t)" for i in range(n_ac)]
    fp = free.copy()
    for k, nm in enumerate(names):
        src = numeric.index(nm)
        fp[(3 * n_ac + k) * N:(3 * n_ac + k + 1) * N] = free[(3 * n_ac + src) * N:(3 * n_ac + src + 1) * N]
    ra, ja, ca, ga = a.evaluate(free)
    rb, jb, cb, gb = b.evaluate(fp)
    np.testing.assert_array_equal(ra, rb); np.testing.assert_array_equal(ja, jb); assert ca == cb
    for k, nm in enumerate(names):
        src = numeric.index(nm)
        np.testing.assert_array_equal(gb[(3 * n_ac + k) * N:(3 * n_ac + k + 1) * N], ga[(3 * n_ac + src) * N:(3 * n_ac + src + 1) * N])
    # opty-dense layout under the same permutation (two problems in one launch: structural zeros laid down once per problem)
    d = CollocationProblem(n_ac, N, h, cost=cs, input_order="opty", layout="dense")
    jd = d.con_jac(np.stack([fp, fp]))
    rd, cd = d.jacobianstructure()
    rc, cc = b.jacobianstructure()
    A = np.zeros((b.num_constraints, b.num_free)); A[rc, cc] = jb
    for q in range(2):
        Bm = np.zeros_like(A); np.add.at(Bm, (rd, cd), jd[q])
        np.testing.assert_array_equal(A, Bm)
    assert jd.shape[1] == (N - 1) * 3 * n_ac * 8 * n_ac and np.count_nonzero(jd[0]) <= 12 * n_ac * (N - 1)


def test_planner_front_ends_and_cost_classes(golden):
    """The mirrored Planner / cost classes used the way the reference scripts use them (06_optyplan.py:177-204,
    test/test_objective.py): known-answer costs of SURVEY appendix C, instance constraints, triangle guess."""
    from d2d_b200 import multiopty_utils as d2mou, opty_utils as d2ou, planner
    g = golden["colloc"]

    class exp(planner.exp_0):
        t1, hz = 20., 50.
    p = planner.Planner(exp)
    assert p.num_nodes == 1001 and p.prob.num_free == 5005 and p.prob.num_constraints == 3006
    sol = g["c3/sol"]
    assert abs(p.prob.obj(sol) - 8.089644746010487e-08) < 1e-18
    assert np.abs(p.prob.con(sol)).max() < 1e-6                       # cached IPOPT solution is feasible
    known = {"bank": (d2ou.CostBank(), 0.09602478183335866), "input": (d2ou.CostInput(12., 1., 50.), 4.801239172564381),
             "obs0": (d2ou.CostObstacle((30, 0), 15., kind=0), 106.87281760768758),
             "obs1": (d2ou.CostObstacle((5, 15), 10., kind=1), 5.801877126038269e-06),
             "composit": (d2ou.CostComposit(((5, 15, 10),), vsp=15., kobs=.5, kvel=.5, kbank=1.), 4.596177031308985)}
    for name, (c, val) in known.items():
        np.testing.assert_allclose(c.cost(sol, p), val, rtol=1e-10, err_msg=name)
        np.testing.assert_allclose(c.cost_grad(sol, p), g[f"cost1/{name}/sol/grad"], rtol=1e-10, atol=1e-300, err_msg=name)
    guess = p.get_initial_guess("tri")
    assert guess.shape == (5005,) and np.isfinite(p.prob.obj(guess))

    class mscen:
        t0, t1, hz = 0., 1.9, 10.
        p0s = tuple(tuple(v) for v in g["m3/p0s"]); p1s = tuple(tuple(v) for v in g["m3/p1s"])
        wind = d2ou.WindField([0.5, -1.0]); vref = 12.; obj_scale = 1.
        cost = d2mou.CostComposit(kvel=70., kbank=1., kobs=0.5, kcol=10., vsp=12., obss=((60., 5., 12.), (-20., 30., 8.)), obs_kind=1, rcol=10.)
    mp = planner.MultiPlanner(mscen)
    assert mp.num_nodes == 20 and mp.acs.nb_aicraft == 3
    free = g["m3/free"]
    np.testing.assert_allclose(mp.prob.con(free), g["m3/residual"], rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(mp.prob.obj(free), g["m3/cost/composit/cost"], rtol=1e-10)
    np.testing.assert_allclose(mscen.cost.cost_grad(free, mp), g["m3/cost/composit/grad"], rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(d2mou.CostCollision(r=10.).cost(free, mp), g["m3/cost/collision/cost"], rtol=1e-10)
    with pytest.raises(ValueError):                             # this scenario carries no input bounds
        mp.run()
    mscen.phi_constraint, mscen.v_constraint = (-0.6, 0.6), (9., 15.)
    mp = planner.MultiPlanner(mscen)
    info = mp.run()                                             # solved on the engine (tests/test_gpu_shooting.py covers the solver)
    assert np.abs(mp.prob.con(mp.solution)[:3 * 3 * 19]).max() < 1e-9 and info["outer"] >= 1


def test_cuda_graph_replay_matches_direct_evaluation(golden):
    import torch
    from d2d_b200 import get_engine
    from d2d_b200.collocation import CollocationProblem, CostSpec
    g = golden["colloc"]
    eng = get_engine()
    prob = CollocationProblem(1, 1001, 0.02, inst=_inst(g, "c3"), cost=CostSpec(vsp=12., kvel=1.))
    free = eng.to_device(g["c3/sol"][None].copy())
    replay, out = prob.graph(free)
    free.copy_(eng.to_device(g["c3/free"][None]))             # new iterate written in place, then one replay
    replay(); torch.cuda.synchronize()
    np.testing.assert_allclose(out["res"].cpu().numpy()[0], g["c3/residual"], rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(out["cost"].cpu().numpy()[0], g["cost1/airvel/noisy/cost"], rtol=RTOL)


def test_reference_csv_solutions_are_feasible_and_round_trip(golden, tmp_path):
    """The 4-aircraft planner outputs shipped with the reference (carried in tracker.npz as x/y references are not
    enough; here a synthetic solution is exported and re-imported) keep the CSV column convention of
    07_multioptyplan.py:476-489, and the cached single-aircraft solution loads through compute_or_load."""
    from d2d_b200 import multiopty_utils as d2mou, opty_utils as d2ou, planner
    g = golden["colloc"]

    class mscen:
        t0, t1, hz = 0., 1.9, 10.
        p0s = tuple(tuple(v) for v in g["m3/p0s"]); p1s = tuple(tuple(v) for v in g["m3/p1s"])
        wind = d2ou.WindField([0.5, -1.0]); vref = 12.; obj_scale = 1.
        cost = d2mou.CostInput(vsp=12., kv=1., kphi=1.)
    mp = planner.MultiPlanner(mscen)
    mp.solution = g["m3/free"].copy()
    fn = tmp_path / "plan.csv"
    mp.save_csv(fn)
    import pandas as pd
    df = pd.read_csv(fn)
    assert list(df.columns[:6]) == ["time", "x_1", "y_1", "psi_1", "phi_1", "v_1"] and len(df) == 20
    mp2 = planner.MultiPlanner(mscen)
    mp2.load_csv(fn)
    np.testing.assert_allclose(mp2.solution, g["m3/free"], rtol=1e-13, atol=1e-15)      # text round trip
    np.testing.assert_allclose(mp2.prob.con(mp2.solution), g["m3/residual"], rtol=1e-10, atol=1e-9)

    class exp(planner.exp_0):
        t1, hz = 20., 50.
    p = planner.Planner(exp)
    npz = tmp_path / "optyplan_exp0_1_3.npz"
    sol = g["c3/sol"]; N = 1001
    np.savez(npz, sol_time=np.linspace(0, 20, N), sol_x=sol[:N], sol_y=sol[N:2 * N], sol_psi=sol[2 * N:3 * N], sol_phi=sol[3 * N:4 * N],
             sol_v=sol[4 * N:], wind=np.zeros((N, 2)))
    planner.compute_or_load(p, filename=str(npz))
    assert np.abs(p.prob.con(p.solution)).max() < 1e-6
    planner.compute_or_load(p, force_recompute=True, filename=str(tmp_path / "new.npz"))     # solves on the engine and caches
    q = planner.Planner(exp)
    planner.compute_or_load(q, filename=str(tmp_path / "new.npz"))
    np.testing.assert_array_equal(q.solution, p.solution)
    assert np.abs(q.prob.con(q.solution)).max() < 1e-6


@pytest.mark.parametrize("n_ac,N,n_prob", [(2, 33, 1), (3, 64, 2), (8, 100, 3), (16, 97, 2), (17, 40, 1), (5, 31, 70), (33, 20, 1),
                                           (16, 97, 200), (3, 65, 300), (7, 150, 120), (2, 500, 40), (9, 100, 200), (2, 20, 65536)])
def test_all_pairs_kernel_shapes_against_oracle(n_ac, N, n_prob):
    """colloc_pairs_kernel (every unordered pair once, exponentials handed over through shared-memory slots): even / odd
    aircraft counts, fewer aircraft than warps, more than two aircraft per warp, ragged last tile, the two-kernel cost
    reduction of large batches (n_prob >= 64), the one-dimensional grid of the largest call (65536 problems), and the ordered fallback beyond
    the shared-memory budget (33 aircraft).
    n_ac <= 16 takes the instantiation whose phase-A gradients wait in registers, larger counts the shared-memory one."""
    from oracle import d2d_oracle as orc
    from d2d_b200.collocation import CollocationProblem, CostSpec
    rng = np.random.default_rng(100 + n_ac)
    h = 0.05
    free = rng.normal(0, 6., (n_prob, 5 * n_ac * N)); free[:, 4 * n_ac * N:] = 12 + rng.normal(0, 1, (n_prob, n_ac * N))
    for obstacles in ([], [(1., 2., 6.), (-4., 3., 5.)]):
        spec = dict(vsp=12., kvel=3., kbank=2., kcol=10., rcol=8., pairs="all", kobs=1.5 if obstacles else 0., obstacles=obstacles, obs_kind=1)
        cs = CostSpec(vsp=12., kvel=3., kbank=2., kcol=10., rcol=8., all_pairs=True, kobs=1.5 if obstacles else 0., obstacles=obstacles, obs_kind=1)
        inst = [(k, 0, 0.5 * k) for k in range(3 * n_ac)]
        prob = CollocationProblem(n_ac, N, h, wind=(1., 2.), inst=inst, cost=cs)
        res, jac, cost, grad = prob.evaluate(free)
        for p in sorted({0, 1, 2, n_prob - 1} & set(range(n_prob))):
            np.testing.assert_allclose(res[p], orc.colloc_residual(free[p], N, n_ac, h, (1., 2.), inst), rtol=RTOL, atol=1e-10)
            np.testing.assert_allclose(jac[p][:-len(inst)], orc.colloc_jac_compact(free[p], N, n_ac, h).reshape(-1), rtol=RTOL)
            co, go = orc.cost_and_grad(free[p], N, n_ac, spec, multi=True)
            np.testing.assert_allclose(cost[p], co, rtol=RTOL)
            np.testing.assert_allclose(grad[p], go, rtol=RTOL, atol=1e-13)
        # cost-only and gradient-only calls agree with the fused call; repeated calls are bit-identical (fixed summation order)
        np.testing.assert_array_equal(prob.obj(free), cost)
        np.testing.assert_array_equal(prob.obj_grad(free), grad)


@pytest.mark.parametrize("world,n_prob", [(8, 1), (2, 1), (4, 3)])
def test_fused_peer_evaluation_emulated_on_one_gpu(golden, world, n_prob):
    """d2dx_colloc_eval_peer with every rank in this process (one exchange buffer and one stream per rank on the same
    GPU, so the kernels really wait on each other's flags): C4 split by aircraft = the unsharded evaluation, every rank
    ends with the same total cost, the second evaluation (next epoch) equals the first, no wait timed out."""
    from d2d_b200.collocation import CollocationProblem, CostSpec
    from d2d_b200 import distributed
    g = golden["colloc"]
    n_ac, N, h = 16, 500, 0.02
    inst = _inst(g, "c4")
    rng = np.random.default_rng(7)
    free = np.stack([g["c4/free"] + (0. if p == 0 else rng.normal(0, 0.5, g["c4/free"].shape)) for p in range(n_prob)])
    cs = CostSpec(vsp=12., kvel=70., kbank=1., kcol=10., rcol=10., all_pairs=True, kobs=0.5, obstacles=[(60., 5., 12.)], obs_kind=1)
    full = CollocationProblem(n_ac, N, h, inst=inst, cost=cs)
    res, jac, cost, grad = full.evaluate(free)
    out = distributed.emulate_peer_eval(n_ac, N, h, (0., 0.), inst, cs, free, world=world, replays=3)
    assert all(st["timeouts"] == 0 and st["evaluations"] == 3 for st in out["status"]), out["status"]
    np.testing.assert_allclose(out["residual"], res, rtol=0, atol=1e-14)
    np.testing.assert_allclose(out["jac"], jac, rtol=1e-15, atol=0)
    np.testing.assert_allclose(out["grad"], grad, rtol=1e-13, atol=1e-16)
    for r in range(world):
        np.testing.assert_array_equal(out["cost"][r], out["cost"][0])
        np.testing.assert_allclose(out["cost"][r], cost, rtol=1e-13)


def test_cost_bank_max_mode_against_reference_golden(golden):
    """CostBank with use_mean = False (d2d/opty_utils.py:72,78-81): obj_scale * max(phi^2), one gradient entry at the first
    maximum; fixtures from the unmodified reference class."""
    from d2d_b200 import opty_utils
    g = golden["colloc"]
    N = 1001

    class P:
        num_nodes, obj_scale = N, 2.5
        _slice_x, _slice_y, _slice_psi, _slice_phi, _slice_v = (slice(k * N, (k + 1) * N) for k in range(5))
    c = opty_utils.CostBank(); c.use_mean = False
    for tag, fr in (("sol", g["c3/sol"]), ("noisy", g["c3/free"])):
        np.testing.assert_allclose(c.cost(fr, P), g[f"cost1/bankmax/{tag}/cost"], rtol=1e-15)
        np.testing.assert_array_equal(c.cost_grad(fr, P), g[f"cost1/bankmax/{tag}/grad"])
    tie = np.zeros(5 * N); tie[3 * N + 7] = -0.3; tie[3 * N + 400] = 0.3          # equal squares: np.argmax takes the first
    gr = c.cost_grad(tie, P)
    assert gr[3 * N + 7] == 2.5 * 2 * -0.3 and np.count_nonzero(gr) == 1


@pytest.mark.parametrize("mode", ["pair01", "nocol", "cost_only"])
def test_fused_peer_evaluation_other_cost_modes(golden, mode):
    """The fused sharded kernel in the reference's own collision mode (aircraft 0 and 1 only -- they live on different ranks
    here), without any collision term (only the cost sums are exchanged), and asked for the cost alone."""
    from d2d_b200.collocation import CollocationProblem, CostSpec
    from d2d_b200 import distributed, _lib
    n_ac, N, h, world = 4, 75, 0.05, 4
    rng = np.random.default_rng(21)
    free = rng.normal(0, 5., (2, 5 * n_ac * N)); free[:, 4 * n_ac * N:] = 12 + rng.normal(0, 1, (2, n_ac * N))
    inst = [(k, 0, 0.25 * k) for k in range(3 * n_ac)]
    if mode == "nocol":
        cs = CostSpec(vsp=12., kvel=3., kbank=2., kobs=1.5, obstacles=[(1., 2., 6.)], obs_kind=1)
    else:
        cs = CostSpec(vsp=12., kvel=3., kbank=2., kcol=10., rcol=8., all_pairs=False, kobs=1.5, obstacles=[(1., 2., 6.)], obs_kind=0)
    full = CollocationProblem(n_ac, N, h, wind=(0.5, -1.), inst=inst, cost=cs)
    res, jac, cost, grad = full.evaluate(free)
    out = distributed.emulate_peer_eval(n_ac, N, h, (0.5, -1.), inst, cs, free, world=world, replays=2)
    assert all(st["timeouts"] == 0 for st in out["status"])
    np.testing.assert_allclose(out["residual"], res, rtol=0, atol=1e-13)
    np.testing.assert_allclose(out["jac"], jac, rtol=1e-14, atol=0)
    np.testing.assert_allclose(out["grad"], grad, rtol=1e-12, atol=1e-15)
    for r in range(world):
        np.testing.assert_allclose(out["cost"][r], cost, rtol=1e-13)


def test_new_entry_points_reject_bad_arguments():
    """d2dx_peer_create / d2dx_colloc_eval_peer / d2dx_ddp_solve / d2dx_cost_bank_max validate before they launch."""
    import ctypes as C
    from d2d_b200 import _lib, get_engine
    from d2d_b200.collocation import CollocationProblem, CostSpec
    eng = get_engine()
    lib = _lib.lib
    p = C.c_void_p()
    assert lib.d2dx_peer_create(eng.h, 0, 0, 1, 4, 10, C.byref(p)) == 1            # world 0
    assert lib.d2dx_peer_create(eng.h, 2, 2, 1, 4, 10, C.byref(p)) == 1            # rank out of range
    assert lib.d2dx_peer_create(eng.h, 17, 0, 1, 4, 10, C.byref(p)) == 1           # more ranks than the exchange supports
    prob = CollocationProblem(2, 10, 0.1, cost=CostSpec(vsp=12., kvel=1.))
    pe = eng.peer_create(2, 0, 1, 2, 10)                                           # never connected
    with pytest.raises(_lib.D2dxError, match="not connected"):
        eng.colloc_eval_peer(pe, prob.c, 1, 0, eng.zeros(50), _lib.EVAL_ALL, eng.zeros(60), eng.zeros(220), eng.zeros(1), eng.zeros(50))
    pe.close()
    with pytest.raises(_lib.D2dxError, match="n_ac = 1"):
        eng.ddp_solve(prob.c, 1, (-0.5, 0.5, 9., 14.), None, eng.zeros(1, 3), eng.zeros(1, 3), eng.zeros(1, 2, 10), eng.zeros(1, 3, 10), eng.zeros(1, 8))
    one = CollocationProblem(1, 10, 0.1, cost=CostSpec(vsp=12., kvel=1.))
    with pytest.raises(_lib.D2dxError):
        eng.ddp_solve(one.c, 1, (0.5, -0.5, 9., 14.), None, eng.zeros(1, 3), eng.zeros(1, 3), eng.zeros(1, 2, 10), eng.zeros(1, 3, 10), eng.zeros(1, 8))
    with pytest.raises(_lib.D2dxError):
        eng.cost_bank_max(eng.zeros(1, 50), 45, 10, 1.0)                           # phi slice runs past the free vector


def test_sixteen_aircraft_instantiation_with_opty_order_and_partial_calls():
    """The 16-aircraft instantiation of colloc_pairs_kernel (compile-time round counts, halo column, prefetched node inputs)
    under opty's name-sorted input order (phi10 .. phi15 before phi2): equal to the numeric-order problem on the permuted free
    vector, equal to the oracle, and consistent between fused and partial (residual only / Jacobian only / gradient only)
    calls; N = 70 leaves a ragged last tile and a first tile whose halo column is unused."""
    from oracle import d2d_oracle as orc
    from d2d_b200.collocation import CollocationProblem, CostSpec
    n_ac, N, h, n_prob = 16, 70, 0.05, 3
    rng = np.random.default_rng(16)
    free = rng.normal(0, 6., (n_prob, 5 * n_ac * N)); free[:, 4 * n_ac * N:] = 12 + rng.normal(0, 1, (n_prob, n_ac * N))
    cs = CostSpec(vsp=12., kvel=3., kbank=2., kcol=10., rcol=8., all_pairs=True, kobs=1.5, obstacles=[(1., 2., 6.)], obs_kind=1)
    inst = [(k, 0, 0.5 * k) for k in range(3 * n_ac)]
    a = CollocationProblem(n_ac, N, h, wind=(1., 2.), inst=inst, cost=cs)
    b = CollocationProblem(n_ac, N, h, wind=(1., 2.), inst=inst, cost=cs, input_order="opty")
    numeric = [f"phi{i}(t)" for i in range(n_ac)] + [f"v{i}(t)" for i in range(n_ac)]
    names = sorted(numeric)                                     # opty sorts the input symbols by name
    src = [numeric.index(nm) for nm in names]
    fp = free.copy()
    for k, s_ in enumerate(src):
        fp[:, (3 * n_ac + k) * N:(3 * n_ac + k + 1) * N] = free[:, (3 * n_ac + s_) * N:(3 * n_ac + s_ + 1) * N]
    ra, ja, ca, ga = a.evaluate(free)
    rb, jb, cb, gb = b.evaluate(fp)
    np.testing.assert_array_equal(ra, rb); np.testing.assert_array_equal(ja, jb); np.testing.assert_array_equal(ca, cb)
    np.testing.assert_array_equal(gb[:, :3 * n_ac * N], ga[:, :3 * n_ac * N])
    for k, s_ in enumerate(src):
        np.testing.assert_array_equal(gb[:, (3 * n_ac + k) * N:(3 * n_ac + k + 1) * N], ga[:, (3 * n_ac + s_) * N:(3 * n_ac + s_ + 1) * N])
    spec = dict(vsp=12., kvel=3., kbank=2., kcol=10., rcol=8., pairs="all", kobs=1.5, obstacles=[(1., 2., 6.)], obs_kind=1)
    for p in range(n_prob):
        np.testing.assert_allclose(ra[p], orc.colloc_residual(free[p], N, n_ac, h, (1., 2.), inst), rtol=RTOL, atol=1e-10)
        np.testing.assert_allclose(ja[p][:-len(inst)], orc.colloc_jac_compact(free[p], N, n_ac, h).reshape(-1), rtol=RTOL)
        co, go = orc.cost_and_grad(free[p], N, n_ac, spec, multi=True)
        np.testing.assert_allclose(ca[p], co, rtol=RTOL)
        np.testing.assert_allclose(ga[p], go, rtol=RTOL, atol=1e-13)
    np.testing.assert_array_equal(a.con(free), ra)
    np.testing.assert_array_equal(a.con_jac(free), ja)
    np.testing.assert_array_equal(a.obj(free), ca)
    np.testing.assert_array_equal(a.obj_grad(free), ga)
