"""Multi-aircraft planner solves, coupled second-order (method="ddp") against augmented-Lagrangian L-BFGS (method="lbfgs"), on
upstream's experiments (07_multioptyplan.py) and the mission's phase-2 problem; plus a population of 1024 four-aircraft problems
in one launch.  Per experiment and method: wall time of MultiPlanner.run (n_starts = 8), cost of the kept solution, feasible starts,
minimum separation between aircraft.  After one warm-up run of each, the two methods alternate, `--repeats` times.

    python scripts/time_ddp_multi.py --out profiles/r4_ddp_multi.json [--repeats 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "drone-sim-python_b200")]

EXPERIMENTS = [("exp_1_0", 0), ("exp_2", 0), ("exp_4", 0), ("exp_5", 0), ("exp_5", 1), ("exp_5_1", 0), ("gvf_trial_3ac", 0), ("trap_4", 0)]
X1_F = ((0, 40, 0, 0, 12), (25, 40, 0, 0, 12), (25, -40, 0, 0, 12), (0, -40, 0, 0, 12))      # mission.full_sim's phase-2 boundary states
X2_F = ((75, 40, 0, 0, 12), (100, 40, 0, 0, 12), (100, -40, 0, 0, 12), (75, -40, 0, 0, 12))


def scenario(name):
    from d2d_b200 import mission, multiopty_scenarios as S
    if name == "trap_4":
        s = mission.trap_4
        s.t1, s.p0s, s.p1s = 6, X1_F, X2_F
        return s
    return getattr(S, name)


def run_once(name, case, method, n_starts):
    import torch
    from d2d_b200 import planner as pl
    exp = scenario(name)
    exp.set_case(case)
    p = pl.MultiPlanner(exp)
    p.configure(tol=exp.tol, max_iter=exp.max_iter)
    guess = p.get_initial_guess("tri")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    info = p.run(initial_guess=guess, n_starts=n_starts, method=method)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    n = p.acs.nb_aicraft
    sep = min([np.hypot(p.sol_x[a] - p.sol_x[b], p.sol_y[a] - p.sol_y[b]).min() for a in range(n) for b in range(a)] or [float("inf")])
    if info["method"] == "ddp":
        feas = int(np.isin(info["flag"], (2, 4)).sum())
    else:
        feas = int((info["c_max"] < 100 * min(exp.tol, 1e-6)).sum())
    return {"time_s": dt, "cost": float(p.prob.obj(p.solution)), "feasible": bool(info["feasible"]), "feasible_starts": feas,
            "starts": int(len(info["c_max"])), "min_separation": float(sep), "con": float(np.abs(p.prob.con(p.solution)).max())}


def population(P=1024, seed=7):
    import torch
    from d2d_b200 import planner as pl, shooting
    s = scenario("trap_4")
    p = pl.MultiPlanner(s)
    p0, p1 = p._boundary_states()
    rng = np.random.default_rng(seed)
    p1s = p1[None] + np.stack([rng.uniform(-8, 8, (P, 4)), rng.uniform(-8, 8, (P, 4)), rng.uniform(-0.3, 0.3, (P, 4))], 1)
    nlp = shooting.ShootingNLP(p.prob, p0, p1s, s.phi_constraint, s.v_constraint, P=P, state_box=(-150, 150, -150, 150, 1000.))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, info = shooting.solve_ddp(nlp, 0., 12., ctol=1e-8, retries=0)
    torch.cuda.synchronize()
    return {"time_s": time.perf_counter() - t0, "solved": int((info["flag"] == 2).sum()), "P": P, "median_sweeps": float(np.median(info["iterations_each"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--n-starts", type=int, default=8)
    a = ap.parse_args()
    import torch
    gpu = {"name": torch.cuda.get_device_name(0)}
    try:
        gpu["power_limit_clock"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                                  capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        gpu["power_limit_clock"] = "unknown"
    rows = []
    for name, case in EXPERIMENTS:
        for m in ("ddp", "lbfgs"):                                     # warm-up: module loads, graph captures
            run_once(name, case, m, a.n_starts)
        res = {"ddp": [], "lbfgs": []}
        for _ in range(a.repeats):
            for m in ("ddp", "lbfgs"):
                res[m].append(run_once(name, case, m, a.n_starts))
        row = {"experiment": name, "case": case}
        for m, rs in res.items():
            row[m] = {"time_s": [r["time_s"] for r in rs], **{k: rs[-1][k] for k in ("cost", "feasible", "feasible_starts", "starts", "min_separation", "con")}}
        rows.append(row)
        print(json.dumps(row), flush=True)
    population()                                                       # warm-up
    pop = [population() for _ in range(a.repeats)]
    print(json.dumps({"population": pop}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"gpu": gpu, "n_starts": a.n_starts, "experiments": rows, "population": pop}, f, indent=1)


if __name__ == "__main__":
    main()
