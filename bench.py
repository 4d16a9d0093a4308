#!/usr/bin/env python3
"""Headline benchmark: closed-loop aircraft-steps/s on the Monte-Carlo sweep (BASELINE.json configs[4], SURVEY 8d
config C5): 10^6 aircraft-scenarios per GPU x 10^4 RK4 steps, dt = 0.01 s, random circles / wind / initial states,
DFFF controller, log decimated x100.  One bench "step" = one full sweep.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # the CUDA engine
    python bench.py ... --dump-outputs bench_outputs               # also write the last timed sweep's results as .npy files
    python bench.py --impl reference ...                           # the CPU arm (C port of the oracle, all host threads)

Prints ONE JSON line (value = device-resident throughput, e2e = through the public host-buffer API with H2D/D2H inside
the timed region, roofline, cpu_baseline, clocks, gpu_launches)."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time as _time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "drone-sim-python_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "closed-loop aircraft-steps/s"
UNIT = "aircraft-steps/s"
# Executed fp64 flop per aircraft-step of rollout_dfff_kernel<CIRCLE> (DADD + DMUL + 2 x DFMA thread-instructions
# from the ncu capture under profiles/, divided by scenarios x steps); see DESIGN.md "Roofline accounting".
FP64_FLOP_PER_STEP = float(os.environ.get("D2DX_FLOP_PER_STEP", "672"))
# From the same capture (profiles/r2i_rollout_dfff_circle.md, one launch of 1e6 scenarios x 400 steps, log x100 = the default
# bench launch): dram__bytes_read.sum + dram__bytes_write.sum, and the fp64 pipe's active fraction.
NCU_TRAFFIC_BYTES_DEFAULT_LAUNCH = 181.10e6 + 323.17e6
NCU_TRAFFIC_CONFIG = (10 ** 6, 10 ** 4, 100, 25)       # (scenarios, steps, log_every, chunks) the capture was taken at
NCU_FP64_PIPE_ACTIVE = 0.770
LOG_BYTES_PER_LOGGED_SAMPLE = 56          # 5 state + 2 input doubles


def workload(B, seed):
    """C5 population (SURVEY 8d): circles c ~ U([-50,50]^2), r ~ U(20,60), v ~ U(10,15), alpha0 ~ U(0,2pi);
    wind ~ N(0, 2.5^2) per axis, redrawn while |w| > 0.4 v; X0 = flat state(t=0) + N(0, diag(5,5,.2,.05,.5)^2)."""
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(-50, 50, B), rng.uniform(-50, 50, B)
    r, v, a0 = rng.uniform(20, 60, B), rng.uniform(10, 15, B), rng.uniform(0, 2 * np.pi, B)
    wind = rng.normal(0, 2.5, (B, 2))
    for _ in range(64):
        bad = np.hypot(wind[:, 0], wind[:, 1]) > 0.4 * v
        if not bad.any():
            break
        wind[bad] = rng.normal(0, 2.5, (int(bad.sum()), 2))
    noise = rng.normal(0, 1, (B, 5)) * np.array([5, 5, 0.2, 0.05, 0.5])
    return dict(cx=cx, cy=cy, r=r, v=v, a0=a0, wind=wind, noise=noise)


def flat_state0(w):
    """Flat state at t = 0 of every circle (closed form of d2d/guidance.py:23-47 on d2d/trajectory.py:153-160);
    workload generation only -- both arms start from these X0."""
    om = w["v"] / w["r"]
    ca, sa = np.cos(w["a0"]), np.sin(w["a0"])
    y0 = np.stack([w["cx"] + w["r"] * ca, w["cy"] + w["r"] * sa], 1)
    y1 = np.stack([om * w["r"] * -sa, om * w["r"] * ca], 1)
    y2 = np.stack([om ** 2 * w["r"] * -ca, om ** 2 * w["r"] * -sa], 1)
    vax, vay = y1[:, 0] - w["wind"][:, 0], y1[:, 1] - w["wind"][:, 1]
    va = np.sqrt(vax ** 2 + vay ** 2)
    phi = np.arctan((y2[:, 1] * vax - y2[:, 0] * vay) / va / 9.81)
    return np.stack([y0[:, 0], y0[:, 1], np.arctan2(vay, vax), phi, va], 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[2 + k].lower().startswith("active") for r in self.rows)]
        pw = [float(r[6]) for r in self.rows if len(r) >= 7 and r[6].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows and self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(pw) if pw else None}


def cpu_port_run(B, T_steps, seed, nthreads=0, reps=1):
    """The oracle's C port on the host cores over a bounded sample of the same workload; returns (steps/s, cores, text)."""
    from oracle import c_oracle as co
    w = workload(B, seed)
    X0 = flat_state0(w) + w["noise"]
    ty, par = co.circle_par(w["cx"], w["cy"], w["r"], w["v"], w["a0"])
    time = np.arange(T_steps + 1) * 0.01
    cores = nthreads or co.max_threads()
    best = 0.
    for _ in range(reps):
        t0 = _time.perf_counter()
        out = co.rollout(time, ty, par, w["wind"], X0, want_log=False, nthreads=cores)
        dt = _time.perf_counter() - t0
        best = max(best, B * T_steps / dt)
    return best, cores, f"first {B} scenarios x {T_steps} steps of the C5 population (seed {seed}), no log, {cores} threads", out


def python_port_rate():
    """The NumPy/SciPy oracle (the reference's own numerics: SciPy CARE every step) on one core, tiny sample."""
    from oracle import d2d_oracle as orc
    w = workload(2, 12345)
    X0 = flat_state0(w) + w["noise"]
    time = np.arange(151) * 0.01
    t0 = _time.perf_counter()
    for b in range(2):
        orc.run_simulation(time, orc.Circle([w["cx"][b], w["cy"][b]], w["r"][b], w["v"][b], alpha0=w["a0"][b]), w["wind"][b], X0[b])
    return 2 * 150 / (_time.perf_counter() - t0)


def _timed(fn, reps, warm=3):
    """average seconds per call of fn on the current stream (CUDA events, after `warm` untimed calls)"""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


DUMP_SCENARIOS = 4096
DUMP_BYTES = 64 << 20


def dump_outputs(path, mc, seed):
    """Writes what the timed sweep (MonteCarloRollout.run_device) left in HBM, under the names MonteCarloRollout.run()
    returns them by, as float64 .npy files: the population statistics whole, every per-scenario array for the same sample
    of at most DUMP_SCENARIOS scenarios (sorted indices drawn from `seed`, so equal arguments give an equal sample) in
    run()'s layout, at most DUMP_BYTES in all.  Two builds run with the same arguments can then be compared file by file;
    pop_sum_sq_err is summed with one atomicAdd per warp, so it may differ in its last bits from run to run."""
    import torch
    per_scenario = 8 * (mc.n_rows * (5 + (2 if mc.d_Ulog is not None else 0)) + 5 + 3)
    S = min(mc.B, DUMP_SCENARIOS, DUMP_BYTES // per_scenario)
    if S < 1:
        raise SystemExit(f"--dump-outputs: the log of one scenario ({per_scenario} bytes) exceeds {DUMP_BYTES} bytes; raise --log-every")
    idx = torch.from_numpy(np.sort(np.random.default_rng(seed).choice(mc.B, S, replace=False))).to(mc.d_Xf.device)
    arrays = {"X_final": mc.d_Xf[:, idx].T, "sum_sq_err": mc.d_ss[idx], "max_err": mc.d_mx[idx], "flags": mc.d_flags[idx],
              "pop_sum_sq_err": mc.d_pop[:1], "pop_max_err": mc.d_pop[1:], "X_log": mc.d_Xlog[:, :, idx]}
    if mc.d_Ulog is not None:
        arrays["U_log"] = mc.d_Ulog[:, :, idx]
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.to(torch.float64).cpu().numpy())


C4 = dict(n_ac=16, N=500, h=0.02)


def _c4_cost():
    from d2d_b200.collocation import CostSpec
    return CostSpec(vsp=12., kvel=70., kbank=1., kcol=10., rcol=10., all_pairs=True)


def core_metrics(eng, hbm_peak, fp64_peak, world, rank, seed):
    """The rest of BASELINE.json's metric at EVERY N (SURVEY 8d/8e): collocation evals/s with the problems sharded over the
    ranks (no data-path collective), the formation rollout sharded by formation, and -- for N > 1 -- ONE C4 problem and a
    batch of C4 problems sharded by AIRCRAFT through the fused peer-memory kernel, checked against rank 0's unsharded
    evaluation.  Every rank runs its share; times are CUDA events, max over ranks; rank 0 returns the aggregate."""
    import torch
    import torch.distributed as dist
    from d2d_b200 import _lib
    from d2d_b200.collocation import CollocationProblem, CostSpec
    from d2d_b200.simulation import chain_incidence
    out, checks = {}, {}

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=eng.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    rng = np.random.default_rng(seed + 1000 * rank)
    # (1) batched collocation, problems sharded over ranks: each rank evaluates its own n_prob problems per launch
    for tag, n_ac, N, h, n_prob, cost in (
            ("c3_batch4096", 1, 1001, 0.02, 4096, CostSpec(vsp=12., kvel=1.)),
            ("c4_batch256_allpairs", C4["n_ac"], C4["N"], C4["h"], 256, _c4_cost())):
        prob = CollocationProblem(n_ac, N, h, inst=[(k, 0, 0.) for k in range(3 * n_ac)], cost=cost)
        free = eng.to_device(rng.normal(0, 3., (n_prob, prob.num_free)) + 12. * (np.arange(prob.num_free) >= 4 * n_ac * N))
        bufs = prob.buffers(n_prob)
        sync_all()
        dt = max_over_ranks(_timed(lambda: prob.evaluate_device(free, _lib.EVAL_ALL, bufs), 20))
        bytes_alg = 200.0 * n_ac * N * n_prob                      # SURVEY 8d: 200 B per aircraft-node, compact layout
        line = {"evals_per_s": world * n_prob / dt, "ms_per_launch": dt * 1e3, "problems_per_gpu": n_prob,
                "aircraft_nodes_per_launch": n_ac * N * n_prob, "sharding": f"by problem x{world}, no collective",
                "roofline": {"bound": "hbm", "achieved": bytes_alg / dt / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": bytes_alg / dt / 1e9 / hbm_peak,
                             "algorithmic_bytes_per_launch": bytes_alg}}
        if n_ac > 1:       # the pair terms make this launch fp64 / issue work as well: executed fp64 flop from the ncu capture
            flop = 548.0 * n_ac * N * n_prob                       # profiles/r2h_colloc_c4_batch256_allpairs.md (16 aircraft, all pairs)
            line["roofline"]["fp64"] = {"achieved": flop / dt / 1e12, "peak": fp64_peak, "unit": "TFLOP/s", "frac": flop / dt / 1e12 / fp64_peak,
                                        "flop_per_aircraft_node": 548.0}
            line["roofline"]["note"] = ("neither roof binds: 847 warp instructions per warp and aircraft-node at 56 % of the issue slots, 32 resident "
                                        "warps per SM (64 registers, 49 KB of shared memory per block) -- latency of the dependent fp64 chains")
        out[tag] = line
        del prob, free, bufs
    # (2) formation rollout, config C2 replicated, formations sharded over ranks (whole waves per GPU)
    n_ac, T = 6, 1200
    F = eng.sm_count * 5 * (eng.formation_threads_per_sm // 32)        # whole waves: 5 formations per warp
    M = F * n_ac
    X0 = eng.to_device(np.ascontiguousarray(np.tile(np.array([20, 30, -np.pi / 2, 0, 10.]), (M, 1)).T))
    c, r, ac = eng.zeros(2, M), eng.to_device(np.full(M, 60.)), eng.to_device(np.stack([np.full(M, 0.01), np.full(M, 1.)]))
    z = np.ones(n_ac - 1) * 2 * np.pi / n_ac
    Xf = eng.empty(5, M)
    sync_all()
    dt = max_over_ranks(_timed(lambda: eng.rollout_formation(n_ac, chain_incidence(n_ac), z, X0, c, r, ac, 4e-4, 15, 20, 15., 0.05, 0, T - 1, 5, X_final=Xf), 3))
    # executed fp64 flop per aircraft-step (5 RK4 sub-steps + DCF + GVF), ncu: profiles/r1_final_formation_c2.md
    flop = 1743.0 * M * (T - 1)                  # profiles/r2i_formation_c2.md
    out["formation_c2_batch"] = {"aircraft_steps_per_s": world * M * (T - 1) / dt, "rk4_substeps_per_s": world * M * (T - 1) * 5 / dt,
                                 "formations_per_gpu": F, "ms_per_launch": dt * 1e3, "sharding": f"by formation x{world}, no collective",
                                 "roofline": {"bound": "fp64", "achieved": flop / dt / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                                              "frac": flop / dt / 1e12 / fp64_peak, "flop_per_aircraft_step": 1743.0}}
    del X0, c, r, ac, Xf
    # (3) ONE C4 problem (and a batch of 64) sharded by aircraft over the ranks: fused peer-memory kernel, CUDA graph
    rng0 = np.random.default_rng(seed)                                # the same problems on every rank
    n_ac, N, h = C4["n_ac"], C4["N"], C4["h"]
    nf = 5 * n_ac * N
    PB = 64
    free_all = rng0.normal(0, 30., (PB, nf)); free_all[:, 4 * n_ac * N:] = 12. + rng0.normal(0, 1, (PB, n_ac * N))
    inst = [(3 * a + k, 0, float(a + k)) for a in range(n_ac) for k in range(3)]
    full = CollocationProblem(n_ac, N, h, inst=inst, cost=_c4_cost())
    fd1, fdB = eng.to_device(free_all[:1].copy()), eng.to_device(free_all)
    b1, bB = full.buffers(1), full.buffers(PB)
    replay1, _ = full.graph(fd1)
    t1 = _timed(replay1, 200, warm=20)
    tB = _timed(lambda: full.evaluate_device(fdB, _lib.EVAL_ALL, bB), 50)
    alg1 = 200.0 * n_ac * N
    out["c4_single_allpairs"] = {"evals_per_s": 1.0 / t1, "us_per_eval": t1 * 1e6, "how": "one GPU, CUDA-graph replay of the fused evaluation",
                                 "roofline": {"bound": "launch latency", "achieved": alg1 / t1 / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": alg1 / t1 / 1e9 / hbm_peak}}
    out["c4_batch64_allpairs_one_gpu"] = {"evals_per_s": PB / tB, "us_per_launch": tB * 1e6}
    if world > 1 and n_ac % world == 0:
        try:
            from d2d_b200.distributed import ShardedCollocation, shard_range
            sc1 = ShardedCollocation(n_ac, N, h, (0., 0.), inst, _c4_cost(), engine=eng, max_prob=1)
            scB = ShardedCollocation(n_ac, N, h, (0., 0.), inst, _c4_cost(), engine=eng, max_prob=PB)
            fl1 = eng.to_device(free_all[0, sc1.shard.idx_free].copy())
            flB = eng.to_device(np.ascontiguousarray(free_all[:, scB.shard.idx_free]))
            rep1, o1 = sc1.graph(fl1)
            repB, oB = scB.graph(flB)
            sync_all()
            ts1 = max_over_ranks(_timed(rep1, 200, warm=20))
            sync_all()
            tsB = max_over_ranks(_timed(repB, 50, warm=5))
            sync_all()
            st1, stB = sc1.check(), scB.check()
            rep1(); torch.cuda.synchronize()
            tl = sc1.peer.timeline()                            # rank 0's phase stamps of one more evaluation (ns since its kernel start)
            # parity: every rank's shard of the batch against rank 0's unsharded evaluation of the same problems
            full.evaluate_device(fdB, _lib.EVAL_ALL, bB)
            diffs = []
            for name, mine, idx in (("res", oB[0], scB.shard.idx_con), ("jac", oB[1], scB.shard.idx_jac), ("grad", oB[3], scB.shard.idx_free)):
                ref = bB[name][:, torch.from_numpy(idx).to(eng.device)]
                diffs.append(float((mine - ref).abs().max().item()))
            diffs.append(float((oB[2] - bB["cost"]).abs().max().item() / bB["cost"].abs().max().item()))
            worst = max_over_ranks(max(diffs))
            checks["sharded_c4_max_abs_diff"] = worst
            checks["sharded_c4_peer_timeouts"] = int(max_over_ranks(float(st1["timeouts"] + stB["timeouts"])))
            sharded_line = {"evals_per_s": 1.0 / ts1, "us_per_eval": ts1 * 1e6, "aircraft_per_gpu": n_ac // world, "one_gpu_us_per_eval": t1 * 1e6,
                            "how": "one kernel per rank and evaluation: positions and cost sums as peer-memory stores over NVLink, CUDA-graph replay",
                            "timeline_ns_rank0": tl,
                            "roofline": {"bound": "launch + NVLink flag latency", "achieved": alg1 / ts1 / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                         "frac": alg1 / ts1 / 1e9 / hbm_peak}}
            out["c4_single_sharded_by_aircraft"] = sharded_line
            # the same 64 problems sharded by PROBLEM instead (PB / world each, no exchange at all): how a batch should be split
            lo, hi = shard_range(PB, world, rank)
            fdP = eng.to_device(free_all[lo:hi].copy())
            bP = full.buffers(hi - lo)
            sync_all()
            tP = max_over_ranks(_timed(lambda: full.evaluate_device(fdP, _lib.EVAL_ALL, bP), 50))
            out["c4_batch64_sharded_by_problem"] = {"evals_per_s": PB / tP, "us_per_launch": tP * 1e6, "one_gpu_us_per_launch": tB * 1e6,
                                                    "speedup_vs_one_gpu": tB / tP, "problems_per_gpu": hi - lo}
            out["c4_batch64_sharded_by_aircraft"] = {"evals_per_s": PB / tsB, "us_per_launch": tsB * 1e6, "one_gpu_us_per_launch": tB * 1e6,
                                                     "speedup_vs_one_gpu": tB / tsB,
                                                     "exchange_bytes_in_per_gpu": 2 * 16.0 * (n_ac - n_ac // world) * N * PB,
                                                     "roofline": {"bound": "hbm", "achieved": alg1 * PB / world / tsB / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                                                  "frac": alg1 * PB / world / tsB / 1e9 / hbm_peak,
                                                                  "note": "per-GPU algorithmic bytes (1/world of each problem) over the launch time; every rank "
                                                                          "receives the positions of all other aircraft of all problems (exchange_bytes_in_per_gpu, "
                                                                          "self-validating 16-byte words): a batch is better split by problem, aircraft "
                                                                          "sharding is for the latency of ONE problem"}}
            del sc1, scB
        except Exception as e:                              # e.g. no peer access between the GPUs of this box: keep every other number
            out["c4_single_sharded_by_aircraft"] = {"error": f"{type(e).__name__}: {e}"}
            checks["sharded_c4_error"] = f"{type(e).__name__}"
    return out, checks


def secondary_metrics(eng, hbm_peak):
    """Single-GPU extras beyond BASELINE.json's metric (SURVEY 8f rows, single-problem latencies, CPU figures)."""
    import torch
    from d2d_b200 import _lib
    from d2d_b200.collocation import CollocationProblem, CostSpec
    out = {}
    timed = lambda fn, reps: _timed(fn, reps)
    rng = np.random.default_rng(12345)
    for tag, n_ac, N, h, n_prob, cost in (("c3_single", 1, 1001, 0.02, 1, CostSpec(vsp=12., kvel=1.)),):
        prob = CollocationProblem(n_ac, N, h, inst=[(k, 0, 0.) for k in range(3 * n_ac)], cost=cost)
        free = eng.to_device(rng.normal(0, 3., (n_prob, prob.num_free)) + 12. * (np.arange(prob.num_free) >= 4 * n_ac * N))
        bufs = prob.buffers(n_prob)
        dt = timed(lambda: prob.evaluate_device(free, _lib.EVAL_ALL, bufs), 200)
        bytes_alg = 200.0 * n_ac * N * n_prob
        replay, _ = prob.graph(free)
        out[tag] = {"graph_replay_evals_per_s": 1.0 / timed(replay, 200), "evals_per_s": n_prob / dt, "ms_per_launch": dt * 1e3,
                    "roofline": {"bound": "launch latency", "achieved": bytes_alg / dt / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": bytes_alg / dt / 1e9 / hbm_peak}}
    # CPU figure for the collocation path: the NumPy oracle (lambdified-EoM class of the survey) on one core, C3
    try:
        from oracle import d2d_oracle as orc
        N3 = 1001
        f3 = rng.normal(0, 3., 5 * N3) + 12. * (np.arange(5 * N3) >= 4 * N3)
        t0 = _time.perf_counter()
        reps = 50
        for _ in range(reps):
            orc.colloc_residual(f3, N3, 1, 0.02, (0., 0.), [(k, 0, 0.) for k in range(3)])
            orc.colloc_jac_compact(f3, N3, 1, 0.02)
            orc.cost_and_grad(f3, N3, 1, dict(vsp=12., kvel=1.))
        out["c3_cpu_numpy_1core"] = {"evals_per_s": reps / (_time.perf_counter() - t0), "kind": "port", "cores": 1}
    except Exception as e:
        out["c3_cpu_numpy_1core"] = {"error": str(e)}
    # C5's second population (SURVEY 8d): randomised min-snap polynomials, POLY-specialised rollout kernel, 2000 steps
    from d2d_b200.simulation import chain_incidence  # noqa: F401
    from d2d_b200 import trajectory as ddt
    from d2d_b200.simulation import MonteCarloRollout
    Bp, Tp, dur = 500000, 2000, 33.65
    Y0 = np.zeros((Bp, 2, 4)); Y1 = np.zeros((Bp, 2, 4))
    a0, a1 = rng.uniform(-0.5, 0.5, Bp), rng.uniform(1.0, 2.0, Bp)
    Y0[:, 0, 0], Y0[:, 1, 0] = rng.uniform(-20, 20, Bp), rng.uniform(-20, 20, Bp)
    Y0[:, 0, 1], Y0[:, 1, 1] = 10 * np.cos(a0), 10 * np.sin(a0)
    Y1[:, 0, 0], Y1[:, 1, 0] = Y0[:, 0, 0] + rng.uniform(150, 250, Bp), Y0[:, 1, 0] + rng.uniform(150, 250, Bp)
    Y1[:, 0, 1], Y1[:, 1, 1] = 10 * np.cos(a1), 10 * np.sin(a1)
    msb = ddt.MinSnapBatch.from_boundaries(Y0, Y1, dur)
    mcp = MonteCarloRollout(Bp, np.arange(Tp + 1) * 0.01, _lib.SEG_POLY, log_every=100, n_chunks=2, host_log=False)
    parp = np.zeros((_lib.SEG_NPAR, Bp)); parp[1:9] = msb.coefs0[:, 0].T; parp[9:17] = msb.coefs0[:, 1].T
    X0p = np.stack([Y0[:, 0, 0] + 1., Y0[:, 1, 0] - 1., a0, 0 * a0, 0 * a0 + 10.], 1)
    mcp.set_inputs(parp, np.zeros((Bp, 2)), X0p); mcp.upload()
    dtp = timed(mcp.run_device, 3)
    out["c5_minsnap_population"] = {"aircraft_steps_per_s": Bp * Tp / dtp, "scenarios": Bp, "steps": Tp, "ms_per_sweep": dtp * 1e3,
                                    "unconverged_or_nonfinite": int(mcp.d_flags.ne(0).sum().item())}
    del mcp
    # the generic (mixed / composite) instantiation rollout_dfff_kernel<-1>: patrol_3-style composites (line, circle arc, slalom),
    # 75 776 scenarios x 2942 steps; the segment table is walked per step (fmod + search) and the parameter column reloaded on a switch
    try:
        from d2d_b200 import scenario as dds
        scen = dds.get("patrol_3")
        scen = scen[0] if isinstance(scen, tuple) else scen
        Bc = eng.sm_count * 512
        trajs = [scen.trajs[k % len(scen.trajs)] for k in range(Bc)]
        X0c = np.stack([np.asarray(scen.X0s[k % len(scen.trajs)], dtype=np.float64) for k in range(Bc)]) + rng.normal(0, 1, (Bc, 5)) * np.array([2, 2, .1, .02, .2])
        tabc = eng.table(ddt.pack(trajs))
        Wc = scen.windfield.sample(0, None)
        X0d, Wd = eng.to_device(np.ascontiguousarray(X0c.T)), eng.to_device(np.ascontiguousarray(np.tile(np.asarray(Wc, float), (Bc, 1)).T))
        acd, tdc = eng.to_device(np.stack([np.full(Bc, 0.01), np.full(Bc, 1.)])), eng.to_device(np.ascontiguousarray(scen.time, dtype=np.float64))
        Xfc, flc = eng.empty(5, Bc), eng.zeros(Bc, dtype=torch.int32)
        Tc = len(scen.time) - 1
        dtc = timed(lambda: eng.rollout_dfff(tabc, X0d, Wd, acd, tdc, 0, Tc, nsub=1, final_control=True, X_final=Xfc, flags=flc), 2)
        out["composite_patrol3_batch"] = {"aircraft_steps_per_s": Bc * Tc / dtc, "scenarios": Bc, "steps": Tc, "ms_per_launch": dtc * 1e3,
                                          "kernel": "rollout_dfff_kernel<-1> (generic: composite trajectories, segment table per step)",
                                          "roofline": {"bound": "fp64", "achieved": Bc * Tc * FP64_FLOP_PER_STEP / dtc / 1e12, "unit": "TFLOP/s",
                                                       "note": "lower bound: counted with the circle kernel's executed flop per step"}}
        del tabc, X0d, Wd, Xfc
    except Exception as e:
        out["composite_patrol3_batch"] = {"error": f"{type(e).__name__}: {e}"}
    # 5-state LQR tracker (SURVEY 8f #1) on sampled circle references: dt 0.1 s, RK4 nsub 10, T = 101 samples
    Mt, Tt = eng.sm_count * 1024, 101
    tt = np.arange(Tt) * 0.1
    rr, vv = rng.uniform(30, 60, Mt), rng.uniform(10, 14, Mt)
    om = vv / rr
    al = om[None, :] * tt[:, None]
    ref = np.stack([rr * np.cos(al), rr * np.sin(al), -vv * np.sin(al), vv * np.cos(al), -vv * om * np.cos(al), -vv * om * np.sin(al)], 1)
    X0t = eng.to_device(np.ascontiguousarray(np.stack([rr + 1., 0 * rr - 1., 0 * rr + np.pi / 2, 0 * rr, vv], 0)))
    refd, wz, act, Xft = eng.to_device(ref), eng.zeros(2, Mt), eng.to_device(np.stack([np.full(Mt, 0.01), np.full(Mt, 1.)])), eng.empty(5, Mt)
    dtt = timed(lambda: eng.rollout_tracker(refd, X0t, wz, act, 0.1, 0, Tt - 1, 10, X_final=Xft), 3)
    out["tracker_lqr5_batch"] = {"aircraft_steps_per_s": Mt * (Tt - 1) / dtt, "rk4_substeps_per_s": Mt * (Tt - 1) * 10 / dtt, "aircraft": Mt, "ms_per_launch": dtt * 1e3}
    # planner NLP solve by single shooting (SURVEY 8f #2).  (a) one Lagrangian+gradient evaluation of a population:
    # forward writes u_phys + states (2+3 doubles) and reads theta (2); adjoint reads theta, u_phys, states (7) and writes
    # the gradient (2): 16 doubles = 128 algorithmic bytes per aircraft-node.  (b) whole solves: exp_0 on the C3 grid.
    from d2d_b200 import planner as pl
    from d2d_b200.shooting import ShootingNLP, solve as shoot_solve
    Ps, Ns = 16384, 1001
    probs = CollocationProblem(1, Ns, 0.02, cost=CostSpec(vsp=12., kvel=1.), multi=False)
    nlp = ShootingNLP(probs, np.zeros((3, 1)), np.array([0., 30., np.pi]).reshape(3, 1), (-0.52, 0.52), (9., 14.), P=Ps)
    th = eng.to_device(rng.uniform(-1., 1., (Ps, nlp.n)))
    dts = timed(lambda: nlp.launch(th), 5)
    out["shoot_eval_batch16384"] = {"evals_per_s": Ps / dts, "aircraft_nodes_per_s": Ps * Ns / dts, "ms_per_eval": dts * 1e3,
                                    "roofline": {"bound": "hbm", "achieved": 128.0 * Ps * Ns / dts / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                                 "frac": 128.0 * Ps * Ns / dts / 1e9 / hbm_peak}}
    del nlp, th

    class exp_c3(pl.exp_0):
        t1, hz = 20., 50.
    _w = pl.Planner(pl.exp_0); _w.configure(tol=1e-8); _w.run()      # untimed: first CUDA-graph capture / module load of the process
    for tag, n_starts in (("planner_solve_c3_single", 1), ("planner_solve_c3_64starts", 64)):
        p = pl.Planner(exp_c3)
        p.configure(tol=1e-8)
        torch.cuda.synchronize(); t0 = _time.perf_counter()
        info = p.run(n_starts=n_starts)
        torch.cuda.synchronize(); dt_solve = _time.perf_counter() - t0
        out[tag] = {"seconds": dt_solve, "iterations": int(info["iterations"]), "evaluations": int(info["nfev"]), "ticks": int(info.get("ticks", 0)),
                    "method": info.get("method"), "starts": int(len(info["c_max"])),
                    "feasible_starts": int((info["c_max"] < 1e-6).sum()), "cost": float(info["cost"][info["best"]]),
                    "constraint_residual_max": float(np.abs(p.prob.con(p.solution)).max())}
    # CPU figure for the planner solve: the oracle's shooting adjoint under SciPy's L-BFGS-B with the same augmented-Lagrangian
    # schedule, one core, exp_0 on the C3 grid (what planner_solve_c3_single does on the GPU)
    try:
        import scipy.optimize as so
        from oracle import d2d_oracle as orc
        Nc, hc = 1001, 0.02
        p0c, p1c = np.zeros((3, 1)), np.array([0., 30., np.pi]).reshape(3, 1)
        lamc, rhoc, uc = np.zeros((3, 1)), 10., np.concatenate([np.full(Nc, 0.1), np.full(Nc, 12.)])
        bnds = [(-np.deg2rad(30.), np.deg2rad(30.))] * Nc + [(9., 14.)] * Nc
        spec_c = dict(vsp=12., kvel=1.)

        def fun(u_):
            L_, dphi_, dv_, _, _ = orc.shoot_value_and_grad(u_[None, :Nc], u_[None, Nc:], p0c, p1c, hc, (0., 0.), spec_c, lamc, rhoc, multi=False)
            return L_, np.concatenate([dphi_[0], dv_[0]])
        t0 = _time.perf_counter(); nit = 0; cprev = None
        for _outer in range(30):
            r_ = so.minimize(fun, uc, jac=True, method="L-BFGS-B", bounds=bnds, options=dict(maxiter=500, ftol=1e-15, gtol=1e-10, maxcor=20))
            uc, nit = r_.x, nit + r_.nit
            _, _, _, cost_c, cc = orc.shoot_value_and_grad(uc[None, :Nc], uc[None, Nc:], p0c, p1c, hc, (0., 0.), spec_c, lamc, rhoc, multi=False)
            cm = np.abs(cc).max()
            if cm < 1e-8:
                break
            lamc = lamc + rhoc * cc
            if cprev is None or cm > 0.25 * cprev:
                rhoc = min(rhoc * 3, 1e6)
            cprev = cm
        out["planner_solve_c3_cpu_scipy_1core"] = {"seconds": _time.perf_counter() - t0, "lbfgs_iterations": int(nit), "cost": float(cost_c),
                                                   "constraint_residual_max": float(cm), "kind": "port", "cores": 1}
    except Exception as e:
        out["planner_solve_c3_cpu_scipy_1core"] = {"error": str(e)}
    # a population of planner problems (exp_0 grid, N = 101) with random terminal targets, solved together
    Pp = 4096
    pe = pl.Planner(pl.exp_0)
    p1 = np.stack([rng.uniform(-10, 10, Pp), rng.uniform(28, 40, Pp), np.pi + rng.uniform(-0.5, 0.5, Pp)], 1).reshape(Pp, 3, 1)
    nlp = ShootingNLP(pe.prob, np.zeros((3, 1)), p1, pl.exp_0.phi_constraint, pl.exp_0.v_constraint, P=Pp)
    th0 = nlp.theta_of(np.full((1, pe.num_nodes), 0.1), np.full((1, pe.num_nodes), 12.))
    torch.cuda.synchronize(); t0 = _time.perf_counter()
    _, info = shoot_solve(nlp, th0, ctol=1e-8)
    torch.cuda.synchronize(); dt_pop = _time.perf_counter() - t0
    out["planner_population_4096_first_order"] = {"seconds": dt_pop, "solved": int((info["flag"] == 2).sum()), "problems": Pp, "ticks": int(info["ticks"]),
                                                  "solved_problems_per_s": float((info["flag"] == 2).sum() / dt_pop),
                                                  "median_iterations": float(np.median(info["iterations_each"])), "method": "AL + L-BFGS on the shooting form"}
    del nlp
    from d2d_b200.shooting import solve_ddp
    nlp = ShootingNLP(pe.prob, np.zeros((3, 1)), p1, pl.exp_0.phi_constraint, pl.exp_0.v_constraint, P=Pp)
    solve_ddp(nlp, 0.1, 12., ctol=1e-8)                                   # untimed: module load
    torch.cuda.synchronize(); t0 = _time.perf_counter()
    _, info = solve_ddp(nlp, 0.1, 12., ctol=1e-8)
    torch.cuda.synchronize(); dt_pop = _time.perf_counter() - t0
    out["planner_population_4096"] = {"seconds": dt_pop, "solved": int((info["flag"] == 2).sum()), "problems": Pp,
                                      "solved_problems_per_s": float((info["flag"] == 2).sum() / dt_pop),
                                      "median_iterations": float(np.median(info["iterations_each"])),
                                      "method": "control-limited DDP, one warp per problem (d2dx_ddp_solve)"}
    del nlp
    # pure-pursuit closed loop (SURVEY 8f #4): 4096 aircraft on the square patrol, 1500 steps, 2000 path samples searched per step
    from d2d_b200 import guidance as ddg, trajectory_factory as ddtf
    from d2d_b200.simulation import pursuit_rollout
    ctl = ddg.PurePursuitControler(ddtf.TrajSquare())
    Bq, Tq = 4096, 1500
    X0q = np.tile(np.array([5., -3., 0.3, 0., 10.]), (Bq, 1)); X0q[:, 0] += rng.uniform(-5, 5, Bq)
    ppd = ctl.device_path()
    X0d, wd, acd = eng.to_device(np.ascontiguousarray(X0q.T)), eng.zeros(2, Bq), eng.to_device(np.stack([np.full(Bq, 0.01), np.full(Bq, 1.)]))
    dtq = timed(lambda: eng.rollout_pursuit(ppd, X0d, wd, acd, 0.01, 0, Tq, 1), 3)
    out["pursuit_square_batch4096"] = {"aircraft_steps_per_s": Bq * Tq / dtq, "path_samples": len(ctl.pts_2d), "ms_per_launch": dtq * 1e3,
                                       "distance_evaluations_per_s": Bq * Tq * len(ctl.pts_2d) / dtq}
    # the three-phase mission of 11_full_sim_case1.py (formation until the stop rule, plan, track, two laps of phase 3)
    try:
        import pandas as pd
        from d2d_b200 import mission
        gt = np.load(os.path.join(ROOT, "tests", "golden", "tracker.npz"))
        cols = {"time": gt["inf/time"]}
        for i in range(4):
            cols[f"x_{i + 1}"], cols[f"y_{i + 1}"], cols[f"psi_{i + 1}"] = gt["inf/x_ref"][:, i], gt["inf/y_ref"][:, i], 0 * gt["inf/time"]
        t0 = _time.perf_counter()
        om = mission.full_sim(pd.DataFrame(cols), t_sim_end=150)
        out["mission_case1"] = {"seconds": _time.perf_counter() - t0, "phase1_end_s": float(om["phase1"][5]), "simulated_s": float(om["time"][-1]),
                                "rows": int(len(om["time"]))}
    except Exception as e:                                    # the fixture is test data; the bench line does not depend on it
        out["mission_case1"] = {"error": str(e)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="d2dx", choices=["d2dx", "reference"])
    ap.add_argument("--scenarios", type=int, default=int(os.environ.get("D2DX_BENCH_B", 10 ** 6)), help="aircraft-scenarios per GPU")
    ap.add_argument("--horizon", type=int, default=int(os.environ.get("D2DX_BENCH_T", 10 ** 4)), help="RK4 steps per scenario")
    ap.add_argument("--log-every", type=int, default=100)
    ap.add_argument("--chunks", type=int, default=25, help="launches per sweep (the log rows of a chunk are copied out while the next chunk computes)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--core-only", action="store_true", help="skip the single-GPU extras (planner solves, tracker, pursuit, CPU figures)")
    ap.add_argument("--seed", type=int, default=12345)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed sweep (a fixed sample of the "
                                                          "scenarios, at most 64 MB) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "d2dx":
        ap.error("--dump-outputs applies to the CUDA engine (--impl d2dx)")
    args.warmup = max(args.warmup, 0)
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": "C5 Monte-Carlo sweep: DFFF closed loop on random circles", "scenarios_per_gpu": args.scenarios,
              "rk4_steps": args.horizon, "dt": 0.01, "nsub": 1, "log_every": args.log_every, "parallelism": f"scenario-sharded x{world}",
              "l2_policy": "inputs exceed L2 (>= 176 MB of per-scenario state per sweep; compute-bound kernel)"}

    if args.impl == "reference":
        if rank != 0:
            return
        # bounded sample per step: ~1.5 s per thread-batch; the same population, first scenarios, first 1000 steps
        from oracle import c_oracle as co
        cores = co.max_threads()
        Bc, Tc = 256 * cores, min(1000, args.horizon)
        rates = []
        for k in range(args.warmup + args.steps):
            rate, cores, sample, _ = cpu_port_run(Bc, Tc, args.seed)
            if k >= args.warmup:
                rates.append(rate)
        val = float(np.mean(rates))
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * Bc * Tc / val, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "extrapolated": True,        # a bounded sample of the config's population and horizon is timed; steps/s is size-independent
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "extrapolated": True,
                                 "note": "C port of the oracle (generic 3x3 CARE per step, pthreads); the reference itself is "
                                         "single-threaded Python (366 steps/s/core measured in the survey)"},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return

    # Only the JSON line may reach stdout: libraries (NCCL's version banner, ...) write to fd 1 directly, so fd 1 is pointed
    # at stderr for the whole run and the JSON line goes to a private duplicate of the original stdout.
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback for the engine arm")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    from d2d_b200 import _lib, get_engine
    from d2d_b200.distributed import reduce_population_stats
    from d2d_b200.simulation import MonteCarloRollout

    eng = get_engine()
    B, T_steps = args.scenarios, args.horizon
    time = np.arange(T_steps + 1) * 0.01               # = np.arange(0, (T+1)*0.01, 0.01) sample grid
    w = workload(B, args.seed + rank)
    X0 = flat_state0(w) + w["noise"]
    host_log = not args.no_e2e
    try:
        mc = MonteCarloRollout(B, time, _lib.SEG_CIRCLE, nsub=1, log_every=args.log_every, n_chunks=args.chunks, host_log=host_log)
    except RuntimeError as e:                           # pinned log buffers did not fit: keep the results, drop the host log
        host_log = False
        mc = MonteCarloRollout(B, time, _lib.SEG_CIRCLE, nsub=1, log_every=args.log_every, n_chunks=args.chunks, host_log=False)
        config["host_log"] = f"disabled ({type(e).__name__})"
    par = np.zeros((6, B))
    par[1], par[2], par[3], par[4], par[5] = w["cx"], w["cy"], w["r"], w["v"] / w["r"], w["a0"]
    mc.set_inputs(par, w["wind"], X0)
    mc.upload()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=eng.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    # ---- device-resident throughput (`value`) ----
    for _ in range(args.warmup):
        mc.run_device()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launches
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        evs[k][0].record()
        mc.run_device()
        evs[k][1].record()
    e1.record()
    barrier()
    launches = eng.launches - l0
    ms_total = reduce_max(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    pop = reduce_population_stats(mc.d_pop.clone())
    flags_bad = int(mc.d_flags.ne(0).sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, mc, args.seed)
    ms_per_step = ms_total / max(args.steps, 1)
    total_steps = float(B) * T_steps * world
    value = total_steps / (ms_per_step * 1e-3)
    launches_per_run = mc.launches_per_run
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in evs])) / launches_per_run     # avg duration of ONE launch

    # ---- end-to-end through the host-buffer API (`e2e`) ----
    e2e = None
    if not args.no_e2e:
        mc.run()                                         # warm the copy paths
        barrier()
        t0 = _time.perf_counter()
        n_e2e = max(1, min(args.steps, 3))
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(n_e2e):
            out = mc.run()
        c1.record()
        barrier()
        wall_ms = 1e3 * (_time.perf_counter() - t0)      # run() returns only after every copy has landed
        ms_e2e = reduce_max(max(c0.elapsed_time(c1), wall_ms)) / n_e2e
        e2e = {"value": total_steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(mc.h2d_bytes), "d2h_bytes_per_step": int(mc.d2h_bytes),
               "ms_per_step": ms_e2e, "host_log": host_log, "api": "d2d_b200.simulation.MonteCarloRollout.run (pinned host buffers in/out)"}

    # ---- the same end-to-end sweep with only the STATE log copied out (north_star: "state logs"; the input log stays in HBM) ----
    if e2e is not None and host_log:
        try:
            del mc
            torch.cuda.empty_cache()
            mc = MonteCarloRollout(B, time, _lib.SEG_CIRCLE, nsub=1, log_every=args.log_every, n_chunks=args.chunks, host_log=True, host_log_u=False)
            mc.set_inputs(par, w["wind"], X0)
            mc.run()
            barrier()
            t0 = _time.perf_counter()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(n_e2e):
                mc.run()
            c1.record()
            barrier()
            ms_x = reduce_max(max(c0.elapsed_time(c1), 1e3 * (_time.perf_counter() - t0))) / n_e2e
            e2e["state_log_only"] = {"value": total_steps / (ms_x * 1e-3), "ms_per_step": ms_x, "d2h_bytes_per_step": int(mc.d2h_bytes),
                                     "note": "X log only (5 of the 7 logged doubles per sample); U log left in HBM"}
        except Exception as e:
            e2e["state_log_only"] = {"error": f"{type(e).__name__}: {e}"}
    # ---- the rest of the metric (collocation evals/s, formation, aircraft-sharded C4) on every rank, at every N ----
    hbm_peak = None
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    peak_tf, probe = eng.measure_fp64_peak(details=True)
    core, core_checks = None, {}
    if not args.no_secondary:
        mc = None                                          # the sweep's 6 GB of logs are no longer needed
        torch.cuda.empty_cache()
        try:
            core, core_checks = core_metrics(eng, hbm_peak or 6650.0, peak_tf, world, rank, args.seed)
        except Exception as e:                             # never lose the headline line over a side metric
            core = {"error": f"{type(e).__name__}: {e}"}
    # ---- the host side of `e2e` at this N: every rank copies 1 GiB device -> pinned host at once (what the log copies of
    # MonteCarloRollout.run do); whole-box GB/s = the ceiling of the end-to-end path ----
    d2h_ceiling = None
    if e2e is not None:
        try:
            nb = 1 << 30
            dsrc = torch.empty(nb // 8, dtype=torch.float64, device=eng.device).normal_()
            hdst = torch.empty(nb // 8, dtype=torch.float64).pin_memory()
            best = 1e30
            for _ in range(3):
                barrier()
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(); hdst.copy_(dsrc, non_blocking=True); c1.record(); c1.synchronize()
                best = min(best, reduce_max(c0.elapsed_time(c1)))
            d2h_ceiling = world * nb / (best * 1e-3) / 1e9
            del dsrc, hdst
            e2e["host_d2h_ceiling_gbs"] = d2h_ceiling
            e2e["d2h_floor_ms"] = world * e2e["d2h_bytes_per_step"] / d2h_ceiling / 1e6
            e2e["note"] = ("ms_per_step cannot fall below d2h_floor_ms = all ranks' log bytes / the box's measured concurrent D2H rate "
                           "(host memory / PCIe root, one NUMA node): at 8 GPUs that floor exceeds the compute time")
        except Exception as e:
            e2e["host_d2h_ceiling_error"] = f"{type(e).__name__}: {e}"
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (rollout_dfff_kernel<CIRCLE>) ----
    steps_per_launch = float(B) * (T_steps / launches_per_run)
    ach_tf = steps_per_launch * FP64_FLOP_PER_STEP / (kernel_ms * 1e-3) / 1e12
    log_bytes = steps_per_launch / args.log_every * LOG_BYTES_PER_LOGGED_SAMPLE
    roofline = {"bound": "fp64", "kernel": "rollout_dfff_kernel<CIRCLE>", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": ach_tf / peak_tf, "peak_source": "DFMA probe kernel timed in this run (MEASURED_PEAKS.json has no fp64 figure); nominal 148 SM x 64 FMA x 2 x 1.965 GHz = 37.2",
                "peak_probe": probe,
                "flop_per_aircraft_step": FP64_FLOP_PER_STEP, "kernel_ms": kernel_ms, "steps_per_launch": steps_per_launch,
                "traffic": NCU_TRAFFIC_BYTES_DEFAULT_LAUNCH if (B, T_steps, args.log_every, args.chunks) == NCU_TRAFFIC_CONFIG else None,
                "traffic_note": "ncu dram bytes of one launch at the default sizes (profiles/r2i_rollout_dfff_circle.md); algorithmic bytes = log_bytes_per_launch",
                "fp64_pipe_active_ncu": NCU_FP64_PIPE_ACTIVE, "log_bytes_per_launch": log_bytes,
                "hbm": {"achieved_gbs": log_bytes / (kernel_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak or 6650.0,
                        "peak_source": "measured (MEASURED_PEAKS.json)" if hbm_peak else "fallback"}}
    cpu = None
    if not args.no_cpu and world == 1:               # reported baseline: rank 0 at N = 1 only
        from oracle import c_oracle as co
        cores = co.max_threads()
        rate, cores, sample, _ = cpu_port_run(512 * cores, min(1000, T_steps), args.seed)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "extrapolated": True,
               "python_port_1core": python_port_rate()}
    secondary = core
    if not args.no_secondary and world == 1 and not args.core_only:
        try:
            secondary = {**(core or {}), **secondary_metrics(eng, hbm_peak or 6650.0)}
        except Exception as e:                          # never lose the headline line over a side metric
            secondary = {**(core or {}), "extended_error": f"{type(e).__name__}: {e}"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "secondary": secondary,
            "checks": {**core_checks, "nonfinite_or_unconverged_scenarios": flags_bad, "population_rms_pos_err": float(np.sqrt(pop[0].item() / (B * world * (T_steps + 1)))),
                       "population_max_pos_err": float(pop[1].item())}}
    json_out.write(json.dumps(line) + "\n")
    json_out.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
