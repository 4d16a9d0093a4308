"""Two-GPU tests (skipped on a single-GPU box): the aircraft-sharded collocation evaluation (fused peer-memory kernel over
NVLink and its CUDA-graph replay, against the unsharded evaluation), and scenario-sharded rollouts with the final statistics
reduction."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    return port


def _worker(rank, world, port, free, inst, ret):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), LOCAL_RANK=str(rank), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from d2d_b200 import get_engine, simulation, trajectory
    from d2d_b200.collocation import CostSpec
    from d2d_b200.distributed import ShardedCollocation, reduce_population_stats, shard_range
    eng = get_engine()
    cs = CostSpec(vsp=12., kvel=70., kbank=1., kcol=10., rcol=10., all_pairs=True, kobs=0.5, obstacles=[(60., 5., 12.)], obs_kind=1)
    import copy
    sc = ShardedCollocation(16, 500, 0.02, (0., 0.), inst, copy.copy(cs), engine=eng)            # fused peer-memory kernel (NVLink)
    fl = eng.to_device(free[sc.shard.idx_free])
    res, jac, cost, grad = (t.clone() for t in sc.evaluate(fl))
    replay, outs = sc.graph(fl)                                                                  # the same, replayed from a CUDA graph
    for _ in range(5):
        replay()
    torch.cuda.synchronize()
    st = sc.check()
    assert st["evaluations"] == 7, st      # 1 eager + 1 warm-up before the capture + 5 replays
    for a_, b_ in zip(outs, (res, jac, cost, grad)):
        assert torch.equal(a_, b_)
    # a batch larger than the co-resident grid (160 problems x 16 tiles = 2560 items; 12 blocks x 148 SMs are resident): the
    # persistent item loop of the fused kernel, every rank against its own unsharded evaluation of the same batch
    from d2d_b200.collocation import CollocationProblem
    PB = 160
    rngb = np.random.default_rng(99)
    freeB = free[None] + rngb.normal(0, 0.3, (PB, free.size))
    scB = ShardedCollocation(16, 500, 0.02, (0., 0.), inst, copy.copy(cs), engine=eng, max_prob=PB)
    flB = eng.to_device(np.ascontiguousarray(freeB[:, scB.shard.idx_free]))
    rB, jB, cB, gB = scB.evaluate(flB)
    rB, jB, cB, gB = (t.clone() for t in scB.evaluate(flB))                                      # second evaluation: next epoch, same answer
    assert scB.check()["timeouts"] == 0
    fullB = CollocationProblem(16, 500, 0.02, inst=inst, cost=copy.copy(cs), engine=eng)
    ob = fullB.evaluate_device(eng.to_device(freeB))
    dev = lambda idx: torch.from_numpy(idx).to(eng.device)
    assert float((rB - ob["res"][:, dev(scB.shard.idx_con)]).abs().max()) < 1e-13
    assert torch.allclose(jB, ob["jac"][:, dev(scB.shard.idx_jac)], rtol=1e-14, atol=0)
    assert torch.allclose(gB, ob["grad"][:, dev(scB.shard.idx_free)], rtol=1e-12, atol=1e-15)
    assert torch.allclose(cB, ob["cost"], rtol=1e-13, atol=0)
    # scenario-sharded rollout: each rank its contiguous half of 64 circles, then the one final all-reduce
    rng = np.random.default_rng(0)
    B = 64
    cx, cy, r, v, a0 = rng.uniform(-50, 50, B), rng.uniform(-50, 50, B), rng.uniform(30, 60, B), rng.uniform(10, 12, B), rng.uniform(0, 6, B)
    X0 = np.stack([cx + r * np.cos(a0), cy + r * np.sin(a0), a0 + np.pi / 2, 0 * a0, v], 1)
    lo, hi = shard_range(B, world, rank)
    out = simulation.rollout(np.arange(0, 2., 0.01), trajectory.CircleBatch(cx[lo:hi], cy[lo:hi], r[lo:hi], v[lo:hi], a0[lo:hi]),
                             [0., 0.], X0[lo:hi], return_log=False)
    pop = eng.to_device(np.array([out.pop_sum_sq_err, out.pop_max_err]))
    reduce_population_stats(pop)
    torch.cuda.synchronize()
    ret[rank] = dict(res=res.cpu().numpy(), jac=jac.cpu().numpy(), cost=float(cost.cpu()[0]), grad=grad.cpu().numpy(),
                     idx_free=sc.shard.idx_free, idx_con=sc.shard.idx_con, idx_jac=sc.shard.idx_jac,
                     pop=pop.cpu().numpy(), local=(out.pop_sum_sq_err, out.pop_max_err))
    dist.destroy_process_group()


def test_two_gpu_sharded_collocation_and_rollout(golden):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = max(w for w in (2, 4, 8) if w <= torch.cuda.device_count())      # C4 on 8 GPUs = 2 aircraft per rank
    import torch.multiprocessing as mp
    from d2d_b200.collocation import CollocationProblem, CostSpec
    g = golden["colloc"]
    free = g["c4/free"]
    inst = [(int(k), int(n), v) for (k, n, v) in g["c4/inst"]]
    mgr = mp.Manager(); ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), free, inst, ret), nprocs=world, join=True)
    cs = CostSpec(vsp=12., kvel=70., kbank=1., kcol=10., rcol=10., all_pairs=True, kobs=0.5, obstacles=[(60., 5., 12.)], obs_kind=1)
    full = CollocationProblem(16, 500, 0.02, inst=inst, cost=cs)
    res, jac, cost, grad = full.evaluate(free)
    R, J, G = np.full_like(res, np.nan), np.full_like(jac, np.nan), np.full_like(grad, np.nan)
    for r in range(world):
        o = ret[r]
        R[o["idx_con"]] = o["res"]; J[o["idx_jac"]] = o["jac"]; G[o["idx_free"]] = o["grad"]
        np.testing.assert_allclose(o["cost"], cost, rtol=1e-13)
    np.testing.assert_array_equal(R, res); np.testing.assert_array_equal(J, jac)
    np.testing.assert_allclose(G, grad, rtol=1e-14, atol=1e-16)
    np.testing.assert_allclose(ret[0]["pop"][0], sum(ret[r]["local"][0] for r in range(world)), rtol=1e-13)
    assert ret[0]["pop"][1] == max(ret[r]["local"][1] for r in range(world)) and np.array_equal(ret[0]["pop"], ret[world - 1]["pop"])
