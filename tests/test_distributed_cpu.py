"""Host-side logic of the multi-GPU plumbing without a GPU: the index maps of an aircraft shard against the oracle, and a
world_size-2 gloo run of the population-statistics reduction and the unit partition."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import d2d_oracle as orc

N_AC, N, H, WIND = 4, 12, 0.1, (0.5, -1.)


def test_aircraft_shard_index_maps_against_oracle():
    """Every rank's shard-local problem (free[idx_free], inst_local), evaluated by the oracle and scattered through idx_con /
    idx_jac, reproduces the residual and compact Jacobian of the whole problem."""
    from d2d_b200.distributed import AircraftShard
    rng = np.random.default_rng(4)
    free = rng.normal(0, 6., 5 * N_AC * N); free[4 * N_AC * N:] += 12.
    inst = [(3 * a + k, 0, 1. + a) for a in range(N_AC) for k in range(3)] + [(3 * a + k, N - 1, -1. - a) for a in range(N_AC) for k in range(3)]
    world = 2
    res_o = orc.colloc_residual(free, N, N_AC, H, WIND, inst)
    jac_o = np.concatenate([orc.colloc_jac_compact(free, N, N_AC, H).reshape(-1), np.ones(len(inst))])
    res, jac = np.full_like(res_o, np.nan), np.full_like(jac_o, np.nan)
    for r in range(world):
        sh = AircraftShard(N_AC, N, inst, world, r)
        fl = free[sh.idx_free]
        res[sh.idx_con] = orc.colloc_residual(fl, N, sh.n_own, H, WIND, sh.inst_local)
        jac[sh.idx_jac] = np.concatenate([orc.colloc_jac_compact(fl, N, sh.n_own, H).reshape(-1), np.ones(len(sh.inst_local))])
    np.testing.assert_allclose(res, res_o, rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(jac, jac_o, rtol=1e-13)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    return port


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from d2d_b200.distributed import reduce_population_stats, shard_range
    pop = torch.tensor([float(rank + 1), float(10 * (rank + 1))], dtype=torch.float64)
    reduce_population_stats(pop)
    ret[rank] = dict(pop=pop.numpy().copy(), rng=shard_range(10, world, rank))
    dist.destroy_process_group()


def test_population_stats_two_ranks_gloo():
    world = 2
    mgr = mp.Manager(); ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    for r in range(world):
        np.testing.assert_array_equal(ret[r]["pop"], [3., 20.])          # sum / max over ranks, on every rank
    assert ret[0]["rng"] == (0, 5) and ret[1]["rng"] == (5, 10)
