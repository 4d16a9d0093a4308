"""Multi-GPU plumbing (one process per GPU, torch.distributed): SURVEY section 8(e).

* Rollouts and batched collocation shard by independent unit (scenario / formation / problem): contiguous
  ranges per rank, NO data-path collective; `reduce_population_stats` is the one final all-reduce.
* One multi-aircraft collocation problem shards by aircraft: the only exchange is the aircraft positions
  (n_ac*N*2 doubles) before the pairwise collision terms and the four cost sums; residual / Jacobian / gradient
  rows stay with the rank that owns the aircraft.  The exchange is done by the evaluation kernel itself through
  NVLink peer memory, so the GPUs of the job must have peer access to each other (one NVLink box)."""
import numpy as np
import torch
import torch.distributed as dist

from . import _lib


def shard_range(n_units, world, rank):
    """Contiguous, balanced partition of n_units independent units: [lo, hi) of this rank."""
    base, rem = divmod(int(n_units), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def reduce_population_stats(pop_stats, group=None):
    """pop_stats = [sum of per-scenario sum_sq_err, max of per-scenario max_err] -> whole-job values."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(pop_stats[0:1], op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(pop_stats[1:2], op=dist.ReduceOp.MAX, group=group)
    return pop_stats


class AircraftShard:
    """Index bookkeeping of one rank's slice of an n_ac-aircraft problem (planner layout, 07_multioptyplan.py:41-47)."""

    def __init__(self, n_ac, N, inst, world, rank):
        self.n_ac, self.N, self.world, self.rank = n_ac, N, world, rank
        self.a_lo, self.a_hi = shard_range(n_ac, world, rank)
        self.n_own = self.a_hi - self.a_lo
        own = range(self.a_lo, self.a_hi)
        blk = lambda b: np.arange(b * N, (b + 1) * N)
        self.idx_free = np.concatenate([blk(3 * a + k) for a in own for k in range(3)] +
                                       [blk(3 * n_ac + a) for a in own] + [blk(4 * n_ac + a) for a in own]) if self.n_own else np.zeros(0, np.int64)
        rblk = lambda e: np.arange(e * (N - 1), (e + 1) * (N - 1))
        n_def = 3 * n_ac * (N - 1)
        self.inst_global = [k for k, (var, _, _) in enumerate(inst) if self.a_lo <= var // 3 < self.a_hi]
        self.inst_local = [(inst[k][0] - 3 * self.a_lo, inst[k][1], inst[k][2]) for k in self.inst_global]
        self.idx_con = np.concatenate([rblk(3 * a + e) for a in own for e in range(3)] + [n_def + np.array(self.inst_global, dtype=np.int64)]) \
            if self.n_own else np.zeros(0, np.int64)
        nnz_def = 12 * n_ac * (N - 1)
        self.idx_jac = np.concatenate([np.arange(12 * a * (N - 1), 12 * (a + 1) * (N - 1)) for a in own] +
                                      [nnz_def + np.array(self.inst_global, dtype=np.int64)]) if self.n_own else np.zeros(0, np.int64)


class ShardedCollocation:
    """Aircraft-sharded evaluation of ONE problem (or a batch of `max_prob` problems) across the ranks of `group`.
    Every rank must own the same number of aircraft.

    ONE kernel per evaluation and rank: positions and cost partials travel as peer-memory stores over NVLink, each value
    tagged with the evaluation number (d2dx_colloc_eval_peer, include/d2dx.h); `graph()` captures it in a CUDA graph.
    connect=True maps every rank's exchange buffer through CUDA IPC over torch.distributed; with connect=False the
    caller connects the exchange objects itself (`emulate_peer_eval`: every rank in one process)."""

    def __init__(self, n_ac, N, h, wind, inst, cost, obj_scale=1., engine=None, group=None, world=None, rank=None,
                 max_prob=1, connect=True):
        from .collocation import CollocationProblem
        from .engine import get_engine
        self.group = group
        self.world = world if world is not None else (dist.get_world_size(group) if dist.is_initialized() else 1)
        self.rank = rank if rank is not None else (dist.get_rank(group) if dist.is_initialized() else 0)
        if n_ac % self.world:
            raise ValueError(f"{n_ac} aircraft do not split evenly over {self.world} ranks")
        self.n_ac, self.N, self.max_prob = n_ac, N, int(max_prob)
        self.shard = AircraftShard(n_ac, N, list(inst), self.world, self.rank)
        self.eng = e = engine or get_engine()
        cost.in_div = n_ac                                   # CostInput normalises by the TOTAL aircraft count
        self.local = CollocationProblem(self.shard.n_own, N, h, wind=wind, inst=self.shard.inst_local, cost=cost,
                                        obj_scale=obj_scale, layout="compact", multi=True, engine=e)
        P = self.max_prob
        self.res = e.empty(P, self.local.num_constraints); self.jac = e.empty(P, self.local.nnz)
        self.grad = e.empty(P, self.local.num_free); self.cost = e.zeros(P)
        self.peer = e.peer_create(self.world, self.rank, P, n_ac, N)
        if connect and self.world > 1:
            handles = [None] * self.world
            dist.all_gather_object(handles, self.peer.ipc_handle(), group=group)
            self.peer.connect_ipc(handles)
            dist.barrier(group=group)                        # nobody launches before every rank has mapped every buffer

    def evaluate(self, free_local, what=_lib.EVAL_ALL):
        """free_local: this rank's slice (device tensor, shard-local planner layout), (num_free_local,) or
        (n_prob, num_free_local).  Returns (residual_local, jac_local, cost_total, grad_local) as device tensors (leading
        problem axis only for 2-D input)."""
        single = free_local.dim() == 1
        n_prob = 1 if single else free_local.shape[0]
        self.eng.colloc_eval_peer(self.peer, self.local.c, n_prob, self.shard.a_lo, free_local, what, self.res, self.jac, self.cost,
                                  self.grad)
        if single:
            return self.res[0], self.jac[0], self.cost[:1], self.grad[0]
        return self.res[:n_prob], self.jac[:n_prob], self.cost[:n_prob], self.grad[:n_prob]

    def graph(self, free_local, what=_lib.EVAL_ALL):
        """Captures one evaluation in a CUDA graph: returns (replay, outputs).  Every rank must replay the same number of
        times."""
        out = self.evaluate(free_local, what)                 # warm-up outside the capture (every rank: one evaluation)
        torch.cuda.synchronize(self.eng.device)
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=self.eng.device)
        with torch.cuda.graph(g, stream=side):
            self.evaluate(free_local, what)
        return g.replay, out

    def check(self):
        """Raises if a peer ever failed to answer (the kernel gives up after ~1 s per wait instead of hanging)."""
        st = self.peer.status()
        if st["timeouts"]:
            raise RuntimeError(f"rank {self.rank}: {st['timeouts']} peer waits timed out; outputs are invalid")
        return st


def emulate_peer_eval(n_ac, N, h, wind, inst, cost, free, world, engine=None, replays=2):
    """The fused peer-memory evaluation with every rank in THIS process on ONE GPU: `world` exchange buffers connected by
    plain pointers, one stream per rank so that the kernels are co-resident and really wait on each other's flags.
    free: (n_prob, 5 n_ac N).  Returns the reassembled global vectors of the last of `replays` evaluations."""
    import copy
    from .engine import get_engine
    eng = engine or get_engine()
    inst = list(inst)
    free = np.asarray(free, dtype=np.float64).reshape(-1, 5 * n_ac * N)
    P = len(free)
    scs = [ShardedCollocation(n_ac, N, h, wind, inst, copy.copy(cost), engine=eng, world=world, rank=r, max_prob=P, connect=False)
           for r in range(world)]
    for sc in scs:
        sc.peer.connect_local([q.peer for q in scs])
    fls = [eng.to_device(np.ascontiguousarray(free[:, sc.shard.idx_free])) for sc in scs]
    streams = [torch.cuda.Stream(device=eng.device) for _ in scs]
    torch.cuda.synchronize(eng.device)
    for _ in range(replays):
        for sc, fl, st in zip(scs, fls, streams):
            with torch.cuda.stream(st):
                sc.evaluate(fl)
    torch.cuda.synchronize(eng.device)
    n_con, nnz = 3 * n_ac * (N - 1) + len(inst), 12 * n_ac * (N - 1) + len(inst)
    out = {"residual": np.zeros((P, n_con)), "jac": np.zeros((P, nnz)), "grad": np.zeros((P, free.shape[1])), "cost": [], "status": []}
    for sc in scs:
        out["residual"][:, sc.shard.idx_con] = sc.res.cpu().numpy()
        out["jac"][:, sc.shard.idx_jac] = sc.jac.cpu().numpy()
        out["grad"][:, sc.shard.idx_free] = sc.grad.cpu().numpy()
        out["cost"].append(sc.cost.cpu().numpy().copy())
        out["status"].append(sc.peer.status())
    return out
