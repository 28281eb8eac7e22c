"""Multi-GPU plumbing: one process per GPU, instances sharded by contiguous global index ranges.

SURVEY.md §8(e): environment instances never interact, so the data path needs NO collective. Rank g owns global
instances [offset_g, offset_g + n_g) and compiles its tables with ``instance_offset = offset_g`` so every Philox draw is
keyed on the GLOBAL instance id — the union of the shards is bit-identical to a single-GPU run of the whole batch.

Shared learner (BASELINE config 5, ``scenario.shared_q``): each rank learns into its own replica of the per-agent
tables (include/rlrm_b200.h, "Shared learner") and every ``sync_every`` lockstep iterations the replicas are merged by
parameter averaging: an NCCL all-gather of the 25.6 KB replicas (4 x 400 x 4 floats; latency-bound over NVLink) summed in
rank order, so the merged table does not depend on the collective's reduction order (``merge_replicas``). The reference has no shared learner; this rule is this repo's specification.

The compute backend is injected (``engine_factory``) so the host logic here is testable on CPU with gloo
(tests/test_dist_gloo.py plugs the oracle in); the product default is engine.Engine (CUDA only).
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist

from .tables import Scenario, compile_scenario


def shard_range(n_total: int, rank: int, world: int) -> Tuple[int, int]:
    """(offset, count) of rank's contiguous shard; the first ``n_total % world`` ranks get one extra instance."""
    base, rem = divmod(int(n_total), int(world))
    count = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return offset, count


_gather_buffers = {}


def merge_replicas(q: torch.Tensor, world: int, group=None, engine=None) -> None:
    """q <- (q_0 + q_1 + ... + q_{world-1}) / world, summed in RANK ORDER on every rank. A plain all_reduce(SUM) leaves
    the association order to NCCL's ring/tree, which for more than two ranks changes the last bit; greedy tie-breaks then
    diverge. The tables are tiny (25.6 KB for config 5), so gathering them costs the same latency as reducing them and
    makes the merged table independent of the collective algorithm.

    On the GPU (``engine`` given, NCCL): ONE all-gather into a persistent [world, n] buffer + ONE hand-written rank-ordered
    reduce kernel (rlrm_merge_replicas) — two launches per merge. Without an engine (CPU / gloo tests of the host logic) the
    same sum is formed with torch ops."""
    if engine is not None and q.is_cuda:
        import ctypes as C

        from ._lib import check

        n = q.numel()
        key = (q.device, world, n)
        buf = _gather_buffers.get(key)
        if buf is None:
            buf = _gather_buffers[key] = torch.empty((world, n), dtype=torch.float32, device=q.device)
        dist.all_gather_into_tensor(buf, q.view(-1), group=group)
        check(engine.L.rlrm_merge_replicas(engine.h, buf.data_ptr(), world, n, q.data_ptr(),
                                           C.c_void_p(torch.cuda.current_stream(q.device).cuda_stream)))
        return
    parts = [torch.empty_like(q) for _ in range(world)]
    dist.all_gather(parts, q.contiguous(), group=group)
    acc = parts[0].clone()
    for part in parts[1:]:
        acc.add_(part)
    q.copy_(acc.div_(world))


def _default_engine_factory(compiled, n_local, device, **kw):
    from .engine import Engine

    return Engine(compiled, n_local, device=device, **kw)


class ShardedTrainer:
    def __init__(self, scenario: Scenario, n_instances_total: int, sync_every: Optional[int] = None, device=None,
                 engine_factory: Callable = _default_engine_factory, group=None, sweep=None):
        """sweep: a hyper-parameter sweep over the whole batch (engine.Engine): setting g covers global instances
        [g * n_total / len(sweep), (g + 1) * n_total / len(sweep)). Settings are keyed on the global id, so every rank
        uploads the same list and trains its shard's part of each group."""
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.n_total = int(n_instances_total)
        self.offset, self.n_local = shard_range(self.n_total, self.rank, self.world)
        if self.n_local == 0:
            raise ValueError("more ranks than environment instances")
        self.scenario = scenario
        self.shared = bool(scenario.shared_q)
        self.sync_every = int(sync_every) if (self.shared and sync_every) else 0
        self.compiled = compile_scenario(scenario, instance_offset=self.offset)
        if sweep is None:
            self.engine = engine_factory(self.compiled, self.n_local, device)
        else:
            if self.n_total % len(sweep):
                raise ValueError("n_instances_total must be a multiple of len(sweep)")
            self.engine = engine_factory(self.compiled, self.n_local, device, sweep=sweep, sweep_group=self.n_total // len(sweep))
        self.t = 0
        self.syncs = 0

    def reset(self):
        self.engine.reset()

    def _merge_tables(self):
        """Parameter averaging of the shared-table replicas (the only collective on the learning path)."""
        if self.world > 1:
            eng = self.engine if hasattr(self.engine, "L") and getattr(self.engine.q, "is_cuda", False) else None
            merge_replicas(self.engine.q, self.world, self.group, engine=eng)
        self.syncs += 1

    def train(self, n_iters: int, learn: bool = True):
        """n_iters lockstep iterations on this rank's shard; shared learner: merge every `sync_every` iterations."""
        if not (self.shared and self.sync_every and learn):
            self.engine.train(n_iters, learn=learn, t0=self.t)
            self.t += n_iters
            return
        done = 0
        while done < n_iters:
            to_sync = self.sync_every - (self.t % self.sync_every)
            chunk = min(to_sync, n_iters - done)
            self.engine.train(chunk, learn=learn, t0=self.t)
            self.t += chunk
            done += chunk
            if self.t % self.sync_every == 0:
                self._merge_tables()

    def global_counters(self):
        """(active agent-steps, episodes, successes) summed over all ranks — a counter reduction, not a data-path step."""
        s = self.engine.stats_numpy()
        vals = torch.tensor([int(self.engine.total_active_steps()), int(s["episodes"].sum()), int(s["successes"].sum())], dtype=torch.int64)
        if self.world > 1:
            dev = self.engine.q.device
            vals = vals.to(dev)
            dist.all_reduce(vals, op=dist.ReduceOp.SUM, group=self.group)
            vals = vals.cpu()
        return tuple(int(v) for v in vals)
