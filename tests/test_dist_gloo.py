"""CPU, world_size 2 over gloo: the sharding / merge-schedule logic of dist.ShardedTrainer, with the C oracle plugged in
as the compute backend (the CUDA Engine is the product backend; the host logic under test is identical)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class OracleEngine:
    """Adapter giving the oracle the slice of engine.Engine's interface that ShardedTrainer uses."""

    def __init__(self, compiled, n_local, device=None):
        import oracle as O

        self.o = O.Oracle(compiled, n_local, "f32")
        self.q = torch.from_numpy(self.o.q)  # shares memory with the oracle's table

    def reset(self):
        self.o.reset()

    def train(self, n_iters, learn=True, t0=0):
        self.o.train(t0, n_iters, learn=learn)

    def stats_numpy(self):
        return self.o.stats

    def total_active_steps(self):
        return self.o.total_active_steps()


def _worker(rank, world, port, shared, out_dir):
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import multiagent_rlrm_b200 as P
    from multiagent_rlrm_b200.dist import ShardedTrainer

    sc = P.scenario_config5(shared=shared)
    tr = ShardedTrainer(sc, 37, sync_every=8 if shared else None, engine_factory=lambda c, n, d: OracleEngine(c, n))
    tr.reset()
    tr.train(21)
    tr.train(19)
    counters = tr.global_counters()
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), q=tr.engine.o.q, slot=tr.engine.o.slot, offset=tr.offset, n=tr.n_local,
             counters=np.array(counters), syncs=tr.syncs)
    dist.destroy_process_group()


def _free_port():
    """A port nothing listens on now, so that runs sharing a host do not collide on a fixed rendezvous port."""
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(shared, tmp_path):
    mp.spawn(_worker, args=(2, _free_port(), shared, str(tmp_path)), nprocs=2, join=True)
    return [np.load(os.path.join(tmp_path, f"r{r}.npz")) for r in range(2)]


def test_shard_ranges_cover_everything():
    from multiagent_rlrm_b200.dist import shard_range

    for n, w in ((37, 2), (65536, 8), (5, 4), (1048576, 8)):
        spans = [shard_range(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and sum(c for _, c in spans) == n
        for (o0, c0), (o1, _c1) in zip(spans, spans[1:]):
            assert o0 + c0 == o1


def test_sharded_per_instance_tables_equal_single_process(tmp_path):
    """No collective on the data path: the union of two shards == one process running all 37 instances."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    parts = _run(False, tmp_path)
    sc = P.scenario_config5(shared=False)
    o = O.Oracle(P.compile_scenario(sc), 37, "f32")
    o.reset()
    o.train(0, 40)
    assert [int(p["offset"]) for p in parts] == [0, 19] and [int(p["n"]) for p in parts] == [19, 18]
    assert np.array_equal(np.concatenate([p["slot"] for p in parts]), o.slot)
    assert np.array_equal(np.concatenate([p["q"] for p in parts]), o.q)
    total = (o.total_active_steps(), int(o.stats["episodes"].sum()), int(o.stats["successes"].sum()))
    assert tuple(parts[0]["counters"]) == total == tuple(parts[1]["counters"])


def test_shared_learner_replicas_are_averaged_every_k(tmp_path):
    """Shared learner: replicas diverge between merges and are identical right after one (t = 40 is a multiple of 8)."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    parts = _run(True, tmp_path)
    assert np.array_equal(parts[0]["q"], parts[1]["q"])
    assert int(parts[0]["syncs"]) == 5 == int(parts[1]["syncs"])
    # restate the schedule in one process: two replicas, averaged every 8 iterations
    sc = P.scenario_config5(shared=True)
    reps = [O.Oracle(P.compile_scenario(sc, instance_offset=off), n, "f32") for off, n in ((0, 19), (19, 18))]
    for r in reps:
        r.reset()
    for t0 in range(0, 40, 8):
        for r in reps:
            r.train(t0, 8)
        mean = (reps[0].q + reps[1].q) / np.float32(2)
        for r in reps:
            r.q[...] = mean
    assert np.array_equal(parts[0]["q"], reps[0].q)
    assert np.array_equal(np.concatenate([p["slot"] for p in parts]), np.concatenate([r.slot for r in reps]))
