#!/usr/bin/env python
"""bench.py — agent-steps/sec (env step + RM transition + Q update) of the fused lockstep kernel.

Workload (BASELINE.json configs[2]): 65,536 batched FrozenLake map1 instances x 2 agents PER GPU, slippery (80/10/10),
built-in A->B->C reward machine, per-instance Q tables (QLearning lr=1, gamma=.99, eps=.01, init 2, use_qrm=True — the
reference driver's learner). One bench "step" = one fused launch of `--iters` lockstep iterations over the whole batch.
Multi-GPU (`torchrun`, one rank per GPU) shards independent instances: no data-path collective, weak scaling.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--iters T] [--instances N] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (see the keys in main()). Besides the headline it carries: `configs` (every other BASELINE configuration,
measured in the same run: config 3 on float64 tables, config 2 batched, config 4 sparse-exact / dense-faithful, config 5 with
per-instance tables and with the shared learner — 1,048,576 instances in TOTAL sharded over the ranks, K sweep and merge time at
N > 1), `e2e` (host buffers through rlrm_train_host), `e2e_call_by_call` (one launch per driver-loop iteration, rlrm_iterate),
`dropin_n1` (BASELINE configs[0] through the reference's driver loop on the N = 1 drop-in classes next to the live Python
reference), `roofline` (frac = algorithmic bytes, dram_frac = ncu DRAM bytes, bound per workload) and `cpu_baseline` (the C port
and the live Python reference on the box's host cores). `--workload` runs any single workload of WORKLOADS as the headline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "agent-steps/sec (env+RM+Q update)"
UNIT = "agent-steps/s"
# algorithmic bytes per active agent-step (SURVEY.md §8d): QRM nQ=4: cell block s 64 + cell block s' 64 + 3 writes x 4 B
# = 140; plain QL: Q[s,:] 16 + Q[s',:] 16 + 4 = 36; dense Q(lambda): (q + e) read + write = 4 * S*A * 4 B


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS),
                    help="cfg3 = the headline (BASELINE configs[2]); the others are extra measured lines")
    ap.add_argument("--iters", type=int, default=None, help="lockstep iterations per launch (= per bench step)")
    ap.add_argument("--instances", type=int, default=None, help="environment instances per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=None,
                    help="target CPU time of one CPU sample (default: 12 s for cpu_baseline, 60 s / steps for --impl reference)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (the other BASELINE configurations)")
    ap.add_argument("--no-call-by-call", action="store_true", help="skip the per-iteration API measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline engine's state (Q tables, slot words, epsilon, episode "
                         "statistics) for a fixed sample of instances to DIR/<name>.npy; with several ranks, rank 0's instances")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed; it needs --impl b200")
    return args


# name -> (description, BASELINE config, default instances/GPU, default iters/launch, algorithmic bytes per active
#          agent-step (SURVEY.md §8d), dominant kernel)
WORKLOADS = {
    "cfg3": ("FrozenLake map1 (10x10), 2 agents, slippery 80/10/10, RM A->B->C (10/15/20), QLearning lr=1 gamma=.99 eps=.01 "
             "init=2 use_qrm=True, per-instance Q tables, auto-reset",
             "configs[2]: 65,536 batched FrozenLake map1 instances x 2 agents, slippery, per-instance Q-tables",
             65536, 2048, 140, "train_qrm4_kernel<FrozenLake>"),
    "cfg3_ql": ("FrozenLake map1, 2 agents, slippery, RM A->B->C, QLearning lr=.1 gamma=.99 eps=.01 init=2 use_qrm=False, "
                "per-instance Q tables, auto-reset",
                "configs[2] companion (plain Q-learning variant, SURVEY.md §8d)", 65536, 2048, 36, "train_ql_fast_kernel<FrozenLake>"),
    "cfg3_f64": ("FrozenLake map1 (10x10), 2 agents, slippery 80/10/10, RM A->B->C (10/15/20), QLearning lr=1 gamma=.99 eps=.01 "
                 "init=2 use_qrm=True, per-instance Q tables in FLOAT64 (the reference's own np.zeros arithmetic: bit-identical to the "
                 "unmodified reference), auto-reset",
                 "configs[2] on the reference's native float64 tables", 65536, 2048, 2 * 128 + 3 * 8, "train_qrm_block_kernel<FrozenLake,double>"),
    "cfg3_ql_f64": ("FrozenLake map1, 2 agents, slippery, RM A->B->C, QLearning lr=.1 gamma=.99 eps=.01 init=2 use_qrm=False, "
                    "per-instance Q tables in FLOAT64, auto-reset",
                    "configs[2] companion (plain Q-learning) on float64 tables", 65536, 2048, 32 + 32 + 8, "train_kernel<FrozenLake,QL,double>"),
    "cfg2_batch": ("OfficeWorld map1 (12x9), 1 agent at (2,7), slip hp=.8, RM 'A -> C -> B -> D, reward on D' (5 states, the --rm-spec "
                   "fixture of configs[1]), QLearning lr=.1 gamma=.9 eps=.1 init=2 use_qrm=False, per-instance Q tables, auto-reset",
                   "configs[1] batched (the reference case itself is N=1 and is a parity test, not a bench line)",
                   131072, 2048, 36, "train_ql_fast_kernel<OfficeWorld>"),
    "cfg2_batch_qrm": ("OfficeWorld map1 (12x9), 1 agent at (2,7), slip hp=.8, RM 'A -> C -> B -> D, reward on D' (5 states), QLearning "
                       "lr=.1 gamma=.9 eps=.1 init=2 use_qrm=True, per-instance Q tables, auto-reset",
                       "configs[1] batched, QRM variant", 131072, 2048, 2 * 5 * 16 + 4 * 4, "train_qrmn_kernel<OfficeWorld,5>"),
    "cfg4": ("OfficeWorld map1 (12x9), 4 agents, slip hp=.8, plants -100, synthetic 12-state completed chain RM (108 "
             "transitions), QLearningLambda gamma=.9 lambda=.9 lr=.1 eps=.1 init 0, SPARSE-EXACT traces (live entries only; "
             "bit-identical to the dense sweep)",
             "configs[3]: OfficeWorld 12-state RM, 262,144 instances x 4 agents, Q(lambda) traces",
             262144, 64, None, "train_qlambda_sparse_kernel<OfficeWorld>"),
    "cfg4_dense": ("OfficeWorld map1 (12x9), 4 agents, slip hp=.8, plants -100, synthetic 12-state completed chain RM (108 "
                   "transitions), QLearningLambda gamma=.9 lambda=.9 lr=.1 eps=.1 init 0, dense-faithful trace sweep",
                   "configs[3]: OfficeWorld 12-state RM, 262,144 instances x 4 agents, Q(lambda) traces",
                   262144, 4, 4 * 1296 * 4 * 4, "train_qlambda_kernel<OfficeWorld>"),
    "cfg4_qrm": ("OfficeWorld map1 (12x9), 4 agents, slip hp=.8, plants -100, synthetic 12-state completed chain RM, QLearning "
                 "lr=.1 gamma=.9 eps=.1 init=2 use_qrm=True (11 counterfactual updates per step), per-instance Q tables",
                 "configs[3]'s environment and reward machine with the QRM learner (generic / lane-group QRM kernel for nQ > 5)",
                 65536, 512, 2 * 12 * 16 + 4 * 11, "train_qrm_block_kernel<OfficeWorld,12>"),
    "ow_exp6_qrm": ("OfficeWorld map1 built-in task exp6 (A-B-C-D-E then coffee + e-mail to office, 10 RM states), 2 agents at "
                    "(2,7),(6,3), slip hp=.8, QLearning lr=.1 gamma=.9 eps=.1 init=2 use_qrm=True, per-instance Q tables",
                    "office_main --experiment exp6 batched (not a BASELINE configuration; the largest built-in machine)",
                    65536, 1024, 2 * 10 * 16 + 4 * 9, "train_qrm_block_kernel<OfficeWorld,10>"),
    "ow12_shared": ("OfficeWorld map1 (12x9), 2 agents at (2,7),(6,3), slip hp=.8, synthetic 12-state completed chain RM, QLearning lr=.1 "
                    "gamma=.9 eps=.1 init=2 use_qrm=True, ONE table per agent index per GPU (shared learner; 10,368 entries: 218 KB of "
                    "tables + accumulators in shared memory)",
                    "configs[3]'s environment and machine with configs[4]'s shared learner (not a BASELINE configuration)",
                    262144, 64, 2 * 12 * 16 + 4 * 11, "shared_train_kernel<OfficeWorld,QRM> (persistent cooperative; shared-memory wavefront bound)"),
    "ow12x4_shared": ("OfficeWorld map1 (12x9), 4 agents, slip hp=.8, synthetic 12-state completed chain RM, QLearning lr=.1 gamma=.9 eps=.1 "
                      "init=2 use_qrm=True, ONE table per agent index per GPU (shared learner; 20,736 entries = 435 KB of tables + "
                      "accumulators: partitioned over the distributed shared memory of 2-block clusters)",
                      "configs[3]'s environment, machine and agent count with configs[4]'s shared learner (not a BASELINE configuration)",
                      262144, 64, 2 * 12 * 16 + 4 * 11, "shared_train_cluster_kernel<OfficeWorld,QRM,2> (persistent cooperative, DSMEM)"),
    "cfg5_tables": ("FrozenLake map1, 4 agents, slippery, RM A->B->C, QLearning use_qrm=True, per-instance Q tables",
                    "configs[4] HBM-bound companion: 1M FrozenLake instances x 4 agents, per-instance tables",
                    1048576, 256, 140, "train_qrm4_kernel<FrozenLake>"),
    "cfg5_shared": ("FrozenLake map1, 4 agents, slippery, RM A->B->C, QLearning use_qrm=True, ONE table per agent index per GPU "
                    "(shared learner, synchronous proposal averaging), all-reduced every 64 iterations",
                    "configs[4]: 1M FrozenLake instances x 4 agents, shared-learner Q-table allreduce over NVLink every K steps",
                    1048576, 64, 140, "shared_propose_kernel<FrozenLake,QRM> + apply_shared_kernel (shared-memory wavefront bound, not HBM)"),
}


def scenario(workload):
    import multiagent_rlrm_b200 as P

    def cfg2(qrm):
        sc = P.scenario_config2(True)
        sc.algo = "qrm" if qrm else "ql"
        return sc

    def cfg4_qrm():
        sc = P.scenario_config4()
        sc.algo, sc.learning_rate, sc.q_init = "qrm", 0.1, 2.0
        return sc

    def exp6():
        return P.scenario_for_experiment("map1", "exp6", starts=[(2, 7), (6, 3)], algo="qrm", learning_rate=0.1, gamma=0.9,
                                         stochastic=True, high_prob=0.8, epsilon_start=0.1, epsilon_end=0.1, epsilon_decay=1.0,
                                         q_init=2.0, seed=1234)

    def ow12_shared():
        sc = cfg4_qrm()
        sc.starts, sc.shared_q = sc.starts[:1] + [(6, 3)], True
        return sc

    def ow12x4_shared():
        sc = cfg4_qrm()
        sc.shared_q = True
        return sc

    def f64(sc):
        sc.table_dtype = "f64"
        return sc

    return {"cfg3_f64": lambda: f64(P.scenario_config3(True)), "cfg3_ql_f64": lambda: f64(P.scenario_config3(False)),
            "ow12_shared": ow12_shared, "ow12x4_shared": ow12x4_shared, "cfg3": lambda: P.scenario_config3(True), "cfg3_ql": lambda: P.scenario_config3(False),
            "cfg2_batch": lambda: cfg2(False), "cfg2_batch_qrm": lambda: cfg2(True),
            "cfg4": P.scenario_config4, "cfg4_dense": P.scenario_config4, "cfg4_qrm": cfg4_qrm, "ow_exp6_qrm": exp6, "cfg5_tables": lambda: P.scenario_config5(False),
            "cfg5_shared": lambda: P.scenario_config5(True)}[workload]()


def resolve_defaults(args):
    w = WORKLOADS[args.workload]
    if args.instances is None:
        args.instances = w[2]
    if args.iters is None:
        args.iters = w[3]
    return args


def workload_config(args, world):
    desc, base, _n, _t, _b, _k = WORKLOADS[args.workload]
    sc = scenario(args.workload)
    agents = len(sc.starts)
    g = sc.grid()
    n_rm = sc.reward_machine().numbers_state()
    table_bytes = g.width * g.height * n_rm * 4 * (8 if sc.table_dtype == "f64" else 4) * (2 if sc.algo == "qlambda" else 1)
    per_gpu = table_bytes * agents * (1 if sc.shared_q else args.instances)
    return {
        "workload": desc,
        "baseline_config": base,
        "instances_per_gpu": args.instances,
        "agents": agents,
        "iters_per_step": args.iters,
        "table_bytes_per_gpu": per_gpu,
        "l2_policy": ("inputs larger than L2 (%.1f GB of tables per GPU vs 126 MB L2); no explicit flush" % (per_gpu / 1e9))
                     if per_gpu > 126e6 else "tables are L2-resident by design (shared learner); state arrays are streamed",
        "sharding": f"independent instances, {world} rank(s), "
                    + ("shared tables merged every 64 iterations (NCCL all_gather_into_tensor + rank-ordered reduce kernel)"
                       if sc.shared_q else "no data-path collective"),
    }


# --------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (the reference is pure Python and does not travel to the GPU box; oracle/rlrm_oracle.c is
# its plain-C restatement, pinned bit-exactly to the live reference by tests/golden)
# --------------------------------------------------------------------------------------------------------------------
def _cpu_worker(job):
    algo, n_inst, iters, offset = job  # `algo` is the workload name
    import multiagent_rlrm_b200 as P
    import oracle as O

    c = P.compile_scenario(scenario(algo), instance_offset=offset)
    o = O.Oracle(c, n_inst, scenario(algo).table_dtype)
    o.reset()
    t0 = time.perf_counter()
    o.train(0, iters)
    dt = time.perf_counter() - t0
    return o.total_active_steps(), n_inst * c.n_agents * iters, dt


def cpu_port_throughput(algo, seconds, procs):
    """All `procs` host cores, each an independent batch of instances through the C oracle (the only way the reference
    'batches' is independent processes, BASELINE.md §3)."""
    import multiprocessing as mp

    import oracle as O

    O.build()
    # calibrate one core
    import multiagent_rlrm_b200 as P

    agents = len(scenario(algo).starts)
    heavy = scenario(algo).algo == "qlambda"  # dense trace sweep: ~1e4x more work per step
    a, s, dt = _cpu_worker((algo, 8 if heavy else 256, 16 if heavy else 256, 0))
    rate = s / max(dt, 1e-6)  # slot-steps/s/core
    iters = 32 if heavy else 512
    n_inst = max(4, int(rate * seconds / (iters * agents)))
    jobs = [(algo, n_inst, iters, k * n_inst) for k in range(procs)]
    t0 = time.perf_counter()
    if procs > 1:
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    else:
        res = [_cpu_worker(jobs[0])]
    wall = time.perf_counter() - t0
    active = sum(r[0] for r in res)
    slots = sum(r[1] for r in res)
    busy = max(r[2] for r in res)
    return {
        "value": active / busy,
        "unit": UNIT,
        "cores": procs,
        "kind": "port",
        "sample": f"{procs} process(es) x {n_inst} instances x {agents} agents x {iters} iterations of the same workload through "
                  f"oracle/rlrm_oracle.c (float32 tables); {slots / busy:.3e} slot-steps/s; wall {wall:.1f}s",
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    per_step = args.cpu_seconds if args.cpu_seconds else max(1.0, min(10.0, 60.0 / max(1, args.steps + args.warmup)))
    vals, last = [], None
    for k in range(args.warmup + args.steps):
        last = cpu_port_throughput(args.workload, per_step, procs)
        if k >= args.warmup:
            vals.append(last["value"])
    value = sum(vals) / len(vals)
    last["value"] = value
    last["reference_python"] = reference_python_throughput(args.workload, min(8.0, max(1.0, per_step)), procs)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": scenario(args.workload).table_dtype, "data": "synthetic", "config": workload_config(args, 1), "cpu_baseline": last,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference is pure Python/NumPy (≈1e4 agent-steps/s/core, BASELINE.md §2) and cannot travel to the GPU box; "
                "this arm times its bit-exact plain-C restatement on all host cores",
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = f"/tmp/rlrm_clocks_{os.getpid()}.csv"
        self.proc = None
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.remove(self.path)
        except OSError:
            pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_capture(workload):
    """What the committed ncu --set full capture of this workload's dominant kernel measured (profiles/traffic.json, written by
    profiles/scripts/make_traffic.py from profiles/<round>/*_raw.csv): DRAM bytes per active agent-step, cache hit rates,
    pipe utilisation, the file and commit it came from. NOT measured in this run (ncu cannot run inside a timed bench)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(workload)
    except Exception:
        return None


# what bounds the dominant kernel of each workload (ncu evidence under profiles/, DESIGN.md section 6); `frac` is always
# computed against the HBM peak with SURVEY 8d's algorithmic bytes — it is an HBM-utilisation figure only where bound = hbm
BOUND = {
    "cfg3": "issue/latency (carried cell block: most algorithmic bytes never leave registers; issue slots 58 %, DRAM 27 % of peak)",
    "cfg3_ql": "latency (one dependent 16-byte gather per step at 6.9 warps per scheduler)",
    "cfg3_f64": "latency (128-byte cell block fetched after every move) / fp64 pipe",
    "cfg3_ql_f64": "latency (one dependent 32-byte gather per step)",
    "cfg2_batch": "latency (one dependent 16-byte gather per step)",
    "cfg2_batch_qrm": "latency on the row loads after a move, then L1 wavefronts",
    "cfg4": "issue (trace lists stay L1/L2-resident)",
    "cfg4_dense": "hbm",
    "cfg4_qrm": "smem-latency (cell block in shared memory, fetched by one TMA bulk copy per thread + mbarrier: short scoreboard 47 % of the stalls, L1 wavefront pipe 52 %)",
    "ow_exp6_qrm": "smem-wavefront (cell block in shared memory: short scoreboard 50 % of the stalls, L1 wavefront pipe 73 %), then the block fetch after a move",
    "cfg5_tables": "issue/latency",
    "cfg5_shared": "smem-wavefront (random 16-byte shared-memory gathers + proposal atomics); tables live on chip, not HBM",
    "ow12_shared": "smem-wavefront (random 16-byte shared-memory gathers + proposal atomics); tables live on chip, not HBM",
    "ow12x4_shared": "distributed-shared-memory latency / wavefronts (half of the row gathers and proposal atomics go to the peer SM); tables live on chip, not HBM",
}


class Runner:
    """One workload on this rank's GPU: engine, optional shared-learner merge schedule, device-timed steps, e2e on host buffers."""

    def __init__(self, workload, instances, iters, rank, world, dev, offset=None, sync_every=0):
        import multiagent_rlrm_b200 as P
        from multiagent_rlrm_b200.engine import Engine

        self.workload, self.instances, self.iters, self.world, self.dev = workload, instances, iters, world, dev
        self.sc = scenario(workload)
        self.c = P.compile_scenario(self.sc, instance_offset=rank * instances if offset is None else offset)  # Philox keyed on the GLOBAL instance id
        self.eng = Engine(self.c, instances, device=dev, qlambda_sparse=(workload == "cfg4"))
        self.eng.reset()
        self.n_slots = instances * self.c.n_agents
        self.sync_every = sync_every if (self.sc.shared_q and world > 1) else 0
        self.merge_events = []

    def train(self, n_iters, timed=False):
        import torch

        from multiagent_rlrm_b200.dist import merge_replicas

        if not self.sync_every:
            self.eng.train(n_iters)
            return
        done = 0
        while done < n_iters:  # shared learner: parameter averaging every sync_every iterations (dist.ShardedTrainer's rule)
            chunk = min(self.sync_every, n_iters - done)
            self.eng.train(chunk)
            done += chunk
            if timed:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            merge_replicas(self.eng.q, self.world, engine=self.eng)
            if timed:
                e1.record()
                self.merge_events.append((e0, e1))

    def barrier(self):
        import torch
        import torch.distributed as dist

        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def run(self, steps, warmup, e2e_steps, rank0_sampler=None, dump_dir=None):
        import torch
        import torch.distributed as dist

        eng = self.eng
        for _ in range(warmup):
            self.train(self.iters)
        self.barrier()
        launches0, steps0 = eng.launches, eng.total_active_steps()
        work0 = int(eng.tr_work.sum()) if eng.sparse else 0
        sampler = rank0_sampler() if rank0_sampler else None
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        self.barrier()
        ev[0].record()
        for k in range(steps):
            self.train(self.iters, timed=True)
            ev[k + 1].record()
        self.barrier()
        clocks = sampler.stop() if sampler else None
        elapsed_ms = ev[0].elapsed_time(ev[-1])
        per_launch_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(steps)]
        merge_ms = [a.elapsed_time(b) for a, b in self.merge_events]
        active = eng.total_active_steps() - steps0
        launches = eng.launches - launches0
        mean_live = ((int(eng.tr_work.sum()) - work0) / max(1, self.n_slots * self.iters * steps)) if eng.sparse else None
        if dump_dir:  # before the e2e window below trains the same engine further
            dump_outputs(eng, dump_dir)

        # ---- end to end: the public API call on HOST (pinned) buffers, copies inside the timed region ----------------
        e2e = None
        if e2e_steps:
            n = self.n_slots
            host_slot = torch.empty(n, dtype=torch.int64).pin_memory()
            host_eps = torch.empty(n, dtype=torch.float64).pin_memory()
            host_stats = torch.empty((n, 32), dtype=torch.uint8).pin_memory()
            host_slot.copy_(eng.slot); host_eps.copy_(eng.epsilon)

            def host_active():  # finished episodes' agent_steps (stats) + running episodes' agent_steps (slot words), on the host
                return int(host_stats.view(torch.int64)[:, 0].sum()) + int(((host_slot >> 16) & 0xFFFF).sum())

            def one():
                if not self.sync_every:
                    eng.train_host(self.iters, host_stats, host_slot, host_eps)
                    return
                from multiagent_rlrm_b200.dist import merge_replicas

                done = 0
                while done < self.iters:
                    chunk = min(self.sync_every, self.iters - done)
                    eng.train_host(chunk, host_stats, host_slot, host_eps)
                    done += chunk
                    merge_replicas(eng.q, self.world, engine=eng)

            one()  # warm
            self.barrier()
            a0 = host_active()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                one()
            torch.cuda.synchronize(self.dev)
            e2e_s = time.perf_counter() - t0
            e2e = {"active": host_active() - a0, "seconds": e2e_s, "steps": e2e_steps, "h2d": host_slot.numel() * 8 + host_eps.numel() * 8,
                   "d2h": host_stats.numel() + host_slot.numel() * 8 + host_eps.numel() * 8}

        merge_total = sum(merge_ms)
        if self.world > 1:
            t = torch.tensor([elapsed_ms, e2e["seconds"] if e2e else 0.0, merge_total], dtype=torch.float64, device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            elapsed_ms, e2e_s_max, merge_total = float(t[0]), float(t[1]), float(t[2])
            cnt = torch.tensor([active, e2e["active"] if e2e else 0, launches], dtype=torch.int64, device=self.dev)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
            active, e2e_active, launches = int(cnt[0]), int(cnt[1]), int(cnt[2])
            if e2e:
                e2e["seconds"], e2e["active"] = e2e_s_max, e2e_active
        return {"elapsed_ms": elapsed_ms, "per_launch_ms": per_launch_ms, "active": active, "launches": launches, "mean_live": mean_live,
                "e2e": e2e, "clocks": clocks, "merge_ms_total": merge_total, "n_merges": len(merge_ms), "steps": steps}


def dump_outputs(eng, out_dir, budget=48 << 20):
    """What a caller of Engine.train holds after the last timed step, as DIR/<name>.npy: the Q tables (table dtype), the decoded
    slot words, epsilon, the running episode return and the episode statistics (integers as exact float64), for a seeded sample
    of instances sized to keep the files under `budget` bytes (all instances when they fit; shared tables are written whole).
    The sample depends only on the instance count and the table shape, so runs with the same arguments write the same
    entries and two builds can be compared file by file. instances.npy holds indices into this engine's own instances: with
    several ranks only rank 0 writes, and its indices are also the global instance ids."""
    import numpy as np
    import torch

    from multiagent_rlrm_b200 import _abi as abi
    from multiagent_rlrm_b200.engine import STATS_DTYPE

    eng.sync_tables()  # sparse Q(lambda) keeps the live q values in its trace lists until they are written back
    N, A = eng.N, eng.A
    shared = bool(eng.cfg.shared_q)
    q_bytes = eng.q.numel() * eng.q.element_size()
    per_instance = (0 if shared else q_bytes // N) + 8 + A * 13 * 8  # its tables, its index, 13 float64 entries per agent slot
    room = budget - 15 * 128 - (q_bytes if shared else 0)  # 15 files, each with a 128-byte .npy header
    n = min(N, max(1, room // per_instance))
    idx = np.arange(N) if n == N else np.sort(np.random.default_rng(0).choice(N, size=n, replace=False))
    it = torch.from_numpy(idx).to(eng.q.device)
    rows = eng.q.shape[1:]  # per-instance tables are stored instance-major: (N * A, S, 4), or (N, rows, 4) with per-agent machines
    q = eng.q if shared else eng.q.reshape(N, -1, *rows)[it].reshape(-1, *rows)
    slot = eng.slot.view(N, A)[it].cpu().numpy().view(np.uint64)
    stats = eng.stats.view(N, A, 32)[it].cpu().numpy().reshape(-1).view(STATS_DTYPE).reshape(n, A)
    out = {"instances": idx, "q": q.cpu().numpy(),
           "epsilon": eng.epsilon.view(N, A)[it].cpu().numpy(), "ep_return": eng.ep_return.view(N, A)[it].cpu().numpy()}
    for name, shift, mask in (("cell", abi.SLOT_CELL_SHIFT, 0xFFFF), ("agent_steps", abi.SLOT_STEPS_SHIFT, 0xFFFF),
                              ("timestep", abi.SLOT_TIME_SHIFT, 0xFFFF), ("rm_state", abi.SLOT_RMSTATE_SHIFT, 0xFF),
                              ("flags", abi.SLOT_FLAGS_SHIFT, 0xFF)):
        out["slot_" + name] = (slot >> np.uint64(shift)) & np.uint64(mask)
    for name in STATS_DTYPE.names:
        out["stats_" + name] = stats[name]
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr if arr.dtype in (np.float32, np.float64) else arr.astype(np.float64))


def random_gather_peak(eng, block_bytes, reps=5):
    """What this GPU's memory system delivers for the ACCESS PATTERN of the per-instance-table kernels: independent gathers of random,
    aligned `block_bytes` blocks spread over the engine's whole resident Q table, eight in flight per thread, read-only and with a
    4-byte write-back per gather (rlrm_probe_random_gather, a measurement aid of the library; it rewrites values it has just read,
    so it runs on a scratch copy of the tables). The streaming copy peak of MEASURED_PEAKS.json is not reachable by scattered
    16-64-byte accesses; this is the second denominator the kernel's DRAM traffic is read against."""
    import ctypes as C

    import torch

    from multiagent_rlrm_b200._lib import check

    dev = eng.q.device
    scratch = eng.q.clone()
    sink = torch.zeros(4, dtype=torch.int32, device=dev)
    n_bytes = scratch.numel() * scratch.element_size()
    n_gathers = min(1 << 26, max(1 << 22, 4 * (n_bytes // block_bytes)))
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    out = {"block_bytes": block_bytes, "gathers": n_gathers, "table_bytes": n_bytes,
           "how": "rlrm_probe_random_gather on a copy of the engine's Q tables: 64 gathers per thread, 8 in flight, best of 5 (CUDA events); "
                  "GB/s counts the gathered blocks only (32-byte sector granularity makes the DRAM traffic of 16-byte blocks twice that)"}
    for write, key in ((0, "read_GBps"), (1, "read_write_GBps")):
        best = None
        for _ in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            check(eng.L.rlrm_probe_random_gather(dev.index or 0, scratch.data_ptr(), n_bytes, block_bytes, n_gathers, write, sink.data_ptr(), stream))
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        out[key] = n_gathers * block_bytes / (best * 1e-3) / 1e9
        out[key.replace("GBps", "gathers_per_s")] = n_gathers / (best * 1e-3)
    del scratch
    return out


def summarise(workload, r, res, world, peak, peak_src):
    """One measured entry (headline or `configs` block) from Runner.run's numbers."""
    steps, iters = res["steps"], r.iters
    value = res["active"] / (res["elapsed_ms"] * 1e-3)
    bytes_per = WORKLOADS[workload][4]
    if bytes_per is None:  # sparse-exact Q(lambda): 32 + 16 * (mean live traces), SURVEY.md 8(d), measured in this run
        bytes_per = 32 + 16 * res["mean_live"]
    kernel_ms = sum(res["per_launch_ms"]) / len(res["per_launch_ms"])  # this rank's average step duration (CUDA events)
    active_per_launch_rank = (res["active"] / world) / steps
    achieved = bytes_per * active_per_launch_rank / (kernel_ms * 1e-3) / 1e9
    cap = ncu_capture(workload) or {}
    dram_b = cap.get("dram_bytes_per_active_step")
    dram_gbs = dram_b * active_per_launch_rank / (kernel_ms * 1e-3) / 1e9 if dram_b else None
    roof = {"bound": BOUND.get(workload, "hbm"), "roofline": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "dram_GBps": dram_gbs, "dram_frac": (dram_gbs / peak) if dram_gbs else None,
            "traffic": (dram_b * active_per_launch_rank) if dram_b else None,
            "traffic_source": cap.get("source"), "ncu": cap.get("ncu"), "peak_source": peak_src, "kernel": WORKLOADS[workload][5],
            "algorithmic_bytes_per_active_agent_step": bytes_per, "active_agent_steps_per_launch": active_per_launch_rank,
            "launch_ms": kernel_ms,
            "note": "frac = SURVEY 8d algorithmic bytes / step time / HBM peak; dram_frac = DRAM bytes the committed ncu capture "
                    "measured per active agent-step (traffic_source) x this run's rate / HBM peak — the real HBM utilisation"}
    if res["mean_live"] is not None:
        roof.update({"mean_live_traces": res["mean_live"],
                     "dense_equivalent_GBps": (4 * 1296 * 4 * 4) * active_per_launch_rank / (kernel_ms * 1e-3) / 1e9,
                     "sparse_note": "achieved uses the sparse algorithm's own bytes (32 + 16*L, SURVEY 8d); dense_equivalent is what the "
                                    "reference's dense sweep would have moved for the same steps, NOT achieved bandwidth; the lists stay "
                                    "cache-resident across the iterations of a launch, so frac can exceed 1. The e2e window runs AFTER the "
                                    "device-timed one, i.e. later in training with a different mean list length, so e2e_over_value mixes "
                                    "the copy cost with that drift"})
    out = {"value": value, "unit": UNIT, "ms_per_step": res["elapsed_ms"] / steps, "steps": steps, "instances_per_gpu": r.instances,
           "agents": r.c.n_agents, "iters_per_step": iters, "gpu_launches": res["launches"],
           "slot_steps_per_s": world * r.n_slots * iters * steps / (res["elapsed_ms"] * 1e-3),
           "active_fraction": res["active"] / (world * r.n_slots * iters * steps), "roofline": roof,
           "baseline_config": WORKLOADS[workload][1]}
    if res["e2e"]:
        e = res["e2e"]
        out["e2e"] = {"value": e["active"] / e["seconds"], "unit": UNIT, "h2d_bytes_per_step": e["h2d"], "d2h_bytes_per_step": e["d2h"],
                      "api": "Engine.train_host -> rlrm_train_host (pinned host slot/epsilon in+out, stats out)"}
        out["e2e_over_value"] = out["e2e"]["value"] / value
        # the e2e window runs after the device-timed one, i.e. later in training, where the share of active (not waiting) agents
        # and, for sparse Q(lambda), the list lengths differ: the TIME ratio isolates what the host copies cost
        out["e2e"]["ms_per_step"] = e["seconds"] * 1e3 / e["steps"]
        out["e2e_time_ratio"] = out["ms_per_step"] / out["e2e"]["ms_per_step"]
    if r.sync_every:
        out["collective"] = {"op": "NCCL all_gather_into_tensor of the replicas + rank-ordered reduce kernel (rlrm_merge_replicas)",
                             "sync_every": r.sync_every, "merges": res["n_merges"],
                             "merge_ms": res["merge_ms_total"] / max(1, res["n_merges"]),
                             "collective_share": res["merge_ms_total"] / res["elapsed_ms"]}
    return out


def call_by_call(c, sc, instances, dev):
    """The reference's per-iteration granularity, end to end on host buffers, two ways: (1) rlrm_iterate — ONE launch per
    driver-loop iteration that writes the step record (4 B) and reward (8 B) per agent straight into page-locked host
    memory, one stream synchronisation per iteration; (2) the five separate calls of the reference loop (select_action ->
    step -> update_policy -> reset), each one C-ABI call, with the actions / observations / rewards / done flags copied to
    the host every iteration."""
    import torch

    from multiagent_rlrm_b200.vec import BatchedRMEnvironment

    env = BatchedRMEnvironment(c, instances, device=dev)
    eng = env.engine
    env.reset()
    for _ in range(50):
        env.iterate()
    a0, n_loop = eng.total_active_steps(), 400
    torch.cuda.synchronize(dev)
    ts = time.perf_counter()
    chk = 0
    for _ in range(n_loop):
        rec, rew = env.iterate()           # synchronised: the host owns the record now
        chk ^= int(rec[0, 0])              # touch it
    dt = time.perf_counter() - ts
    fused = {"value": (eng.total_active_steps() - a0) / dt, "unit": UNIT, "iterations": n_loop, "us_per_iteration": dt / n_loop * 1e6,
             "launches_per_iteration": 1, "d2h_bytes_per_iteration": rec.numel() * 4 + rew.numel() * 8, "h2d_bytes_per_iteration": 0,
             "api": "vec.BatchedRMEnvironment.iterate -> rlrm_iterate (select + step + update + masked reset in one launch; record and "
                    "reward written in place into page-locked host memory; one stream synchronisation per iteration)"}
    del env

    env = BatchedRMEnvironment(c, instances, device=dev)
    h_act = torch.empty((instances, c.n_agents), dtype=torch.uint8).pin_memory()
    h_cell = torch.empty((instances, c.n_agents), dtype=torch.int64).pin_memory()
    h_rew = torch.empty((instances, c.n_agents), dtype=torch.float64).pin_memory()
    h_done = torch.empty((instances, c.n_agents), dtype=torch.bool).pin_memory()
    fl = sc.driver == "frozen_lake_main"
    n_active = torch.zeros((), dtype=torch.int64, device=dev)  # agents that actually stepped (executed != 5), on the device

    def loop(n):
        states, _ = env.reset()
        for _ in range(n):
            actions = env.select_action(states)
            h_act.copy_(actions, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            actions = h_act.to(dev, non_blocking=True)
            new_states, rewards, term, trunc, infos = env.step(actions)
            n_active.add_((env._rec["executed"] != 5).sum())
            h_cell.copy_(new_states["cell"], non_blocking=True)
            h_rew.copy_(rewards, non_blocking=True)
            h_done.copy_(term | trunc, non_blocking=True)
            env.update_policy(env.driver_states(states, new_states), actions, rewards, new_states, (term | trunc) if fl else term, infos)
            states = new_states
            over = env.episode_over(term, trunc)
            env.reset(mask=over)
            states = env._obs(env._cells())
            torch.cuda.current_stream(dev).synchronize()

    prev = None
    for _ in range(8):  # warm up until the per-iteration time stops improving (lazy kernel loading on a fresh box)
        tw = time.perf_counter()
        loop(20)
        torch.cuda.synchronize(dev)
        tw = time.perf_counter() - tw
        if prev is not None and tw > 0.8 * prev:
            break
        prev = tw
    n_active.zero_()
    n_loop = 100
    torch.cuda.synchronize(dev)
    ts = time.perf_counter()
    loop(n_loop)
    dt = time.perf_counter() - ts
    unfused = {"value": int(n_active) / dt, "unit": UNIT, "iterations": n_loop, "us_per_iteration": dt / n_loop * 1e6,
               "h2d_bytes_per_iteration": h_act.numel(),
               "d2h_bytes_per_iteration": h_act.numel() + h_cell.numel() * 8 + h_rew.numel() * 8 + h_done.numel(),
               "api": "vec.BatchedRMEnvironment select_action / step / update_policy / reset (one C-ABI call each), host round trip every iteration"}
    del env
    return fused, unfused


def reference_python_throughput(workload, seconds, procs):
    """The REAL reference (its Python sources staged into the git-ignored oracle/_ref by __graft_entry__.build) on `procs` host
    processes, own PCG64 randomness, float64 tables: BASELINE.md section 3's baseline of record. None when it is not staged."""
    import multiprocessing as mp

    try:
        import ref_harness as H

        if not H.reference_available():
            return None
        import time_reference_python as T

        sc = scenario(workload).to_dict()
        mode = "fixed" if sc["driver"] == "frozen_lake_main" else "episode"
        jobs = [(workload, dict(sc, seed=sc["seed"] + k), seconds, 10**9, mode) for k in range(procs)]
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(T.run_case, jobs)
        return {"value": sum(r["active_agent_steps_per_s"] for r in res), "unit": UNIT, "cores": procs, "kind": "reference",
                "per_core": sum(r["active_agent_steps_per_s"] for r in res) / procs,
                "sample": f"{procs} independent processes x {seconds:.0f} s of the live Python reference classes (multiagent_rlrm, float64 "
                          f"tables, its own driver loop restated) on the same workload"}
    except Exception as exc:  # the staged reference is optional
        return {"unavailable": repr(exc)[:200]}


def dropin_n1(seconds=2.0):
    """BASELINE configs[0] (frozen_lake_main --map map1: 2 agents, built-in RM, QRM learner) through the reference's OWN driver loop
    on this repo's reference-shaped N = 1 classes (device-backed: one launch per step, look-ahead selection in the update launch)
    and, when the reference sources are staged (oracle/_ref), on the live Python reference — same host, same process, own PCG64
    randomness. One object instance per call: this is the compatibility layer, not the throughput path."""
    try:
        here = os.path.dirname(os.path.abspath(__file__))
        for sub in ("tests", os.path.join("profiles", "scripts")):
            if os.path.join(here, sub) not in sys.path:
                sys.path.insert(0, os.path.join(here, sub))
        import multiagent_rlrm_b200 as P
        import time_dropin_n1 as T
        from dropin_builder import build_b200

        d = P.scenario_config1().to_dict()
        rm_env, env, agents = build_b200(d)
        T.loop(rm_env, env, agents, True, d["seed"], 0.5)  # warm
        out = {"workload": "configs[0]: frozen_lake_main map1, 2 agents, built-in RM A->B->C, QLearning use_qrm=True, one instance",
               "b200_dropin": T.loop(rm_env, env, agents, True, d["seed"], seconds)}
        try:
            import numpy as np
            import ref_harness as H

            if H.reference_available():
                r_env, r_e, r_agents = H.build_reference(d, np.float64)
                T.loop(r_env, r_e, r_agents, True, d["seed"], 0.3)
                out["python_reference"] = T.loop(r_env, r_e, r_agents, True, d["seed"], seconds)
                out["dropin_over_reference"] = out["b200_dropin"]["active_agent_steps_per_s"] / out["python_reference"]["active_agent_steps_per_s"]
        except Exception as exc:  # the staged reference is optional
            out["python_reference"] = {"unavailable": repr(exc)[:200]}
        return out
    except Exception as exc:  # never fatal for the bench line
        return {"error": repr(exc)[:300]}


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    from multiagent_rlrm_b200.dist import shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    peak, peak_src = measured_peak()

    # ---- headline ------------------------------------------------------------------------------------------------------
    shared = scenario(args.workload).shared_q
    r = Runner(args.workload, args.instances, args.iters, rank, world, dev, sync_every=64 if shared else 0)
    res = r.run(args.steps, args.warmup, max(3, args.steps // 2), (lambda: ClockSampler(local_rank)) if rank == 0 else None,
                dump_dir=args.dump_outputs if rank == 0 else None)
    head = summarise(args.workload, r, res, world, peak, peak_src)
    if not r.sc.shared_q and r.sc.algo != "qlambda":  # per-instance tables read by scattered row / cell-block gathers
        try:
            blk = 16 if r.sc.algo == "ql" else min(64, 16 * r.c.n_rm_states)  # a row, or (up to) a 64-byte cell block
            g = random_gather_peak(r.eng, blk)
            head["roofline"]["random_gather"] = g
            steps_per_s = head["value"] / world
            g["kernel_gathers_per_s"] = steps_per_s  # one row / cell-block gather (+ write-back) per active agent-step
            g["kernel_over_probe"] = steps_per_s / g["read_write_gathers_per_s"]
        except Exception as exc:  # a yardstick, never fatal
            head["roofline"]["random_gather"] = {"error": repr(exc)[:200]}
    stepwise = unfused = n1 = None
    if world == 1 and args.workload in ("cfg3", "cfg3_ql") and not args.no_call_by_call:
        stepwise, unfused = call_by_call(r.c, r.sc, args.instances, dev)
        n1 = dropin_n1()
    del r
    torch.cuda.empty_cache()

    # ---- every other BASELINE configuration, short measured entries (same timing rules) -------------------------------------
    configs = {}
    if args.workload == "cfg3" and not args.no_configs:
        n_total5 = 1048576
        off5, n5 = shard_range(n_total5, rank, world)
        plan = [  # name, workload, instances on this rank, global offset (None = rank * instances), iters, steps, sync_every, scaling
            ("cfg3_f64", "cfg3_f64", 65536, None, 2048, 5, 0, "weak"),  # the headline workload on the reference's own float64 tables
            ("cfg2_batch", "cfg2_batch", 131072, None, 2048, 5, 0, "weak"),
            ("cfg4_sparse", "cfg4", 262144, None, 64, 5, 0, "weak"),
            ("cfg4_dense", "cfg4_dense", 262144, None, 4, 3, 0, "weak"),
            ("cfg5_tables", "cfg5_tables", n5, off5, 256, 5, 0, "strong"),
            ("cfg5_shared", "cfg5_shared", n5, off5, 256, 5, 64, "strong"),
        ]
        if world > 1:
            plan += [("cfg5_shared_K16", "cfg5_shared", n5, off5, 256, 3, 16, "strong"),
                     ("cfg5_shared_K256", "cfg5_shared", n5, off5, 256, 3, 256, "strong"),
                     ("cfg5_shared_weak", "cfg5_shared", n_total5, None, 256, 3, 64, "weak")]
        for name, wl, inst, off, iters, steps, k_sync, scaling in plan:
            try:
                rr = Runner(wl, inst, iters, rank, world, dev, offset=off, sync_every=k_sync)
                rs = rr.run(steps, 3, 2)
                entry = summarise(wl, rr, rs, world, peak, peak_src)
                entry["scaling"] = scaling
                entry["sharding"] = (f"{n_total5} instances in total over {world} rank(s) (dist.shard_range)" if scaling == "strong"
                                     else f"{inst} instances per rank") + \
                                    (f"; shared tables merged every {k_sync} iterations: NCCL all_gather_into_tensor + rank-ordered reduce kernel"
                                     if (k_sync and world > 1) else ("; shared tables, single replica (no collective at 1 GPU)" if k_sync else
                                                                     "; no data-path collective"))
                configs[name] = entry
                del rr
            except Exception as exc:  # a config that does not fit must not take the headline down
                configs[name] = {"error": repr(exc)[:300]}
            torch.cuda.empty_cache()

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            procs = os.cpu_count() or 1
            cpu = cpu_port_throughput(args.workload, args.cpu_seconds or 12.0, procs)
            cpu["reference_python"] = reference_python_throughput(args.workload, 8.0, procs)
        cfgd = workload_config(args, world)
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": scenario(args.workload).table_dtype, "data": "synthetic", "config": cfgd,
            "slot_steps_per_s": head["slot_steps_per_s"], "active_fraction": head["active_fraction"],
            "clocks": res["clocks"], "e2e": head.get("e2e"), "e2e_call_by_call": stepwise, "e2e_call_by_call_unfused": unfused, "dropin_n1": n1,
            "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "cpu_baseline": cpu, "configs": configs,
        }
        if "collective" in head:
            line["collective"] = head["collective"]
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = resolve_defaults(parse_args())
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
