"""B200 measurement of softmax exploration (rlrm_set_exploration) against epsilon-greedy on the same kernel.

For config 3 QRM (FrozenLake map1, 2 agents, 65,536 instances), config 2 batched (OfficeWorld, 1 agent, 131,072 instances,
slippery) and config 4 sparse Q(lambda) (OfficeWorld chain of 12, 4 agents, 262,144 instances), three engines per workload:
  softmax          temperature 0.5: the generic kernel (train_kernel<..., SOFTMAX = true>) or train_qlambda_sparse_kernel<.., true>
  epsilon_generic  epsilon-greedy on the same kernel family (config.reserved bit 0 forces the generic kernel for QL / QRM)
  epsilon_default  epsilon-greedy as the library routes it (the specialised kernel where one applies: context only)
Launches of the engines alternate within each round and the order flips every round. Rates are active agent-steps per second
(env.agent_steps summed over slots, as bench.py counts them), timed with CUDA events around whole launches; the card's name,
power limit and maximum SM clock are read in the same run.

usage: python profiles/r06/softmax_bench.py [--rounds 5] [--launches 3] [--out r06_softmax_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import multiagent_rlrm_b200 as P  # noqa: E402
from multiagent_rlrm_b200.engine import Engine  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return {"query": q, "value": r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unavailable"}


def timed(e, iters, launches):
    before = e.total_active_steps()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(launches):
        e.train(iters)
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / 1e3, e.total_active_steps() - before


WORKLOADS = {  # name -> (scenario, instances, iterations per launch, Engine keywords)
    "cfg3_qrm": (lambda: P.scenario_config3(True), 65536, 2048, {}),
    "cfg2_batch": (lambda: P.scenario_config2(True), 131072, 2048, {}),
    "cfg4_sparse_qlambda": (P.scenario_config4, 262144, 64, {"qlambda_sparse": True}),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=3)
    ap.add_argument("--temperature", type=float, default=0.5)
    ap.add_argument("--out", default="r06_softmax_bench.json", help="where the full result JSON goes (relative to the working directory)")
    a = ap.parse_args()
    res = {"card_before": card(), "temperature": a.temperature, "rounds": a.rounds, "launches_per_round": a.launches, "workloads": {}}
    for name, (make, n, iters, kw) in WORKLOADS.items():
        c = P.compile_scenario(make())
        forced = P.compile_scenario(make())
        forced.config.reserved = 1  # epsilon-greedy on the generic kernel (QL / QRM); Q(lambda) has no other kernel
        engines = {"softmax": Engine(c, n, exploration="softmax", temperature=a.temperature, **kw),
                   "epsilon_generic": Engine(forced, n, **kw), "epsilon_default": Engine(c, n, **kw)}
        for e in engines.values():
            e.reset()
            e.train(iters)  # warm-up: module load, first touch of the tables
        rows = []
        for r in range(a.rounds):
            order = list(engines.items()) if r % 2 == 0 else list(engines.items())[::-1]
            for en, e in order:
                sec, steps = timed(e, iters, a.launches)
                rows.append({"round": r, "engine": en, "seconds": sec, "agent_steps_per_s": steps / sec})
        summary = {}
        for en in engines:
            v = [x["agent_steps_per_s"] for x in rows if x["engine"] == en]
            summary[en] = {"mean": sum(v) / len(v), "min": min(v), "max": max(v)}
        summary["softmax_over_epsilon_generic"] = summary["softmax"]["mean"] / summary["epsilon_generic"]["mean"]
        res["workloads"][name] = {"instances": n, "agents": engines["softmax"].A, "iters_per_launch": iters, "rows": rows, **summary}
        del engines
        torch.cuda.empty_cache()
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: ({w: {x: y for x, y in v.items() if x != "rows"} for w, v in res[k].items()} if k == "workloads" else res[k])
                      for k in res}, indent=1))


if __name__ == "__main__":
    main()
