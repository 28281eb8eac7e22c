"""B200 measurement of hyper-parameter sweeps on config 3 (FrozenLake map1, 2 agents, slippery, QRM: train_qrm4_kernel).

A. Cost of the sweep instantiation alone: 65,536 instances, a uniform engine against a degenerate 16-setting sweep (every setting
   equal to the scenario's, so the dynamics are identical), launches alternated in rounds.
B. The use case: a 16-setting grid (learning rate x epsilon decay) x 4,096 instances as ONE sweep launch, against 16 uniform
   engines of 4,096 instances launched one after the other on the same stream.
Rates are active agent-steps per second (env.agent_steps summed over slots, as bench.py counts them), timed with CUDA events
around whole launches. The card's name, power limit and maximum SM clock are read in the same run. Every compared pair is
also checked for bit-identical state at the end.

usage: python profiles/r05/sweep_bench.py [--iters 2048] [--rounds 5] [--launches 5] [--out r05_sweep_bench.json]
"""
import argparse
import copy
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
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return {"query": q, "value": r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unavailable"}


def active_steps(engines):
    return sum(e.total_active_steps() for e in engines)


def timed(engines, iters, launches):
    """seconds and active agent-steps of `launches` rounds, each round one train(iters) launch per engine in turn"""
    before = active_steps(engines)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(launches):
        for e in engines:
            e.train(iters)
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / 1e3, active_steps(engines) - before


def same_state(a, b, rows=None):
    ra = slice(None) if rows is None else rows
    return all(torch.equal(getattr(a, k).view(a.N, -1)[ra], getattr(b, k).view(b.N, -1))
               for k in ("slot", "epsilon", "q", "ep_return", "stats"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=2048)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=5)
    ap.add_argument("--out", default="r05_sweep_bench.json", help="where the full result JSON goes (relative to the working directory)")
    a = ap.parse_args()
    sc = P.scenario_config3(True)
    res = {"card": card(), "iters_per_launch": a.iters, "rounds": a.rounds, "launches_per_round": a.launches}

    # A: uniform vs degenerate sweep, 65,536 instances
    n, H = 65536, 16
    c = P.compile_scenario(sc)
    uni, swp = Engine(c, n), Engine(c, n, sweep=[{} for _ in range(H)])
    for e in (uni, swp):
        e.reset()
        e.train(a.iters)  # warm-up: module load, first touch of the tables
    rows = []
    for r in range(a.rounds):
        for name, e in (("uniform", uni), ("sweep16_degenerate", swp)) if r % 2 == 0 else (("sweep16_degenerate", swp), ("uniform", uni)):
            sec, steps = timed([e], a.iters, a.launches)
            rows.append({"round": r, "engine": name, "seconds": sec, "agent_steps_per_s": steps / sec})
    rate = lambda name: [x["agent_steps_per_s"] for x in rows if x["engine"] == name]  # noqa: E731
    ru, rs = rate("uniform"), rate("sweep16_degenerate")
    res["A_degenerate_sweep"] = {
        "instances": n, "settings": H, "rows": rows,
        "uniform_mean": sum(ru) / len(ru), "uniform_min": min(ru), "uniform_max": max(ru),
        "sweep_mean": sum(rs) / len(rs), "sweep_min": min(rs), "sweep_max": max(rs),
        "sweep_over_uniform": (sum(rs) / len(rs)) / (sum(ru) / len(ru)),
        "state_identical": same_state(uni, swp),
    }
    del uni, swp
    torch.cuda.empty_cache()

    # B: a real 16-setting grid, one sweep launch vs 16 uniform engines in turn
    k = 4096
    grid = [{"learning_rate": lr, "epsilon_start": 0.5, "epsilon_end": 0.01, "epsilon_decay": d}
            for lr in (0.05, 0.1, 0.5, 1.0) for d in (0.9, 0.99, 0.999, 0.9995)]
    sweep = Engine(c, H * k, sweep=grid)
    singles = []
    for g, s in enumerate(grid):
        scg = copy.deepcopy(sc)
        for key, v in s.items():
            setattr(scg, key, v)
        singles.append(Engine(P.compile_scenario(scg, instance_offset=g * k), k))
    for e in [sweep] + singles:
        e.reset()
        e.train(a.iters)
    rows = []
    for r in range(a.rounds):
        order = (("one_sweep_launch", [sweep]), ("16_uniform_launches", singles))
        for name, es in order if r % 2 == 0 else order[::-1]:
            sec, steps = timed(es, a.iters, a.launches)
            rows.append({"round": r, "engine": name, "seconds": sec, "agent_steps_per_s": steps / sec})
    r1, r16 = rate("one_sweep_launch"), rate("16_uniform_launches")
    rows_b = rows
    res["B_grid_16x4096"] = {
        "settings": grid, "instances_per_setting": k, "rows": rows_b,
        "sweep_mean": sum(r1) / len(r1), "sweep_min": min(r1), "sweep_max": max(r1),
        "uniform16_mean": sum(r16) / len(r16), "uniform16_min": min(r16), "uniform16_max": max(r16),
        "sweep_over_uniform16": (sum(r1) / len(r1)) / (sum(r16) / len(r16)),
        "groups_identical": all(same_state(sweep, e, slice(g * k, (g + 1) * k)) for g, e in enumerate(singles)),
        "success_rate_per_setting": [float(x) for x in (sweep.group_stats()["successes"].double() /
                                                        sweep.group_stats()["episodes"].clamp(min=1).double()).cpu()],
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    summary = {k2: v for k2, v in res.items() if k2 == "card"}
    for part in ("A_degenerate_sweep", "B_grid_16x4096"):
        summary[part] = {k2: v for k2, v in res[part].items() if k2 not in ("rows", "settings", "success_rate_per_setting")}
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
