#!/usr/bin/env python
"""A learning-rate x epsilon-decay grid on BASELINE config 3 (FrozenLake map1, 2 agents, slippery, QRM) trained as ONE
hyper-parameter sweep: every setting gets its own block of instances, all settings advance in the same kernel launch.
Prints the success rate of the finished episodes per setting.

    python examples/sweep_frozen_lake.py --instances-per-setting 1024 --iterations 20000
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import multiagent_rlrm_b200 as P  # noqa: E402
from multiagent_rlrm_b200.engine import Engine  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances-per-setting", type=int, default=1024)
    ap.add_argument("--iterations", type=int, default=20000)
    ap.add_argument("--learning-rates", type=float, nargs="+", default=[0.05, 0.2, 0.5, 1.0])
    ap.add_argument("--epsilon-decays", type=float, nargs="+", default=[0.9, 0.99, 0.999])
    ap.add_argument("--epsilon-start", type=float, default=0.5)
    args = ap.parse_args()

    sc = P.scenario_config3(True)
    grid = [{"learning_rate": lr, "epsilon_start": args.epsilon_start, "epsilon_end": 0.01, "epsilon_decay": d}
            for lr in args.learning_rates for d in args.epsilon_decays]
    k = args.instances_per_setting
    eng = Engine(P.compile_scenario(sc), len(grid) * k, sweep=grid)
    eng.reset()
    done = 0
    while done < args.iterations:
        chunk = min(2000, args.iterations - done)
        eng.train(chunk)
        done += chunk
    g = eng.group_stats()
    episodes, successes = g["episodes"].cpu(), g["successes"].cpu()
    print(f"{len(grid)} settings x {k} instances x {args.iterations} iterations, one launch per {2000} iterations")
    print(f"{'learning_rate':>13} {'epsilon_decay':>13} {'episodes':>10} {'success rate':>12}")
    for s, e, w in zip(eng.sweep, episodes.tolist(), successes.tolist()):
        print(f"{s['learning_rate']:>13g} {s['epsilon_decay']:>13g} {e:>10d} {w / max(e, 1):>12.4f}")


if __name__ == "__main__":
    main()
