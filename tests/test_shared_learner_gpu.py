"""GPU: the shared learner (Scenario.shared_q, BASELINE config 5) on every kernel route, each launch against the C oracle,
bit-exact; which kernel each launch ran; and the schedule-perturbation equality the integer merge rule implies.

rlrm_create / rlrm_train pick one of four routes for a shared table:

  P  shared_train_kernel<ENV, ALGO>                  one persistent cooperative launch, tables in one SM's shared memory
  C  shared_train_cluster_kernel<ENV, ALGO, CL>      the same with the tables partitioned over a cluster of CL = 2 / 4 / 8 blocks
  T  shared_propose_kernel + apply_shared_kernel     per iteration, tables in shared memory (trace, learn = 0, reserved bit 1)
  G  train_kernel<ENV, ALGO, PA, float> + apply      per iteration, global atomics (per-agent machines, visit counts,
                                                     reserved bit 0, tables beyond 8 x 227 KiB, ...)

The merge rule (include/rlrm_b200.h, "Shared learner") makes every route compute the same bits. So:

* `expected_route` restates the admission of rlrm_create and the dispatch of rlrm_train on the host;
* `test_routes` profiles every named scenario, every generated case and both sides of every size boundary in a fresh child
  process and compares the kernels each launch ran with `expected_route`;
* one seeded generator per route (P, P with RLRM_SHARED_BALANCED=1, C2, C4, C8, T, G) draws only cases that route admits,
  with instance counts at block, grid-wrap and chunk edges and fixed-point values whose 2^20-scaled sums carry across 32 bits
  or round half to even; every launch is compared with the oracle;
* `test_cross_route_equality` runs each P and C case again on the other routes and with the tuning switches flipped;
* `test_plan_coverage` (CPU) checks that the default plan reaches every route, instantiation and edge claimed here.

RLRM_SFUZZ_CASES sets the number of cases per route. Case i of a route depends on (route, i) only."""
import copy
import json
import os
import subprocess
import sys
import time
from collections import namedtuple
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import pytest

import multiagent_rlrm_b200 as P
from multiagent_rlrm_b200 import _abi as abi
from multiagent_rlrm_b200.maps import frozen_lake_grid, office_world_grid
from test_fuzz_gpu import random_machine
from test_fuzz_kernels_gpu import _machine, _template_args

DEFAULT_CASES = 6  # per route
N_CASES = int(os.environ.get("RLRM_SFUZZ_CASES", str(DEFAULT_CASES)))
ROUTES = ("P", "Pb", "C2", "C4", "C8", "T", "G")
SLOT_STEPS = 2_000_000  # oracle budget of one case (instances x agents x iterations)
B200_SMS, B200_SMEM_OPTIN = 148, 232448  # the plan is sized for these; the GPU tests read the device's own limits
SHARED_BLOCK = 1024
FL, OW = abi.ENV_FROZEN_LAKE, abi.ENV_OFFICE_WORLD
QL, QRM = abi.ALGO_QL, abi.ALGO_QRM
MAX_RM_STATES, MAX_AGENTS = 32, 8  # include/rlrm_b200.h

# values whose 2^20-scaled proposals straddle 2^32 (high-word add with and without carry), large negatives, round-half-even
# ties of __float2ll_rn / llrintf (2^-21 * 2^20 = 0.5), and values that do not round exactly
EDGE = [4096 + 2 ** -8, 4096 - 2 ** -8, -(4096 + 2 ** -8), -(4096 - 2 ** -8), -3000.0, 2 ** -21, -(2 ** -21), 3 * 2 ** -21,
        -1 / 3, 0.1]


# ----------------------------------------------------------------------------------------------------------------------
# which kernel ran
# ----------------------------------------------------------------------------------------------------------------------
def parse_shared_kernel_name(name: str) -> Optional[Tuple]:
    """(family, template arguments) of a demangled shared-learner or training kernel name; None for any other kernel"""
    import re

    m = re.search(r"\b(shared_\w+_kernel|apply_shared_kernel|train_\w*kernel)\s*([<(])", name)
    if not m:
        return None
    if m.group(2) == "(":
        return m.group(1), ()
    i, depth, j = m.end(), 1, m.end()
    while j < len(name) and depth:
        depth += {"<": 1, ">": -1}.get(name[j], 0)
        j += 1
    return m.group(1), _template_args(name[i:j - 1])


def profiled_kernels(fn) -> List[Tuple]:
    """launched_train_kernels' recipe (tests/test_fuzz_kernels_gpu.py, where its kineto limitation is described) with the
    parser widened to the shared-learner kernels; [] when the profiler recorded no CUDA kernel at all"""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = sorted((e.time_range.start, e.name) for e in prof.events() if e.device_type == DeviceType.CUDA)
    if not evs:
        return []
    return [k for k in (parse_shared_kernel_name(n) for _t, n in evs) if k is not None]


# ----------------------------------------------------------------------------------------------------------------------
# admission and dispatch, restated from rlrm_create / rlrm_train
# ----------------------------------------------------------------------------------------------------------------------
Route = namedtuple("Route", "name kernels per_iteration")  # kernels: of the whole launch, or of each iteration


def _align16(x):
    return (x + 15) & ~15


def blob_bytes(ncell, nQ, nEv, A, per_agent=False, n_free=0):
    """rlrm_create's table blob (rlrm_b200.cu:293-312). The train_qrm4_kernel sections are empty: qrm4_fast excludes shared_q."""
    sec = A if per_agent else 1
    nd = nQ * (nEv + 1) * sec
    off = 0
    for size in (sec * 2 * MAX_RM_STATES * 8, nd * 8, nd * 8, ncell * 8, MAX_AGENTS * 2, ncell, ncell * sec, nd, MAX_RM_STATES * sec,
                 n_free * 2):
        off = _align16(off + size)
    return off


def admission(ncell, nQ, nEv, A, blob, reserved=0, cluster_env=None, max_smem=B200_SMEM_OPTIN, eligible=True, f32=True):
    """(shared_fast, shared_cluster, reserved as rlrm_create leaves it) — rlrm_b200.cu:403-459. `eligible`: shared table,
    not per-agent, not Q(lambda), learning_rate >= 0."""
    n_ent = A * ncell * nQ * 4
    need = blob + n_ent * 21  # :405 Q 4 B + sum 8 B + count 4 B + last 4 B per entry + row max 4 B per 4 entries
    fast = eligible and need <= 227 * 1024 and not reserved & 1 and need <= max_smem  # :407-409
    cl_min = 2
    if cluster_env is not None and int(cluster_env) >= 2:  # :436-437
        cl_min = 8 if int(cluster_env) >= 8 else (4 if int(cluster_env) >= 4 else 2)
        reserved |= 4
    cl = 0
    if eligible and f32 and not reserved & 1 and (not fast or reserved & 4):  # :433, :439
        rows = n_ent // 4
        for c in (2, 4, 8):  # :443-449, the first CL from cl_min on whose partition fits
            if c >= cl_min and _align16(blob) + -(-rows // c) * 84 <= max_smem:
                cl = c
                break
    return fast, cl, reserved


def expected_route(compiled, n, engine_kw, reserved, env, max_smem_optin, num_sms, learn, trace) -> Route:
    """The kernels one rlrm_train launch of a shared-table engine runs: rlrm_create's admission (rlrm_b200.cu:293-312 blob,
    :403-459 persistent / cluster admission) and rlrm_train's dispatch (:846-905). n and num_sms do not change the route
    (the persistent grid is min(blocks, SMs), the cluster grid the co-resident clusters); they are arguments so that a
    change that makes them matter lands here."""
    cfg = compiled.config
    env = env or {}
    assert cfg.shared_q
    A, ncell, nQ, nEv = int(cfg.n_agents), int(cfg.width) * int(cfg.height), int(cfg.n_rm_states), int(cfg.n_events)
    per_agent = bool(cfg.per_agent_rm)
    blob = blob_bytes(ncell, nQ, nEv, A, per_agent, int(cfg.n_free_cells) if cfg.random_starts else 0)
    if env.get("RLRM_FORCE_GENERIC"):
        reserved |= 1  # :223
    eligible = not per_agent and cfg.algo != abi.ALGO_QLAMBDA and cfg.learning_rate >= 0
    fast, cl, reserved = admission(ncell, nQ, nEv, A, blob, reserved, env.get("RLRM_SHARED_CLUSTER"), max_smem_optin, eligible,
                                   cfg.table_dtype == abi.TABLE_F32)
    visits = bool(engine_kw.get("track_visits")) or cfg.learning_rate < 0
    e, a = int(cfg.env_kind), int(cfg.algo)
    persistent_ok = not visits and learn and not trace and not reserved & 2
    if fast and persistent_ok and not (reserved & 4 and cl):  # :849
        return Route("P", [("shared_train_kernel", (e, a))], False)
    if cl and not (fast and not reserved & 4) and persistent_ok:  # :870
        return Route(f"C{cl}", [("shared_train_cluster_kernel", (e, a, cl))], False)
    apply = [("apply_shared_kernel", ())] if learn else []  # :900-903
    if fast and not visits:  # :885
        return Route("T", [("shared_propose_kernel", (e, a))] + apply, True)
    return Route("G", [("train_kernel", (e, a, per_agent, "float", False))] + apply, True)  # :897 -> launch_train :829-833


def launch_kernels(route: Route, iters: int) -> List[Tuple]:
    return route.kernels * (iters if route.per_iteration else 1)


# ----------------------------------------------------------------------------------------------------------------------
# cases
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class Case:
    family: str  # a route of ROUTES, "named", "boundary" or "regression"
    index: object
    sc: P.Scenario
    n: int
    launches: List[Tuple[int, bool, bool]]  # (iterations, learn, trace)
    offset: int = 0
    reserved: int = 0
    env: Dict[str, str] = field(default_factory=dict)
    kw: Dict[str, bool] = field(default_factory=dict)  # Engine keywords: track_visits, with_stats
    tags: Tuple[str, ...] = ()

    @property
    def id(self):
        return f"{self.family}-{self.index}"

    def compiled(self):
        c = P.compile_scenario(self.sc, instance_offset=self.offset)
        c.config.reserved = self.reserved
        return c

    def route(self, learn, trace, max_smem=B200_SMEM_OPTIN, num_sms=B200_SMS) -> Route:
        return expected_route(self.compiled(), self.n, self.kw, self.reserved, self.env, max_smem, num_sms, learn, trace)

    def variant(self, **changes):
        v = copy.copy(self)
        for k, x in changes.items():
            setattr(v, k, x)
        return v

    def describe(self):
        sc = self.sc
        per = sc.rm_transitions_per_agent is not None
        return (f"{self.id}: {sc.env}/{sc.map_name} A={len(sc.starts)} {sc.algo} nQ={self.compiled().config.n_rm_states} "
                f"per_agent={per} stoch={sc.stochastic} delay={sc.delay_action} all_slip={sc.all_slip} hp={sc.high_prob} "
                f"driver={sc.driver} rsh={sc.use_rsh and sc.rs_kind} rs={sc.random_start_positions} max_steps={sc.max_steps} "
                f"lr={sc.learning_rate} gamma={sc.gamma} q_init={sc.q_init} n={self.n} off={self.offset} "
                f"reserved={self.reserved} env={self.env} kw={self.kw} launches={self.launches} tags={self.tags}")


def _grid(env, map_name):
    return frozen_lake_grid(map_name) if env == "frozen_lake" else office_world_grid(map_name)


def _free(grid):
    hazards = set(grid.hazards)
    return [(x, y) for y in range(grid.height) for x in range(grid.width) if (x, y) not in hazards]


MAPS = [("frozen_lake", "map1")] + [("office_world", m) for m in ("map0", "map1", "map2", "map3", "map4")]


def _sizes_for(route, rng, env, force_cluster):
    """(env, map, A, nQ) whose table size suits `route` (estimated with nEv = nQ - 1; the compiled case is checked again)"""
    maps = [m for m in MAPS if m[0] == env]
    for _ in range(10000):
        env, map_name = maps[int(rng.integers(len(maps)))]
        g = _grid(env, map_name)
        ncell = g.width * g.height
        A = int(rng.integers(1, 9))
        nQ = int(rng.integers(2, 33)) if rng.random() < 0.5 else int(rng.integers(2, 9))
        if nQ - 1 > len(_free(g)) - A:
            continue
        fast, cl, _r = admission(ncell, nQ, nQ - 1, A, blob_bytes(ncell, nQ, nQ - 1, A))
        if route in ("P", "Pb", "T") and fast:
            return env, map_name, A, nQ
        if route in ("C2", "C4", "C8"):
            want = int(route[1])
            if force_cluster and fast:
                return env, map_name, A, nQ
            if not force_cluster and cl == want:
                return env, map_name, A, nQ
        if route == "G":
            return env, map_name, A, nQ
    raise RuntimeError(route)


def _values(rng, sc, rm, edge):
    """learner settings; with `edge`, q_init and part of the machine's rewards from EDGE"""
    sc.learning_rate = float(rng.choice([1.0, 0.1, 0.37, 0.5]))
    sc.gamma = float(rng.choice([0.9, 0.99, 0.5, 1 / 3]))
    sc.q_init = float(rng.choice([0.0, 2.0, -1.0, 0.1]))
    if edge:
        sc.q_init = float(rng.choice(EDGE))
        rm = [(s, e, d, float(rng.choice(EDGE)) if rng.random() < 0.6 else r) for (s, e, d, r) in rm]
    return rm


def _scenario(rng, route, i, sizes):
    env, map_name, A, nQ = sizes
    free = _free(_grid(env, map_name))
    starts = [free[j] for j in rng.choice(len(free), size=A, replace=False)]
    per_agent = route == "G" and i % 3 == 0 and A > 1
    edge = i % 2 == 0 or rng.random() < 0.3
    if per_agent:  # small machines: the per-agent blob must stay within 48 KB
        machines = [random_machine(rng, free, f"m{a}_") for a in range(A)]
        rm, per = machines[0][0], [m[0] for m in machines]
        detector = sorted({p for m in machines for p in m[1]})
    else:
        rm, ev = _machine(rng, free, nQ, "s", shuffle_names=rng.random() < 0.4)
        per = None
        detector = sorted(set(ev) | ({free[int(rng.integers(len(free)))]} if rng.random() < 0.3 else set()))
    sc = P.Scenario(env=env, map_name=map_name, starts=starts, rm_transitions=rm, rm_transitions_per_agent=per,
                    detector_positions=detector, algo=("ql", "qrm")[i % 2], seed=int(rng.integers(1, 1 << 30)))
    sc.rm_transitions = _values(rng, sc, sc.rm_transitions, edge)
    if per is not None and edge:
        sc.rm_transitions_per_agent = [[(s, e, d, float(rng.choice(EDGE)) if rng.random() < 0.5 else r) for (s, e, d, r) in m]
                                       for m in per]
    sc.shared_q = True
    sc.driver = str(rng.choice(["frozen_lake_main", "office_main"]))
    sc.stochastic = bool(rng.random() < 0.7)
    sc.delay_action = bool(sc.stochastic and rng.random() < 0.25)
    sc.all_slip = bool(env == "office_world" and rng.random() < 0.4)
    sc.high_prob = float(rng.choice([0.0, 1 / 3, 0.6, 0.8, 0.95, 1.0]))
    sc.penalty_amount = float(rng.choice([0, -1, -5.5, -1 / 3, 0.1]))
    sc.plants_penalty = float(rng.choice([-100, -3, 0, -1 / 3]))
    sc.wall_penalty = float(rng.choice([0, -0.25, -2, -1e-3, -1 / 3]))
    sc.terminate_on_plants = bool(rng.random() < 0.3)
    sc.terminate_hit_walls = bool(rng.random() < 0.25)
    sc.max_steps = int(rng.choice([5, 12, 40, 150, 1000]))
    sc.reward_modifier = float(rng.choice([1, 1, 0.5, 3]))
    sc.epsilon_start = float(rng.choice([0.01, 0.3, 1.0]))
    sc.epsilon_end = float(rng.choice([0.01, 0.1]))
    sc.epsilon_decay = float(rng.choice([1.0, 0.9, 0.999]))
    if not per_agent and rng.random() < 0.35:
        sc.use_rsh, sc.rs_kind = True, ("vi", "distance")[(i // 2) % 2]
        sc.rs_gamma, sc.rs_alpha = float(rng.choice([0.9, 0.99])), float(rng.choice([100, 7]))
    sc.random_start_positions = bool(env == "frozen_lake" and rng.random() < 0.3)
    return sc


def _instances(rng, route, i, G):
    """(n, tag): block edges N*G = 1024k +- G (+-1 with one agent), a grid-stride walk that wraps (N*G above SMs x 1024),
    balanced chunks that leave the last blocks short or empty, or a small count"""
    kind = i % 3
    if route in ("P", "Pb", "C2", "C4", "C8") and kind == 2:
        return B200_SMS * SHARED_BLOCK // G + int(rng.choice([1, 3, 33, 200])), "wrap"
    if kind == 1:
        k = int(rng.integers(1, 4))
        return k * SHARED_BLOCK // G + int(rng.choice([-1, 1])), "edge"
    return int(rng.choice([1, 3, 31, 129, 700])), "small"


LENGTHS = (1, 2, 3, 4, 7)


def _launches(rng, route, n, A, only_aux):
    """3-6 launches. Lengths from LENGTHS (every residue mod 3) plus one long launch that fills the oracle budget. P / C
    cases mix in traced and learn = False launches (other routes) between launches of their own route; only_aux: every
    launch traced or not learning (routes T and G reached through them)"""
    k = int(rng.integers(3, 7))
    budget = max(k, min(400, SLOT_STEPS // (n * A)))
    lens = [int(rng.choice(LENGTHS)) for _ in range(k)]
    j = int(rng.integers(k))
    lens[j] = max(lens[j], budget - (sum(lens) - lens[j]))
    aux = [(True, True), (False, False), (False, True)]
    if only_aux:
        kinds = [aux[int(rng.integers(3))] for _ in range(k)]
    elif route in ("T", "G"):
        kinds = [(True, False) if rng.random() < 0.5 else aux[int(rng.integers(3))] for _ in range(k)]
    else:  # own route first and last; aux launches in between
        kinds = [(True, False)] + [(True, False) if rng.random() < 0.5 else aux[int(rng.integers(3))] for _ in range(k - 2)] + [(True, False)]
    return [(ln, lr, tr) for ln, (lr, tr) in zip(lens, kinds)]


def make_case(route, i) -> Case:
    rng = np.random.default_rng(7000 + 1000 * ROUTES.index(route) + i)
    force = route in ("C2", "C4", "C8") and i % 4 in (1, 2)  # natural and forced clusters, each with QL and QRM
    env = ("frozen_lake", "office_world")[(i // 2) % 2]
    for _attempt in range(200):
        sizes = _sizes_for(route, rng, env, force)
        sc = _scenario(rng, route, i, sizes)
        A = len(sc.starts)
        G = 1 << (A - 1).bit_length()
        n, tag = _instances(rng, route, i, G)
        case = Case(route, i, sc, n, [], tags=(tag,))
        if rng.random() < 0.3:
            case.offset = int(rng.choice([1, 31, 1000, 65535, 1 << 20]))
        if rng.random() < 0.2:
            case.kw = {"with_stats": False}
        only_aux = False
        if route == "Pb":
            case.env = {"RLRM_SHARED_BALANCED": "1"}
        if force:
            case.env = {"RLRM_SHARED_CLUSTER": route[1]}
        if route == "T":
            if i % 2 == 0:
                case.reserved = 2
            else:
                only_aux = True
        if route == "G" and sc.rm_transitions_per_agent is None:
            why = i % 3  # 0 is the per-agent case
            if why == 1:
                case.kw = dict(case.kw, track_visits=True)
            elif case.route(True, False).name.startswith("C"):
                only_aux = True  # traced / learn = 0 launches on tables that only fit a cluster
            elif case.route(True, False).name != "G":
                case.reserved = 1
        case.launches = _launches(rng, route, n, A, only_aux)
        want = "P" if route == "Pb" else route
        routes = {case.route(lr, tr).name for _it, lr, tr in case.launches}
        own = [case.route(lr, tr).name for _it, lr, tr in case.launches if lr and not tr]
        if route in ("T", "G"):
            ok = routes == {want}
        else:
            ok = len(own) >= 2 and set(own) == {want}
        if ok:
            return case
    raise RuntimeError(f"no admissible draw for {route}-{i}")


def plan(n_cases=None) -> List[Case]:
    n_cases = N_CASES if n_cases is None else n_cases
    return [make_case(r, i) for r in ROUTES for i in range(n_cases)]


# ---- size boundaries: for each transition P -> C2 -> C4 -> C8 -> G the largest configuration of one route and the smallest
# of the next (chain machines with nQ - 1 events, no per-agent machines; size = table entries, then blob) ----
TRANSITIONS = (("P", "C2"), ("C2", "C4"), ("C4", "C8"), ("C8", "G"))


def _natural_route(ncell, nQ, A):
    blob = blob_bytes(ncell, nQ, nQ - 1, A)
    fast, cl, _r = admission(ncell, nQ, nQ - 1, A, blob)
    return ("P" if fast else (f"C{cl}" if cl else "G")), (A * ncell * nQ * 4, blob)


def boundary_configs():
    """[(transition, side, (env, map, A, nQ))] over every map, A = 1..8 and nQ = 2..32"""
    by_route = {}
    for env, map_name in MAPS:
        g = _grid(env, map_name)
        ncell = g.width * g.height
        for A in range(1, 9):
            for nQ in range(2, 33):
                if nQ - 1 > len(_free(g)) - A:
                    continue
                r, key = _natural_route(ncell, nQ, A)
                by_route.setdefault(r, []).append((key, (env, map_name, A, nQ)))
    out = []
    for lo, hi in TRANSITIONS:
        out.append(((lo, hi), "last", max(by_route[lo])[1]))
        out.append(((lo, hi), "first", min(by_route[hi])[1]))
    return out


def make_boundary_case(j) -> Case:
    (lo, hi), side, (env, map_name, A, nQ) = boundary_configs()[j]
    rng = np.random.default_rng(6100 + j)
    free = _free(_grid(env, map_name))
    while True:
        rm, ev = _machine(rng, free, nQ, "s")
        if len(set(ev)) == nQ - 1:
            break
    starts = [c for c in free if c not in set(ev)][:A]
    sc = P.Scenario(env=env, map_name=map_name, starts=starts, rm_transitions=rm, detector_positions=sorted(set(ev)),
                    algo="qrm" if j % 2 else "ql", learning_rate=0.37, gamma=0.9, q_init=float(EDGE[j % len(EDGE)]),
                    epsilon_start=0.3, epsilon_end=0.1, epsilon_decay=0.999, stochastic=True, max_steps=40, seed=4100 + j,
                    driver="frozen_lake_main" if env == "frozen_lake" else "office_main")
    sc.shared_q = True
    n = 300
    return Case("boundary", f"{lo}{hi}-{side}", sc, n, [(1, True, False), (4, True, False), (2, True, True), (30, True, False)],
                tags=(side, lo if side == "last" else hi))


def boundary_cases() -> List[Case]:
    return [make_boundary_case(j) for j in range(2 * len(TRANSITIONS))]


# ---- the named scenarios the rest of the suite relies on ----
def _office12(agents=4):
    sc = P.scenario_config4()
    sc.algo, sc.learning_rate, sc.q_init, sc.shared_q = "qrm", 0.1, 2.0, True
    if agents == 8:
        sc.starts = sc.starts + [(5, 5), (8, 2), (1, 1), (10, 7)]
    return sc


def _acbd(starts):
    sc = P.scenario_config2(True)
    sc.shared_q, sc.starts = True, starts
    return sc


def _cfg5_ql():
    sc = P.scenario_config5(True)
    sc.algo, sc.learning_rate = "ql", 0.1
    return sc


def _per_agent_shared():
    g = P.frozen_lake_grid("map1").goals
    sc = P.scenario_config5(True)
    sc.starts = [(5, 0), (0, 0), (9, 9)]
    sc.detector_positions = sorted(g.values())
    sc.rm_transitions_per_agent = [P.tables.frozen_lake_abc_transitions(), [("p0", g["B"], "p1", 3.0), ("p1", g["A"], "p2", 7.0)],
                                   [("r0", g["C"], "r1", 1.0)]]
    return sc


def _huge_table():
    """8 agents x 225 cells x a 32-state machine: 57,600 rows, beyond a cluster of 8 x 227 KiB"""
    rng = np.random.default_rng(31)
    free = _free(office_world_grid("map3"))
    rm, ev = _machine(rng, free, 32, "h")
    starts = [c for c in free if c not in set(ev)][:8]
    return P.Scenario(env="office_world", map_name="map3", starts=starts, rm_transitions=rm, detector_positions=sorted(set(ev)),
                      algo="qrm", learning_rate=0.5, gamma=0.9, q_init=1.0, epsilon_start=0.5, epsilon_end=0.1, stochastic=True,
                      max_steps=30, seed=777, shared_q=True)


L1, TR, NL = [(3, True, False)], [(3, True, True)], [(3, False, False)]
NAMED = {
    # name: (scenario, n, reserved, env, Engine keywords, launches, route each launch must take)
    "cfg5": (lambda: P.scenario_config5(True), 3000, 0, {}, {}, L1, "P"),
    "cfg5_trace": (lambda: P.scenario_config5(True), 3000, 0, {}, {}, TR, "T"),  # test_shared_learner_matches_oracle
    "cfg5_no_learn": (lambda: P.scenario_config5(True), 3000, 0, {}, {}, NL, "T"),
    "cfg5_reserved1": (lambda: P.scenario_config5(True), 5000, 1, {}, {}, L1 + TR, "G"),  # ..._generic_path_equals_fast_path
    "cfg5_reserved2": (lambda: P.scenario_config5(True), 3000, 2, {}, {}, L1, "T"),  # ..._persistent_kernel_equals_two_launch_path
    "cfg5_reserved4": (lambda: P.scenario_config5(True), 3000, 4, {}, {}, L1, "C2"),  # cfg5_forced_cluster
    "cfg5_visits": (lambda: P.scenario_config5(True), 3000, 0, {}, {"track_visits": True}, L1, "G"),
    "cfg5_cluster2": (lambda: P.scenario_config5(True), 3000, 0, {"RLRM_SHARED_CLUSTER": "2"}, {}, L1, "C2"),
    "cfg5_cluster4": (lambda: P.scenario_config5(True), 3000, 0, {"RLRM_SHARED_CLUSTER": "4"}, {}, L1, "C4"),
    "cfg5_cluster8": (lambda: P.scenario_config5(True), 3000, 0, {"RLRM_SHARED_CLUSTER": "8"}, {}, L1, "C8"),
    "cfg5_balanced": (lambda: P.scenario_config5(True), 200000, 0, {"RLRM_SHARED_BALANCED": "1"}, {}, L1, "P"),
    "cfg5_one_instance": (lambda: P.scenario_config5(True), 1, 0, {}, {}, TR, "T"),  # ..._with_one_instance_is_the_reference_learner
    "cfg5_ql_trace": (_cfg5_ql, 700, 0, {}, {}, TR, "T"),  # test_options_gpu frozen_ql
    "office12_4agents": (lambda: _office12(4), 2000, 0, {}, {}, L1, "C2"),
    "office12_8agents": (lambda: _office12(8), 2000, 0, {}, {}, L1, "C4"),
    "office12_reserved2": (lambda: _office12(4), 2000, 2, {}, {}, L1, "G"),  # the two-launch side of the cluster comparison
    "office12_trace": (lambda: _office12(4), 700, 0, {}, {}, TR, "G"),  # test_options_gpu office_qrm
    "acbd_ql_2agents": (lambda: _acbd([(2, 7), (6, 3)]), 5000, 0, {}, {}, L1, "P"),  # config 2 QL task
    "acbd_ql_2agents_reserved2": (lambda: _acbd([(2, 7), (6, 3)]), 5000, 2, {}, {}, L1, "T"),
    "acbd_ql_forced": (lambda: _acbd([(2, 7), (6, 3), (0, 0)]), 2500, 4, {}, {}, L1, "C2"),
    "acbd_ql_forced_reserved2": (lambda: _acbd([(2, 7), (6, 3), (0, 0)]), 2500, 2, {}, {}, L1, "T"),
    "per_agent": (_per_agent_shared, 300, 0, {}, {}, L1 + TR, "G"),
    "huge_table": (_huge_table, 64, 0, {}, {}, L1, "G"),
}


def named_case(name) -> Case:
    make, n, reserved, env, kw, launches, _route = NAMED[name]
    return Case("named", name, make(), n, list(launches), reserved=reserved, env=dict(env), kw=dict(kw))


# the variants test_cross_route_equality runs a P / C case on
def cross_variants(case: Case) -> List[Case]:
    flip = {"RLRM_SHARED_BALANCED": "0" if case.env.get("RLRM_SHARED_BALANCED") == "1" else "1"}
    out = [case.variant(reserved=2, index=f"{case.index}/reserved2"), case.variant(reserved=1, index=f"{case.index}/reserved1"),
           case.variant(env=dict(case.env, **flip), index=f"{case.index}/balanced{flip['RLRM_SHARED_BALANCED']}")]
    own = case.route(True, False).name
    force = "2" if own == "P" else ("8" if own in ("C2", "C4") else None)
    if force is not None:
        out.append(case.variant(env=dict(case.env, RLRM_SHARED_CLUSTER=force), index=f"{case.index}/cluster{force}"))
    return out


PERSISTENT = ("P", "Pb", "C2", "C4", "C8")


def cross_cases() -> List[Case]:
    return [c for c in plan() if c.family in PERSISTENT]


# ----------------------------------------------------------------------------------------------------------------------
# the GPU runs
# ----------------------------------------------------------------------------------------------------------------------
class _Env:
    """the switches rlrm_create reads, set while an Engine is built (restored afterwards)"""

    KEYS = ("RLRM_SHARED_BALANCED", "RLRM_SHARED_CLUSTER", "RLRM_FORCE_GENERIC")

    def __init__(self, env):
        self.env = env

    def __enter__(self):
        self.saved = {k: os.environ.pop(k, None) for k in self.KEYS}
        os.environ.update(self.env)

    def __exit__(self, *exc):
        for k in self.KEYS:
            os.environ.pop(k, None)
            if self.saved[k] is not None:
                os.environ[k] = self.saved[k]


def _engine(case: Case):
    from multiagent_rlrm_b200.engine import Engine

    with _Env(case.env):
        eng = Engine(case.compiled(), case.n, **case.kw)
    eng.reset()
    return eng


def _device_limits():
    import torch

    p = torch.cuda.get_device_properties(0)
    return p.shared_memory_per_block_optin, p.multi_processor_count


def _state(eng, trace_out):
    """every state array of a shared-table engine as bytes"""
    out = {"slot": eng.slot, "epsilon": eng.epsilon, "q": eng.q, "ep_return": eng.ep_return}
    if eng.stats is not None:
        out["stats"] = eng.stats
    if eng.visits is not None:
        out["visits"] = eng.visits
    if trace_out is not None:
        out["trace"] = trace_out
    return {k: v.cpu().numpy().tobytes() for k, v in out.items()}


def run_case(case: Case):
    """every launch of the case against the oracle, bit for bit"""
    import oracle as O

    eng = _engine(case)
    c = case.compiled()
    o = O.Oracle(c, case.n, "f32", track_visits=bool(case.kw.get("track_visits")))
    o.reset()
    info = case.describe()
    t0 = 0
    for li, (iters, learn, trace) in enumerate(case.launches):
        tr = eng.train(iters, learn=learn, trace=trace)
        tr_o = o.train(t0, iters, learn, trace)
        where = (info, f"launch {li} (t0={t0}, {iters} iterations, learn={learn}, trace={trace})")
        if trace:
            assert np.array_equal(tr.cpu().numpy().view(np.uint32), tr_o), (where, "trace")
        assert np.array_equal(eng.slot.cpu().numpy().view(np.uint64), o.slot), (where, "slot")
        assert eng.epsilon.cpu().numpy().tobytes() == o.epsilon.tobytes(), (where, "epsilon")
        assert eng.q.cpu().numpy().tobytes() == o.q.tobytes(), (where, "q")
        assert eng.ep_return.cpu().numpy().tobytes() == o.ep_return.tobytes(), (where, "ep_return")
        if eng.stats is not None:
            st = eng.stats_numpy()
            for f in O.STATS_DTYPE.names:
                assert st[f].reshape(-1).tobytes() == o.stats[f].reshape(-1).tobytes(), (where, "stats." + f)
        if o.visits is not None:
            assert np.array_equal(eng.visits.cpu().numpy().view(np.uint32), o.visits), (where, "visits")
        assert int(eng.acc_cnt.abs().sum()) == 0 and int(eng.acc_sum.abs().sum()) == 0, (where, "accumulators left dirty")
        t0 += iters


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("index", range(N_CASES))
def test_shared_case_matches_oracle(route, index, cuda_device):
    run_case(make_case(route, index))


@pytest.mark.gpu
@pytest.mark.parametrize("j", range(2 * len(TRANSITIONS)))
def test_size_boundary_matches_oracle(j, cuda_device):
    run_case(make_boundary_case(j))


@pytest.mark.gpu
def test_shared_table_visit_counts_count_every_proposal(cuda_device):
    """Regression: under a shared table every instance's update counts a visit of the one shared entry (update_q increments
    the count atomically). On the first iteration all instances stand on the same start cells."""
    case = Case("regression", "visits", P.scenario_config5(True), 3000, [(1, True, False), (2, True, True), (40, True, False)],
                kw={"track_visits": True})
    run_case(case)
    case = Case("regression", "visits_qrm_office12", _office12(4), 1000, [(1, True, False), (7, True, False)], kw={"track_visits": True})
    run_case(case)


@pytest.mark.gpu
@pytest.mark.parametrize("route", PERSISTENT)
@pytest.mark.parametrize("index", range(N_CASES))
def test_cross_route_equality(route, index, cuda_device):
    """Each P / C case again on route T (reserved bit 1), route G (reserved bit 0), with RLRM_SHARED_BALANCED flipped and
    with the cluster kernel forced: every launch leaves the same bits as the primary run (which run_case checks against the
    oracle). The merge rule sums integers, so no schedule may change a result."""
    case = make_case(route, index)
    engines = [(case, _engine(case))] + [(v, _engine(v)) for v in cross_variants(case)]
    for li, (iters, learn, trace) in enumerate(case.launches):
        states = [(v, _state(e, e.train(iters, learn=learn, trace=trace))) for v, e in engines]
        ref = states[0][1]
        for v, s in states[1:]:
            for k in ref:
                assert s[k] == ref[k], (v.describe(), f"launch {li}", k)


# ---- routes, profiled in a fresh child process ----
def route_cases() -> List[Case]:
    """everything whose route the suite relies on: the named scenarios, every generated case, every cross-route variant
    and both sides of every size boundary"""
    out = [named_case(n) for n in NAMED]
    for case in plan():
        out.append(case)
        if case.family in PERSISTENT:
            out.extend(cross_variants(case))
    return out + boundary_cases()


def _route_launches(case):
    """the case's launch kinds with at most 2 iterations each (the route does not depend on the length)"""
    return [(min(it, 2), lr, tr) for it, lr, tr in case.launches]


def _route_child(lo, hi):
    """child process: profile cases [lo, hi) of route_cases(), one profiler session over all launches of a case, and print
    {id: kernels in launch order} as JSON"""
    res = {}
    for case in route_cases()[lo:hi]:
        eng = _engine(case)

        def launches():
            for it, lr, tr in _route_launches(case):
                eng.train(it, learn=lr, trace=tr)

        res[case.id] = profiled_kernels(launches)
        del eng
    print("ROUTES " + json.dumps(res))


ROUTE_CHUNK = 40  # cases per child process: keeps each process short (see launched_train_kernels for kineto's dropouts)


@pytest.mark.gpu
def test_routes(cuda_device):
    """The kernels each launch of every route case ran, against expected_route. The profiling runs in fresh child
    processes, where kineto keeps the kernel records (see launched_train_kernels in tests/test_fuzz_kernels_gpu.py)."""
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    cases = route_cases()
    max_smem, num_sms = _device_limits()
    got = {}
    for lo in range(0, len(cases), ROUTE_CHUNK):
        code = (f"import sys; sys.path[:0] = {[here, root, os.path.join(root, 'oracle')]!r}; "
                f"import test_shared_learner_gpu as T; T._route_child({lo}, {lo + ROUTE_CHUNK})")
        flags = ["-s"] if sys.flags.no_user_site else []
        t = time.time()
        res = subprocess.run([sys.executable, *flags, "-c", code], capture_output=True, text=True, timeout=600, cwd=root)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
        line = [x for x in res.stdout.splitlines() if x.startswith("ROUTES ")]
        assert line, res.stdout[-3000:] + res.stderr[-3000:]
        got.update(json.loads(line[-1][len("ROUTES "):]))
        print(f"route cases [{lo}, {lo + ROUTE_CHUNK}): {time.time() - t:.1f} s")
    seen = set()
    for case in cases:
        ran = got.get(case.id)
        assert ran, (case.describe(), "torch.profiler recorded no kernel for this case (see launched_train_kernels)")
        want, names = [], []
        for it, lr, tr in _route_launches(case):
            r = case.route(lr, tr, max_smem, num_sms)
            want += [[f, list(a)] for f, a in launch_kernels(r, it)]
            names.append(r.name)
        assert ran == want, (case.describe(), names, ran)
        seen.update(names)
        if case.family == "named":
            assert NAMED[case.index][6] in names, (case.id, names)
    assert seen == {"P", "C2", "C4", "C8", "T", "G"}, seen


# ----------------------------------------------------------------------------------------------------------------------
# the plan's coverage (CPU)
# ----------------------------------------------------------------------------------------------------------------------
def test_plan_coverage():
    """Every case is admitted by its route, and the default plan reaches every route x environment x algorithm, CL 2 / 4 / 8,
    balanced 0 / 1, per-agent machines, both shaping kinds, random starts, visit counts, A = 1..8, the wrap and edge
    instance counts, every value edge, every launch length mod 3 and both sides of every size boundary."""
    cases = plan(max(N_CASES, DEFAULT_CASES))
    ids = [c.id for c in cases]
    assert len(ids) == len(set(ids))
    combos, cls, balanced, per_agent, shaping, edges, mods, agents, tags = set(), set(), set(), False, set(), set(), set(), set(), set()
    random_starts = visits = no_stats = offset = False
    for case in cases:
        c = case.compiled()
        sc = case.sc
        A = len(sc.starts)
        G = 1 << (A - 1).bit_length()
        want = "P" if case.family == "Pb" else case.family
        own = [case.route(lr, tr) for _it, lr, tr in case.launches if lr and not tr] or [case.route(lr, tr) for _it, lr, tr in case.launches]
        assert {r.name for r in own} == {want}, case.describe()
        assert 3 <= len(case.launches) <= 6, case.describe()
        assert case.n * A * sum(it for it, _l, _t in case.launches) <= SLOT_STEPS + case.n * A * 30, case.describe()
        combos.add((want, int(c.config.env_kind), int(c.config.algo)))
        for r in own:
            if r.name.startswith("C"):
                cls.add(int(r.name[1]))
        if want == "P":
            balanced.add(case.env.get("RLRM_SHARED_BALANCED", "0"))
        if case.family == "G" and own[0].kernels[0][1][2]:
            per_agent = True
        if sc.use_rsh:
            shaping.add((sc.rs_kind, want[0]))
        random_starts |= bool(sc.random_start_positions)
        visits |= bool(case.kw.get("track_visits"))
        no_stats |= case.kw.get("with_stats") is False
        offset |= case.offset != 0
        agents.add(A)
        tag = case.tags[0]
        tags.add((want[0], tag))
        if tag == "wrap":
            assert case.n * G > B200_SMS * SHARED_BLOCK, case.describe()
        if tag == "edge":
            assert (case.n * G) % SHARED_BLOCK in (G, SHARED_BLOCK - G) or A == 1, case.describe()
        if case.family == "Pb" and tag == "wrap":  # balanced chunks: the last blocks get short or empty ranges
            total, grid = case.n * G, B200_SMS
            chunk = ((-(-total // grid)) + 31) & ~31
            assert chunk * (grid - 1) >= total or total % chunk, case.describe()
        vals = [sc.q_init] + [r for (_s, _e, _d, r) in sc.rm_transitions]
        for m in sc.rm_transitions_per_agent or []:
            vals += [r for (_s, _e, _d, r) in m]
        edges |= {v for v in vals if v in EDGE}
        mods |= {it % 3 for it, _l, _t in case.launches}
        assert case.sc.learning_rate is not None
    for route in ("P", "C2", "C4", "C8", "T", "G"):
        for e in (FL, OW):
            for a in (QL, QRM):
                assert (route, e, a) in combos, (route, e, a)
    assert cls == {2, 4, 8} and balanced == {"0", "1"} and per_agent
    assert {k for k, _r in shaping} == {"vi", "distance"} and {r for _k, r in shaping} >= {"P", "C", "T"}
    assert random_starts and visits and no_stats and offset
    assert agents == set(range(1, 9))
    for r in ("P", "C"):
        assert {(r, "wrap"), (r, "edge"), (r, "small")} <= tags, (r, tags)
    assert set(EDGE) <= edges, set(EDGE) - edges
    assert mods == {0, 1, 2}
    assert any(lr == 1.0 for lr in (c.sc.learning_rate for c in cases))
    assert {len(c.sc.starts) for c in cases if c.family in ("C2", "C4", "C8")} >= {1, 8}
    assert any(list(c.compiled().qrm_states) != sorted(c.compiled().qrm_states) for c in cases if c.sc.algo == "qrm")
    office = [c.sc for c in cases if c.sc.env == "office_world"]
    assert {sc.map_name for sc in office} == {"map0", "map1", "map2", "map3", "map4"}
    assert any(sc.all_slip for sc in office) and any(sc.delay_action for sc in office)
    assert {c.sc.driver for c in cases} == {"frozen_lake_main", "office_main"}
    assert any(c.sc.terminate_on_plants for c in cases) and any(c.sc.terminate_hit_walls for c in cases)
    assert any(not c.sc.stochastic for c in cases) and 5 in {c.sc.max_steps for c in cases}
    # both sides of every size boundary, and the sides are adjacent routes
    b = boundary_cases()
    for case in b:
        side, route = case.tags
        assert case.route(True, False).name == route, case.describe()
    assert {(cs.tags[1]) for cs in b} == {"P", "C2", "C4", "C8", "G"}
    # every cross-route variant leaves its primary's route
    for case in cross_cases():
        names = {v.route(True, False).name for v in cross_variants(case)}
        assert {"T", "G"} <= names or "G" in names, (case.describe(), names)


def test_shared_kernel_name_parsing():
    assert parse_shared_kernel_name("void shared_train_kernel<1, 0>(KP, DState, unsigned long long, int, unsigned long long*, int*, float*)") == \
        ("shared_train_kernel", (1, 0))
    assert parse_shared_kernel_name("void shared_train_cluster_kernel<0, 1, 8>(KP, DState, unsigned long long, int, unsigned long long*, "
                                    "int*, float*)") == ("shared_train_cluster_kernel", (0, 1, 8))
    assert parse_shared_kernel_name("apply_shared_kernel(KP, DState)") == ("apply_shared_kernel", ())
    assert parse_shared_kernel_name("void train_kernel<0, 1, true, float, false>(KP)") == ("train_kernel", (0, 1, True, "float", False))
    assert parse_shared_kernel_name("void reset_kernel<0>(KP, DState)") is None
