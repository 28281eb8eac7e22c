"""GPU: seeded random cases for each specialised training kernel, every launch against the C oracle, bit-exact; and which
kernel each launch ran.

The specialised kernels (train_qrm4_kernel, train_qrmn_kernel, train_qrm_block_kernel, train_ql_fast_kernel) are picked
by rlrm_create's admission conditions. The uniform draws of test_fuzz_gpu.py rarely meet them, and a result comparison
alone cannot tell whether a launch ran the kernel it was meant to test. So:

* `launched_train_kernels` reads the names of the kernels a call launched from the CUDA activity trace of torch.profiler;
* `test_named_scenario_routes` pins the kernel of the named scenarios the rest of the suite relies on;
* one generator per family draws only cases that family admits (machine size and state order, table type, shaping,
  random starts) and spreads them over environments, maps, agents, drivers, slip models, penalties, termination flags,
  learner settings, instance counts around warp and block edges, instance offsets and hyper-parameter sweeps. Every case
  runs 3-5 launches mixing learn / trace; after each launch every state array is compared with the oracle and the launch
  must have run the family's kernel with the expected template arguments;
* `test_plan_coverage` (CPU) checks that the plan reaches every instantiation the GPU tests claim to cover.

RLRM_KFUZZ_CASES sets the number of cases per family. Case i of a family depends on (family, i) only, so a larger count
adds cases and keeps the default ones."""
import copy
import os
import re
from collections import namedtuple
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np
import pytest

import multiagent_rlrm_b200 as P
from multiagent_rlrm_b200 import _abi as abi
from multiagent_rlrm_b200.maps import frozen_lake_grid, office_world_grid
from test_fuzz_gpu import random_machine

DEFAULT_CASES = 16  # per family; the qrm_block plan needs 16 to reach NU x type x fetch variant
N_CASES = int(os.environ.get("RLRM_KFUZZ_CASES", str(DEFAULT_CASES)))
FAMILIES = ("qrm4", "qrmn", "qrm_block", "ql_fast")
KERNEL = {"qrm4": "train_qrm4_kernel", "qrmn": "train_qrmn_kernel", "qrm_block": "train_qrm_block_kernel",
          "ql_fast": "train_ql_fast_kernel", "generic": "train_kernel"}
B200_SMS = 148  # the plan's MINB 8 cases are sized for this; the GPU tests read the device's own count
TRAIN_BLOCK = 128
SLOT_STEPS = 2_000_000  # oracle budget of one ordinary case (instances x agents x iterations)

# values whose float32 and float64 roundings differ: exercise the host's float32 step records against the oracle
ODD = [0.1, -1 / 3, 1e-3, -5.5]


# ----------------------------------------------------------------------------------------------------------------------
# which kernel ran
# ----------------------------------------------------------------------------------------------------------------------
Kernel = namedtuple("Kernel", "family args name")


def _template_args(s: str) -> Tuple:
    """'0, true, float, 7' -> (0, True, 'float', 7); nested brackets stay one argument"""
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch in "<(":
            depth += 1
        elif ch in ">)":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur)
            cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur)
    vals = []
    for tok in (t.strip() for t in out):
        if tok in ("true", "false"):
            vals.append(tok == "true")
        elif re.fullmatch(r"-?\d+[uUlL]*", tok):
            vals.append(int(re.match(r"-?\d+", tok).group(0)))
        else:
            vals.append(tok)
    return tuple(vals)


def parse_kernel_name(name: str) -> Optional[Kernel]:
    """Family and template arguments of a demangled kernel name, e.g. 'void train_qrm4_kernel<0, true, true, false, 7,
    false>(KP, ...)'; None when the family does not start with train_."""
    m = re.search(r"\b(train_\w+)\s*<", name)
    if not m:
        m = re.search(r"\b(train_\w+)\s*\(", name)
        return Kernel(m.group(1), (), name) if m else None
    i, depth = m.end(), 1
    j = i
    while j < len(name) and depth:
        depth += {"<": 1, ">": -1}.get(name[j], 0)
        j += 1
    return Kernel(m.group(1), _template_args(name[i:j - 1]), name)


def launched_train_kernels(fn) -> List[Kernel]:
    """Run fn() under torch.profiler with CUDA activity tracing and return the train_* kernels it launched, in launch order.
    The library launches from a ctypes-loaded shared object; CUPTI records its kernels as it records torch's own.

    Fails when the profiler recorded no kernel at all: an empty trace would make every route check pass vacuously.

    Known limitation (torch 2.11, CUDA 12.8, B200): late in a long-running process kineto discards the kernel records of a
    session as "Out-of-range" of its capture window. Its log shows them, and torch's own kernels are dropped the same way.
    The runtime-API records (cudaLaunchKernel) of the same session are kept. Device memory is not the cause: with 188 of
    191 GB free and after torch.cuda.empty_cache() the records are still dropped. Neither padding the window with 0.3 s on
    both sides nor TEARDOWN_CUPTI=0 brings them back. In a process that profiles one small torch kernel every 7.6 s, the
    kernels go missing from about 18 s on, in some sessions and not others. A full `pytest -m gpu tests` run keeps them
    through this file and tests/test_gpu_parity.py, and loses them by tests/test_sweep_gpu.py (about 70 s in). So every
    route check lives in the files that run early, and a dropout fails here with this message instead of passing."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = [(e.time_range.start, e.name) for e in prof.events() if e.device_type == DeviceType.CUDA]
    assert evs, ("torch.profiler recorded no CUDA kernel for this call; see launched_train_kernels for when kineto drops them "
                 "(run the test earlier in the process, or alone)")
    return [k for k in (parse_kernel_name(n) for _t, n in sorted(evs, key=lambda e: e[0])) if k is not None]


# ----------------------------------------------------------------------------------------------------------------------
# the routing of the named scenarios
# ----------------------------------------------------------------------------------------------------------------------
FL, OW = abi.ENV_FROZEN_LAKE, abi.ENV_OFFICE_WORLD


def _office_task(exp, algo):
    return P.scenario_for_experiment("map1", exp, starts=[(2, 7), (6, 3), (0, 0)], algo=algo, learning_rate=0.1, gamma=0.9,
                                     stochastic=True, epsilon_start=0.1, epsilon_end=0.1, epsilon_decay=1.0, q_init=2.0,
                                     wall_penalty=-0.5, max_steps=200, seed=97)


def _named(name, num_sms):
    """name -> (scenario, n, Engine keywords, config.reserved, expected kernel family, expected template arguments without
    the trailing SWEEP flag) for one learning launch without a trace"""
    if name == "cfg3_qrm":
        return P.scenario_config3(True), 256, {}, 0, "train_qrm4_kernel", (FL, True, True, False, 7)
    if name == "cfg5_minb8":  # 4 agents, lane groups of 4: more threads than 7 resident blocks per SM hold
        return P.scenario_config5(False), num_sms * 7 * TRAIN_BLOCK // 4 + 1, {}, 0, "train_qrm4_kernel", (FL, True, True, False, 8)
    if name == "exp1":
        return _office_task("exp1", "qrm"), 64, {}, 0, "train_qrmn_kernel", (OW, 3, True, True, False)
    if name == "exp3":
        return _office_task("exp3", "qrm"), 64, {}, 0, "train_qrmn_kernel", (OW, 5, True, True, False)
    if name == "exp5_f32":  # 9 states: 144-byte cell blocks
        return _office_task("exp5", "qrm"), 64, {}, 0, "train_qrm_block_kernel", (OW, 11, "float", False)
    if name == "cfg3_f64":  # 4 states in float64: 128-byte cell blocks
        sc = P.scenario_config3(True)
        sc.table_dtype = "f64"
        return sc, 64, {}, 0, "train_qrm_block_kernel", (FL, 3, "double", False)
    if name == "chain12":  # 12 states: 192-byte cell blocks
        sc = P.scenario_config4()
        sc.algo, sc.learning_rate, sc.q_init = "qrm", 0.1, 2.0
        return sc, 64, {}, 0, "train_qrm_block_kernel", (OW, 11, "float", True)
    if name == "cfg3_ql":
        return P.scenario_config3(False), 256, {}, 0, "train_ql_fast_kernel", (FL, True, True, False)
    if name == "cfg2":
        return P.scenario_config2(True), 256, {}, 0, "train_ql_fast_kernel", (OW, True, True, False)
    generic = ("train_kernel", (FL, abi.ALGO_QRM, False, "float"))
    if name == "reserved_generic":
        return (P.scenario_config3(True), 64, {}, 1) + generic
    if name == "track_visits":
        return (P.scenario_config3(True), 64, {"track_visits": True}, 0) + generic
    if name == "lr_none":
        sc = P.scenario_config3(True)
        sc.learning_rate = None
        return (sc, 64, {}, 0) + generic
    raise KeyError(name)


NAMED = ["cfg3_qrm", "cfg5_minb8", "exp1", "exp3", "exp5_f32", "cfg3_f64", "chain12", "cfg3_ql", "cfg2", "reserved_generic",
         "track_visits", "lr_none"]


def _num_sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.gpu
@pytest.mark.parametrize("sweep", [False, True])
@pytest.mark.parametrize("name", NAMED)
def test_named_scenario_routes(name, sweep, cuda_device):
    """The kernel each named scenario of the suite runs on; under a sweep the same family in its SWEEP instantiation."""
    from multiagent_rlrm_b200.engine import Engine

    sc, n, kw, reserved, family, args = _named(name, _num_sms())
    c = P.compile_scenario(sc)
    c.config.reserved = reserved
    if sweep:
        kw = dict(kw, sweep=[{"epsilon_start": 0.3}, {"epsilon_end": 0.05}], sweep_group=(n + 1) // 2)
    eng = Engine(c, n, **kw)
    eng.reset()
    got = launched_train_kernels(lambda: eng.train(3))
    assert [(k.family, k.args) for k in got] == [(family, args + (sweep,))], [k.name for k in got]


@pytest.mark.gpu
def test_sweep_setting_without_learning_rate_routes_to_generic(cuda_device):
    """learning_rate None needs visit counts, which only the generic kernel keeps: one such setting sends the whole sweep there"""
    from multiagent_rlrm_b200.engine import Engine

    eng = Engine(P.compile_scenario(P.scenario_config3(True)), 64, sweep=[{"learning_rate": 0.5}, {"learning_rate": None}])
    eng.reset()
    got = launched_train_kernels(lambda: eng.train(3))
    assert [(k.family, k.args) for k in got] == [("train_kernel", (FL, abi.ALGO_QRM, False, "float", True))], [k.name for k in got]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["qrm4_minb7", "ql_fast", "qrmn_3", "qrmn_5", "qrm_block_f32", "qrm_block_f64", "qrm_block_f32_cpasync",
                                  "qrm_block_f64_cpasync", "shaping_qrm"])
def test_forced_generic_sweep_engines_run_different_kernels(name, cuda_device):
    """The two engines test_forced_generic_equals_fast_path_under_a_sweep (tests/test_sweep_gpu.py) compares: the fast one runs its
    family's SWEEP instantiation, the one with config.reserved bit 0 the generic kernel's. The check lives here rather than
    in that test because kineto drops kernel records by the time that file runs in a full suite (see launched_train_kernels)."""
    from test_sweep_gpu import _case, _engine

    sc, sets, k, _iters, kw = _case(name)
    n = len(sets) * k
    fast, gen = _engine(sc, n, sweep=sets, **kw), _engine(sc, n, reserved=1, sweep=sets, **kw)
    fast.reset(); gen.reset()
    kf = launched_train_kernels(lambda: fast.train(5, trace=True))
    kg = launched_train_kernels(lambda: gen.train(5, trace=True))
    assert [(x.family, x.args[-1]) for x in kg] == [("train_kernel", True)], kg
    assert len(kf) == 1 and kf[0].family != "train_kernel" and kf[0].args[-1] is True, kf


# ----------------------------------------------------------------------------------------------------------------------
# admission, restated from rlrm_create (used to redraw until a case belongs to its family; the route check confirms it)
# ----------------------------------------------------------------------------------------------------------------------
def admitted(c, lr_none=False) -> str:
    cfg = c.config
    if cfg.learning_rate < 0 or lr_none or cfg.shared_q or cfg.per_agent_rm:
        return "generic"
    f32 = cfg.table_dtype == abi.TABLE_F32
    rsh = bool(cfg.use_rsh) and c.phi is not None
    nq, nqrm = int(cfg.n_rm_states), int(cfg.n_qrm_states)
    identity = [int(x) for x in c.qrm_states[:nqrm]] == list(range(nqrm))
    if cfg.algo == abi.ALGO_QRM:
        plain = f32 and not rsh and not cfg.random_starts and identity
        if plain and nq == 4 and nqrm == 3:
            return "qrm4"
        if plain and nq in (3, 5) and nqrm == nq - 1:
            return "qrmn"
        if 2 <= nq <= 16 and 1 <= nqrm <= 15:
            return "qrm_block"
    if cfg.algo == abi.ALGO_QL and f32 and not rsh and not cfg.random_starts:
        return "ql_fast"
    return "generic"


def block_bytes(cfg):
    return int(cfg.n_rm_states) * (32 if cfg.table_dtype == abi.TABLE_F64 else 16)


def nu_of(n_qrm):
    return 3 if n_qrm <= 3 else 7 if n_qrm <= 7 else 11 if n_qrm <= 11 else 15


def zero_probability_outcome(cfg) -> bool:
    """a stochastic slip model with an outcome of probability 0 (equal consecutive cumulative thresholds)"""
    if not cfg.stochastic or cfg.slip_n < 2:
        return False
    thr = [0] + [int(cfg.slip_thr[j]) for j in range(cfg.slip_n - 1)] + [1 << 32]
    return any(a == b for a, b in zip(thr, thr[1:]))


# ----------------------------------------------------------------------------------------------------------------------
# the case generators
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class Case:
    family: str
    index: int
    sc: P.Scenario
    n: int
    offset: int
    launches: List[Tuple[int, bool, bool]]  # (iterations, learn, trace)
    sweep: Optional[List[dict]] = None
    group: Optional[int] = None
    tma: Optional[str] = None  # RLRM_QRMB_TMA forced for this case

    @property
    def id(self):
        return f"{self.family}-{self.index}"

    def compiled(self, offset=None):
        return P.compile_scenario(self.sc, instance_offset=self.offset if offset is None else offset)

    def describe(self):
        sc = self.sc
        return (f"{self.id}: {sc.env}/{sc.map_name} A={len(sc.starts)} {sc.algo} {sc.table_dtype} stoch={sc.stochastic} "
                f"delay={sc.delay_action} all_slip={sc.all_slip} hp={sc.high_prob} driver={sc.driver} rsh={sc.use_rsh} "
                f"rs={sc.random_start_positions} max_steps={sc.max_steps} n={self.n} off={self.offset} "
                f"launches={self.launches} sweep={self.sweep} k={self.group} tma={self.tma}")


def _long_machine(rng, cells, k, tag):
    """random_machine's recipe (a rewarded chain over distinct cells plus self-loops / resets / shortcuts) for chains of
    any length k; zero-padded names keep the sort order of the states equal to the chain order"""
    ev = [cells[i] for i in rng.choice(len(cells), size=k, replace=False)]
    name = lambda i: f"{tag}{i:02d}"  # noqa: E731
    trs = [(name(i), ev[i], name(i + 1), float(rng.choice([0, 1, 2.5, 10, -1]))) for i in range(k)]
    extra = []
    p = min(0.25, 3.0 / k)
    for i in range(k):
        for j in range(k):
            if j != i and rng.random() < p:
                kind = rng.integers(0, 3)
                dst = name(i) if kind == 0 else (name(0) if kind == 1 else name(min(i + 2, k)))
                extra.append((name(i), ev[j], dst, float(rng.choice([0, -0.5, 1]))))
    return trs[:-1] + extra + trs[-1:], ev


def _machine(rng, cells, n_states, tag, shuffle_names=False):
    """a machine with n_states states (n_states - 1 chain events); rewards partly replaced by values that round differently
    in float32; shuffle_names renames the states so that their index order (sorted names) is not the chain order"""
    k = n_states - 1
    if k <= 5:
        while True:
            rm, ev = random_machine(rng, cells, tag)
            if len(ev) == k:
                break
    else:
        rm, ev = _long_machine(rng, cells, k, tag)
    if rng.random() < 0.6:
        rm = [(s, e, d, float(rng.choice(ODD + [r]))) for (s, e, d, r) in rm]
    if shuffle_names:
        states = list(dict.fromkeys([x for (s, _e, d, _r) in rm for x in (s, d)]))
        perm = rng.permutation(len(states))
        new = {st: (st if st == rm[0][0] else f"{tag}x{perm[i]:02d}") for i, st in enumerate(states)}
        rm = [(new[s], e, new[d], r) for (s, e, d, r) in rm]
    return rm, ev


def _scenario(rng, family, i):
    """one draw of a scenario for `family`, before the admission check"""
    if i % 8 == 0:
        env = "office_world"  # the zero-probability slip outcome cases
    elif i % 8 == 4:
        env = "frozen_lake"
    else:
        env = "frozen_lake" if rng.random() < 0.5 else "office_world"
    map_name = "map1" if env == "frozen_lake" else str(rng.choice(["map0", "map1", "map2", "map3", "map4"]))
    grid = frozen_lake_grid(map_name) if env == "frozen_lake" else office_world_grid(map_name)
    hazards = set(grid.hazards)
    free = [(x, y) for y in range(grid.height) for x in range(grid.width) if (x, y) not in hazards]
    A = int(rng.integers(1, 9))
    starts = [free[j] for j in rng.choice(len(free), size=A, replace=False)]
    dtype = "f32"
    shuffle = False
    if family == "qrm4":
        n_states = 4
    elif family == "qrmn":
        n_states = 3 if i % 2 == 0 else 5
    elif family == "ql_fast":
        n_states = int(rng.integers(2, 7))
    else:  # qrm_block: NU bucket and table type from the case index (all 16 NU x type x fetch combinations in 16 cases)
        b = (i // 4) % 4
        nu_lo, nu_hi = [(2, 4), (5, 8), (9, 12), (13, 16)][(i % 4 + b) % 4]
        n_states = int(rng.integers(nu_lo, nu_hi + 1))
        dtype = "f64" if b % 2 else "f32"
        shuffle = rng.random() < 0.5
    rm, ev = _machine(rng, free, n_states, "s", shuffle_names=shuffle)
    detector = sorted(set(ev) | ({free[int(rng.integers(len(free)))]} if rng.random() < 0.3 else set()))
    sc = P.Scenario(env=env, map_name=map_name, starts=starts, rm_transitions=rm, detector_positions=detector,
                    algo="ql" if family == "ql_fast" else "qrm", seed=int(rng.integers(1, 1 << 30)), table_dtype=dtype)
    sc.driver = str(rng.choice(["frozen_lake_main", "office_main"]))
    if family == "ql_fast" and i % 4 == 1:
        sc.driver = "frozen_lake_main"  # first-iteration aliasing of the observation (RLRM_FLAG_FIRST)
    sc.stochastic = i % 3 != 1
    sc.delay_action = bool(sc.stochastic and rng.random() < 0.25)
    sc.all_slip = bool(env == "office_world" and rng.random() < 0.4)
    sc.high_prob = float(rng.choice([0.0, 1 / 3, 0.6, 0.8, 0.95, 1.0]))
    if i % 8 == 0:
        sc.delay_action, sc.high_prob = False, float(rng.choice([0.0, 1.0]))
    sc.penalty_amount = float(rng.choice([0, -1, -5.5, -1 / 3, 0.1]))
    sc.plants_penalty = float(rng.choice([-100, -3, 0, -1 / 3]))
    sc.wall_penalty = float(rng.choice([0, -0.25, -2, -1e-3, -1 / 3]))
    sc.terminate_on_plants = bool(rng.random() < 0.3)
    sc.terminate_hit_walls = bool(rng.random() < 0.25)
    sc.max_steps = int(rng.choice([12, 40, 150, 1000]))
    sc.reward_modifier = float(rng.choice([1, 1, 0.5, 3, 0.1]))
    sc.gamma = float(rng.choice([0.9, 0.99, 0.5, 1 / 3]))
    sc.q_init = float(rng.choice([0.0, 2.0, -1.0, 0.1]))
    sc.epsilon_start = float(rng.choice([0.01, 0.3, 1.0]))
    sc.epsilon_end = float(rng.choice([0.01, 0.1]))
    sc.epsilon_decay = float(rng.choice([1.0, 0.9, 0.999]))
    sc.learning_rate = float(rng.choice([1.0, 0.1, 0.37, 0.5]))
    if family == "qrm_block":
        if rng.random() < 0.3:
            sc.use_rsh, sc.rs_kind = True, str(rng.choice(["vi", "distance"]))
            sc.rs_gamma, sc.rs_alpha = float(rng.choice([0.9, 0.99])), float(rng.choice([100, 7]))
        sc.random_start_positions = bool(env == "frozen_lake" and rng.random() < 0.3)
    return sc


def _sweep(rng, sc):
    sets = []
    for _ in range(int(rng.integers(2, 5))):
        s = {}
        if rng.random() < 0.7:
            s["learning_rate"] = float(rng.choice([1.0, 0.05, 0.37, 0.9]))
        if not sc.use_rsh and rng.random() < 0.6:  # shaping potentials are built with the scenario's discount
            s["gamma"] = float(rng.choice([0.8, 0.9, 0.99, 1 / 3]))
        if rng.random() < 0.3:
            s["lambd"] = float(rng.choice([0.0, 0.5, 0.9]))
        if rng.random() < 0.6:
            s["epsilon_start"] = float(rng.choice([0.05, 0.6, 1.0]))
        if rng.random() < 0.5:
            s["epsilon_end"] = float(rng.choice([0.02, 0.1, 0.2]))
        if rng.random() < 0.5:
            s["epsilon_decay"] = float(rng.choice([0.9, 0.95, 1.0]))
        sets.append(s)
    return sets


def _launches(rng, total, all_four):
    """3-5 launches (4-5 with all_four) whose (learn, trace) pairs are distinct for the first four"""
    k = int(rng.integers(4, 6)) if all_four else int(rng.integers(3, 6))
    kinds = [(bool(x >> 1), bool(x & 1)) for x in rng.permutation(4)]
    kinds = (kinds + [kinds[int(rng.integers(4))]])[:k]
    cuts = sorted(rng.choice(np.arange(1, total), size=k - 1, replace=False)) if total > k else list(range(1, k))
    sizes = np.diff([0] + list(cuts) + [max(total, k)])
    return [(int(s), lr, tr) for s, (lr, tr) in zip(sizes, kinds)]


def make_case(family, i) -> Case:
    rng = np.random.default_rng(9000 + 1000 * FAMILIES.index(family) + i)
    for _attempt in range(200):
        sc = _scenario(rng, family, i)
        if admitted(P.compile_scenario(sc)) == family:
            break
    else:
        raise RuntimeError(f"no admissible draw for {family}-{i}")
    n = int(rng.choice([1, 31, 32, 33, 127, 128, 129, 1000]))
    sweep = group = None
    offset = 0
    if i % 4 == 3:
        sweep = _sweep(rng, sc)
        offset = int(rng.integers(1, n + 1)) if rng.random() < 0.5 else 0
        H = len(sweep)
        group = -(-(offset + n) // H)
        group += int(rng.integers(0, 3))
        if group % 32 == 0:
            group += 1  # group edges inside warps
    elif rng.random() < 0.35:
        offset = int(rng.choice([1, 31, 1000, 65535, 1 << 20]))
    A = len(sc.starts)
    total = min(int(rng.choice([150, 400, 700, 1500])), max(20, SLOT_STEPS // (n * A)))
    launches = _launches(rng, total, all_four=i < 3)
    tma = None
    if family == "qrm_block":
        want = (i // 8) % 2 == 1  # fetch variant from the case index; forced when the block size would pick the other
        natural = block_bytes(P.compile_scenario(sc).config) >= 192
        if want != natural or rng.random() < 0.3:
            tma = "1" if want else "0"
    return Case(family, i, sc, n, offset, launches, sweep, group, tma)


def make_minb8_case(j, num_sms=B200_SMS) -> Case:
    """qrm4 above the MINB 8 threshold (more than 7 resident blocks per SM of threads) of a device with num_sms SMs, about
    200 iterations"""
    rng = np.random.default_rng(8800 + j)
    while True:
        sc = _scenario(rng, "qrm4", 2 + 3 * j)  # stochastic, FrozenLake / OfficeWorld as drawn
        sc.starts = sc.starts[:2] if len(sc.starts) >= 2 else sc.starts
        if admitted(P.compile_scenario(sc)) == "qrm4":
            break
    G = 1 if len(sc.starts) == 1 else 2
    n = num_sms * 7 * TRAIN_BLOCK // G + 1025 + 512 * j  # a few blocks above the threshold, not a multiple of the block
    launches = _launches(rng, 200, all_four=False)
    sweep = group = None
    if j == 1:
        sweep = _sweep(rng, sc)
        group = -(-n // len(sweep)) + 5
    return Case("qrm4", 100 + j, sc, n, 0, launches, sweep, group)


def plan(n_cases=None) -> List[Case]:
    n_cases = N_CASES if n_cases is None else n_cases
    return [make_case(f, i) for f in FAMILIES for i in range(n_cases)] + [make_minb8_case(j) for j in range(2)]


def _lane_group(case):
    """threads per instance: the agent count rounded up to a power of two"""
    return 1 << (len(case.sc.starts) - 1).bit_length()


def expected_kernel(case, c, learn, trace, num_sms):
    cfg = c.config
    env, stoch, sw = int(cfg.env_kind), bool(cfg.stochastic), case.sweep is not None
    if case.family == "qrm4":
        minb = 8 if case.n * _lane_group(case) > num_sms * 7 * TRAIN_BLOCK else 7
        return KERNEL["qrm4"], (env, stoch, learn, trace, minb, sw)
    if case.family == "qrmn":
        return KERNEL["qrmn"], (env, int(cfg.n_rm_states), stoch, learn, trace, sw)
    if case.family == "qrm_block":
        tma = block_bytes(cfg) >= 192 if case.tma is None else case.tma == "1"
        t = "double" if cfg.table_dtype == abi.TABLE_F64 else "float"
        return KERNEL["qrm_block"], (env, nu_of(int(cfg.n_qrm_states)), t, tma, sw)
    return KERNEL["ql_fast"], (env, stoch, learn, trace, sw)


# ----------------------------------------------------------------------------------------------------------------------
# the GPU comparison
# ----------------------------------------------------------------------------------------------------------------------
def _setting_scenario(sc, s):
    scg = copy.deepcopy(sc)
    for k, v in s.items():
        setattr(scg, k, v)
    return scg


def _oracles(case, eng):
    """(local instance range, oracle) pairs covering the engine: one oracle per sweep group the engine's global ids
    [offset, offset + n) touch, built on that group's setting at the group's first global id"""
    import oracle as O

    if case.sweep is None:
        return [((0, case.n), O.Oracle(case.compiled(), case.n))]
    out = []
    lo_g, hi_g = case.offset, case.offset + case.n
    for g, s in enumerate(eng.sweep):
        lo, hi = max(lo_g, g * case.group), min(hi_g, (g + 1) * case.group)
        if lo < hi:
            c = P.compile_scenario(_setting_scenario(case.sc, s), instance_offset=lo)
            out.append(((lo - case.offset, hi - case.offset), O.Oracle(c, hi - lo)))
    assert sum(hi - lo for (lo, hi), _o in out) == case.n
    return out


def _run_case(case, monkeypatch):
    import oracle as O
    from multiagent_rlrm_b200.engine import Engine

    if case.tma is not None:
        monkeypatch.setenv("RLRM_QRMB_TMA", case.tma)
    c = case.compiled()
    eng = Engine(c, case.n, sweep=case.sweep, sweep_group=case.group)
    A = eng.A
    oracles = _oracles(case, eng)
    eng.reset()
    for _r, o in oracles:
        o.reset()
    info = case.describe()
    num_sms = _num_sms()
    t0 = 0
    for li, (iters, learn, trace) in enumerate(case.launches):
        box = {}
        ran = launched_train_kernels(lambda: box.update(tr=eng.train(iters, learn=learn, trace=trace)))
        fam, args = expected_kernel(case, c, learn, trace, num_sms)
        assert [(k.family, k.args) for k in ran] == [(fam, args)], (info, li, [k.name for k in ran])
        tr = box["tr"].cpu().numpy().view(np.uint32) if trace else None
        q = eng.q.cpu().numpy().reshape(case.n * A, -1)
        slot = eng.slot.cpu().numpy().view(np.uint64)
        eps, ret = eng.epsilon.cpu().numpy(), eng.ep_return.cpu().numpy()
        st = eng.stats_numpy()
        for (lo, hi), o in oracles:
            tr_o = o.train(t0, iters, learn, trace)
            sl = slice(lo * A, hi * A)
            where = (info, f"launch {li} (t0={t0}, {iters} iterations, learn={learn}, trace={trace}), instances [{lo}, {hi})")
            if trace:
                assert np.array_equal(tr[:, sl], tr_o), (where, "trace")
            assert np.array_equal(slot[sl], o.slot), (where, "slot")
            assert eps[sl].tobytes() == o.epsilon.tobytes(), (where, "epsilon")
            assert q[sl].tobytes() == o.q.reshape(hi * A - lo * A, -1).tobytes(), (where, "q")
            assert ret[sl].tobytes() == o.ep_return.tobytes(), (where, "ep_return")
            for f in O.STATS_DTYPE.names:
                assert st[f][sl].tobytes() == o.stats[f].tobytes(), (where, "stats." + f)
        t0 += iters
    return oracles


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("index", range(N_CASES))
def test_kernel_case_matches_oracle(family, index, cuda_device, monkeypatch):
    _run_case(make_case(family, index), monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("j", [0, 1])
def test_qrm4_minb8_case_matches_oracle(j, cuda_device, monkeypatch):
    _run_case(make_minb8_case(j, _num_sms()), monkeypatch)


# ----------------------------------------------------------------------------------------------------------------------
# the plan's coverage (CPU)
# ----------------------------------------------------------------------------------------------------------------------
def test_plan_coverage():
    """Every case is admitted by its family, and the default plan reaches every instantiation the GPU tests claim."""
    cases = plan(max(N_CASES, DEFAULT_CASES))
    seen = {f: set() for f in FAMILIES}
    envs = {f: set() for f in FAMILIES}
    zero_p = {f: 0 for f in FAMILIES}
    sweeps = {f: 0 for f in FAMILIES}
    nq, block, minb8 = set(), set(), 0
    ids = set()
    for case in cases:
        assert case.id not in ids
        ids.add(case.id)
        c = case.compiled()
        assert admitted(c) == case.family, case.describe()
        assert 3 <= len(case.launches) <= 5 and all(it > 0 for it, _l, _t in case.launches), case.describe()
        if case.index < 100:
            assert case.n in (1, 31, 32, 33, 127, 128, 129, 1000)
            assert case.n * c.n_agents * sum(it for it, _l, _t in case.launches) <= max(SLOT_STEPS, 20 * case.n * c.n_agents)
        if case.sweep is not None:
            sweeps[case.family] += 1
            assert 2 <= len(case.sweep) <= 4 and len(case.sweep) * case.group >= case.offset + case.n
            if case.sc.use_rsh:
                assert all("gamma" not in s for s in case.sweep)
        envs[case.family].add(int(c.config.env_kind))
        zero_p[case.family] += zero_probability_outcome(c.config)
        for iters, learn, trace in case.launches:
            fam, args = expected_kernel(case, c, learn, trace, B200_SMS)
            seen[case.family].add((bool(c.config.stochastic), learn, trace))
            if case.family == "qrmn":
                nq.add(args[1])
            if case.family == "qrm_block":
                block.add(args[1:4])
            if case.family == "qrm4" and args[4] == 8:
                minb8 += 1
    everything = {(s, l, t) for s in (False, True) for l in (False, True) for t in (False, True)}
    for f in FAMILIES:
        assert seen[f] == everything, (f, everything - seen[f])
        assert envs[f] == {FL, OW}, f
        assert zero_p[f] > 0, f
        assert sweeps[f] > 0, f
    assert nq == {3, 5}
    assert block == {(nu, t, tma) for nu in (3, 7, 11, 15) for t in ("float", "double") for tma in (False, True)}, block
    assert minb8 > 0
    # the scenario dimensions the generators draw from: a change to them must not drop a value unnoticed
    office = [c.sc for c in cases if c.sc.env == "office_world"]
    frozen = [c.sc for c in cases if c.sc.env == "frozen_lake"]
    assert {sc.map_name for sc in office} == {"map0", "map1", "map2", "map3", "map4"}
    assert {sc.high_prob for sc in office if sc.stochastic and not sc.delay_action} == {0.0, 1 / 3, 0.6, 0.8, 0.95, 1.0}
    assert any(sc.all_slip and sc.stochastic and not sc.delay_action for sc in office)
    assert any(sc.delay_action for sc in office) and any(sc.delay_action for sc in frozen)
    assert {c.sc.max_steps for c in cases} == {12, 40, 150, 1000}
    for values in ([sc.penalty_amount for sc in frozen], [sc.plants_penalty for sc in office], [sc.wall_penalty for sc in office]):
        assert 0 in values and any(v != 0 for v in values), values
    assert any(sc.terminate_on_plants for sc in office) and any(sc.terminate_hit_walls for sc in office)
    assert any(len(c.sc.starts) == 1 for c in cases) and any(len(c.sc.starts) == 8 for c in cases)
    assert any(any(r in ODD for (_s, _e, _d, r) in c.sc.rm_transitions) for c in cases)
    blocks = [c for c in cases if c.family == "qrm_block"]
    assert any(list(c.compiled().qrm_states) != sorted(c.compiled().qrm_states) for c in blocks)  # states in any index order
    assert any(c.sc.use_rsh and c.sc.rs_kind == "vi" for c in blocks) and any(c.sc.use_rsh and c.sc.rs_kind == "distance" for c in blocks)
    assert any(c.sc.random_start_positions for c in blocks)
    assert any(c.sc.driver == "frozen_lake_main" for c in cases if c.family == "ql_fast")
    assert any(c.offset for c in cases if c.sweep is None) and any(c.offset for c in cases if c.sweep is not None)


def test_kernel_name_parsing():
    k = parse_kernel_name("void train_qrm4_kernel<0, true, true, false, 7, false>(KP, DState, unsigned long long, int, unsigned int*, Sweep)")
    assert k.family == "train_qrm4_kernel" and k.args == (0, True, True, False, 7, False)
    k = parse_kernel_name("void train_qrm_block_kernel<1, 11, double, true, true>(KP, DState, unsigned long long, int, int, unsigned int*, Sweep)")
    assert k.family == "train_qrm_block_kernel" and k.args == (1, 11, "double", True, True)
    assert parse_kernel_name("void reset_kernel<0>(KP, DState)") is None
    assert parse_kernel_name("void train_kernel<1, 1, false, float, false>(KP)").args == (1, 1, False, "float", False)
