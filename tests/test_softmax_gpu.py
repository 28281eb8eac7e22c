"""GPU: softmax exploration (rlrm_set_exploration) against its CPU oracle (tests/softmax_oracle.c), bit for bit.

* `test_select_boundaries`: for random rows, float32 / float64 tables and every n_actions, the thresholds T_j come from the
  oracle and w1 = T_j - 1, T_j, T_j + 1 is injected through rlrm_select_action and rlrm_update_list_select; the device must
  choose j, j + 1, j + 1. A one-ULP difference between the device's and the oracle's exp that moves a decision fails here.
* `test_softmax_case_matches_oracle`: seeded random cases of QL, QRM and dense / sparse Q(lambda) over both environments and
  drivers, float32 / float64 tables, per-agent machines, shaping, random starts, visit counts, sweeps and instance offsets, 3-5
  launches mixing learn / trace; after every launch slot, epsilon, Q, traces, visits, running return, stats and trace equal
  the oracle's. `test_plan_coverage` (CPU) checks what the plan reaches. RLRM_SMFUZZ_CASES sets the number of cases per family.
* `test_routes`: under softmax every launch runs train_kernel or a Q(lambda) kernel with SOFTMAX = true; after
  kind = 0 the scenario runs its epsilon-greedy kernel again (profiled in fresh child processes, see launched_train_kernels).
* equalities: iterate() == train(1), iterate_unfused == train, 300 + save / load + 300 == 600, and softmax then kind = 0 ==
  a handle that never set it; ABI errors."""
import copy
import ctypes as C
import json
import os
import subprocess
import sys
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import pytest

import multiagent_rlrm_b200 as P
from multiagent_rlrm_b200 import _abi as abi
from multiagent_rlrm_b200.maps import frozen_lake_grid, office_world_grid
from test_fuzz_gpu import random_machine

FAMILIES = ("ql", "qrm", "qlambda", "qlambda_sparse")
N_CASES = int(os.environ.get("RLRM_SMFUZZ_CASES", "12"))
TEMPS = (0.02, 0.3, 1.0, 7.5)


# ----------------------------------------------------------------------------------------------------------------------
# boundaries of the selection
# ----------------------------------------------------------------------------------------------------------------------
def _select_engine(real, n_actions, n, tau):
    from multiagent_rlrm_b200.engine import Engine

    sc = P.Scenario(env="frozen_lake", map_name="map1", starts=[(0, 0)], rm_transitions=[("u0", (1, 1), "u1", 1.0)],
                    detector_positions=[(1, 1)], algo="ql", seed=11, table_dtype=real)
    c = P.compile_scenario(sc)
    c.config.n_actions = n_actions
    eng = Engine(c, n, exploration="softmax", temperature=tau, host_control=False)
    eng.reset()
    return eng


def _random_rows(rng, n, n_actions, dt):
    rows = rng.choice([0.0, 1.0, -1.0, 0.5, 0.25, -3000.0, 1e-3, 2.0, 0.1], size=(n, 4)).astype(dt)
    tweak = rng.random((n, 4)) < 0.3
    rows[tweak] += rng.standard_normal(int(tweak.sum())).astype(dt)
    rows[:, n_actions:] = rng.choice([100.0, -100.0, 0.0], size=(n, 4 - n_actions)).astype(dt)  # unused entries are ignored
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("n_actions", [1, 2, 3, 4])
def test_select_boundaries(real, n_actions, cuda_device):
    import softmax_oracle as SO
    import torch

    rng = np.random.default_rng(31 * n_actions + (real == "f64"))
    dt = np.float32 if real == "f32" else np.float64
    n = 600
    for tau in TEMPS:
        eng = _select_engine(real, n_actions, n, tau)
        rows = _random_rows(rng, n, n_actions, dt)
        cell = int(eng.slots_numpy()["cell"][0, 0])
        enc = cell * int(eng.cfg.n_rm_states)
        q = eng.q.cpu().numpy()
        q[:, enc, :] = rows
        eng.q.copy_(torch.from_numpy(q))
        w1 = np.zeros(n, dtype=np.uint64)
        want = np.zeros(n, dtype=np.int64)
        for i in range(n):
            thr = SO.softmax_thresholds(rows[i, :n_actions], tau, real)
            if thr.size == 0:
                w1[i] = rng.integers(0, 1 << 32)
                continue
            j = int(rng.integers(thr.size))
            w1[i] = min(max(int(thr[j]) + int(rng.integers(-1, 2)), 0), (1 << 32) - 1)
            want[i] = int(np.sum(w1[i] >= thr))
        draws = rng.integers(0, 1 << 32, size=(n, 1, 4), dtype=np.uint64)
        draws[:, 0, 1] = w1
        draws = torch.from_numpy(draws.astype(np.uint32).view(np.int32))
        got = eng.select_action(draws=draws).cpu().numpy().reshape(-1)
        assert np.array_equal(got, want), (real, n_actions, tau, np.nonzero(got != want)[0][:5])
        # the same selections through rlrm_update_list_select (n = 0: selection only), on a page-locked request
        buf = torch.zeros(C.sizeof(abi.SelectReq), dtype=torch.uint8).pin_memory()
        req = abi.SelectReq.from_buffer(buf.numpy())
        d32 = draws.numpy().view(np.uint32)
        for i in range(0, n, 7):
            req.state, req.best, req.epsilon, req.seq = enc, 0, 1.0, i + 1
            for k in range(4):
                req.draws[k] = int(d32[i, 0, k])
            P_check(eng.L.rlrm_update_list_select(eng.h, C.byref(eng.state), i, 0, None, buf.data_ptr(), eng._stream()))
            eng.sync()
            assert req.done_seq == i + 1 and req.action == want[i], (real, n_actions, tau, i, req.action, want[i])
        # greedy evaluation stays the first argmax
        best = eng.select_action(draws=draws, best=True).cpu().numpy().reshape(-1)
        assert np.array_equal(best, np.argmax(rows, axis=1))


def P_check(rc):
    from multiagent_rlrm_b200._lib import check

    check(rc)


# ----------------------------------------------------------------------------------------------------------------------
# training cases against the oracle
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class Case:
    family: str
    index: int
    sc: object
    n: int
    offset: int
    tau: float
    launches: list
    sweep: Optional[list]
    group: Optional[int]
    track_visits: bool

    @property
    def id(self):
        return f"{self.family}-{self.index}"

    def compiled(self):
        return P.compile_scenario(self.sc, instance_offset=self.offset)

    def describe(self):
        sc = self.sc
        return (f"{self.id}: {sc.env}/{sc.map_name} A={len(sc.starts)} {sc.algo} {sc.table_dtype} per_agent="
                f"{sc.rm_transitions_per_agent is not None} rsh={sc.use_rsh} rs={sc.random_start_positions} driver={sc.driver} "
                f"stoch={sc.stochastic} lr={sc.learning_rate} n={self.n} off={self.offset} tau={self.tau} sweep={self.sweep} "
                f"k={self.group} visits={self.track_visits} launches={self.launches}")


def make_case(family, i) -> Case:
    rng = np.random.default_rng(7100 + 1000 * FAMILIES.index(family) + i)
    env = "frozen_lake" if i % 2 == 0 else "office_world"
    map_name = "map1" if env == "frozen_lake" else str(rng.choice(["map0", "map1", "map2", "map3", "map4"]))
    grid = frozen_lake_grid(map_name) if env == "frozen_lake" else office_world_grid(map_name)
    hazards = set(grid.hazards)
    free = [(x, y) for y in range(grid.height) for x in range(grid.width) if (x, y) not in hazards]
    A = int(rng.integers(2 if i % 4 == 1 else 1, 5))
    starts = [free[j] for j in rng.choice(len(free), size=A, replace=False)]
    algo = "qlambda" if family.startswith("qlambda") else family
    per = None
    if i % 4 == 1:
        machines = [random_machine(rng, free, f"m{a}_") for a in range(A)]
        rm, per = machines[0][0], [m[0] for m in machines]
        detector = sorted({p for m in machines for p in m[1]})
    else:
        rm, ev = random_machine(rng, free, "s")
        detector = sorted(set(ev))
    sc = P.Scenario(env=env, map_name=map_name, starts=starts, rm_transitions=rm, rm_transitions_per_agent=per,
                    detector_positions=detector, algo=algo, seed=int(rng.integers(1, 1 << 30)),
                    table_dtype="f64" if i % 3 == 2 else "f32")
    sc.driver = "frozen_lake_main" if (i // 2) % 2 == 0 else "office_main"
    sc.stochastic = bool(rng.random() < 0.7)
    sc.all_slip = bool(env == "office_world" and rng.random() < 0.3)
    sc.penalty_amount = float(rng.choice([0, -1, -5.5]))
    sc.wall_penalty = float(rng.choice([0, -0.25]))
    sc.max_steps = int(rng.choice([12, 40, 150]))
    sc.gamma = float(rng.choice([0.9, 0.99, 0.5]))
    sc.q_init = float(rng.choice([0.0, 2.0, -1.0, 0.1]))
    sc.epsilon_start, sc.epsilon_end, sc.epsilon_decay = 0.5, 0.05, float(rng.choice([1.0, 0.9]))
    track_visits = False
    if algo == "qlambda":
        sc.learning_rate, sc.lambd = float(rng.choice([0.1, 0.5])), float(rng.choice([0.0, 0.5, 0.9]))
        if family == "qlambda" and i % 6 == 5:
            sc.learning_rate = None
    else:
        sc.learning_rate = None if i % 6 == 5 else float(rng.choice([1.0, 0.1, 0.37]))
        track_visits = i % 6 == 4
        if i % 4 == 3:
            sc.use_rsh, sc.rs_kind = True, str(rng.choice(["vi", "distance"]))
            sc.rs_gamma, sc.rs_alpha = sc.gamma, float(rng.choice([100, 7]))
    sc.random_start_positions = bool(env == "frozen_lake" and i % 4 == 2)
    n = int(rng.choice([1, 7, 33, 128, 257]))
    sweep = group = None
    offset = 0
    if i % 3 == 1:
        sweep = [{"epsilon_decay": 0.95}, {"lambd": 0.3, "learning_rate": 0.2}, {"epsilon_start": 1.0}][: int(rng.integers(2, 4))]
        offset = int(rng.integers(0, n + 1))
        group = -(-(offset + n) // len(sweep)) + int(rng.integers(0, 3))
    elif rng.random() < 0.4:
        offset = int(rng.choice([1, 31, 1000, 1 << 20]))
    total = int(rng.choice([150, 400]))
    k = int(rng.integers(3, 6))
    kinds = [(bool(x >> 1), bool(x & 1)) for x in rng.permutation(4)]
    kinds = (kinds + [kinds[0]])[:k]
    cuts = sorted(rng.choice(np.arange(1, total), size=k - 1, replace=False))
    launches = [(int(s), lr, tr) for s, (lr, tr) in zip(np.diff([0] + cuts + [total]), kinds)]
    return Case(family, i, sc, n, offset, float(TEMPS[i % len(TEMPS)]), launches, sweep, group, track_visits)


def plan(n_cases=None) -> List[Case]:
    n_cases = N_CASES if n_cases is None else n_cases
    return [make_case(f, i) for f in FAMILIES for i in range(n_cases)]


def _engine(case, **kw):
    from multiagent_rlrm_b200.engine import Engine

    return Engine(case.compiled(), case.n, sweep=case.sweep, sweep_group=case.group, track_visits=case.track_visits,
                  qlambda_sparse=case.family == "qlambda_sparse", exploration="softmax", temperature=case.tau, **kw)


def _oracles(case, eng):
    """(local instance range, oracle) pairs: one oracle per sweep group the engine's global ids touch"""
    import softmax_oracle as SO

    kw = dict(temperature=case.tau, track_visits=case.track_visits)
    if case.sweep is None:
        return [((0, case.n), SO.SoftmaxOracle(case.compiled(), case.n, **kw))]
    out = []
    for g, s in enumerate(eng.sweep):
        lo, hi = max(case.offset, g * case.group), min(case.offset + case.n, (g + 1) * case.group)
        if lo < hi:
            scg = copy.deepcopy(case.sc)
            for key, v in s.items():
                setattr(scg, key, v)
            out.append(((lo - case.offset, hi - case.offset), SO.SoftmaxOracle(P.compile_scenario(scg, instance_offset=lo), hi - lo, **kw)))
    assert sum(hi - lo for (lo, hi), _o in out) == case.n
    return out


def _run_case(case):
    import oracle as O

    eng = _engine(case)
    A = eng.A
    oracles = _oracles(case, eng)
    eng.reset()
    for _r, o in oracles:
        o.reset()
    t0 = 0
    for li, (iters, learn, trace) in enumerate(case.launches):
        tr = eng.train(iters, learn=learn, trace=trace)
        tr = tr.cpu().numpy().view(np.uint32) if trace else None
        e = eng.sync_tables(with_traces=True)
        q = eng.q.cpu().numpy().reshape(case.n, -1)
        vis = eng.visits.cpu().numpy().view(np.uint32).reshape(case.n, -1) if eng.visits is not None else None
        e = e.cpu().numpy().reshape(case.n, -1) if e is not None else None
        slot = eng.slot.cpu().numpy().view(np.uint64)
        eps, ret = eng.epsilon.cpu().numpy(), eng.ep_return.cpu().numpy()
        st = eng.stats_numpy()
        for (lo, hi), o in oracles:
            tr_o = o.train(t0, iters, learn, trace)
            sl = slice(lo * A, hi * A)
            where = (case.describe(), f"launch {li} (t0={t0}, {iters} iterations, learn={learn}, trace={trace}), instances [{lo}, {hi})")
            if trace:
                assert np.array_equal(tr[:, sl], tr_o), (where, "trace")
            assert np.array_equal(slot[sl], o.slot), (where, "slot")
            assert eps[sl].tobytes() == o.epsilon.tobytes(), (where, "epsilon")
            if case.family == "qlambda_sparse":  # sparse traces: equal up to the sign of zero
                assert np.array_equal(q[lo:hi].reshape(-1), o.q.reshape(-1)), (where, "q")
                assert np.array_equal(e[lo:hi].reshape(-1), o.e.reshape(-1)), (where, "e")
            else:
                assert q[lo:hi].tobytes() == o.q.tobytes(), (where, "q")
                if e is not None:
                    assert e[lo:hi].tobytes() == o.e.tobytes(), (where, "e")
            if o.visits is not None:
                assert np.array_equal(vis[lo:hi].reshape(-1), o.visits.reshape(-1)), (where, "visits")
            assert ret[sl].tobytes() == o.ep_return.tobytes(), (where, "ep_return")
            for f in O.STATS_DTYPE.names:
                assert st[f][sl].tobytes() == o.stats[f].tobytes(), (where, "stats." + f)
        t0 += iters
    return eng


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("index", range(N_CASES))
def test_softmax_case_matches_oracle(family, index, cuda_device):
    _run_case(make_case(family, index))


def test_plan_coverage():
    """CPU: the default plan reaches every family x environment x driver x table type, per-agent machines, shaping, random
    starts, visit counts, learning_rate None, sweeps, instance offsets, every temperature and learn / trace mixes"""
    cases = plan(12)
    seen = set()
    for c in cases:
        sc = c.sc
        seen.update({("env", c.family, sc.env), ("driver", c.family, sc.driver), ("dtype", c.family, sc.table_dtype),
                     ("tau", c.tau), ("sweep", c.family, c.sweep is not None), ("offset", c.offset > 0)})
        if sc.rm_transitions_per_agent is not None:
            seen.add(("per_agent", c.family))
        if sc.use_rsh:
            seen.add(("rsh", c.family))
        if sc.random_start_positions:
            seen.add(("random_starts", c.family))
        if sc.learning_rate is None:
            seen.add(("lr_none", c.family))
        if c.track_visits:
            seen.add(("visits", c.family))
        assert 3 <= len(c.launches) <= 5
        for _it, lr, tr in c.launches:
            seen.add(("launch", lr, tr))
    for f in FAMILIES:
        for env in ("frozen_lake", "office_world"):
            assert ("env", f, env) in seen, (f, env)
        for drv in ("frozen_lake_main", "office_main"):
            assert ("driver", f, drv) in seen, (f, drv)
        for dt in ("f32", "f64"):
            assert ("dtype", f, dt) in seen, (f, dt)
        for s in (False, True):
            assert ("sweep", f, s) in seen, (f, s)
        assert ("per_agent", f) in seen and ("random_starts", f) in seen, f
    for f in ("ql", "qrm"):
        assert ("rsh", f) in seen and ("visits", f) in seen and ("lr_none", f) in seen, f
    assert ("lr_none", "qlambda") in seen
    assert all(("tau", t) in seen for t in TEMPS) and ("offset", True) in seen
    assert all(("launch", lr, tr) in seen for lr in (False, True) for tr in (False, True))


# ----------------------------------------------------------------------------------------------------------------------
# routes, profiled in fresh child processes
# ----------------------------------------------------------------------------------------------------------------------
ROUTE_NAMED = ["cfg3_qrm", "exp1", "exp3", "exp5_f32", "cfg3_f64", "chain12", "cfg3_ql", "cfg2", "track_visits", "lr_none"]


def _route_scenarios():
    """(id, scenario, n, Engine keywords) of the named scenarios with a specialised or generic epsilon-greedy kernel, with and
    without a sweep, and the Q(lambda) ones dense and sparse"""
    from test_fuzz_kernels_gpu import _named

    out = []
    for name in ROUTE_NAMED:
        sc, n, kw, _reserved, _fam, _args = _named(name, 148)
        out.append((name, sc, n, kw))
        out.append((name + "+sweep", sc, n, dict(kw, sweep=[{"epsilon_start": 0.3}, {"learning_rate": 0.2}], sweep_group=(n + 1) // 2)))
    for sparse in (False, True):
        sc = P.scenario_config4()
        sc.max_steps = 60
        out.append((f"qlambda_sparse={sparse}", sc, 64, {"qlambda_sparse": sparse}))
        out.append((f"qlambda_sparse={sparse}+sweep", sc, 64, {"qlambda_sparse": sparse, "sweep": [{"lambd": 0.5}, {}], "sweep_group": 32}))
    return out


def _route_child():
    """child process: per scenario the kernels of (a) a fresh epsilon-greedy engine, (b) a softmax engine, (c) the same engine
    after kind = 0, as JSON"""
    from multiagent_rlrm_b200.engine import Engine
    from test_fuzz_kernels_gpu import launched_train_kernels

    res = {}
    for name, sc, n, kw in _route_scenarios():
        c = P.compile_scenario(sc)
        base, soft = Engine(c, n, **kw), Engine(c, n, exploration="softmax", temperature=0.5, **kw)
        base.reset(); soft.reset()

        def run(e):
            return [[k.family, list(k.args)] for k in launched_train_kernels(lambda: (e.train(2), e.train(1, learn=False, trace=True)))]

        got = {"base": run(base), "softmax": run(soft)}
        soft.set_exploration("epsilon_greedy")
        got["back"] = run(soft)
        res[name] = got
    print("ROUTES " + json.dumps(res))


@pytest.mark.gpu
def test_routes(cuda_device):
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    code = f"import sys; sys.path[:0] = {[here, root, os.path.join(root, 'oracle')]!r}; import test_softmax_gpu as T; T._route_child()"
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable, *flags, "-c", code], capture_output=True, text=True, timeout=900, cwd=root)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    line = [x for x in res.stdout.splitlines() if x.startswith("ROUTES ")]
    assert line, res.stdout[-3000:] + res.stderr[-3000:]
    got = json.loads(line[-1][len("ROUTES "):])
    specialised = 0
    for name, _sc, _n, kw in _route_scenarios():
        r = got[name]
        assert len(r["base"]) == 2 and len(r["softmax"]) == 2, (name, r)
        sweep = "sweep" in kw
        for fam, args in r["softmax"]:  # the SOFTMAX flag follows SWEEP; train_kernel's epsilon-greedy instantiations have neither
            assert fam in ("train_kernel", "train_qlambda_kernel", "train_qlambda_sparse_kernel") and args[-2:] == [sweep, True], (name, fam, args)
            assert fam != "train_kernel" or len(args) == 6, (name, fam, args)
        for fam, args in r["base"]:
            assert not (fam == "train_kernel" and len(args) == 6) and not (fam.startswith("train_qlambda") and args[-1]), (name, fam, args)
        specialised += r["base"][0][0] not in ("train_kernel", "train_qlambda_kernel", "train_qlambda_sparse_kernel")
        assert r["back"] == r["base"], (name, r)
    assert specialised >= 12, specialised  # the specialised families really were in play


# ----------------------------------------------------------------------------------------------------------------------
# equalities and ABI errors
# ----------------------------------------------------------------------------------------------------------------------
def _state_bytes(eng, keys=None):
    eng.sync_tables()
    keys = [k for k in (keys or eng._STATE_TENSORS) if getattr(eng, k) is not None]
    return {k: getattr(eng, k).cpu().numpy().tobytes() for k in keys}


EQ_CASES = [("ql", 0), ("qrm", 1), ("qlambda", 2), ("qrm", 6), ("ql", 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("family,index", EQ_CASES)
def test_iterate_equals_train(family, index, cuda_device):
    import torch

    case = make_case(family, index)
    a, b = _engine(case), _engine(case)
    a.reset(); b.reset()
    a.train(120)
    rec = torch.zeros(case.n * a.A, dtype=torch.int32, device=a.device)
    for _ in range(120):
        b.iterate(record=rec, sync=False)
    assert _state_bytes(a) == _state_bytes(b)


@pytest.mark.gpu
@pytest.mark.parametrize("family,index", EQ_CASES)
def test_iterate_unfused_equals_train(family, index, cuda_device):
    case = make_case(family, index)
    a, b = _engine(case), _engine(case)
    a.reset(); b.reset()
    a.train(120)
    for _ in range(120):
        b.iterate_unfused()
    # the call-by-call entry points keep no running return or statistics (as in test_random_scenario_call_by_call_equals_fused)
    keys = ("slot", "epsilon", "q", "e", "visits")
    assert _state_bytes(a, keys) == _state_bytes(b, keys)


@pytest.mark.gpu
@pytest.mark.parametrize("family,index", EQ_CASES + [("qlambda_sparse", 4)])
def test_checkpoint_resume(family, index, cuda_device):
    case = make_case(family, index)
    a, b = _engine(case), _engine(case)
    a.reset(); b.reset()
    a.train(600)
    b.train(300)
    sd = b.state_dict()
    c = _engine(case)
    c.load_state_dict(sd)
    c.train(300)
    assert _state_bytes(a) == _state_bytes(c)
    from multiagent_rlrm_b200.engine import Engine

    for kw in ({}, {"exploration": "softmax", "temperature": case.tau * 2}):
        d = Engine(case.compiled(), case.n, sweep=case.sweep, sweep_group=case.group, track_visits=case.track_visits,
                   qlambda_sparse=case.family == "qlambda_sparse", **kw)
        with pytest.raises(ValueError, match="exploration"):
            d.load_state_dict(sd)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg3_qrm", "cfg3_ql", "exp3", "chain12"])
def test_softmax_then_epsilon_greedy_equals_never_set(name, cuda_device):
    from multiagent_rlrm_b200.engine import Engine
    from test_fuzz_kernels_gpu import _named

    sc, n, kw, _r, _f, _a = _named(name, 148)
    c = P.compile_scenario(sc)
    a, b = Engine(c, n, **kw), Engine(c, n, exploration="softmax", temperature=0.1, **kw)
    b.set_exploration("epsilon_greedy")
    a.reset(); b.reset()
    for e in (a, b):
        e.train(200)
        e.train(50, learn=False, trace=True)
        e.iterate()
    assert _state_bytes(a) == _state_bytes(b)
    assert b.state_dict()["exploration"] == "epsilon_greedy"


@pytest.mark.gpu
def test_set_exploration_errors(cuda_device):
    from multiagent_rlrm_b200.engine import Engine

    eng = Engine(P.compile_scenario(P.scenario_config3(True)), 4)
    L = eng.L
    ERR_ARG, ERR_UNSUPPORTED = -1, -3  # RLRM_ERR_ARG, RLRM_ERR_UNSUPPORTED
    for kind, tau in [(2, 1.0), (-1, 1.0), (1, 0.0), (1, -1.0), (1, float("nan")), (1, float("inf")), (1, 1e-320)]:
        assert L.rlrm_set_exploration(eng.h, kind, tau) == ERR_ARG, (kind, tau)
    assert L.rlrm_set_exploration(eng.h, 1, 0.5) == 0
    assert L.rlrm_set_exploration(eng.h, 0, float("nan")) == 0  # the temperature is not read for epsilon-greedy
    shared = Engine(P.compile_scenario(P.scenario_config5(True)), 4)
    assert L.rlrm_set_exploration(shared.h, 1, 0.5) == ERR_UNSUPPORTED
    assert L.rlrm_set_exploration(shared.h, 0, 1.0) == 0
    with pytest.raises(P_error()):
        Engine(P.compile_scenario(P.scenario_config5(True)), 4, exploration="softmax", temperature=1.0)
    with pytest.raises(ValueError):
        Engine(P.compile_scenario(P.scenario_config3(True)), 4, exploration="boltzmann")


def P_error():
    from multiagent_rlrm_b200._lib import RlrmError

    return RlrmError
