"""CPU: host-side logic — C-ABI surface (struct layout, exported symbols, loud failure without CUDA), map parsers,
Reward Machine bookkeeping, encoders, agent plumbing, the table compiler (brute force against the live reference when
its sources are present) and the slip-threshold arithmetic."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT

import multiagent_rlrm_b200 as P
from multiagent_rlrm_b200 import _abi as abi
from multiagent_rlrm_b200 import maps, tables
from ref_harness import REFERENCE_MISSING, REFERENCE_ROOT, reference_available

HEADER = os.path.join(ROOT, "include", "rlrm_b200.h")
HAVE_REF = reference_available()


# ---------------------------------------------------------------------------------------------- C ABI
def test_ctypes_structs_match_the_header(tmp_path):
    fields = {
        "rlrm_config_t": [f for f, _ in abi.Config._fields_],
        "rlrm_tables_t": [f for f, _ in abi.Tables._fields_],
        "rlrm_stats_t": [f for f, _ in abi.Stats._fields_],
        "rlrm_state_t": [f for f, _ in abi.State._fields_],
        "rlrm_step_out_t": [f for f, _ in abi.StepOut._fields_],
        "rlrm_eval_t": [f for f, _ in abi.Eval._fields_],
        "rlrm_select_req_t": [f for f, _ in abi.SelectReq._fields_],
        "rlrm_experience_t": [f for f, _ in abi.Experience._fields_],
    }
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){"]
    for st, fs in fields.items():
        lines.append(f'printf("{st} %zu\\n", sizeof({st}));')
        for f in fs:
            lines.append(f'printf("{st}.{f} %zu\\n", offsetof({st}, {f}));')
    lines.append("return 0;}")
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(src)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for st, cls in (("rlrm_config_t", abi.Config), ("rlrm_tables_t", abi.Tables), ("rlrm_stats_t", abi.Stats),
                    ("rlrm_state_t", abi.State), ("rlrm_step_out_t", abi.StepOut), ("rlrm_eval_t", abi.Eval),
                    ("rlrm_select_req_t", abi.SelectReq), ("rlrm_experience_t", abi.Experience)):
        assert int(out[st]) == C.sizeof(cls), st
        for f, _ in cls._fields_:
            assert int(out[f"{st}.{f}"]) == getattr(cls, f).offset, f"{st}.{f}"
    assert C.sizeof(abi.Stats) == 32 and C.sizeof(abi.SelectReq) == 48 and C.sizeof(abi.Experience) == 24


def test_library_loads_and_exports_every_declared_symbol():
    from multiagent_rlrm_b200 import _lib

    declared = set(re.findall(r"\b(rlrm_[a-z_]+)\s*\(", open(HEADER).read()))
    assert declared == set(abi.EXPORTED_SYMBOLS)
    _lib.build()
    L = _lib.load()
    for name in declared:
        assert hasattr(L, name), name
    assert L.rlrm_abi_version() == abi.ABI_VERSION


def test_fails_loudly_without_cuda():
    import torch

    if torch.cuda.is_available():
        pytest.skip("only meaningful on a box without a GPU")
    from multiagent_rlrm_b200 import _lib
    from multiagent_rlrm_b200.engine import Engine

    c = P.compile_scenario(P.scenario_config1())
    with pytest.raises(RuntimeError, match="CUDA"):
        Engine(c, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        P.QLearning(gamma=0.9, action_selection="greedy", learning_rate=1.0, state_space_size=4, action_space_size=4)
    L = _lib.load()
    h = C.c_void_p()
    t = c.tables_struct()
    assert L.rlrm_create(C.byref(c.config), C.byref(t), 0, C.byref(h)) == -2  # RLRM_ERR_CUDA
    assert b"no CPU fallback" in L.rlrm_last_error()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "multiagent-rl-rm_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(import|from)\s+(oracle|ref_harness|philox)\b", src, re.M), fn


# ---------------------------------------------------------------------------------------------- maps
def _tup(x):
    return [tuple(p) for p in x]


def test_ascii_maps_equal_reference_parsers_output():
    ref = json.load(open(os.path.join(GOLDEN_DIR, "maps.json")))
    for name, want in ref["frozen_lake"].items():
        holes, goals, dims = maps.parse_frozen_lake_rows(maps.FROZEN_LAKE_MAPS[name])
        assert holes == _tup(want["holes"]) and dims == tuple(want["dims"])
        assert goals == {k: tuple(v) for k, v in want["goals"].items()}
    for name, want in ref["office_world"].items():
        rows, grid_size, start = maps.OFFICE_WORLD_MAPS[name]
        coords, goals, walls = maps.parse_office_rows(rows)
        for k in ("plant", "coffee", "letter", "empty_cell"):
            assert coords[k] == _tup(want["coordinates"][k]), (name, k)
        assert goals == {k: tuple(v) for k, v in want["goals"].items()}
        assert walls == [(tuple(a), tuple(b)) for a, b in want["walls"]], name
        assert tuple(grid_size) == tuple(want["grid_size"]) and tuple(start) == tuple(want["start"])


def test_emoji_front_ends_round_trip():
    """/root/reference/tests/test_utils_encoding.py:49-69 style: tiny maps through the emoji parsers."""
    holes, goals, dims = P.parse_map_emoji("A 🟩\n⛔ B")
    assert holes == [(0, 1)] and goals == {"A": (0, 0), "B": (1, 1)} and dims == (2, 2)
    for name, (rows, _gs, _st) in maps.OFFICE_WORLD_MAPS.items():
        assert P.parse_office_world(maps.emoji_from_ascii_rows(rows)) == maps.parse_office_rows(rows), name
    rows = maps.FROZEN_LAKE_MAPS["map1"]
    assert P.parse_map_emoji(maps.emoji_from_ascii_rows(rows)) == maps.parse_frozen_lake_rows(rows)


@pytest.mark.skipif(not HAVE_REF, reason=REFERENCE_MISSING)
def test_emoji_parsers_equal_live_reference():
    sys.path[:0] = [os.path.join(ROOT, "oracle", "ref_shim"), REFERENCE_ROOT]
    from multiagent_rlrm.environments.frozen_lake.config_frozen_lake import config as fc
    from multiagent_rlrm.environments.office_world.config_office import config as oc
    from multiagent_rlrm.utils.utils import parse_map_emoji, parse_office_world

    for m in oc["maps"].values():
        assert P.parse_office_world(m["layout"]) == parse_office_world(m["layout"])
    for m in fc["maps"].values():
        assert P.parse_map_emoji(m["layout"]) == parse_map_emoji(m["layout"])


# ---------------------------------------------------------------------------------------------- reward machine
class _StubDetector:
    def __init__(self, event=None):
        self.event = event

    def detect_event(self, state):
        return state.get("event", self.event)


def _linear_rm():
    return P.RewardMachine({("q0", "a"): ("q1", 1), ("q1", "b"): ("qf", 2)}, _StubDetector())


def test_reward_machine_known_answers():
    """/root/reference/tests/test_reward_machine.py:12-50"""
    rm = _linear_rm()
    assert rm.get_current_state() == "q0" and rm.numbers_state() == 3 and rm.get_state_index("q0") == 0
    assert rm.step({"event": "a"}) == 1 and rm.get_current_state() == "q1"
    assert rm.step({"event": "b"}) == 2 and rm.get_current_state() == "qf"
    assert rm.step({"event": "a"}) == 0 and rm.get_current_state() == "qf"
    assert rm.get_reward_for_non_current_state("q0", "a") == ("q1", 1) and rm.get_current_state() == "qf"
    assert rm.get_reward_for_non_current_state("q0", "zzz") == (None, 0)
    assert rm.get_state_from_index(1) == "q1"
    assert rm.reset_to_initial_state() == "q0" and rm.get_current_state() == "q0"
    rm2 = P.RewardMachine({("q0", ("x", 1)): ("q1", 5)}, _StubDetector())
    assert rm2.get_reward_for_non_current_state("q0", ["x", 1]) == ("q1", 5)  # list event -> tuple
    assert rm.get_final_state() == "qf" and rm.get_all_states() == ["q0", "q1", "qf"]
    with pytest.raises(ValueError):
        rm.get_state_from_index(17)


def test_reward_machine_constructor_signature():
    """/root/reference/tests/test_reward_machine_api.py:6-17 guards the (transitions, event_detector) signature."""
    import inspect

    assert list(inspect.signature(P.RewardMachine.__init__).parameters)[1:] == ["transitions", "event_detector"]


def test_index_map_is_initial_first_then_lexicographic():
    tr = {}
    for i in range(11):
        tr[(f"q{i}", (i, 0))] = (f"q{i + 1}", 0)
    rm = P.RewardMachine(tr, P.PositionEventDetector({(i, 0) for i in range(11)}))
    assert rm.state_indices == {"q0": 0, "q1": 1, "q10": 2, "q11": 3, "q2": 4, "q3": 5, "q4": 6, "q5": 7, "q6": 8, "q7": 9,
                                "q8": 10, "q9": 11}
    assert rm.get_all_states() == [f"q{i}" for i in range(12)] and rm.get_final_state() == "q11"
    t = rm.compile_tables(12, 1)
    assert t["n_states"] == 12 and t["final"] == 3 and list(t["qrm_states"]) == [0, 1, 4, 5, 6, 7, 8, 9, 10, 11, 2]


def test_compiled_rm_tables_equal_dict_lookups():
    for sc in (P.scenario_config1(), P.scenario_config2(), P.scenario_config4()):
        c = P.compile_scenario(sc)
        rm, W = c.rm, c.config.width
        inv = {v: k for k, v in rm.state_indices.items()}
        for q in range(c.n_rm_states):
            for cell in range(c.config.width * c.config.height):
                pos = (cell % W, cell // W)
                ev = rm.event_detector.detect_event({"pos_x": pos[0], "pos_y": pos[1]})
                want_state, want_r = rm.get_reward_for_non_current_state(inv[q], ev)
                lab = c.label[cell]
                col = c.config.n_events if lab == abi.EVENT_NONE else lab
                assert (lab == abi.EVENT_NONE) == (ev is None)
                d = c.delta[q, col]
                if want_state is None:
                    assert d == abi.NO_TRANSITION
                else:
                    assert d == rm.state_indices[want_state] and c.rq[q, col] == want_r and c.rcf[q, col] == want_r


# ---------------------------------------------------------------------------------------------- encoders / agent
class _Problem:
    grid_width, grid_height = 4, 5


def test_state_encoder_known_answers():
    """/root/reference/tests/test_state_encoder_frozen_lake.py:21-43 ; tests/test_utils_encoding.py:24-36"""
    ag = P.AgentRL("a", _Problem())
    ag.set_reward_machine(P.RewardMachine({("q0", "e"): ("q0", 0)}, _StubDetector()))
    enc = P.StateEncoderFrozenLake(ag)
    assert enc.encode({"pos_x": 1, "pos_y": 2}, "q0") == (9, {"s": 9, "q": 0})
    ag.set_reward_machine(P.RewardMachine({("q0", "e"): ("q1", 0)}, _StubDetector()))
    assert enc.decode(19) == ({"pos_x": 1, "pos_y": 2}, {"q": "q1"})
    with pytest.raises(ValueError):
        enc.encode({"pos_x": 3, "pos_y": 5}, "q1")

    class P2:
        grid_width, grid_height = 2, 2

    ag2 = P.AgentRL("b", P2())
    ag2.set_reward_machine(P.RewardMachine({("q0", "e"): ("q0", 0)}, _StubDetector()))
    assert P.encode_state(ag2, {"pos_x": 1, "pos_y": 1}, "q0") == 3
    # time-augmented variants (/root/reference/tests/test_utils_encoding.py:24-47)
    from multiagent_rlrm_b200.encoders import encode_state_time, encode_state_with_time

    class P3:
        grid_width, grid_height, max_time = 2, 2, 3

    ag3 = P.AgentRL("c", P3())
    ag3.set_reward_machine(P.RewardMachine({("q0", None): ("q0", 0)}, _StubDetector()))
    state = {"pos_x": 1, "pos_y": 1, "timestamp": 1, "timestep": 2}
    assert encode_state_with_time(ag3, state, "q0") == 3 * 3 + 1 and encode_state_time(ag3, state, "q0") == 3 * 3 + 2

    class P4:
        grid_width, grid_height, max_time = 1, 1, 1

    ag4 = P.AgentRL("d", P4())
    ag4.set_reward_machine(P.RewardMachine({("q0", None): ("q0", 0)}, _StubDetector()))
    zero = {"pos_x": 0, "pos_y": 0, "timestamp": 0, "timestep": 0}
    with pytest.raises(ValueError):
        encode_state_with_time(ag4, zero | {"timestamp": 2}, "q0")
    with pytest.raises(ValueError):
        encode_state_time(ag4, zero | {"timestep": 2}, "q0")


class _DummyAlgo:
    def __init__(self):
        self.calls = []

    def choose_action(self, encoded_state, best=False, **kw):
        self.calls.append(("choose", encoded_state, best, kw))
        return 2

    def update(self, *args, **kw):
        self.calls.append(("update", args, kw))
        return "sentinel"


def test_agent_select_and_update_plumbing():
    """/root/reference/tests/test_agent_rl.py:57-101 ; tests/test_agent_rl_actions.py:17-27"""
    ag = P.AgentRL("a", _Problem())
    ag.add_action_encoder(P.ActionEncoderFrozenLake(ag))
    ag.add_state_encoder(P.StateEncoderFrozenLake(ag))
    ag.set_reward_machine(P.RewardMachine({("q0", "e"): ("q1", 1)}, _StubDetector()))
    algo = _DummyAlgo()
    ag.set_learning_algorithm(algo)
    assert [a.name for a in ag.get_actions()] == ["up", "down", "left", "right"]
    act = ag.select_action({"pos_x": 1, "pos_y": 0})
    assert act.name == "left" and algo.calls[-1][1] == 2  # enc = (0*4+1)*2 + 0
    out = ag.update_policy({"pos_x": 1, "pos_y": 0}, act, 1.5, {"pos_x": 0, "pos_y": 0}, True,
                           infos={"prev_q": "q0", "q": "q1", "Renv": 0.5, "RQ": 1.0})
    assert out == "sentinel"
    _, args, kw = algo.calls[-1]
    assert args == (2, 1, 2, 1.5, True) and kw["info"]["prev_q"] == 0 and kw["info"]["q"] == 1 and kw["info"]["prev_s"] == 1
    with pytest.raises(P.UPValueError):
        ag.action("jump")
    with pytest.raises(Exception, match="Encoder not set"):
        P.AgentRL("x", _Problem()).select_action({"pos_x": 0, "pos_y": 0})


def test_reward_machine_caches_follow_mutation_of_the_transition_dict():
    """_states_in_order / get_state_from_index are cached (the reference re-derives them on every call); configuration code
    builds machines by inserting transitions and by replacing the dicts, and the caches must follow both."""
    from multiagent_rlrm_b200.reward_machine import PositionEventDetector, RewardMachine

    rm = RewardMachine({("a", (0, 0)): ("b", 1.0)}, PositionEventDetector({(0, 0), (1, 1)}))
    assert rm.numbers_state() == 2 and rm.get_all_states() == ["a", "b"] and rm.get_state_from_index(1) == "b"
    rm.transitions[("b", (1, 1))] = ("c", 2.0)                      # grown in place
    assert rm.numbers_state() == 3 and rm.get_all_states() == ["a", "b", "c"] and rm.get_final_state() == "c"
    rm.state_indices = rm._generate_state_indices()
    assert rm.get_state_from_index(2) == "c"
    rm.transitions = {("x", (0, 0)): ("y", 0.5), ("y", (1, 1)): ("z", 0.5), ("z", (0, 0)): ("x", 0.0)}   # replaced, same size
    assert rm.get_all_states() == ["x", "y", "z"] and rm.numbers_state() == 3
    rm.state_indices = {"x": 0, "y": 1, "z": 2}                     # replaced, same size as before
    assert rm.get_state_from_index(2) == "z" and rm.get_state_from_index(0) == "x"
    with pytest.raises(ValueError):
        rm.get_state_from_index(7)
    states = rm.get_all_states()
    states.append("junk")                                            # callers own the list they get
    assert rm.get_all_states() == ["x", "y", "z"]


# ---------------------------------------------------------------------------------------------- table compiler
def test_slip_thresholds_equal_numpy_searchsorted():
    rng = np.random.default_rng(0)
    for probs in ([0.8, 0.1, 0.1], [0.6, 0.36, 0.02, 0.02], [0.7, 0.1, 0.1, 0.1], [0.9, 0.05, 0.05], [1 / 3, 1 / 3, 1 / 3]):
        thr = tables.slip_thresholds(probs)
        cdf = np.cumsum(np.array(probs, dtype=np.float64))
        cdf /= cdf[-1]
        ks = np.concatenate([rng.integers(0, 1 << 32, 20000, dtype=np.uint64),
                             np.array([t + d for t in thr for d in (-1, 0, 1) if 0 <= t + d < (1 << 32)], dtype=np.uint64),
                             np.array([0, (1 << 32) - 1], dtype=np.uint64)])
        want = np.searchsorted(cdf, ks.astype(np.float64) / 4294967296.0, side="right")
        got = sum((ks >= np.uint64(t)).astype(np.int64) for t in thr)
        assert np.array_equal(want, got), probs


@pytest.mark.skipif(not HAVE_REF, reason=REFERENCE_MISSING)
@pytest.mark.parametrize("env_name", ["frozen_lake", "office_world"])
def test_move_tables_equal_reference_apply_action(env_name):
    """Brute force: for every cell and action the compiled next_cell / blocked bit equals what the reference's
    apply_action / is_wall_collision do (ma_frozen_lake.py:224-242 ; ma_office.py:269-309)."""
    import ref_harness as H

    sc = P.scenario_config3() if env_name == "frozen_lake" else P.scenario_config4()
    c = P.compile_scenario(sc)
    rm_env, env, agents = H.build_reference(sc.to_dict())
    ag = agents[0]
    W, Hh = env.grid_width, env.grid_height
    assert (W, Hh) == (c.config.width, c.config.height)
    for y in range(Hh):
        for x in range(W):
            for a, name in enumerate(("up", "down", "left", "right")):
                ag.set_position(x, y)
                env.apply_action(ag, name)
                nx, ny = ag.get_position()
                assert c.next_cell[y * W + x, a] == ny * W + nx, (x, y, name)
                if env_name == "office_world":
                    ag.set_position(x, y)
                    assert env.is_wall_collision(ag, name) == (c.next_cell[y * W + x, a] == y * W + x)
    hazards = set(env.holes) if env_name == "frozen_lake" else set(env.plants)
    assert {(i % W, i // W) for i in np.flatnonzero(c.cell_flags & 1)} == hazards


@pytest.mark.skipif(not HAVE_REF, reason=REFERENCE_MISSING)
def test_slip_tables_equal_reference_probability_mappings():
    import ref_harness as H

    names = ("up", "down", "left", "right", "wait")
    cases = []
    for delay in (False, True):
        sc = P.scenario_config3(); sc.delay_action = delay
        cases.append(sc)
    for delay, allslip, hp in ((False, False, 0.8), (False, True, 0.7), (True, False, 0.8)):
        sc = P.scenario_config4(); sc.delay_action, sc.all_slip, sc.high_prob = delay, allslip, hp
        cases.append(sc)
    for sc in cases:
        c = P.compile_scenario(sc)
        _, env, _ = H.build_reference(sc.to_dict())
        mapping = env._stochastic_action_probability_mapping() if sc.env == "frozen_lake" else env.get_action_probability_mapping()
        for a in range(4):
            outs, probs = mapping[names[a]]
            assert [names[c.config.slip_outcome[a][j]] for j in range(len(outs))] == list(outs)
            assert list(c.config.slip_thr)[: len(probs) - 1] == tables.slip_thresholds(probs)
            assert c.config.slip_n == len(probs)


# ---------------------------------------------------------------------------------------------- built-in OfficeWorld tasks
def test_builtin_office_experiments_known_answers():
    """config_office.py:292-470: exp4 on map1 is A -> B -> C -> D with the reward on the last link (SURVEY.md §8 constants)."""
    from multiagent_rlrm_b200.experiments import OPTIMAL, get_experiment_for_map, scenario_for_experiment

    exp = get_experiment_for_map("map1", "exp4")
    assert list(exp["transitions"].items()) == [(("state0", (1, 7)), ("state1", 0)), (("state1", (1, 1)), ("state2", 0)),
                                                (("state2", (10, 1)), ("state3", 0)), (("state3", (10, 7)), ("state4", 1))]
    assert exp["positions"] == {(1, 7), (1, 1), (10, 1), (10, 7)}
    assert get_experiment_for_map("map1", "exp1")["transitions"][("state0", (8, 6))] == ("state1", 0)  # second coffee machine
    assert get_experiment_for_map("map1", "no such experiment") is None
    assert get_experiment_for_map("map4", "exp6")["transitions"] == get_experiment_for_map("map4", "exp7")["transitions"]
    assert OPTIMAL["map1;exp4"] == 30 and OPTIMAL["map1;exp1"] == 15
    sc = scenario_for_experiment("map1", "exp3", starts=[(2, 7)], algo="qrm")
    c = P.compile_scenario(sc)
    assert c.config.n_rm_states == 5 and c.config.rm_final == 4 and c.config.n_events == 4


@pytest.mark.skipif(not HAVE_REF, reason=REFERENCE_MISSING)
def test_builtin_office_experiments_equal_live_reference():
    import ast

    import ref_harness as H

    H._import_reference()  # puts the stub packages and the reference tree on sys.path
    from multiagent_rlrm.environments.office_world.config_office import config, get_experiment_for_map as ref_get

    from multiagent_rlrm_b200.experiments import OPTIMAL, get_experiment_for_map

    for mp in config["maps"]:
        for exp in ("exp0", "exp0_simply", "exp1", "exp2", "exp3", "exp4", "exp5", "exp6", "exp7", "unknown"):
            r, m = ref_get(mp, exp), get_experiment_for_map(mp, exp)
            if r is None:
                assert m is None
                continue
            assert list(r["transitions"].items()) == list(m["transitions"].items()), (mp, exp)  # insertion order matters
            assert r["positions"] == m["positions"] and r["description"] == m["description"], (mp, exp)
    src = open(os.path.join(REFERENCE_ROOT, "multiagent_rlrm", "environments", "office_world", "office_main.py")).read()
    node = next(n for n in ast.parse(src).body if isinstance(n, ast.Assign) and getattr(n.targets[0], "id", "") == "OPTIMAL")
    assert ast.literal_eval(node.value) == OPTIMAL


# ---------------------------------------------------------------------------------------------- reward shaping (f3)
def test_distance_reward_shaping_known_answers():
    """/root/reference/tests/test_reward_machine_shaping.py: qf -> 0, one step away -> -alpha, two steps -> -2 alpha"""
    rm = P.RewardMachine({("q0", "a"): ("q1", 0), ("q1", "b"): ("qf", 1)}, _StubDetector())
    rm.add_distance_reward_shaping(gamma=0.9, rs_gamma=0.9, alpha=5)
    assert rm.potentials == {"q0": -10, "q1": -5, "qf": 0}
    assert rm.get_distance("q0") == 2 and rm.get_distance("qf") == 0
    lonely = P.RewardMachine({("q0", "a"): ("q0", 0), ("q1", "b"): ("qf", 1)}, _StubDetector())
    assert lonely.get_distance("q0") == 999999


def test_value_iteration_shaping_known_answers():
    rm = P.builtin_frozen_lake_rm({"A": (4, 4), "B": (0, 0), "C": (4, 8)}) if hasattr(P, "builtin_frozen_lake_rm") else None
    from multiagent_rlrm_b200.reward_machine import builtin_frozen_lake_rm

    rm = builtin_frozen_lake_rm({"A": (4, 4), "B": (0, 0), "C": (4, 8)})
    rm.add_reward_shaping(0.99, 0.9)
    # V(state2) = 20, V(state1) = 15 + .9*20 = 33, V(state0) = 10 + .9*33 = 39.7 ; potentials are -V
    assert rm.potentials == {"state0": -(10 + 0.9 * (15 + 0.9 * 20)), "state1": -(15 + 0.9 * 20), "state2": -20, "state3": 0}


@pytest.mark.skipif(not HAVE_REF, reason=REFERENCE_MISSING)
def test_potentials_equal_live_reference():
    import contextlib
    import io

    import ref_harness as H

    for sc in (P.scenario_config1(), P.scenario_config2(), P.scenario_config4()):
        _, _, agents = H.build_reference(sc.to_dict())
        ref_rm = agents[0].get_reward_machine()
        mine = sc.reward_machine()
        with contextlib.redirect_stdout(io.StringIO()):
            ref_rm.add_reward_shaping(sc.gamma, 0.9)
        mine.add_reward_shaping(sc.gamma, 0.9)
        assert mine.potentials == ref_rm.potentials
        ref_rm.add_distance_reward_shaping(sc.gamma, 0.9, alpha=7)
        mine.add_distance_reward_shaping(sc.gamma, 0.9, alpha=7)
        assert mine.potentials == ref_rm.potentials
        # the public pieces add_reward_shaping is made of (reward_machine.py:280-345)
        assert mine.get_delta_u() == ref_rm.get_delta_u()
        dr_mine, dr_ref = mine.get_delta_r(), ref_rm.get_delta_r()
        assert {u: {v: (f.get_type(), f.get_reward(None)) for v, f in d.items()} for u, d in dr_mine.items()} == \
               {u: {v: (f.get_type(), f.get_reward(None)) for v, f in d.items()} for u, d in dr_ref.items()}
        with contextlib.redirect_stdout(io.StringIO()):
            v_ref = ref_rm.value_iteration(list(ref_rm.state_indices), ref_rm.get_delta_u(), dr_ref, ref_rm.get_final_state(), 0.8)
        assert mine.value_iteration(list(mine.state_indices), mine.get_delta_u(), dr_mine, mine.get_final_state(), 0.8) == v_ref


# ---------------------------------------------------------------------------------------------- N = 1 host plumbing (no device)
def test_learner_word_blocks_follow_the_generator_stream():
    """_own_words hands out self.rng's 32-bit words four at a time from 64-word blocks: the sequence equals four-word requests on
    an identical generator, across block boundaries, and a block drawn from a generator that was replaced is dropped."""
    from multiagent_rlrm_b200.learners import _TabularBase

    obj = object.__new__(_TabularBase)  # no device: only the word plumbing is exercised
    obj.rng = np.random.default_rng(42)
    ref = np.random.default_rng(42)
    for _ in range(40):  # 160 words = 2.5 blocks
        assert obj._own_words() == ref.integers(0, 1 << 32, size=4, dtype=np.uint64).tolist()
    obj.rng = np.random.default_rng(7)  # reseeded: the rest of the old block must not be used
    ref = np.random.default_rng(7)
    assert obj._own_words() == ref.integers(0, 1 << 32, size=4, dtype=np.uint64).tolist()


def test_env_slip_words_are_buffered_without_changing_the_stream():
    """BaseEnvironment._slip_words reads env.rng in blocks holding a whole number of steps: word 3 of every agent's draw block
    equals per-step requests of n words on an identical generator; reset() installs a new generator and a new block."""
    env = P.MultiAgentFrozenLake(width=4, height=4, holes=[])
    for k in range(3):
        env.add_agent(P.AgentRL(f"a{k}", env))
    env.rng = np.random.default_rng(5)
    ref = np.random.default_rng(5)
    out = np.zeros(12, dtype=np.uint32)
    for _ in range(50):  # 150 words: several blocks of 63
        env._slip_words(out)
        assert out[3::4].tolist() == ref.integers(0, 1 << 32, size=3, dtype=np.uint64).astype(np.uint32).tolist()
    env.rng = np.random.default_rng(6)
    ref = np.random.default_rng(6)
    env._slip_words(out)
    assert out[3::4].tolist() == ref.integers(0, 1 << 32, size=3, dtype=np.uint64).astype(np.uint32).tolist()


def test_agent_action_index_cache_follows_the_action_list():
    from multiagent_rlrm_b200.actions import ActionRL

    ag = P.AgentRL("a", None)
    up, down, left = ActionRL("up"), ActionRL("down"), ActionRL("left")
    ag.add_action(up)
    ag.add_action(down)
    assert (ag.actions_idx(up), ag.actions_idx(down), ag.actions_idx(left)) == (0, 1, None)
    ag.add_action(left)                      # the list grew
    assert ag.actions_idx(left) == 2
    ag.actions_[0], ag.actions_[1] = down, up  # same length, other order
    assert (ag.actions_idx(up), ag.actions_idx(down)) == (1, 0)
    assert ag.name == "a" and ag.get_reward_machine() is None and ag.get_actions() is ag.actions_
