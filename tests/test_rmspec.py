"""CPU: the RM-spec compile path (SURVEY.md §8 f1): spec file + map name -> RewardMachine -> device tables.
Known answers restated from the reference's tests, and a differential test against the live reference pipeline."""
import json
import os
import sys

import numpy as np
import pytest

from conftest import ROOT

import multiagent_rlrm_b200 as P
from multiagent_rlrm_b200 import rmspec as R
from ref_harness import REFERENCE_MISSING, REFERENCE_ROOT, reference_available

FIX = os.path.join(ROOT, "tests", "fixtures")
HAVE_REF = reference_available()


def _partial():
    return R.RMSpec.from_dict({"name": "partial", "env_id": "env", "version": "1.0", "states": ["q0", "q1"], "initial_state": "q0",
                               "terminal_states": ["q1"], "event_vocabulary": ["e1", "e2"],
                               "transitions": [{"from_state": "q0", "event": "e1", "to_state": "q1", "reward": 1}]})


def test_completion_full_cartesian_and_defaults():
    """/root/reference/tests/test_rmgen_completion.py:22-55"""
    spec, report = R.complete_missing_transitions(_partial(), default_reward=0.0)
    assert report["added"] == 3 and len(spec.transitions) == 4
    assert any((t.from_state, t.event, t.to_state, t.reward) == ("q0", "e1", "q1", 1) for t in spec.transitions)
    spec, _ = R.complete_missing_transitions(_partial(), default_reward=0.5)
    assert next(t for t in spec.transitions if (t.from_state, t.event) == ("q1", "e2")).reward == 0.5
    spec, _ = R.complete_missing_transitions(_partial(), terminal_self_loop=True)
    assert any((t.from_state, t.event, t.to_state) == ("q1", "e1", "q1") for t in spec.transitions)
    spec, rep = R.complete_missing_transitions(_partial(), terminal_self_loop=False)
    assert rep["added"] == 1 and not any(t.from_state == "q1" for t in spec.transitions)


def test_load_and_compile_with_passthrough_detector(tmp_path):
    """/root/reference/tests/test_rmspec_io.py:10-18 (fixture rewritten: two-step machine ending on at(G))"""
    p = tmp_path / "simple.json"
    p.write_text(json.dumps({"name": "s", "env_id": "OfficeWorld ", "version": "1.0", "states": ["q0", "q1", "q2"],
                             "initial_state": "q0", "terminal_states": ["q2"], "event_vocabulary": ["at(K)", "at(G)"],
                             "transitions": [{"from_state": "q0", "event": "at(K)", "to_state": "q1", "reward": 0},
                                             {"from_state": "q1", "event": "at(G)", "to_state": "q2", "reward": "r1"}]}))
    spec = R.load_rmspec(p)
    assert spec.env_id == "officeworld"
    rm = R.compile_reward_machine(spec)
    assert isinstance(rm, P.RewardMachine)
    assert rm.get_reward_for_non_current_state("q1", "at(G)") == ("q2", 1.0)
    assert rm.step({"event": "at(K)"}) == 0 and rm.get_current_state() == "q1"
    with pytest.raises(FileNotFoundError):
        R.load_rmspec(tmp_path / "nope.json")
    bad = tmp_path / "bad.json"
    bad.write_text("{not json")
    with pytest.raises(ValueError):
        R.load_rmspec(bad)


def test_validation_errors():
    d = _partial().to_dict()
    for mutate, msg in ((lambda x: x.update(initial_state="zz"), "initial_state"),
                        (lambda x: x["transitions"].append({"from_state": "q0", "event": "e1", "to_state": "q0", "reward": 0}), "Non-deterministic"),
                        (lambda x: x["transitions"].append({"from_state": "q1", "event": "e2", "to_state": "q1", "reward": 2}), "Terminal transitions"),
                        (lambda x: x.update(event_vocabulary=["e1", "e1"]), "Duplicate event")):
        dd = json.loads(json.dumps(d))
        mutate(dd)
        with pytest.raises(R.ValidationError, match=msg):
            R.compile_reward_machine(R.RMSpec.from_dict(dd))


def test_officeworld_event_normalisation():
    """/root/reference/tests/test_officeworld_event_context.py:15-64 ; tests/test_frozenlake_event_context.py"""
    ctx = R.build_officeworld_context("map1")
    spec = {"name": "b", "env_id": "officeworld", "version": "1.0", "states": ["q0", "q1", "q2", "q3", "q4"], "initial_state": "q0",
            "terminal_states": ["q4"], "event_vocabulary": ["A", "B", "C", "D"],
            "transitions": [{"from_state": f"q{i}", "event": e, "to_state": f"q{i + 1}", "reward": int(i == 3)} for i, e in enumerate("ABCD")]}
    out = R.normalize_rmspec_events(spec, ctx)
    assert out["event_vocabulary"] == ["at(A)", "at(B)", "at(C)", "at(D)"]
    assert [t["event"] for t in out["transitions"]] == ["at(A)", "at(B)", "at(C)", "at(D)"]
    syn = R.normalize_rmspec_events({"event_vocabulary": [" At( Office )"], "transitions": [{"event": "office"}]}, ctx)
    assert syn["event_vocabulary"] == ["at(O)"] and syn["transitions"][0]["event"] == "at(O)"
    with pytest.raises(R.UnknownEventError, match="Unknown event 'at\\(G\\)'"):
        R.normalize_rmspec_events({"event_vocabulary": ["at(G)"], "transitions": []}, ctx)
    fl = R.normalize_rmspec_events({"event_vocabulary": ["A", "B"], "transitions": [{"event": "A"}]}, R.build_frozenlake_context("map1"))
    assert fl["event_vocabulary"] == ["at(A)", "at(B)"] and fl["transitions"][0]["event"] == "at(A)"


def test_env_id_enforcement_and_autofix(capsys):
    """/root/reference/tests/test_officeworld_env_id_enforcement.py"""
    spec = R.RMSpec.from_dict({"name": "t", "env_id": "officework", "version": "1.0", "states": ["q0", "q1"], "initial_state": "q0",
                               "terminal_states": [], "event_vocabulary": ["A"],
                               "transitions": [{"from_state": "q0", "event": "A", "to_state": "q4", "reward": 1.0}]})
    spec = R.enforce_env_id(spec, "officeworld", reason="--rm-spec is set")
    assert spec.env_id == "officeworld" and "overriding env_id" in capsys.readouterr().out
    spec = R.autofix_rmspec_states_for_officeworld(spec)
    assert spec.states == ["q0", "q1", "q4"] and spec.terminal_states == ["q4"]
    R.validate_spec(R.normalize_rmspec_events(spec, R.build_officeworld_context("map1")))
    loop = R.RMSpec.from_dict({"name": "t", "env_id": "officeworld", "version": "1.0", "states": ["q0", "q1"], "initial_state": "q0",
                               "terminal_states": ["q1"], "event_vocabulary": ["A", "B"],
                               "transitions": [{"from_state": "q0", "event": "A", "to_state": "q1", "reward": 0},
                                               {"from_state": "q1", "event": "B", "to_state": "q1", "reward": 1}]})
    fixed = R.autofix_terminal_reward_violations_for_officeworld(loop)
    assert fixed.states == ["q0", "q1", "q2"] and fixed.terminal_states == ["q2"]
    assert (fixed.transitions[1].from_state, fixed.transitions[1].to_state, fixed.transitions[1].reward) == ("q1", "q2", 1.0)


def test_spec_files_compile_to_the_baseline_scenarios():
    """The authored spec fixtures reproduce the BASELINE config machines and their device tables."""
    rm, _ = R.load_reward_machine(os.path.join(FIX, "officeworld_acbd.json"), "office_world", "map1")
    want = P.scenario_config2().reward_machine()
    assert list(rm.transitions.items()) == list(want.transitions.items())
    sc, rm12 = R.scenario_from_rmspec(os.path.join(FIX, "officeworld_chain12.json"), P.scenario_config4(), complete_missing_transitions=True)
    c_spec, c_ref = P.compile_scenario(sc), P.compile_scenario(P.scenario_config4())
    assert len(rm12.transitions) == 108 and rm12.get_final_state() == "q11"
    assert rm12.state_indices == c_ref.rm.state_indices
    for name in ("label", "delta", "rq", "rcf", "qrm_states"):
        assert np.array_equal(getattr(c_spec, name), getattr(c_ref, name)), name
    rm3, _ = R.load_reward_machine(os.path.join(FIX, "frozenlake_abc.json"), "frozen_lake", "map1")
    c3, c1 = P.compile_scenario(P.scenario_config1(), rm=rm3), P.compile_scenario(P.scenario_config1())
    for name in ("label", "delta", "rq", "rcf", "qrm_states"):
        assert np.array_equal(getattr(c3, name), getattr(c1, name)), name
    assert c3.config.rm_final == c1.config.rm_final == 3


@pytest.mark.skipif(not HAVE_REF, reason=REFERENCE_MISSING)
@pytest.mark.parametrize("fixture,env,complete", [("officeworld_acbd.json", "office_world", False), ("officeworld_acbd.json", "office_world", True),
                                                  ("officeworld_chain12.json", "office_world", True), ("frozenlake_abc.json", "frozen_lake", False),
                                                  ("frozenlake_abc.json", "frozen_lake", True), ("REF:frozenlake_linear.json", "frozen_lake", True)])
def test_pipeline_equals_live_reference(fixture, env, complete, capsys):
    """Same spec file through the reference's runner pipeline (office_main.py:487-515 / frozen_lake_main.py:133-183)."""
    sys.path[:0] = [os.path.join(ROOT, "oracle", "ref_shim"), REFERENCE_ROOT]
    from multiagent_rlrm.environments.frozen_lake.config_frozen_lake import config as fc
    from multiagent_rlrm.environments.frozen_lake.detect_event import PositionEventDetector
    from multiagent_rlrm.environments.frozen_lake.event_context import build_frozenlake_context
    from multiagent_rlrm.environments.office_world.config_office import config as oc
    from multiagent_rlrm.environments.office_world.event_context import build_officeworld_context
    from multiagent_rlrm.rmgen import io as rio
    from multiagent_rlrm.rmgen import normalize as rnorm
    from multiagent_rlrm.utils.utils import parse_map_emoji, parse_office_world

    path = os.path.join(REFERENCE_ROOT, "tests", "fixtures", fixture[4:]) if fixture.startswith("REF:") else os.path.join(FIX, fixture)
    if not os.path.exists(path):  # the staged copy under oracle/_ref holds the reference's package, not its tests/
        pytest.skip(f"{path} is not in the reference tree")
    spec = rio.load_rmspec(path)
    if env == "office_world":
        spec = rnorm.enforce_env_id(spec, "officeworld", reason="t")
        ctx = build_officeworld_context("map1")
        assert ctx == R.build_officeworld_context("map1")
        spec = rnorm.normalize_rmspec_events(spec, ctx)
        spec = rnorm.autofix_rmspec_states_for_officeworld(spec)
        spec = rnorm.autofix_terminal_reward_violations_for_officeworld(spec)
        coords, goals, _ = parse_office_world(oc["maps"]["map1"]["layout"])
        mapping = {}
        for label, pos in goals.items():
            mapping[f"at({label})"] = pos
            mapping[label] = pos
        mapping["office"] = mapping["at(office)"] = goals["O"]
        mapping["coffee"] = mapping["at(coffee)"] = list(coords["coffee"])
        for k in ("letter", "email", "at(letter)", "at(email)"):
            mapping[k] = list(coords["letter"])
        assert mapping == R.officeworld_event_mapping("map1")
        positions = set(oc["maps"]["map1"]["position_map"](coords, goals))
    else:
        spec = rnorm.enforce_env_id(spec, "frozenlake", reason="t")
        ctx = build_frozenlake_context("map1")
        assert ctx == R.build_frozenlake_context("map1")
        spec = rnorm.normalize_rmspec_events(spec, ctx)
        _, goals, _ = parse_map_emoji(fc["maps"]["map1"]["layout"])
        mapping = {}
        for label, pos in goals.items():
            mapping[f"at({label})"] = pos
            mapping[label] = pos
        positions = set(goals.values())
    for m in mapping.values():
        positions.update(m if isinstance(m, list) else [m])
    ref_rm = rio.compile_reward_machine(spec, event_detector=PositionEventDetector(positions), event_mapping=mapping,
                                        complete_missing_transitions=complete)
    rm, _ = R.load_reward_machine(path, env, "map1", complete_missing_transitions=complete)
    assert list(rm.transitions.items()) == list(ref_rm.transitions.items())
    assert rm.state_indices == ref_rm.state_indices and rm.initial_state == ref_rm.initial_state
    assert rm.get_final_state() == ref_rm.get_final_state() and rm.get_all_states() == ref_rm.get_all_states()
    assert set(rm.event_detector.positions) == set(ref_rm.event_detector.positions)


def test_per_agent_spec_files_compile_to_per_agent_tables(tmp_path):
    """frozen_lake_main.py --rm-spec-a1 / --rm-spec-a2: one spec per agent -> per-agent table sections."""
    a2 = tmp_path / "a2.json"
    a2.write_text(json.dumps({"name": "a2", "env_id": "frozenlake", "version": "1.0", "states": ["p0", "p1", "p2"], "initial_state": "p0",
                              "terminal_states": ["p2"], "event_vocabulary": ["C", "A"],
                              "transitions": [{"from_state": "p0", "event": "C", "to_state": "p1", "reward": 3},
                                              {"from_state": "p1", "event": "A", "to_state": "p2", "reward": 7}]}))
    rm1, _ = R.load_reward_machine(os.path.join(FIX, "frozenlake_abc.json"), "frozen_lake", "map1")
    rm2, _ = R.load_reward_machine(a2, "frozen_lake", "map1")
    c = P.compile_scenario(P.scenario_config3(True), rm=[rm1, rm2])
    cfg = c.config
    assert cfg.per_agent_rm == 1 and list(cfg.agent_n_rm_states)[:2] == [4, 3] and list(cfg.agent_rm_final)[:2] == [3, 2]
    assert list(cfg.agent_n_qrm)[:2] == [3, 2] and cfg.n_rm_states == 4 and c.agent_rows == [400, 300]
    assert c.delta.shape == (2, 4, cfg.n_events + 1) and c.label.shape == (2, 100)
    uniform = P.compile_scenario(P.scenario_config3(True))
    assert np.array_equal(c.delta[0], uniform.delta) and np.array_equal(c.rq[0], uniform.rq)
    g = P.frozen_lake_grid("map1").goals
    col = {ev: k for k, ev in enumerate(c.events)}
    assert c.delta[1, 0, col[g["C"]]] == 1 and c.rq[1, 1, col[g["A"]]] == 7.0 and c.delta[1, 0, col[g["A"]]] == 255


def test_export_round_trip_and_passthrough_machine(tmp_path):
    """rmgen/exporter.py: export_spec_to_file writes what load_rmspec reads; build_reward_machine runs on the spec's own events."""
    spec = R.load_rmspec(os.path.join(FIX, "officeworld_acbd.json"))
    out = tmp_path / "nested" / "dir" / "spec.json"
    R.export_spec_to_file(spec, out)
    assert R.load_rmspec(out).to_dict() == spec.to_dict()
    rm = R.build_reward_machine(spec)
    assert rm.initial_state == spec.initial_state and rm.get_state_index(spec.initial_state) == 0
    first = spec.transitions[0]
    assert rm.step({"event": first.event}) == first.reward and rm.get_current_state() == first.to_state
    assert rm.step({"event": "not in the vocabulary"}) == 0 and rm.get_current_state() == first.to_state


@pytest.mark.skipif(not HAVE_REF, reason=REFERENCE_MISSING)
@pytest.mark.parametrize("fixture", ["officeworld_acbd.json", "officeworld_chain12.json", "frozenlake_abc.json"])
def test_exporter_equals_live_reference(fixture, tmp_path):
    sys.path[:0] = [os.path.join(ROOT, "oracle", "ref_shim"), REFERENCE_ROOT]
    from multiagent_rlrm.rmgen import exporter as rexp
    from multiagent_rlrm.rmgen import io as rio

    path = os.path.join(FIX, fixture)
    mine, theirs = tmp_path / "mine.json", tmp_path / "theirs.json"
    R.export_spec_to_file(R.load_rmspec(path), mine)
    rexp.export_spec_to_file(rio.load_rmspec(path), theirs)
    assert mine.read_bytes() == theirs.read_bytes()  # the on-disk format, byte for byte
    from multiagent_rlrm.rmgen.summary import format_rmspec_summary as ref_summary

    for kw in ({}, {"agent_names": ["a1"], "source": "x.json"}, {"agent_names": ["a1", "a2"], "max_core_transition_lines": 2},
               {"max_core_transition_lines": None}):
        assert R.format_rmspec_summary(R.load_rmspec(path), **kw) == ref_summary(rio.load_rmspec(path), **kw)
    a, b = R.build_reward_machine(R.load_rmspec(path)), rexp.build_reward_machine(rio.load_rmspec(path))
    assert list(a.transitions.items()) == list(b.transitions.items()) and a.state_indices == b.state_indices
    assert a.initial_state == b.initial_state and a.get_final_state() == b.get_final_state()


# ---- known answers of the reference's remaining spec tests --------------------------------------------------------------
_BASE = {"name": "reward_test", "env_id": "env", "version": "1.0", "states": ["q0", "q1"], "initial_state": "q0",
         "terminal_states": ["q1"], "event_vocabulary": ["e"]}


@pytest.mark.parametrize("raw,expected", [("r0", 0.0), ("r1", 1.0), ("r0.5", 0.5), ("1", 1.0), (2, 2.0)])
def test_reward_strings_and_env_id_normalisation(raw, expected):
    """/root/reference/tests/test_rmgen_rewards.py:28-49"""
    spec = R.RMSpec.from_dict({**_BASE, "transitions": [{"from_state": "q0", "event": "e", "to_state": "q1", "reward": raw}]})
    assert spec.transitions[0].reward == expected
    with pytest.raises(ValueError):
        R.RMSpec.from_dict({**_BASE, "transitions": [{"from_state": "q0", "event": "e", "to_state": "q1", "reward": "not_a_number"}]})
    upper = R.RMSpec.from_dict({**_BASE, "env_id": "OfficeWorld ", "transitions": [{"from_state": "q0", "event": "e", "to_state": "q1", "reward": 0}]})
    assert upper.env_id == "officeworld"


def test_semantic_limits_known_answers():
    """/root/reference/tests/test_rmgen_semantics.py:14-62 (the checks the generation pipeline applies to a spec)"""
    two_rewards = R.RMSpec.from_dict({"name": "pos_limit", "env_id": "env", "version": "1.0", "states": ["q0"], "initial_state": "q0",
                                      "terminal_states": [], "event_vocabulary": ["e1", "e2"],
                                      "transitions": [{"from_state": "q0", "event": "e1", "to_state": "q0", "reward": 1},
                                                      {"from_state": "q0", "event": "e2", "to_state": "q0", "reward": 1}]})
    R.validate_spec(two_rewards)
    with pytest.raises(R.ValidationError):
        R.validate_semantics(two_rewards, max_positive_reward_transitions=1)
    terminal_reward = R.RMSpec.from_dict({"name": "terminal_reward", "env_id": "env", "version": "1.0", "states": ["q0"],
                                          "initial_state": "q0", "terminal_states": ["q0"], "event_vocabulary": ["e1"],
                                          "transitions": [{"from_state": "q0", "event": "e1", "to_state": "q0", "reward": 1}]})
    with pytest.raises(R.ValidationError):
        R.validate_semantics(terminal_reward, terminal_reward_must_be_zero=True)
    R.validate_semantics(terminal_reward, terminal_reward_must_be_zero=False)


def test_summary_known_answers():
    """/root/reference/tests/test_rmspec_summary.py:8-34"""
    spec = R.RMSpec(name="core_only", env_id="officeworld", version="1.0", states=["q0", "q1"], initial_state="q0", terminal_states=["q1"],
                    event_vocabulary=["at(C)", "at(E)"],
                    transitions=[R.TransitionSpec("q0", "at(C)", "q1", 0.0), R.TransitionSpec("q0", "at(E)", "q0", 0.0)])
    text = R.format_rmspec_summary(spec)
    assert "core_transitions_count: 1" in text and "q0 --at(C)--> q1" in text and "q0 --at(E)--> q0" not in text
    acbd = R.format_rmspec_summary(R.load_rmspec(os.path.join(FIX, "officeworld_acbd.json")), agent_names=["agent0"], source="f.json")
    assert "env_id: officeworld" in acbd and "reward=1.0" in acbd and acbd.splitlines()[0] == "Reward Machine summary (from f.json)"


def test_reward_machine_extras_known_answers():
    """/root/reference/tests/test_reward_machine_extras.py:12-25"""
    import multiagent_rlrm_b200 as P

    class Detector:
        def detect_event(self, _state):
            return None

    rm = P.RewardMachine({("q0", "a"): ("q1", 0)}, Detector())
    assert rm.get_distance("q_missing") == 999999
    V = rm.value_iteration(list(rm.state_indices.keys()), rm.get_delta_u(), rm.get_delta_r(), rm.get_final_state(), gamma=0.9)
    assert V[rm.get_final_state()] == 0
