"""Edge cases: lane groups with idle lanes (3 agents), the maximum agent count (8), the maximum grid (32x32 = 1024
cells), a 32-state reward machine with 63 event cells, instance counts that do not fill a warp/block, and the C ABI's
argument validation. GPU tests compare with the (reference-pinned) oracle; validation tests run on CPU."""
import ctypes as C

import numpy as np
import pytest

import multiagent_rlrm_b200 as P
from multiagent_rlrm_b200 import _abi as abi
from multiagent_rlrm_b200.maps import GridSpec
from multiagent_rlrm_b200.tables import Scenario, frozen_lake_abc_transitions


def _big_grid(env):
    rng = np.random.default_rng(5)
    W = H = 32
    cells = [(x, y) for y in range(H) for x in range(W)]
    hazards = [cells[i] for i in rng.choice(len(cells), 60, replace=False) if cells[i] not in ((0, 0), (31, 31), (5, 5), (9, 20))]
    walls = []
    if env == "office_world":
        for _ in range(120):
            x, y = int(rng.integers(0, W - 1)), int(rng.integers(0, H - 1))
            a, b = ((x, y), (x + 1, y)) if rng.random() < 0.5 else ((x, y), (x, y + 1))
            walls += [(a, b), (b, a)]
    return GridSpec(env, W, H, hazards=hazards, walls=walls)


def _rm32(grid, n_states=32, n_events=63):
    rng = np.random.default_rng(9)
    free = [(x, y) for y in range(grid.height) for x in range(grid.width) if (x, y) not in set(grid.hazards)]
    events = [free[i] for i in rng.choice(len(free), n_events, replace=False)]
    tr = []
    for i in range(n_states - 1):
        tr.append((f"s{i:02d}", events[i], f"s{i + 1:02d}", float(i % 3)))
    for i in range(n_states):  # extra branches, loops back, event-less states
        for ev in events[40 + (i % 5): 63: 7]:
            if (f"s{i:02d}", ev) not in {(s, e) for s, e, _t, _r in tr}:
                tr.append((f"s{i:02d}", ev, f"s{(i * 7 + 3) % n_states:02d}", -0.5))
    tr.append((f"s{n_states - 2:02d}", events[39], f"s{n_states - 1:02d}", 10.0))
    return tr, events


def edge_scenarios():
    out = {}
    sc = P.scenario_config3(True)
    sc.starts = [(5, 0), (0, 0), (9, 9)]
    out["fl_3_agents_qrm"] = (sc, None, 333, 700)
    sc = P.scenario_config3(False)
    sc.starts = [(5, 0), (0, 0), (9, 9), (7, 3), (9, 0), (0, 9), (5, 5), (2, 3)]
    out["fl_8_agents_ql"] = (sc, None, 77, 700)
    g = _big_grid("frozen_lake")
    tr, ev = _rm32(g)
    sc = Scenario(env="frozen_lake", starts=[(0, 0), (31, 31), (5, 5)], rm_transitions=tr, detector_positions=ev, stochastic=True,
                  delay_action=True, penalty_amount=-3, algo="qrm", learning_rate=0.5, gamma=0.95, epsilon_start=0.3,
                  epsilon_end=0.05, epsilon_decay=0.9, q_init=1.0, driver="frozen_lake_main", seed=3)
    out["fl_32x32_rm32_qrm"] = (sc, g, 130, 1300)
    g = _big_grid("office_world")
    tr, ev = _rm32(g, 12, 40)
    sc = Scenario(env="office_world", starts=[(0, 0), (9, 20)], rm_transitions=tr, detector_positions=ev, stochastic=True, all_slip=True,
                  high_prob=0.6, wall_penalty=-0.25, plants_penalty=-7, algo="ql", learning_rate=None, gamma=0.9, epsilon_start=0.5,
                  epsilon_end=0.1, epsilon_decay=0.99, q_init=0.5, driver="office_main", seed=4)
    out["ow_32x32_lr_none_ql"] = (sc, g, 130, 1300)
    sc = P.scenario_config1()
    sc.starts = [(5, 0)]
    out["one_instance_one_agent"] = (sc, None, 1, 2500)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(edge_scenarios()))
def test_edge_case_matches_oracle(name, cuda_device):
    import oracle as O
    from multiagent_rlrm_b200.engine import Engine

    sc, grid, n, iters = edge_scenarios()[name]
    c = P.compile_scenario(sc, grid=grid)
    eng, o = Engine(c, n), O.Oracle(c, n, "f32")
    eng.reset(); o.reset()
    tr_g = eng.train(iters, trace=True)
    tr_o = o.train(0, iters, trace=True)
    assert np.array_equal(tr_g.cpu().numpy().view(np.uint32), tr_o), name
    assert np.array_equal(eng.q.cpu().numpy(), o.q) and np.array_equal(eng.slot.cpu().numpy().view(np.uint64), o.slot)
    assert np.array_equal(eng.epsilon.cpu().numpy(), o.epsilon)
    if o.visits is not None:
        assert np.array_equal(eng.visits.cpu().numpy().view(np.uint32), o.visits)
    # and the same through the call-by-call entry points
    eng2 = Engine(c, n)
    eng2.reset()
    for _ in range(40):
        eng2.iterate_unfused()
    o2 = O.Oracle(c, n, "f32")
    o2.reset(); o2.train(0, 40)
    assert np.array_equal(eng2.q.cpu().numpy(), o2.q) and np.array_equal(eng2.slot.cpu().numpy().view(np.uint64), o2.slot)


def test_three_agent_oracle_matches_live_reference():
    """CPU: the oracle on a 3-agent instance equals the live reference (skipped without the reference sources)."""
    import oracle as O
    import ref_harness as H

    if not H.reference_available():
        pytest.skip(H.REFERENCE_MISSING)

    sc, _g, _n, _t = edge_scenarios()["fl_3_agents_qrm"]
    ref = H.run_reference(sc.to_dict(), 2, 400)
    o = O.Oracle(P.compile_scenario(sc), 2, "f32")
    o.reset(); o.reset()
    tr = O.unpack_trace(o.train(0, 400, trace=True), 2, 3)
    for k in ("action", "cell", "q", "term", "trunc"):
        assert np.array_equal(tr[k], ref[k].astype(np.int32)), k
    assert np.array_equal(o.q.reshape(ref["q_final"].shape), ref["q_final"])


def test_create_rejects_bad_arguments():
    """rlrm_create validates its arguments before touching the device (error codes, never exceptions)."""
    from multiagent_rlrm_b200 import _lib

    _lib.build()
    L = _lib.load()

    def create(mutate):
        c = P.compile_scenario(P.scenario_config1())
        t = c.tables_struct()
        mutate(c.config, t)
        h = C.c_void_p()
        rc = L.rlrm_create(C.byref(c.config), C.byref(t), 0, C.byref(h))
        if rc == 0:
            L.rlrm_destroy(h)
        return rc, L.rlrm_last_error().decode()

    for mutate, text in ((lambda cfg, t: setattr(cfg, "abi_version", 99), "abi_version"),
                         (lambda cfg, t: setattr(cfg, "n_agents", 9), "n_agents"),
                         (lambda cfg, t: setattr(cfg, "width", 200), "width*height"),
                         (lambda cfg, t: setattr(cfg, "n_rm_states", 33), "n_rm_states"),
                         (lambda cfg, t: setattr(cfg, "n_actions", 5), "n_actions"),
                         (lambda cfg, t: setattr(cfg, "algo", 7), "algo"),
                         (lambda cfg, t: setattr(t, "delta", None), "null table"),
                         (lambda cfg, t: setattr(cfg, "rm_final", 4), "rm_final"),
                         (lambda cfg, t: setattr(cfg, "max_steps", 70000), "max_steps"),
                         (lambda cfg, t: setattr(cfg, "table_dtype", 2), "table_dtype")):
        rc, msg = create(mutate)
        assert rc == -1 and text in msg, (rc, msg)

    # table CONTENTS are validated too: the kernels follow these indices without bounds checks
    def create_with(field, index, value):
        c = P.compile_scenario(P.scenario_config1())
        arr = getattr(c, field)
        arr.reshape(-1)[index] = value
        t = c.tables_struct()
        h = C.c_void_p()
        rc = L.rlrm_create(C.byref(c.config), C.byref(t), 0, C.byref(h))
        if rc == 0:
            L.rlrm_destroy(h)
        return rc, L.rlrm_last_error().decode()

    for field, index, value, text in (("next_cell", 17, 100, "next_cell"), ("start_cell", 1, 400, "start_cell"),
                                      ("label", 5, 3, "label"), ("delta", 2, 4, "delta"), ("qrm_states", 1, 9, "qrm_states")):
        rc, msg = create_with(field, index, value)
        assert rc == -1 and text in msg, (field, rc, msg)
    c = P.compile_scenario(P.scenario_config3(True))
    c.config.slip_outcome[2][1] = 7
    t = c.tables_struct()
    h = C.c_void_p()
    assert L.rlrm_create(C.byref(c.config), C.byref(t), 0, C.byref(h)) == -1 and "slip_outcome" in L.rlrm_last_error().decode()
    assert L.rlrm_create(None, None, 0, None) == -1
    with pytest.raises(ValueError):
        P.compile_scenario(P.scenario_config1(), grid=GridSpec("frozen_lake", 40, 40))
    sc = P.scenario_config1()
    sc.starts = [(0, 0)] * 9
    with pytest.raises(ValueError):
        P.compile_scenario(sc)


def test_value_iteration_rejects_bad_arguments():
    """rlrm_value_iteration needs no handle: its argument checks run before any device work."""
    from multiagent_rlrm_b200 import _lib

    L = _lib.load()
    buf = (C.c_double * 64)()
    p = C.addressof(buf)
    ok = dict(device=0, n=4, n_out=1, prob=p, nxt=p, rew=p, done=p, gamma=0.9, theta=1e-3, rel=0, sweeps=10, V=p, Q=p, pol=p, work=p)

    def call(**kw):
        a = {**ok, **kw}
        return L.rlrm_value_iteration(a["device"], a["n"], a["n_out"], a["prob"], a["nxt"], a["rew"], a["done"], a["gamma"], a["theta"],
                                      a["rel"], a["sweeps"], a["V"], a["Q"], a["pol"], a["work"], None, None)

    for kw, text in (({"prob": None}, "null"), ({"work": None}, "null"), ({"n": 0}, "n_states"), ({"n_out": 0}, "n_states"),
                     ({"theta": 0.0}, "theta"), ({"sweeps": 0}, "theta")):
        assert call(**kw) == -1 and text in L.rlrm_last_error().decode(), kw


@pytest.mark.gpu
def test_round2_entry_points_reject_bad_arguments(cuda_device):
    """rlrm_iterate / rlrm_update_list / rlrm_merge_replicas and the float64 table mode: error codes, never a crash."""
    import torch

    from multiagent_rlrm_b200._lib import RlrmError
    from multiagent_rlrm_b200.engine import Engine

    sc = P.scenario_config5(True)
    sc.table_dtype = "f64"
    with pytest.raises(RlrmError, match="float32"):     # the shared learner is specified on float32 tables
        Engine(P.compile_scenario(sc), 4)
    eng = Engine(P.compile_scenario(P.scenario_config5(True)), 8)
    eng.reset()
    L, st, stream = eng.L, C.byref(eng.state), eng._stream()
    rew = torch.zeros(8 * 4, dtype=torch.float64).pin_memory()
    assert L.rlrm_iterate(eng.h, st, 0, 1, None, rew.data_ptr(), stream) == -3 and "shared" in L.rlrm_last_error().decode()
    rec, none = eng.iterate()                           # record only: fine
    assert none is None and rec.shape == (32,)
    ex = (C.c_uint8 * 24)()
    assert L.rlrm_update_list(eng.h, st, 0, 1, C.addressof(ex), stream) == -3   # proposals need the synchronous iteration
    g = torch.zeros(2 * eng.q.numel(), device="cuda:0")
    assert L.rlrm_merge_replicas(eng.h, None, 2, eng.q.numel(), eng.q.data_ptr(), stream) == -1
    assert L.rlrm_merge_replicas(eng.h, g.data_ptr(), 0, eng.q.numel(), eng.q.data_ptr(), stream) == -1
    assert L.rlrm_merge_replicas(eng.h, g.data_ptr(), 2, eng.q.numel(), eng.q.data_ptr(), stream) == 0
    assert L.rlrm_stream_sync(None, stream) == -1 and L.rlrm_stream_sync(eng.h, stream) == 0
    assert float(eng.q.abs().sum()) == 0.0              # mean of two zero replicas
    plain = Engine(P.compile_scenario(P.scenario_config3(False)), 8)
    plain.reset()
    st2 = C.byref(plain.state)
    assert L.rlrm_update_list(plain.h, st2, 16, 1, C.addressof(ex), stream) == -1 and "slot" in L.rlrm_last_error().decode()
    assert L.rlrm_update_list(plain.h, st2, 0, 1, None, stream) == -1
    assert L.rlrm_update_list(plain.h, st2, 0, 0, None, stream) == 0            # an empty list is a no-op
    sp = Engine(P.compile_scenario(P.scenario_config4()), 2, qlambda_sparse=True)
    assert L.rlrm_update_list(sp.h, C.byref(sp.state), 0, 1, C.addressof(ex), stream) == -3  # needs dense traces
    with pytest.raises(RuntimeError, match="host_control"):
        plain.step_host([0] * 16)
    with pytest.raises(ValueError, match="table_dtype"):
        P.QLearning(gamma=0.9, action_selection="greedy", learning_rate=0.1, state_space_size=4, action_space_size=4, table_dtype="f16")
    big = P.scenario_config4()                          # 8 agents x 32-state machines x 60 events would exceed the 48 KB table blob
    assert P.compile_scenario(big).config.table_dtype == 0


@pytest.mark.gpu
def test_value_iteration_reports_non_convergence(cuda_device):
    """gamma = 1 with a rewarded self-loop never converges: RLRM_ERR_UNSUPPORTED after max_sweeps, as an exception in Python."""
    from multiagent_rlrm_b200._lib import RlrmError
    from multiagent_rlrm_b200.mdp_vi import value_iteration_arrays

    prob = np.ones((2, 4, 1))
    nxt = np.zeros((2, 4, 1), dtype=np.int32)
    rew = np.ones((2, 4, 1))
    done = np.zeros((2, 4, 1), dtype=np.uint8)
    with pytest.raises(RlrmError, match="did not converge"):
        value_iteration_arrays(prob, nxt, rew, done, gamma=1.0, theta=1e-3, max_sweeps=50)
    V, pol, Q, sweeps = value_iteration_arrays(prob, nxt, rew, done, gamma=0.5, theta=1e-9)
    assert np.allclose(V.cpu().numpy(), 2.0, atol=1e-8) and sweeps > 10  # 1 / (1 - 0.5)
    with pytest.raises(ValueError):
        value_iteration_arrays(prob, nxt + 5, rew, done)


@pytest.mark.gpu
def test_state_validation_errors(cuda_device):
    """check_state: every entry point refuses an incomplete or misaligned rlrm_state_t with an error code and a message."""
    import torch

    from multiagent_rlrm_b200 import _lib
    from multiagent_rlrm_b200.engine import Engine

    L = _lib.load()

    def rc_msg(eng, **override):
        st = abi.State.from_buffer_copy(bytes(eng.state))
        for k, v in override.items():
            setattr(st, k, v)
        rc = L.rlrm_train(eng.h, C.byref(st), 0, 1, 1, None, None)
        return rc, L.rlrm_last_error().decode()

    eng = Engine(P.compile_scenario(P.scenario_config3(True)), 8)
    eng.reset()
    assert rc_msg(eng)[0] == 0
    for override, text in (({"slot": None}, "slot"), ({"q": None}, "state.q is required"), ({"n_instances": 0}, "n_instances"),
                           ({"q": eng.q.data_ptr() + 4}, "32-byte aligned")):
        rc, msg = rc_msg(eng, **override)
        assert rc == -1 and text in msg, (override, rc, msg)
    assert L.rlrm_train(eng.h, C.byref(eng.state), 0, -1, 1, None, None) == -1

    sc = P.scenario_config3(False)
    sc.learning_rate = None
    lr_none = Engine(P.compile_scenario(sc), 8)
    rc, msg = rc_msg(lr_none, visits=None)
    assert rc == -1 and "visits" in msg

    qlam = Engine(P.compile_scenario(P.scenario_config4()), 4)
    rc, msg = rc_msg(qlam, e=None)
    assert rc == -1 and "Q(lambda) needs" in msg
    sparse = Engine(P.compile_scenario(P.scenario_config4()), 4, qlambda_sparse=True)
    rc, msg = rc_msg(sparse, tr_cap=10)
    assert rc == -1 and "tr_cap" in msg

    shared = Engine(P.compile_scenario(P.scenario_config5(True)), 8)
    rc, msg = rc_msg(shared, acc_sum=None)
    assert rc == -1 and "acc_sum" in msg
    torch.cuda.synchronize()
