"""GPU parity tests (run on the B200 box: pytest -m gpu). Every comparison is bit-exact: environment / RM / event /
reward / done traces, epsilon, statistics and float32 Q / trace tables of the CUDA path (through the C ABI) against
(a) the golden fixtures generated from the live reference and (b) the CPU oracle on the same seeded inputs."""
import numpy as np
import pytest

from conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu


def _engine(compiled, n, **kw):
    from multiagent_rlrm_b200.engine import Engine

    return Engine(compiled, n, device="cuda:0", **kw)


def _trace(tr, n, a):
    import oracle as O

    return O.unpack_trace(tr.cpu().numpy().view(np.uint32), n, a)


@pytest.mark.parametrize("name", golden_names())
def test_fused_kernel_matches_reference_golden(name, cuda_device):
    """Every fixture recorded from the live reference, float32-cast tables AND the reference's native float64 tables
    (`*_f64`: the device runs its float64 table mode, RLRM_TABLE_F64) — traces and final tables bit for bit."""
    import multiagent_rlrm_b200 as P

    meta, ref = load_golden(name)
    sc = P.Scenario.from_dict(meta["scenario"])
    sc.table_dtype = meta["real"]
    c = P.compile_scenario(sc)
    n, t = meta["n_instances"], meta["n_iters"]
    eng = _engine(c, n)
    for _ in range(meta["pre_resets"] + 1):
        eng.reset()
    tr = _trace(eng.train(t, trace=True), n, c.n_agents)
    for k in ("action", "cell", "q", "term", "trunc"):
        assert np.array_equal(tr[k], ref[k].astype(np.int32)), f"{name}: {k}"
    q = eng.q.cpu().numpy().reshape(ref["q_final"].shape)
    assert q.dtype == ref["q_final"].dtype == (np.float64 if meta["real"] == "f64" else np.float32)
    assert np.array_equal(q, ref["q_final"]), f"{name}: Q"
    if "e_final" in ref:
        assert np.array_equal(eng.e.cpu().numpy().reshape(ref["e_final"].shape), ref["e_final"]), f"{name}: traces"
    assert np.array_equal(eng.stats_numpy()["episodes"].reshape(n, -1)[:, 0], ref["episode_end"].sum(axis=0))


def _compare_with_oracle(eng, o, what=""):
    import oracle as O

    assert np.array_equal(eng.slot.cpu().numpy().view(np.uint64), o.slot), what + " slot state"
    assert np.array_equal(eng.epsilon.cpu().numpy(), o.epsilon), what + " epsilon"
    assert np.array_equal(eng.q.cpu().numpy(), o.q), what + " Q"
    if o.e is not None:
        assert np.array_equal(eng.e.cpu().numpy(), o.e), what + " traces"
    if o.visits is not None:
        assert np.array_equal(eng.visits.cpu().numpy().view(np.uint32), o.visits), what + " visits"
    assert np.array_equal(eng.ep_return.cpu().numpy(), o.ep_return), what + " ep_return"
    s = eng.stats_numpy()
    for f in O.STATS_DTYPE.names:
        assert np.array_equal(s[f], o.stats[f]), what + " stats." + f


def _scenarios_medium():
    import multiagent_rlrm_b200 as P

    out = {
        "cfg3_qrm": (P.scenario_config3(True), 2048, 1500),
        "cfg3_ql": (P.scenario_config3(False), 2048, 1500),
        "cfg5_qrm_4agents": (P.scenario_config5(False), 1024, 1200),
        "cfg2_office_slip": (P.scenario_config2(True), 1024, 1500),
    }
    sc = P.scenario_config4()
    sc.algo, sc.learning_rate, sc.q_init = "qrm", 0.1, 2.0
    out["office_chain12_qrm"] = (sc, 512, 1200)
    out["cfg4_qlambda"] = (P.scenario_config4(), 24, 1100)
    sc = P.scenario_config3(False)
    sc.learning_rate, sc.epsilon_start, sc.epsilon_end, sc.epsilon_decay = None, 0.6, 0.05, 0.97
    out["fl_lr_none_epsdecay"] = (sc, 512, 1500)
    sc = P.scenario_config5(False)
    sc.random_start_positions = True
    out["fl_random_starts_qrm"] = (sc, 1500, 1200)
    g = P.frozen_lake_grid("map1").goals
    for algo, lr in (("qrm", 1.0), ("ql", 0.2)):
        sc = P.scenario_config3(algo == "qrm")
        sc.algo, sc.learning_rate, sc.starts, sc.detector_positions = algo, lr, [(5, 0), (0, 0), (9, 9)], sorted(g.values())
        sc.rm_transitions_per_agent = [P.tables.frozen_lake_abc_transitions(), [("p0", g["C"], "p1", 3.0), ("p1", g["A"], "p2", 7.0)],
                                       [("w0", g["B"], "w1", 1.0), ("w1", g["A"], "w2", 1.0), ("w2", g["C"], "w3", 1.0),
                                        ("w3", g["B"], "w4", 5.0), ("w1", g["C"], "w0", -1.0)]]
        out[f"fl_per_agent_rms_{algo}"] = (sc, 700, 1300)
        if algo == "qrm":  # agents with different machines + potential-based shaping (one phi section per agent)
            import copy

            sh = copy.deepcopy(sc)
            sh.use_rsh, sh.rs_kind, sh.learning_rate = True, "vi", 0.5
            out["fl_per_agent_rms_shaping_qrm"] = (sh, 300, 1300)
        else:      # agents with different machines + Q(lambda) (per-agent table sizes in the trace sweeps)
            import copy

            ql = copy.deepcopy(sc)
            ql.algo, ql.lambd, ql.learning_rate, ql.q_init = "qlambda", 0.8, 0.2, 0.0
            out["fl_per_agent_rms_qlambda"] = (ql, 40, 1100)
    return out


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("name", list(_scenarios_medium().keys()))
def test_fused_kernel_matches_oracle(name, dtype, cuda_device):
    import multiagent_rlrm_b200 as P
    import oracle as O

    sc, n, t = _scenarios_medium()[name]
    sc.table_dtype = dtype
    c = P.compile_scenario(sc)
    eng = _engine(c, n)
    o = O.Oracle(c, n, dtype)
    eng.reset(); o.reset()
    # several launches with odd lengths: state must carry across launches exactly
    t0 = 0
    for chunk in (1, 7, t - 8 - 300, 300):
        tr_g = eng.train(chunk, trace=True)
        tr_o = o.train(t0, chunk, trace=True)
        assert np.array_equal(tr_g.cpu().numpy().view(np.uint32), tr_o), f"{name}: trace chunk starting at {t0}"
        t0 += chunk
    _compare_with_oracle(eng, o, name)


def _office_task(exp, algo, stochastic=True):
    import multiagent_rlrm_b200 as P

    return P.scenario_for_experiment("map1", exp, starts=[(2, 7), (6, 3), (0, 0)], algo=algo, learning_rate=0.1 if stochastic else 1.0,
                                     gamma=0.9, stochastic=stochastic, epsilon_start=0.1, epsilon_end=0.1, epsilon_decay=1.0, q_init=2.0,
                                     wall_penalty=-0.5, max_steps=200, seed=97)


def _shaped_qrm():
    import multiagent_rlrm_b200 as P

    sc = P.scenario_config3(True)
    sc.use_rsh, sc.rs_kind, sc.rs_alpha, sc.learning_rate = True, "distance", 5, 0.5
    return sc


@pytest.mark.parametrize("name", ["cfg3_qrm", "cfg5_qrm_4agents", "cfg3_ql", "office_exp1_qrm", "office_exp3_qrm", "office_exp4_qrm_det",
                                  "office_exp2_ql", "office_exp5_qrm", "office_exp6_qrm", "office_exp6_qrm_det", "office_chain12_qrm",
                                  "fl_random_starts_qrm", "fl_shaping_qrm"])
def test_generic_kernel_equals_specialised(name, cuda_device):
    """config.reserved bit 0 forces the generic train_kernel; it must agree bit-for-bit with the specialised kernels
    (train_qrm4_kernel, train_qrmn_kernel<3 / 5 RM states>, train_ql_fast_kernel, and train_qrm_block_kernel for machines with
    more states / permuted state order / shaping / random starts) — and both with the oracle."""
    import multiagent_rlrm_b200 as P
    import oracle as O
    from test_fuzz_kernels_gpu import launched_train_kernels

    if name == "fl_shaping_qrm":
        sc, n, t = _shaped_qrm(), 400, 1500
    elif name.startswith("office_exp"):
        sc = {"office_exp1_qrm": lambda: _office_task("exp1", "qrm"), "office_exp3_qrm": lambda: _office_task("exp3", "qrm"),
              "office_exp4_qrm_det": lambda: _office_task("exp4", "qrm", False), "office_exp2_ql": lambda: _office_task("exp2", "ql"),
              "office_exp5_qrm": lambda: _office_task("exp5", "qrm"), "office_exp6_qrm": lambda: _office_task("exp6", "qrm"),
              "office_exp6_qrm_det": lambda: _office_task("exp6", "qrm", False)}[name]()
        n, t = 300, 1500
    else:
        sc, n, t = _scenarios_medium()[name]
    c_fast, c_gen = P.compile_scenario(sc), P.compile_scenario(sc)
    c_gen.config.reserved = 1
    a, b = _engine(c_fast, n), _engine(c_gen, n)
    a.reset(); b.reset()
    out = {}
    ka = launched_train_kernels(lambda: out.update(a=a.train(t, trace=True)))
    kb = launched_train_kernels(lambda: out.update(b=b.train(t, trace=True)))
    # the comparison means something only if the two engines ran different kernels. The helper relies on CUPTI's kernel records,
    # which torch.profiler drops in processes that have run for a minute or more (see launched_train_kernels): this file runs
    # early enough in the suite, and a dropout fails loudly instead of passing
    assert [k.family for k in kb] == ["train_kernel"] and len(ka) == 1 and ka[0].family != "train_kernel", (ka, kb)
    ta, tb = out["a"], out["b"]
    assert np.array_equal(ta.cpu().numpy(), tb.cpu().numpy())
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy())
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())
    assert np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy())
    o = O.Oracle(c_fast, n, "f32")
    o.reset()
    o.train(0, t)
    assert np.array_equal(a.q.cpu().numpy().reshape(-1), o.q.reshape(-1)) and np.array_equal(a.slot.cpu().numpy().view(np.uint64), o.slot)
    assert int(o.stats["episodes"].sum()) > 0


@pytest.mark.parametrize("name", ["cfg3_qrm", "cfg5_qrm_4agents", "office_exp1_qrm", "office_exp3_qrm", "office_exp6_qrm", "office_chain12_qrm",
                                  "fl_random_starts_qrm", "fl_shaping_qrm"])
def test_float64_block_kernel_equals_generic_and_oracle(name, cuda_device):
    """Float64 tables (the reference's own arithmetic): QRM takes train_qrm_block_kernel<.., double> (cell block of two 16-byte
    chunks per row in shared memory); it must agree bit-for-bit with the generic float64 kernel (config.reserved bit 0) and
    with the float64 oracle — traces, tables, slot words and statistics."""
    import copy

    import torch

    import multiagent_rlrm_b200 as P
    import oracle as O

    if name == "fl_shaping_qrm":
        sc, n, t = _shaped_qrm(), 400, 1500
    elif name.startswith("office_exp"):
        sc, n, t = _office_task(name.split("_")[1], "qrm"), 300, 1500
    else:
        sc, n, t = _scenarios_medium()[name]
    sc = copy.deepcopy(sc)
    sc.table_dtype = "f64"
    c_fast, c_gen = P.compile_scenario(sc), P.compile_scenario(sc)
    c_gen.config.reserved = 1
    a, b = _engine(c_fast, n), _engine(c_gen, n)
    a.reset(); b.reset()
    ta, tb = a.train(t, trace=True), b.train(t, trace=True)
    a.train(137); b.train(137)  # a second launch picks the state up from memory
    assert a.q.dtype == torch.float64
    assert np.array_equal(ta.cpu().numpy(), tb.cpu().numpy())
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy())
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())
    assert np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy())
    o = O.Oracle(c_fast, n, "f64")
    o.reset()
    o.train(0, t + 137)
    assert np.array_equal(a.q.cpu().numpy().reshape(-1), o.q.reshape(-1)) and np.array_equal(a.slot.cpu().numpy().view(np.uint64), o.slot)
    assert int(o.stats["episodes"].sum()) > 0


@pytest.mark.parametrize("tma", ["0", "1"])
@pytest.mark.parametrize("name,dtype", [("cfg3_qrm", "f64"), ("office_exp3_qrm", "f64"), ("office_exp6_qrm", "f32"), ("office_chain12_qrm", "f32"),
                                        ("office_chain12_qrm", "f64"), ("fl_shaping_qrm", "f32"), ("fl_random_starts_qrm", "f64")])
def test_block_kernel_fetch_variants_equal_oracle(name, dtype, tma, cuda_device, monkeypatch):
    """train_qrm_block_kernel fetches the cell block either with one cp.async per 16-byte chunk or with ONE bulk copy per thread
    (cp.async.bulk + mbarrier; the library picks it from 192-byte blocks on). RLRM_QRMB_TMA forces either variant for every
    block size and table type: traces, tables, slot words and statistics must equal the oracle in both."""
    import copy

    import multiagent_rlrm_b200 as P
    import oracle as O

    monkeypatch.setenv("RLRM_QRMB_TMA", tma)
    if name == "fl_shaping_qrm":
        sc, n, t = _shaped_qrm(), 300, 900
    elif name.startswith("office_exp"):
        sc, n, t = _office_task(name.split("_")[1], "qrm"), 300, 900
    else:
        sc, n, t = _scenarios_medium()[name]
    sc = copy.deepcopy(sc)
    sc.table_dtype = dtype
    c = P.compile_scenario(sc)
    a = _engine(c, n)
    a.reset()
    ta = a.train(t, trace=True)
    a.train(77)
    o = O.Oracle(c, n, dtype)
    o.reset()
    to = o.train(0, t, trace=True)
    o.train(t, 77)
    assert np.array_equal(ta.cpu().numpy().view(np.uint32), to)
    assert np.array_equal(a.q.cpu().numpy().reshape(-1), o.q.reshape(-1)) and np.array_equal(a.slot.cpu().numpy().view(np.uint64), o.slot)
    assert np.array_equal(a.stats_numpy()["episodes"], o.stats["episodes"]) and int(o.stats["episodes"].sum()) > 0


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("name", ["cfg3_qrm", "cfg3_ql", "cfg2_office_slip", "cfg4_qlambda", "fl_per_agent_rms_qrm",
                                  "fl_per_agent_rms_ql", "fl_random_starts_qrm", "fl_per_agent_rms_qlambda", "fl_per_agent_rms_shaping_qrm"])
def test_unfused_entry_points_equal_fused(name, dtype, cuda_device):
    """select -> step -> update -> reset through the separate C-ABI calls == the fused persistent kernel."""
    import multiagent_rlrm_b200 as P

    sc, n, _ = _scenarios_medium()[name]
    sc.table_dtype = dtype
    n = min(n, 256)
    iters = 260 if name != "cfg4_qlambda" else 60
    c = P.compile_scenario(sc)
    a, b = _engine(c, n), _engine(c, n)
    a.reset(); b.reset()
    tr = _trace(a.train(iters, trace=True), n, c.n_agents)
    for it in range(iters):
        actions, rec, _over = b.iterate_unfused()
        assert np.array_equal(actions.cpu().numpy().astype(np.int32), tr["action"][it]), f"action at {it}"
        assert np.array_equal(rec["cell"].cpu().numpy().view(np.uint16).reshape(n, -1).astype(np.int32), tr["cell"][it])
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy())
    assert np.array_equal(a.epsilon.cpu().numpy(), b.epsilon.cpu().numpy())
    if a.e is not None:
        assert np.array_equal(a.e.cpu().numpy(), b.e.cpu().numpy())


def test_injected_draws_equal_philox(cuda_device):
    """The draws= injection path consumes the same words the in-kernel Philox generates."""
    import torch

    import multiagent_rlrm_b200 as P
    import philox

    sc = P.scenario_config3(True)
    c = P.compile_scenario(sc)
    n = 128
    a, b = _engine(c, n), _engine(c, n)
    a.reset(); b.reset()
    for it in range(120):
        d = torch.from_numpy(philox.draws(sc.seed, it, n, c.n_agents).astype(np.int64)).to(torch.int32).cuda().contiguous()
        a.iterate_unfused(draws=d.view(-1))
        b.iterate_unfused()
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy())


def test_full_size_config3_windows_match_oracle(cuda_device):
    """BASELINE config 3 at full size (65,536 instances x 2 agents): instances are independent and keyed on their
    global id, so windows of the batch must equal the oracle run with the matching instance_offset."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    sc = P.scenario_config3(True)
    c = P.compile_scenario(sc)
    n, iters = 65536, 700
    eng = _engine(c, n)
    eng.reset()
    eng.train(iters)
    slots = eng.slot.cpu().numpy().view(np.uint64).reshape(n, 2)
    q = eng.q.cpu().numpy().reshape(n, 2, -1)
    stats = eng.stats_numpy().reshape(n, 2)
    for start in (0, 31337, 65536 - 48):
        cw = P.compile_scenario(sc, instance_offset=start)
        o = O.Oracle(cw, 48, "f32")
        o.reset()
        o.train(0, iters)
        assert np.array_equal(slots[start:start + 48].reshape(-1), o.slot)
        assert np.array_equal(q[start:start + 48].reshape(o.q.shape), o.q)
        assert np.array_equal(stats["active_steps"][start:start + 48].reshape(-1), o.stats["active_steps"])
    # size-independent invariants of the whole batch
    s = eng.slots_numpy()
    assert (s["timestep"][:, 0] == s["timestep"][:, 1]).all()          # the shared env.timestep stays replicated
    assert (s["timestep"] <= 1001).all() and (s["agent_steps"] <= s["timestep"]).all()
    assert int(stats["active_steps"].sum()) <= n * 2 * iters
    assert np.isfinite(q).all()


def test_shared_learner_matches_oracle(cuda_device):
    """BASELINE config 5 shared-learner mode (one table per agent index, synchronous proposal averaging):
    the integer accumulation makes the CUDA result independent of thread order, so it equals the oracle bit for bit."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    sc = P.scenario_config5(shared=True)
    c = P.compile_scenario(sc)
    n, iters = 3000, 160
    eng = _engine(c, n)
    o = O.Oracle(c, n, "f32")
    eng.reset(); o.reset()
    tr_g = eng.train(iters, trace=True)
    tr_o = o.train(0, iters, trace=True)
    assert np.array_equal(tr_g.cpu().numpy().view(np.uint32), tr_o)
    _compare_with_oracle(eng, o, "shared learner")
    assert int(eng.acc_cnt.abs().sum()) == 0 and int(eng.acc_sum.abs().sum()) == 0  # accumulators are left clean


@pytest.mark.parametrize("n,chunks", [(1, (1, 2, 3, 7)), (37, (5, 1, 64)), (3000, (160,)), (200000, (3, 40))])
def test_shared_learner_persistent_kernel_equals_two_launch_path_and_oracle(n, chunks, cuda_device):
    """rlrm_train runs the shared learner's iterations in one cooperative launch (shared_train_kernel: tables in shared
    memory for the whole launch, three global accumulator sets used round-robin, one grid barrier per iteration). It must
    equal the two-launches-per-iteration path (config.reserved bit 1) and the oracle for any launch length and grid size."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    sc = P.scenario_config5(shared=True)
    c_coop, c_two = P.compile_scenario(sc), P.compile_scenario(sc)
    c_two.config.reserved = 2
    a, b = _engine(c_coop, n), _engine(c_two, n)
    o = O.Oracle(c_coop, n, "f32") if n <= 3000 else None
    a.reset(); b.reset()
    if o:
        o.reset()
    t0 = 0
    for chunk in chunks:
        a.train(chunk); b.train(chunk)
        if o:
            o.train(t0, chunk)
        t0 += chunk
        assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy()), f"Q after {t0} iterations"
        assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())
    assert a.launches == len(chunks) + 1 and b.launches > a.launches       # reset + ONE launch per train call
    assert np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy()) and np.array_equal(a.epsilon.cpu().numpy(), b.epsilon.cpu().numpy())
    assert np.array_equal(a.ep_return.cpu().numpy(), b.ep_return.cpu().numpy())
    assert int(a.acc_cnt.abs().sum()) == 0 and int(a.acc_sum.abs().sum()) == 0
    if o:
        _compare_with_oracle(a, o, "persistent shared learner")
    # the OfficeWorld shared learner (plain QL on the 5-state A->C->B->D task) takes the same path
    sc = P.scenario_config2(True)
    sc.shared_q, sc.starts = True, [(2, 7), (6, 3)]
    c1, c2 = P.compile_scenario(sc), P.compile_scenario(sc)
    c2.config.reserved = 2
    a, b = _engine(c1, min(n, 5000)), _engine(c2, min(n, 5000))
    a.reset(); b.reset()
    a.train(90); b.train(90)
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy()) and np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())


@pytest.mark.parametrize("name", ["cfg5_forced_cluster", "office12_4agents", "office12_8agents", "office_acbd_ql_forced"])
def test_shared_learner_cluster_kernel_equals_two_launch_path_and_oracle(name, cuda_device):
    """Shared tables that do not fit in one SM's shared memory are partitioned over the distributed shared memory of a
    thread-block cluster (shared_train_cluster_kernel, 2 / 4 / 8 blocks). It must equal the two-launches-per-iteration path
    (config.reserved bit 1; global-memory proposals for these sizes) and the oracle; `reserved` bit 2 forces it for tables that
    would fit in one SM, where it must also equal the single-block persistent kernel."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    if name == "cfg5_forced_cluster":
        sc, n, force = P.scenario_config5(shared=True), 3000, True
    elif name == "office_acbd_ql_forced":
        sc, n, force = P.scenario_config2(True), 2500, True
        sc.shared_q, sc.starts = True, [(2, 7), (6, 3), (0, 0)]
    else:
        sc, n, force = P.scenario_config4(), 2000, False
        sc.algo, sc.learning_rate, sc.q_init, sc.shared_q = "qrm", 0.1, 2.0, True
        if name == "office12_8agents":
            sc.starts = sc.starts + [(5, 5), (8, 2), (1, 1), (10, 7)]
    c_cl, c_two = P.compile_scenario(sc), P.compile_scenario(sc)
    c_cl.config.reserved = 4 if force else 0
    c_two.config.reserved = 2
    a, b = _engine(c_cl, n), _engine(c_two, n)
    o = O.Oracle(c_cl, n, "f32")
    a.reset(); b.reset(); o.reset()
    t0 = 0
    for chunk in (1, 2, 3, 70):
        a.train(chunk); b.train(chunk); o.train(t0, chunk)
        t0 += chunk
        assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy()), f"{name}: Q after {t0} iterations"
    assert a.launches == 5 and b.launches > a.launches                      # reset + ONE launch per train call
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy()) and np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy())
    assert np.array_equal(a.ep_return.cpu().numpy(), b.ep_return.cpu().numpy())
    assert int(a.acc_cnt.abs().sum()) == 0 and int(a.acc_sum.abs().sum()) == 0
    _compare_with_oracle(a, o, name)
    if force:  # the single-block persistent kernel on the same scenario
        c1 = P.compile_scenario(sc)
        e1 = _engine(c1, n)
        e1.reset()
        e1.train(76)
        assert np.array_equal(e1.q.cpu().numpy(), a.q.cpu().numpy()) and np.array_equal(e1.slot.cpu().numpy(), a.slot.cpu().numpy())


def test_shared_learner_with_one_instance_is_the_reference_learner(cuda_device):
    """Degenerate tie to the reference: N = 1 shared == per-instance tables (which equal the reference trace)."""
    import multiagent_rlrm_b200 as P

    a = _engine(P.compile_scenario(P.scenario_config5(shared=True)), 1)
    b = _engine(P.compile_scenario(P.scenario_config5(shared=False)), 1)
    a.reset(); b.reset()
    ta, tb = a.train(900, trace=True), b.train(900, trace=True)
    assert np.array_equal(ta.cpu().numpy(), tb.cpu().numpy())
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy())
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())


def test_full_size_config4_qlambda_windows_match_oracle(cuda_device):
    """BASELINE config 4 at full size (262,144 OfficeWorld instances x 4 agents, Q(lambda), 43.5 GB of tables):
    windows of the batch equal the oracle run with the matching instance_offset; traces obey their invariants."""
    import torch

    import multiagent_rlrm_b200 as P
    import oracle as O

    sc = P.scenario_config4()
    c = P.compile_scenario(sc)
    n, iters = 262144, 24
    free, _total = torch.cuda.mem_get_info()
    if free < 50e9:
        pytest.skip("needs ~45 GB of free device memory")
    eng = _engine(c, n)
    eng.reset()
    eng.train(iters)
    for start in (0, 200001):
        cw = P.compile_scenario(sc, instance_offset=start)
        o = O.Oracle(cw, 3, "f32")
        o.reset()
        o.train(0, iters)
        sl = slice(start * 4, (start + 3) * 4)
        assert np.array_equal(eng.slot[sl].cpu().numpy().view(np.uint64), o.slot)
        assert np.array_equal(eng.q[sl].cpu().numpy(), o.q)
        assert np.array_equal(eng.e[sl].cpu().numpy(), o.e)
    e = eng.e[: 4096 * 4]
    assert float(e.min()) >= 0.0 and float(e.max()) <= 1.0           # replacing traces live in [0, 1]
    assert int((e != 0).sum(dim=(1, 2)).max()) <= iters                # at most one new trace per step
    del eng
    torch.cuda.empty_cache()


def test_full_size_config5_windows_match_oracle(cuda_device):
    """BASELINE config 5 companion at full size (1,048,576 FrozenLake instances x 4 agents, per-instance tables, 26.8 GB)."""
    import torch

    import multiagent_rlrm_b200 as P
    import oracle as O

    sc = P.scenario_config5(shared=False)
    c = P.compile_scenario(sc)
    n, iters = 1048576, 300
    free, _total = torch.cuda.mem_get_info()
    if free < 32e9:
        pytest.skip("needs ~28 GB of free device memory")
    eng = _engine(c, n)
    eng.reset()
    eng.train(iters)
    for start in (0, 777777, n - 16):
        cw = P.compile_scenario(sc, instance_offset=start)
        o = O.Oracle(cw, 16, "f32")
        o.reset()
        o.train(0, iters)
        sl = slice(start * 4, (start + 16) * 4)
        assert np.array_equal(eng.slot[sl].cpu().numpy().view(np.uint64), o.slot)
        assert np.array_equal(eng.q[sl].cpu().numpy(), o.q)
    assert eng.total_active_steps() <= n * 4 * iters
    del eng
    torch.cuda.empty_cache()


def test_shared_learner_generic_path_equals_fast_path(cuda_device):
    """config.reserved bit 0 forces the global-atomic propose path; it must agree with shared_propose_kernel."""
    import multiagent_rlrm_b200 as P

    sc = P.scenario_config5(shared=True)
    c_fast, c_gen = P.compile_scenario(sc), P.compile_scenario(sc)
    c_gen.config.reserved = 1
    a, b = _engine(c_fast, 5000), _engine(c_gen, 5000)
    a.reset(); b.reset()
    ta, tb = a.train(120, trace=True), b.train(120, trace=True)
    assert np.array_equal(ta.cpu().numpy(), tb.cpu().numpy())
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy())
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy())
    assert np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy())
    assert np.array_equal(a.ep_return.cpu().numpy(), b.ep_return.cpu().numpy())


@pytest.mark.parametrize("name,n,iters", [("cfg4_office_chain12_qlambda", 48, 1300), ("fl_qlambda", 64, 1500),
                                            ("long_office_coffee_qlambda", 8, 12000), ("cfg4_office_chain12_qlambda_f64", 24, 1300),
                                            ("fl_qlambda_lr_none_f64", 32, 1500), ("long_office_coffee_qlambda_f64", 4, 12000)])
def test_sparse_exact_qlambda_equals_dense_and_oracle(name, n, iters, cuda_device):
    """The sparse-exact trace lists (live entries only, q values cached in the list) reproduce the dense sweep of
    QLearningLambda.update bit for bit: vs the dense CUDA kernel and vs the oracle, across several launches, with
    terminated updates and episode resets wiping the lists in between."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    meta, _ref = load_golden(name)
    sc = P.Scenario.from_dict(meta["scenario"])
    sc.table_dtype = meta["real"]
    c = P.compile_scenario(sc)
    sp, de = _engine(c, n, qlambda_sparse=True), _engine(c, n)
    o = O.Oracle(c, n, meta["real"])
    sp.reset(); de.reset(); o.reset()
    t0 = 0
    for chunk in (3, 250, iters - 253):
        ts, td = sp.train(chunk, trace=True), de.train(chunk, trace=True)
        to = o.train(t0, chunk, trace=True)
        assert np.array_equal(ts.cpu().numpy().view(np.uint32), to) and np.array_equal(td.cpu().numpy().view(np.uint32), to)
        t0 += chunk
        e_dense = sp.sync_tables(with_traces=True)
        assert np.array_equal(sp.q.cpu().numpy(), o.q), f"q after {t0}"
        assert np.array_equal(e_dense.cpu().numpy(), o.e), f"traces after {t0}"
        assert np.array_equal(de.q.cpu().numpy(), o.q) and np.array_equal(de.e.cpu().numpy(), o.e)
    assert np.array_equal(sp.slot.cpu().numpy().view(np.uint64), o.slot)
    assert np.array_equal(sp.stats_numpy()["episodes"], o.stats["episodes"])
    live = (o.e != 0).sum(axis=(1, 2))
    assert int(sp.tr_len.max()) <= sp.tr_cap and (sp.tr_len.cpu().numpy() >= live).all()
    # a masked reset flushes and forgets the lists of the selected instances only
    import torch

    mask = torch.zeros(n, dtype=torch.uint8)
    mask[::2] = 1
    sp.reset(mask); o.reset(mask.numpy())
    e_dense = sp.sync_tables(with_traces=True)
    assert np.array_equal(sp.q.cpu().numpy(), o.q) and np.array_equal(e_dense.cpu().numpy(), o.e)
    assert int(sp.tr_len.view(n, -1)[::2].sum()) == 0


@pytest.mark.parametrize("agents", [1, 2, 3, 4])
@pytest.mark.parametrize("n", [1, 3, 5, 37])
def test_sparse_qlambda_lane_layout_ragged_instance_counts(agents, n, cuda_device):
    """The sparse Q(lambda) kernel packs several instances into one warp (eight lanes per agent: 4 / 2 / 1 / 1 instances per warp
    for 1 / 2 / 3 / 4 agents). Instance counts that leave the last warp partly empty, and agent counts that are not a power of
    two, must not change anything: traces, tables, slot words and trace lists against the oracle."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    sc = P.scenario_config4()
    sc.starts = sc.starts[:agents]
    sc.max_steps = 60
    c = P.compile_scenario(sc)
    sp = _engine(c, n, qlambda_sparse=True)
    o = O.Oracle(c, n, "f32")
    sp.reset(); o.reset()
    t0 = 0
    for chunk in (1, 130, 400):
        ts = sp.train(chunk, trace=True)
        to = o.train(t0, chunk, trace=True)
        assert np.array_equal(ts.cpu().numpy().view(np.uint32), to)
        t0 += chunk
    e_dense = sp.sync_tables(with_traces=True)
    assert np.array_equal(sp.q.cpu().numpy(), o.q) and np.array_equal(e_dense.cpu().numpy(), o.e)
    assert np.array_equal(sp.slot.cpu().numpy().view(np.uint64), o.slot)
    assert np.array_equal(sp.stats_numpy()["episodes"], o.stats["episodes"]) and int(o.stats["episodes"].sum()) > 0


@pytest.mark.parametrize("name", ["cfg3_qrm", "cfg3_ql", "cfg2_office_slip"])
def test_batched_reference_style_driver_loop_equals_fused(name, cuda_device):
    """The reference driver loop written with the batched API (vec.BatchedRMEnvironment: reset / select_action / step /
    update_policy with [N, A] tensors) gives the same tables and states as the fused kernel."""
    import multiagent_rlrm_b200 as P

    sc, n, _ = _scenarios_medium()[name]
    n, iters = 192, 220
    env = P.BatchedRMEnvironment(sc, n)
    fused = _engine(P.compile_scenario(sc), n)
    fused.reset()
    fused.train(iters)
    fl = sc.driver == "frozen_lake_main"
    states, _ = env.reset()
    for _ in range(iters):
        actions = env.select_action(states)
        new_states, rewards, terminated, truncated, infos = env.step(actions)
        env.update_policy(env.driver_states(states, new_states), actions, rewards, new_states,
                          (terminated | truncated) if fl else terminated, infos)
        states = new_states
        over = env.episode_over(terminated, truncated)
        if bool(over.any()):
            states, _ = env.reset(mask=over)
    assert np.array_equal(env.engine.slot.cpu().numpy(), fused.slot.cpu().numpy())
    assert np.array_equal(env.q_table.cpu().numpy().reshape(-1), fused.q.cpu().numpy().reshape(-1))
    assert np.array_equal(env.engine.epsilon.cpu().numpy(), fused.epsilon.cpu().numpy())
