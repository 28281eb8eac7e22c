"""GPU: hyper-parameter sweeps (Engine(sweep=...), rlrm_set_sweep). Instance i of a sweep engine must behave bit for bit as
instance i of a uniform engine built with its group's setting; the reference for group g is the uniform CPU oracle on
compile_scenario(scenario with that setting, instance_offset=g*k). One scenario per training-kernel family."""
import copy
import ctypes as C

import numpy as np
import pytest

import multiagent_rlrm_b200 as P

pytestmark = pytest.mark.gpu

# settings that differ in learning rate, discount, lambda and epsilon schedule; {} = the scenario's own
_SETTINGS = [
    {"learning_rate": 0.5, "gamma": 0.9, "lambd": 0.5, "epsilon_start": 0.6, "epsilon_end": 0.05, "epsilon_decay": 0.9},
    {"learning_rate": 0.05, "gamma": 0.99, "lambd": 0.9, "epsilon_start": 0.3, "epsilon_end": 0.1, "epsilon_decay": 0.99},
    {"learning_rate": 0.9, "gamma": 0.8, "lambd": 0.0, "epsilon_start": 1.0, "epsilon_end": 0.02, "epsilon_decay": 0.95},
    {},
]


def _office_task(exp, algo):
    return P.scenario_for_experiment("map1", exp, starts=[(2, 7), (6, 3), (0, 0)], algo=algo, learning_rate=0.1, gamma=0.9,
                                     stochastic=True, epsilon_start=0.1, epsilon_end=0.1, epsilon_decay=1.0, q_init=2.0,
                                     wall_penalty=-0.5, max_steps=200, seed=97)


def _chain12(dtype):
    sc = P.scenario_config4()
    sc.algo, sc.learning_rate, sc.q_init, sc.table_dtype = "qrm", 0.1, 2.0, dtype
    sc.max_steps = 150  # episodes end (truncate) within the run, so the epsilon schedules take effect
    return sc


def _config4():
    sc = P.scenario_config4()
    sc.max_steps = 150
    return sc


def _per_agent(algo):
    g = P.frozen_lake_grid("map1").goals
    sc = P.scenario_config3(True)
    sc.algo, sc.learning_rate = algo, 0.3
    sc.detector_positions = sorted(g.values())
    sc.rm_transitions_per_agent = [P.tables.frozen_lake_abc_transitions(), [("p0", g["B"], "p1", 3.0), ("p1", g["A"], "p2", 7.0)]]
    return sc


def _shaped():
    sc = P.scenario_config3(True)
    sc.use_rsh, sc.rs_kind, sc.rs_alpha, sc.learning_rate = True, "distance", 5, 0.5
    return sc


# name -> (scenario, settings, k, iterations, Engine keyword arguments). The block kernel fetches cell blocks of 192 bytes and more
# with bulk copies (TMA: chain12) and smaller ones with cp.async (exp5's 144 bytes, config 3 in float64: 128 bytes).
def _case(name):
    no_gamma = [{k: v for k, v in s.items() if k != "gamma"} for s in _SETTINGS]
    if name == "qrm4_minb7":
        return P.scenario_config3(True), _SETTINGS, 256, 600, {}
    if name == "qrm4_minb8":  # more than 7 resident blocks per SM of threads: the 64-register instantiation
        return P.scenario_config3(True), _SETTINGS, 17408, 150, {}
    if name == "ql_fast":
        return P.scenario_config3(False), _SETTINGS, 256, 600, {}
    if name == "qrmn_3":
        return _office_task("exp1", "qrm"), _SETTINGS[:3], 128, 600, {}
    if name == "qrmn_5":
        return _office_task("exp3", "qrm"), _SETTINGS[:3], 128, 600, {}
    if name == "qrm_block_f32":
        return _chain12("f32"), _SETTINGS, 64, 500, {}
    if name == "qrm_block_f64":
        return _chain12("f64"), _SETTINGS, 64, 500, {}
    if name == "qrm_block_f32_cpasync":
        return _office_task("exp5", "qrm"), _SETTINGS[:3], 96, 500, {}
    if name == "qrm_block_f64_cpasync":
        sc = P.scenario_config3(True)
        sc.table_dtype = "f64"
        return sc, _SETTINGS, 128, 500, {}
    if name == "cfg2_office_ql":
        return P.scenario_config2(True), _SETTINGS, 128, 600, {}
    if name == "qlambda_dense":
        return _config4(), _SETTINGS[:3], 8, 400, {}
    if name == "qlambda_sparse":
        return _config4(), _SETTINGS[:3], 8, 400, {"qlambda_sparse": True}
    if name == "per_agent_qrm":
        return _per_agent("qrm"), _SETTINGS, 96, 600, {}
    if name == "per_agent_qlambda":
        return _per_agent("qlambda"), _SETTINGS[:3], 8, 300, {}
    if name == "shaping_qrm":
        return _shaped(), no_gamma, 128, 600, {}
    if name == "lr_none":
        sets = copy.deepcopy(_SETTINGS[:3])
        sets[1]["learning_rate"] = None
        return P.scenario_config3(True), sets, 128, 600, {}
    raise KeyError(name)


FAMILIES = ["qrm4_minb7", "qrm4_minb8", "ql_fast", "qrmn_3", "qrmn_5", "qrm_block_f32", "qrm_block_f64", "qrm_block_f32_cpasync",
            "qrm_block_f64_cpasync", "cfg2_office_ql",
            "qlambda_dense", "qlambda_sparse", "per_agent_qrm", "per_agent_qlambda", "shaping_qrm", "lr_none"]


def _engine(sc, n, reserved=0, **kw):
    from multiagent_rlrm_b200.engine import Engine

    c = P.compile_scenario(sc, instance_offset=kw.pop("instance_offset", 0))
    c.config.reserved = reserved
    return Engine(c, n, device="cuda:0", **kw)


def _state(eng):
    """every state array of the engine (host numpy), the sparse traces materialised into q and e"""
    e = eng.sync_tables(with_traces=True)
    out = {"slot": eng.slot, "epsilon": eng.epsilon, "q": eng.q, "ep_return": eng.ep_return, "stats": eng.stats}
    if e is not None:
        out["e"] = e
    if eng.visits is not None:
        out["visits"] = eng.visits
    return {k: v.cpu().numpy() for k, v in out.items()}


def _same_state(a, b):
    sa, sb = _state(a), _state(b)
    assert sa.keys() == sb.keys()
    for k in sa:
        assert sa[k].tobytes() == sb[k].tobytes(), k


def _setting_scenario(sc, s):
    scg = copy.deepcopy(sc)
    for k, v in s.items():
        setattr(scg, k, v)
    return scg


@pytest.mark.parametrize("name", FAMILIES)
def test_sweep_equals_per_group_oracle(name, cuda_device):
    import oracle as O

    sc, sets, k, iters, kw = _case(name)
    H = len(sets)
    eng = _engine(sc, H * k, sweep=sets, **kw)
    eng.reset()
    eng.train(iters // 2)
    eng.train(iters - iters // 2)  # a second launch picks the state up from memory
    st = _state(eng)
    A = eng.A
    episodes = 0
    for g, s in enumerate(eng.sweep):
        cg = P.compile_scenario(_setting_scenario(sc, s), instance_offset=g * k)
        o = O.Oracle(cg, k, track_visits=eng.visits is not None)
        o.reset()
        o.train(0, iters)
        sl = slice(g * k * A, (g + 1) * k * A)
        assert st["slot"].view(np.uint64)[sl].tobytes() == o.slot.tobytes(), (g, "slot")
        assert st["epsilon"][sl].tobytes() == o.epsilon.tobytes(), (g, "epsilon")
        assert st["ep_return"][sl].tobytes() == o.ep_return.tobytes(), (g, "ep_return")
        assert st["stats"][sl].tobytes() == o.stats.tobytes(), (g, "stats")
        rows = st["q"].reshape(H * k, -1)[g * k:(g + 1) * k]
        assert rows.tobytes() == o.q.tobytes(), (g, "q")
        if "e" in st:
            assert st["e"].reshape(H * k, -1)[g * k:(g + 1) * k].tobytes() == o.e.tobytes(), (g, "e")
        if "visits" in st:
            assert st["visits"].reshape(H * k, -1)[g * k:(g + 1) * k].view(np.uint32).tobytes() == o.visits.tobytes(), (g, "visits")
        episodes += int(o.stats["episodes"].sum())
    assert episodes > 0  # episodes ended and restarted: the epsilon schedules took effect


@pytest.mark.parametrize("name", FAMILIES)
def test_degenerate_sweep_equals_uniform_engine(name, cuda_device):
    sc, sets, k, iters, kw = _case(name)
    sets = [{} for _ in sets]  # every setting is the scenario's own
    n = len(sets) * k
    uni, swp = _engine(sc, n, **kw), _engine(sc, n, sweep=sets, **kw)
    uni.reset(); swp.reset()
    ta, tb = uni.train(iters, trace=True), swp.train(iters, trace=True)
    assert np.array_equal(ta.cpu().numpy(), tb.cpu().numpy())
    _same_state(uni, swp)


@pytest.mark.parametrize("name", ["qrm4_minb7", "ql_fast", "qrmn_3", "qrmn_5", "qrm_block_f32", "qrm_block_f64", "qrm_block_f32_cpasync",
                                  "qrm_block_f64_cpasync", "shaping_qrm"])
def test_forced_generic_equals_fast_path_under_a_sweep(name, cuda_device):
    # that these two engines run different kernels is checked by test_forced_generic_sweep_engines_run_different_kernels
    # (tests/test_fuzz_kernels_gpu.py), early in the suite, where the profiler still records kernels
    sc, sets, k, iters, kw = _case(name)
    n = len(sets) * k
    fast, gen = _engine(sc, n, sweep=sets, **kw), _engine(sc, n, reserved=1, sweep=sets, **kw)
    fast.reset(); gen.reset()
    ta, tb = fast.train(iters, trace=True), gen.train(iters, trace=True)
    assert np.array_equal(ta.cpu().numpy(), tb.cpu().numpy())
    _same_state(fast, gen)


@pytest.mark.parametrize("name", ["qrm4_minb7", "qlambda_sparse", "lr_none"])
def test_groups_are_keyed_on_the_global_instance_id(name, cuda_device):
    """two engines on [0, N/2) and [N/2, N) (instance_offset, N/2 splitting a group) together equal one engine of N"""
    sc, sets, k, iters, kw = _case(name)
    H = len(sets)
    n = H * k
    half = n // 2 + 1  # not a group boundary
    whole = _engine(sc, n, sweep=sets, **kw)
    lo = _engine(sc, half, sweep=sets, sweep_group=k, **kw)
    hi = _engine(sc, n - half, sweep=sets, sweep_group=k, instance_offset=half, **kw)
    for e in (whole, lo, hi):
        e.reset()
        e.train(iters)
    sw, sl, sh = _state(whole), _state(lo), _state(hi)
    for key in sw:
        joined = np.concatenate([sl[key].reshape(half, -1), sh[key].reshape(n - half, -1)])
        assert joined.tobytes() == sw[key].reshape(n, -1).tobytes(), key
    gs = whole.group_stats()
    gl, gh = lo.group_stats(), hi.group_stats()
    for f in ("episodes", "successes", "active_steps"):
        assert np.array_equal(gs[f].cpu().numpy(), (gl[f] + gh[f]).cpu().numpy()), f


def test_train_host_chunks_split_a_group(cuda_device):
    """rlrm_train_host pipelines 2 chunks of 300,000 instances; the chunk boundary falls inside group 1 of 3"""
    import torch

    free, _total = torch.cuda.mem_get_info()
    if free < 20e9:
        pytest.skip("needs ~10 GB of free device memory")
    sc = P.scenario_config3(True)
    sets = _SETTINGS[:3]
    n = 600000
    resident, hosted = _engine(sc, n, sweep=sets), _engine(sc, n, sweep=sets)
    resident.reset(); hosted.reset()
    n_slots = n * hosted.A
    host_slot = torch.empty(n_slots, dtype=torch.int64).pin_memory()
    host_eps = torch.empty(n_slots, dtype=torch.float64).pin_memory()
    host_stats = torch.empty((n_slots, 32), dtype=torch.uint8).pin_memory()
    host_slot.copy_(hosted.slot); host_eps.copy_(hosted.epsilon)
    for chunk in (3, 60):
        resident.train(chunk)
        hosted.train_host(chunk, host_stats, host_slot, host_eps)
    _same_state(resident, hosted)
    assert torch.equal(host_slot, resident.slot.cpu()) and torch.equal(host_eps, resident.epsilon.cpu())
    assert torch.equal(host_stats, resident.stats.cpu())


@pytest.mark.parametrize("name", ["qrm4_minb7", "qlambda_dense", "per_agent_qrm", "lr_none"])
def test_iterate_unfused_equals_train_under_a_sweep(name, cuda_device):
    """select / step / update / reset launched one by one (the update and reset kernels take each instance's setting)"""
    sc, sets, k, _iters, kw = _case(name)
    n = len(sets) * k
    fused, unfused = _engine(sc, n, sweep=sets, **kw), _engine(sc, n, sweep=sets, **kw)
    fused.reset(); unfused.reset()
    fused.train(120)
    for _ in range(120):
        unfused.iterate_unfused()
    sf, su = _state(fused), _state(unfused)
    for key in sf:
        if key not in ("ep_return", "stats"):  # the running return and the statistics are kept by the fused kernels only
            assert sf[key].tobytes() == su[key].tobytes(), key


def test_update_list_takes_the_slot_setting(cuda_device):
    """rlrm_update_list on a sweep handle applies the update with the setting of the slot's group"""
    import torch

    from multiagent_rlrm_b200 import _abi as abi
    from multiagent_rlrm_b200._lib import check

    sc = P.scenario_config3(False)
    sets = _SETTINGS[:2]
    swp = _engine(sc, 4, sweep=sets)
    ex = abi.Experience(3, 7, 2, 0, (C.c_uint8 * 6)(), 1.0)
    ex_dev = torch.frombuffer(bytearray(bytes(ex)), dtype=torch.uint8).to("cuda:0")  # the kernel reads the list from device memory
    for slot in (0, 7):  # slot 0: instance 0, group 0; slot 7: instance 3, group 1
        g = (slot // swp.A) // 2
        uni = _engine(_setting_scenario(sc, sets[g]), 4)
        for e in (swp, uni):
            check(e.L.rlrm_update_list(e.h, C.byref(e.state), slot, 1, ex_dev.data_ptr(), e._stream()))
        torch.cuda.synchronize()
        assert torch.equal(swp.q[slot], uni.q[slot]), slot
        assert not torch.equal(swp.q[slot], torch.full_like(swp.q[slot], sc.q_init))


@pytest.mark.parametrize("name", ["qrm4_minb7", "qlambda_sparse"])
def test_checkpoint_resume_under_a_sweep(name, cuda_device, tmp_path):
    import torch

    sc, sets, k, _iters, kw = _case(name)
    n = len(sets) * k
    straight, first = _engine(sc, n, sweep=sets, **kw), _engine(sc, n, sweep=sets, **kw)
    straight.reset(); first.reset()
    straight.train(400)
    first.train(200)
    path = tmp_path / "engine.pt"
    torch.save(first.state_dict(), path)
    resumed = _engine(sc, n, sweep=sets, **kw)
    resumed.load_state_dict(torch.load(path))
    resumed.train(200)
    _same_state(straight, resumed)
    other = copy.deepcopy(sets)
    other[0]["learning_rate"] = 0.25
    with pytest.raises(ValueError):
        _engine(sc, n, sweep=other, **kw).load_state_dict(first.state_dict())
    with pytest.raises(ValueError):
        _engine(sc, n, **kw).load_state_dict(first.state_dict())


def _hyper(lr=0.1):
    from multiagent_rlrm_b200 import _abi as abi

    return (abi.Hyper * 2)(abi.Hyper(lr, 0.9, 0.0, 0.1, 1.0), abi.Hyper(0.5, 0.9, 0.0, 0.1, 1.0))


def test_abi_errors(cuda_device):
    from multiagent_rlrm_b200._lib import RlrmError

    ARG, UNSUPPORTED = -1, -3
    eng = _engine(P.scenario_config3(True), 64)
    L, h = eng.L, eng.h
    assert L.rlrm_set_sweep(h, _hyper(), 2, 0) == ARG  # group_size must be positive
    assert L.rlrm_set_sweep(h, _hyper(), 2, -4) == ARG
    # launch checks: instances not covered by n_sets * group_size
    assert L.rlrm_set_sweep(h, _hyper(), 2, 16) == 0
    assert L.rlrm_train(h, C.byref(eng.state), 0, 10, 1, None, eng._stream()) == ARG
    assert L.rlrm_reset(h, C.byref(eng.state), None, eng._stream()) == ARG
    # rlrm_set_learner does not half-apply on a sweep handle
    assert L.rlrm_set_learner(h, 0.3, 0.9, 0.0) == UNSUPPORTED
    # a learning_rate = None setting needs state.visits
    assert L.rlrm_set_sweep(h, _hyper(-1.0), 2, 32) == 0
    assert L.rlrm_train(h, C.byref(eng.state), 0, 10, 1, None, eng._stream()) == ARG
    # clearing the sweep gives the uniform handle back
    assert L.rlrm_set_sweep(h, None, 0, 0) == 0
    assert L.rlrm_set_learner(h, 0.3, 0.9, 0.0) == 0
    assert L.rlrm_train(h, C.byref(eng.state), 0, 10, 1, None, eng._stream()) == 0
    # the instances of a shared table share one learner
    shared = _engine(P.scenario_config5(True), 64)
    assert shared.L.rlrm_set_sweep(shared.h, _hyper(), 2, 32) == UNSUPPORTED
    with pytest.raises(ValueError):
        _engine(P.scenario_config5(True), 64, sweep=[{}, {}])
    with pytest.raises(RlrmError):
        _engine(P.scenario_config3(True), 64, sweep=[{}, {}]).set_learner(0.2, 0.9)
    with pytest.raises(ValueError):  # n_instances must be a multiple of len(sweep)
        _engine(P.scenario_config3(True), 65, sweep=[{}, {}])
    with pytest.raises(ValueError):  # settings do not cover the engine's instances
        _engine(P.scenario_config3(True), 64, sweep=[{}, {}], sweep_group=16)


def test_group_stats_equals_numpy_reduction(cuda_device):
    sc, sets, k, iters, kw = _case("qrm4_minb7")
    H = len(sets)
    eng = _engine(sc, H * k, sweep=sets)
    eng.reset()
    eng.train(iters)
    gs = eng.group_stats()
    s = eng.stats_numpy().reshape(H, k * eng.A)
    for f in ("episodes", "successes", "active_steps"):
        assert np.array_equal(gs[f].cpu().numpy(), s[f].astype(np.int64).sum(axis=1)), f
    assert np.allclose(gs["return_sum"].cpu().numpy(), s["return_sum"].sum(axis=1), rtol=1e-12, atol=0)
    assert int(gs["episodes"].sum()) > 0
    # one offset shard: groups it does not touch read zero
    hi = _engine(sc, 2 * k, sweep=sets, sweep_group=k, instance_offset=(H - 2) * k)
    hi.reset()
    hi.train(iters)
    gh = hi.group_stats()
    assert np.array_equal(gh["episodes"].cpu().numpy()[:H - 2], np.zeros(H - 2, dtype=np.int64))
    assert np.array_equal(gh["episodes"].cpu().numpy()[H - 2:], gs["episodes"].cpu().numpy()[H - 2:])
