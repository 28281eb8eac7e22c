"""train_qrm4_kernel (QRM with four reward-machine states on float32 tables: BASELINE configs 1, 3 and 5) in the
instantiations the other GPU tests do not reach: without a trace buffer (what Engine.train runs by default and what the
benchmark times), with the 64-register allocation taken when a batch needs more than 7 resident blocks per SM, and on an
OfficeWorld machine (wall and plant penalties in its step records). Every comparison is bit-exact."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _engine(compiled, n):
    from multiagent_rlrm_b200.engine import Engine

    return Engine(compiled, n, device="cuda:0")


def _office_exp0():
    import multiagent_rlrm_b200 as P

    # exp0 is the built-in OfficeWorld machine with 4 states and counterfactual states [0, 1, 2]; wall penalty -0.5 and
    # plants at -100 exercise all four env-reward classes
    return P.scenario_for_experiment("map1", "exp0", starts=[(2, 7), (6, 3), (0, 0)], algo="qrm", learning_rate=0.1, gamma=0.9,
                                     stochastic=True, epsilon_start=0.1, epsilon_end=0.1, epsilon_decay=1.0, q_init=2.0,
                                     wall_penalty=-0.5, max_steps=200, seed=97)


def _assert_qrm4(c):
    assert c.config.n_rm_states == 4 and c.config.n_qrm_states == 3


def _assert_same_engines(a, b, what):
    assert np.array_equal(a.q.cpu().numpy(), b.q.cpu().numpy()), what + " Q"
    assert np.array_equal(a.slot.cpu().numpy(), b.slot.cpu().numpy()), what + " slot words"
    assert np.array_equal(a.epsilon.cpu().numpy(), b.epsilon.cpu().numpy()), what + " epsilon"
    assert np.array_equal(a.ep_return.cpu().numpy(), b.ep_return.cpu().numpy()), what + " ep_return"
    assert np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy()), what + " stats"


def _assert_matches_oracle(eng, o, what):
    import oracle as O

    assert np.array_equal(eng.slot.cpu().numpy().view(np.uint64), o.slot), what + " slot words"
    assert np.array_equal(eng.epsilon.cpu().numpy(), o.epsilon), what + " epsilon"
    assert np.array_equal(eng.q.cpu().numpy(), o.q), what + " Q"
    assert np.array_equal(eng.ep_return.cpu().numpy(), o.ep_return), what + " ep_return"
    s = eng.stats_numpy()
    for f in O.STATS_DTYPE.names:
        assert np.array_equal(s[f], o.stats[f]), what + " stats." + f


@pytest.mark.parametrize("name", ["cfg3_qrm", "cfg5_qrm_4agents", "office_exp0_qrm"])
def test_untraced_equals_traced(name, cuda_device):
    """train(trace=False) runs the TRACE = 0 instantiation; it must leave exactly the state train(trace=True) leaves, in
    learning and in greedy (learn=False) launches of odd lengths."""
    import multiagent_rlrm_b200 as P

    sc, n = {"cfg3_qrm": (P.scenario_config3(True), 2048), "cfg5_qrm_4agents": (P.scenario_config5(False), 1024),
             "office_exp0_qrm": (_office_exp0(), 300)}[name]
    c_a, c_b = P.compile_scenario(sc), P.compile_scenario(sc)
    _assert_qrm4(c_a)
    a, b = _engine(c_a, n), _engine(c_b, n)
    a.reset(); b.reset()
    for chunk, learn in ((1, True), (7, True), (613, True), (37, False), (300, True)):
        a.train(chunk, learn=learn)
        b.train(chunk, learn=learn, trace=True)
        _assert_same_engines(a, b, f"{name} after a {chunk}-iteration launch (learn={learn}):")
    assert int(a.stats_numpy()["episodes"].sum()) > 0


def test_office_exp0_specialised_equals_generic_and_oracle(cuda_device):
    """OfficeWorld exp0 takes train_qrm4_kernel; config.reserved bit 0 forces the generic train_kernel. Both, and the oracle,
    agree bit for bit."""
    import multiagent_rlrm_b200 as P
    import oracle as O

    sc, n, t = _office_exp0(), 300, 1500
    c_fast, c_gen = P.compile_scenario(sc), P.compile_scenario(sc)
    _assert_qrm4(c_fast)
    c_gen.config.reserved = 1
    a, b = _engine(c_fast, n), _engine(c_gen, n)
    a.reset(); b.reset()
    ta, tb = a.train(t, trace=True), b.train(t, trace=True)
    assert np.array_equal(ta.cpu().numpy(), tb.cpu().numpy())
    _assert_same_engines(a, b, "exp0 specialised vs generic:")
    o = O.Oracle(c_fast, n, "f32")
    o.reset()
    o.train(0, t)
    _assert_matches_oracle(a, o, "exp0 vs oracle:")
    assert int(o.stats["episodes"].sum()) > 0


def test_dense_batch_matches_oracle(cuda_device):
    """Config 5 (4 agents) with more threads than 7 resident 128-thread blocks per SM hold: the launch takes the MINB = 8
    instantiation. Untraced launches of odd lengths must match the C oracle."""
    import torch

    import multiagent_rlrm_b200 as P
    import oracle as O

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    c = P.compile_scenario(P.scenario_config5(False))
    _assert_qrm4(c)
    n = sms * 7 * 128 // c.n_agents + 1000
    assert n * c.n_agents > sms * 7 * 128
    eng, o = _engine(c, n), O.Oracle(c, n, "f32")
    eng.reset(); o.reset()
    t0 = 0
    for chunk in (1, 7, 151, 141):
        eng.train(chunk)
        o.train(t0, chunk)
        t0 += chunk
    _assert_matches_oracle(eng, o, "config 5 dense batch:")
    assert int(o.stats["episodes"].sum()) > 0
