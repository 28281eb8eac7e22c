"""train_qrm4_kernel against the C oracle for every lane-group size it runs with: 1 to 8 agents per instance (groups of 1, 2,
4 and 8 lanes, with idle lanes when the agent count is not a power of two), on the slippery map (slip index from padded
thresholds) and the deterministic one. The episode-end test is a fixed xor butterfly whose steps past the group size are
masked off, so a wrong mask ends or continues episodes of one instance on its neighbours' flags. Every comparison is bit-exact."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# free cells of FrozenLake map1, the first four those of BASELINE config 5
_STARTS = [(5, 0), (0, 0), (9, 0), (7, 3), (1, 1), (2, 5), (8, 6), (3, 4)]


@pytest.mark.parametrize("stochastic", [True, False], ids=["slippery", "deterministic"])
@pytest.mark.parametrize("agents", [1, 2, 3, 4, 5, 8])
def test_group_size_matches_oracle(agents, stochastic, cuda_device):
    import multiagent_rlrm_b200 as P
    import oracle as O
    from multiagent_rlrm_b200.engine import Engine

    sc = P.scenario_config3(True)
    sc.starts = _STARTS[:agents]
    sc.stochastic = stochastic
    sc.max_steps = 80  # episodes also end by truncation, which needs every agent of the instance
    sc.epsilon_start = sc.epsilon_end = 0.2
    c = P.compile_scenario(sc)
    assert c.config.n_rm_states == 4 and c.config.n_qrm_states == 3
    n = 301  # the last block is partly empty
    eng, o = Engine(c, n, device="cuda:0"), O.Oracle(c, n, "f32")
    eng.reset(); o.reset()
    t0 = 0
    for chunk in (1, 7, 400):
        eng.train(chunk)
        o.train(t0, chunk)
        t0 += chunk
    assert np.array_equal(eng.slot.cpu().numpy().view(np.uint64), o.slot), "slot words"
    assert np.array_equal(eng.epsilon.cpu().numpy(), o.epsilon), "epsilon"
    assert np.array_equal(eng.q.cpu().numpy(), o.q), "Q"
    assert np.array_equal(eng.ep_return.cpu().numpy(), o.ep_return), "ep_return"
    s = eng.stats_numpy()
    for f in O.STATS_DTYPE.names:
        assert np.array_equal(s[f], o.stats[f]), "stats." + f
    assert int(o.stats["episodes"].sum()) > n
