"""CPU: the Python side of hyper-parameter sweeps — completing and validating the settings list (engine.sweep_settings)."""
import pytest

import multiagent_rlrm_b200 as P
from multiagent_rlrm_b200.engine import SWEEP_KEYS, sweep_settings


def test_missing_keys_come_from_the_scenario():
    sc = P.scenario_config3(True)
    out = sweep_settings(sc, [{"learning_rate": 0.5}, {"gamma": 0.8, "epsilon_start": 1}, {"learning_rate": None}])
    assert [set(s) for s in out] == [set(SWEEP_KEYS)] * 3
    assert out[0]["learning_rate"] == 0.5 and out[0]["gamma"] == sc.gamma and out[0]["epsilon_decay"] == sc.epsilon_decay
    assert out[1]["learning_rate"] == sc.learning_rate and out[1]["gamma"] == 0.8
    assert out[1]["epsilon_start"] == 1.0 and isinstance(out[1]["epsilon_start"], float)
    assert out[2]["learning_rate"] is None


@pytest.mark.parametrize("bad", [[], {}, {"learning_rate": 0.1}, [{"lr": 0.1}], [3], [{"gamma": None}], [{"gamma": "0.9"}],
                                 [{"learning_rate": -0.5}], [{"epsilon_end": True}]])
def test_malformed_sweeps_are_rejected(bad):
    with pytest.raises(ValueError):
        sweep_settings(P.scenario_config3(True), bad)


def test_shared_learner_and_shaping_gamma_are_rejected():
    with pytest.raises(ValueError):
        sweep_settings(P.scenario_config5(True), [{}])
    sc = P.scenario_config3(True)
    sc.use_rsh = True
    assert len(sweep_settings(sc, [{"learning_rate": 0.2}, {"gamma": sc.gamma}])) == 2
    with pytest.raises(ValueError):  # the shaping potentials were built with the scenario's gamma
        sweep_settings(sc, [{"gamma": 0.5}])


def test_sharded_trainer_passes_the_sweep_through():
    from multiagent_rlrm_b200.dist import ShardedTrainer

    seen = {}

    def factory(compiled, n_local, device, **kw):
        seen.update(kw, n_local=n_local)
        return object()

    ShardedTrainer(P.scenario_config3(True), 64, engine_factory=factory, sweep=[{}, {"learning_rate": 0.5}])
    assert seen == {"sweep": [{}, {"learning_rate": 0.5}], "sweep_group": 32, "n_local": 64}
    with pytest.raises(ValueError):
        ShardedTrainer(P.scenario_config3(True), 63, engine_factory=factory, sweep=[{}, {}])
