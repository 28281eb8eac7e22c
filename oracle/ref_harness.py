"""TEST INFRASTRUCTURE — not part of the product path.

Drives the LIVE reference (/root/reference, imported under oracle/ref_shim) through a verbatim restatement of its
two driver loops and records everything the hot path produces, with the randomness INJECTED from Philox words
(oracle/philox.py) through stand-in ``rng`` objects. Used to (1) generate the golden fixtures under tests/golden/
(oracle/gen_golden.py) and (2) validate the C oracle (oracle/rlrm_oracle.c) in this container.
It is never imported by the package, and cannot run on the GPU box (no /root/reference there).

Loop restated:
  FrozenLake  /root/reference/multiagent_rlrm/environments/frozen_lake/frozen_lake_main.py:312, 336-376
  OfficeWorld /root/reference/multiagent_rlrm/environments/office_world/office_main.py:1696-1749
"""
from __future__ import annotations

import copy
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# the original project's source tree (its multiagent_rlrm package, and tests/ for the tests that read the reference's own
# test files): RLRM_REFERENCE_ROOT, else the copy __graft_entry__.build() stages into the git-ignored oracle/_ref/
REFERENCE_ROOT = os.environ.get("RLRM_REFERENCE_ROOT") or os.path.join(_HERE, "_ref")
REFERENCE_MISSING = "needs the original multiagent-rl-rm sources (set RLRM_REFERENCE_ROOT to its checkout)"


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "multiagent_rlrm"))


def _import_reference():
    shim = os.path.join(_HERE, "ref_shim")
    for p in (REFERENCE_ROOT, shim):
        if p not in sys.path:
            sys.path.insert(0, p)
    sys.path.insert(0, _HERE)


ACTIONS = ("up", "down", "left", "right")


class DrawSource:
    """Philox words per (t, instance, agent); t is set by the loop before each lockstep iteration."""

    def __init__(self, seed, n_instances, n_agents, instance_offset=0):
        self.seed, self.n, self.a, self.off = seed, n_instances, n_agents, instance_offset
        self.t = 0
        self._cache = {}

    def start_words(self, i, block):
        """Words that key the random start positions of instance i for the episode whose first step is iteration t."""
        import philox

        T = self.t
        w = philox.philox4x32_10(T & 0xFFFFFFFF, (~(T >> 32)) & 0xFFFFFFFF, (self.off + i) & 0xFFFFFFFF, 0x80000000 | block,
                                 self.seed & 0xFFFFFFFF, (self.seed >> 32) & 0xFFFFFFFF)
        return [int(x) for x in w]

    def words(self, i, a):
        w = self._cache.get(self.t)
        if w is None:
            if len(self._cache) > 4096:
                self._cache.clear()
            import philox

            w = self._cache[self.t] = philox.draws(self.seed, self.t, self.n, self.a, self.off)
        return w[i, a]


class LearnerRNG:
    """Stands in for learner.rng (numpy Generator) inside QLearning.choose_action (qlearning.py:118-143)."""

    def __init__(self, src, i, a):
        self.src, self.i, self.a = src, i, a

    def uniform(self, lo=0.0, hi=1.0):
        return lo + (hi - lo) * (int(self.src.words(self.i, self.a)[0]) / 4294967296.0)

    def words(self):
        """Hook used by this repo's learners (learners.py): the four words of the current (t, instance, agent)."""
        return self.src.words(self.i, self.a)

    def choice(self, seq, p=None):
        w = self.src.words(self.i, self.a)
        if isinstance(seq, range):  # rng.choice(range(A)): uniform random action
            return seq[(int(w[1]) * len(seq)) >> 32]
        seq = list(seq)  # rng.choice(maxs): uniform tie-break
        return seq[(int(w[2]) * len(seq)) >> 32]


class EnvRNG:
    """Stands in for env.rng inside get_stochastic_action (ma_frozen_lake.py:257-262 ; ma_office.py:376-379):
    numpy's Generator.choice(a, p=p) is one uniform + searchsorted(cdf, u, side='right')."""

    def __init__(self, src, i):
        self.src, self.i = src, i
        self.agent_index = 0

    def words(self, agent_index):
        """Hook used by this repo's environments (envs.py)."""
        return self.src.words(self.i, agent_index)

    def shuffle(self, cells):
        """Stands in for rng.shuffle(free_cells) in _sample_start_positions (ma_frozen_lake.py:171): an in-place Fisher-Yates
        shuffle whose k-th swap partner is j = k + ((w_k * (F - k)) >> 32); only the first A entries are ever read."""
        F, w = len(cells), None
        for k in range(min(F - 1, 8)):
            if k % 4 == 0:
                w = self.src.start_words(self.i, k // 4)
            j = k + ((w[k % 4] * (F - k)) >> 32)
            cells[k], cells[j] = cells[j], cells[k]

    def choice(self, actions, p=None):
        u = int(self.src.words(self.i, self.agent_index)[3]) / 4294967296.0
        cdf = np.cumsum(np.array(p, dtype=np.float64))
        cdf /= cdf[-1]
        return actions[int(np.searchsorted(cdf, u, side="right"))]


def build_reference(sc: dict, table_dtype=np.float32):
    """Reference objects for one environment instance of scenario dict `sc` (tables.Scenario.to_dict())."""
    _import_reference()
    from multiagent_rlrm.learning_algorithms.qlearning import QLearning
    from multiagent_rlrm.learning_algorithms.qlearning_lambda import QLearningLambda
    from multiagent_rlrm.multi_agent.agent_rl import AgentRL
    from multiagent_rlrm.multi_agent.reward_machine import RewardMachine
    from multiagent_rlrm.multi_agent.wrappers.rm_environment_wrapper import RMEnvironmentWrapper
    from multiagent_rlrm.utils.utils import parse_map_emoji, parse_office_world

    if sc["env"] == "frozen_lake":
        from multiagent_rlrm.environments.frozen_lake.action_encoder_frozen_lake import ActionEncoderFrozenLake as AEnc
        from multiagent_rlrm.environments.frozen_lake.config_frozen_lake import config as fl_config
        from multiagent_rlrm.environments.frozen_lake.detect_event import PositionEventDetector
        from multiagent_rlrm.environments.frozen_lake.ma_frozen_lake import MultiAgentFrozenLake
        from multiagent_rlrm.environments.frozen_lake.state_encoder_frozen_lake import StateEncoderFrozenLake as SEnc

        holes, goals, (w, h) = parse_map_emoji(fl_config["maps"][sc["map_name"]]["layout"])
        env = MultiAgentFrozenLake(width=w, height=h, holes=holes)
        env.frozen_lake_stochastic = bool(sc["stochastic"])
        env.penalty_amount = sc["penalty_amount"]
        env.delay_action = bool(sc["delay_action"])
        env.random_start_positions = bool(sc.get("random_start_positions", False))
    else:
        from multiagent_rlrm.environments.office_world.action_encoder_office_world import ActionEncoderOfficeWorld as AEnc
        from multiagent_rlrm.environments.office_world.config_office import config as ow_config
        from multiagent_rlrm.environments.office_world.detect_event import PositionEventDetector
        from multiagent_rlrm.environments.office_world.ma_office import MultiAgentOfficeWorld
        from multiagent_rlrm.environments.office_world.state_encoder_office import StateEncoderOfficeWorld as SEnc

        m = ow_config["maps"][sc["map_name"]]
        coords, goals, walls = parse_office_world(m["layout"])
        walls = walls + [(b, a) for (a, b) in walls]  # office_main.py:416
        env = MultiAgentOfficeWorld(
            width=m["grid_size"][1], height=m["grid_size"][0], plants=coords["plant"], coffee=coords["coffee"],
            letters=coords["letter"], walls=walls, plants_penalty_value=sc["plants_penalty"],
            wall_penalty_value=sc["wall_penalty"], terminate_on_plants=bool(sc["terminate_on_plants"]),
            terminate_hit_walls=bool(sc["terminate_hit_walls"]))
        env.all_slip = bool(sc["all_slip"])
        env.stochastic = bool(sc["stochastic"])
        env.high_prob = sc["high_prob"]
        env.delay_action = bool(sc["delay_action"])
    env.max_steps_unused = sc["max_steps"]
    assert sc["max_steps"] == 1000, "the reference hard-codes the 1000-step cap"

    def machine(k):
        trs = sc["rm_transitions"] if not sc.get("rm_transitions_per_agent") else sc["rm_transitions_per_agent"][k]
        tmap = {}
        for (s, e, t, r) in trs:
            tmap[(s, None if e is None else tuple(e))] = (t, r)
        if sc.get("detector_positions") is not None:
            pos = {tuple(p) for p in sc["detector_positions"]}
        else:
            pos = {ev for (_s, ev) in tmap if ev is not None}
        return tmap, pos

    agents = []
    for k, (x, y) in enumerate(sc["starts"]):
        transitions, positions = machine(k)
        ag = AgentRL(f"a{k + 1}", env)
        ag.set_initial_position(x, y)
        ag.add_state_encoder(SEnc(ag))
        ag.add_action_encoder(AEnc(ag))
        rm = RewardMachine(dict(transitions), PositionEventDetector(set(positions)))
        ag.set_reward_machine(rm)
        env.add_agent(ag)
        n_states = env.grid_width * env.grid_height * rm.numbers_state()
        common = dict(state_space_size=n_states, action_space_size=4, learning_rate=sc["learning_rate"],
                      gamma=sc["gamma"], action_selection="greedy", epsilon_start=sc["epsilon_start"],
                      epsilon_end=sc["epsilon_end"], epsilon_decay=sc["epsilon_decay"])
        if sc["algo"] == "qlambda":
            learner = QLearningLambda(lambd=sc["lambd"], **common)
            learner.e_table = learner.e_table.astype(table_dtype)
        else:
            if sc["learning_rate"] is None:
                # QLearning.__init__ formats learning_rate with :0.2f (qlearning.py:37) and cannot take None
                common["learning_rate"] = 0.0
            learner = QLearning(qtable_init=sc["q_init"], use_qrm=(sc["algo"] == "qrm"), **common)
            learner.learning_rate = sc["learning_rate"]
        learner.q_table = np.full(learner.q_table.shape, sc["q_init"], dtype=table_dtype)
        if sc.get("use_rsh") and sc["algo"] != "qlambda":  # QL_RS / QRM_RS (office_main.py:543-573)
            import contextlib
            import io

            learner.use_rsh = True
            with contextlib.redirect_stdout(io.StringIO()):  # value_iteration prints debug lines
                if sc.get("rs_kind", "vi") == "distance":
                    rm.add_distance_reward_shaping(sc["gamma"], sc["rs_gamma"], sc["rs_alpha"])
                else:
                    rm.add_reward_shaping(sc["gamma"], sc["rs_gamma"])
        ag.set_learning_algorithm(learner)
        agents.append(ag)
    rm_env = RMEnvironmentWrapper(env, agents)
    rm_env.reward_modifier = sc["reward_modifier"]
    return rm_env, env, agents


FIELDS_U8 = ("action", "q", "prev_q", "env_term", "rm_term", "term", "trunc", "active", "fail")
FIELDS_I32 = ("cell", "prev_cell", "event_cell", "agent_steps", "timestep")
FIELDS_F64 = ("renv", "rq", "reward", "epsilon", "q_sa")


def _np(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


def run_reference(sc: dict, n_instances: int, n_iters: int, table_dtype=np.float32, pre_resets: int = 1,
                  instance_offset: int = 0, learn: bool = True, snapshot_iters=(), builder=None):
    """Run `n_iters` lockstep iterations (episodes restart back-to-back) for each of `n_instances` independent
    reference environments. Returns dict of arrays shaped [T, N, A] plus final tables [N, A, S, 4]."""
    n_agents = len(sc["starts"])
    src = DrawSource(sc["seed"], n_instances, n_agents, instance_offset)
    out = {k: np.zeros((n_iters, n_instances, n_agents), dtype=np.uint8) for k in FIELDS_U8}
    out.update({k: np.full((n_iters, n_instances, n_agents), -1, dtype=np.int32) for k in FIELDS_I32})
    out.update({k: np.zeros((n_iters, n_instances, n_agents), dtype=np.float64) for k in FIELDS_F64})
    out["episode_end"] = np.zeros((n_iters, n_instances), dtype=np.uint8)
    q_final, e_final, snaps = [], [], {int(t): [] for t in snapshot_iters}
    fl_driver = sc["driver"] == "frozen_lake_main"

    for i in range(n_instances):
        rm_env, env, agents = (builder or build_reference)(sc, table_dtype)
        W = env.grid_width
        for k, ag in enumerate(agents):
            ag.get_learning_algorithm().rng = LearnerRNG(src, i, k)
        index_of = {ag.name: k for k, ag in enumerate(agents)}
        orig_gsa = env.get_stochastic_action

        def gsa(agent, intended, _orig=orig_gsa, _env=env, _idx=index_of):
            _env.rng.agent_index = _idx[agent.name]
            return _orig(agent, intended)

        env.get_stochastic_action = gsa
        def do_reset():
            # env.reset() builds its own np.random.default_rng(seed) and (random_start_positions) shuffles with it before
            # returning (ma_frozen_lake.py:59-64): hand it the stand-in for the duration of the call
            real = np.random.default_rng
            np.random.default_rng = lambda *a, **k: EnvRNG(src, i)
            try:
                return rm_env.reset(sc["seed"])
            finally:
                np.random.default_rng = real

        src.t = 0
        for _ in range(pre_resets):
            do_reset()
        t = 0
        while t < n_iters:
            src.t = t  # the new episode's first step is iteration t
            states, infos = do_reset()
            env.rng = EnvRNG(src, i)  # reset() re-created env.rng (ma_frozen_lake.py:59 ; ma_office.py:96)
            if not fl_driver:
                states = copy.deepcopy(states)  # office_main.py:1700
            while t < n_iters:
                src.t = t
                actions = {}
                for ag in rm_env.agents:
                    actions[ag.name] = ag.select_action(rm_env.env.get_state(ag))
                new_states, rewards, terminated, truncated, infos = rm_env.step(actions)
                for k, ag in enumerate(rm_env.agents):
                    name = ag.name
                    term_arg = (terminated[name] or truncated[name]) if fl_driver else terminated[name]
                    info = infos[name]
                    rm = ag.get_reward_machine()
                    if learn:
                        ag.update_policy(state=states[name], action=actions[name], reward=rewards[name],
                                         next_state=new_states[name], terminated=term_arg, infos=info)
                    a_idx = ag.actions_idx(actions[name])
                    prev_s = info.get("prev_s", new_states[name])
                    o = (t, i, k)
                    out["action"][o] = a_idx
                    out["cell"][o] = new_states[name]["pos_y"] * W + new_states[name]["pos_x"]
                    out["prev_cell"][o] = prev_s["pos_y"] * W + prev_s["pos_x"]
                    out["q"][o] = rm.get_state_index(info["q"])
                    out["prev_q"][o] = rm.get_state_index(info["prev_q"])
                    ev = rm.event_detector.detect_event(new_states[name])
                    out["event_cell"][o] = -1 if ev is None else ev[1] * W + ev[0]
                    out["renv"][o] = info.get("Renv", 0)
                    out["rq"][o] = info["RQ"]
                    out["reward"][o] = rewards[name]
                    out["env_term"][o] = info["env_terminated"]
                    out["rm_term"][o] = info["rm_terminated"]
                    out["term"][o] = terminated[name]
                    out["trunc"][o] = truncated[name]
                    out["active"][o] = env.active_agents[name]
                    out["fail"][o] = env.agent_fail[name]
                    out["agent_steps"][o] = env.agent_steps[name]
                    out["timestep"][o] = env.timestep
                    out["epsilon"][o] = getattr(ag.get_learning_algorithm(), "epsilon", 0.0)
                    enc = out["prev_cell"][o] * rm.numbers_state() + out["prev_q"][o]
                    out["q_sa"][o] = float(ag.get_learning_algorithm().q_table[int(enc), int(a_idx)])
                states = copy.deepcopy(new_states)
                t += 1
                if t in snaps:
                    snaps[t].append(np.stack([_np(ag.get_learning_algorithm().q_table).copy() for ag in agents]))
                if fl_driver:
                    over = all(terminated.values()) or all(truncated.values())
                else:
                    over = all(terminated.values()) or all(truncated.values())
                if over:
                    out["episode_end"][t - 1, i] = 1
                    break
        join = np.concatenate if sc.get("rm_transitions_per_agent") else np.stack  # per-agent machines: tables of S_a rows
        q_final.append(join([_np(ag.get_learning_algorithm().q_table) for ag in agents]))
        if sc["algo"] == "qlambda":
            e_final.append(join([_np(ag.get_learning_algorithm().e_table) for ag in agents]))
    out["q_final"] = np.stack(q_final)
    if e_final:
        out["e_final"] = np.stack(e_final)
    for t, lst in snaps.items():
        out[f"q_at_{t}"] = np.stack(lst)
    return out
