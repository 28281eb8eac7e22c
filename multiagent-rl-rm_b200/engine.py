"""Batched engine: torch-owned device state + thin calls into the C ABI (include/rlrm_b200.h).

This is the batched counterpart of the object graph the reference drivers build
(frozen_lake_main.py:200-295 / office_main.py:400-717): N independent environment instances x A agents, each
agent with its own Reward-Machine state, learner table and epsilon. torch is used for memory, streams and
(in dist.py) torch.distributed only; every computation below is a kernel of csrc/rlrm_b200.cu.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _abi as abi
from ._lib import check, load
from .tables import Compiled

_TORCH_DT = {"uint16": torch.int16, "uint8": torch.uint8, "float64": torch.float64}

EVAL_DTYPE = np.dtype([("cum_gamma", "<f8"), ("disc_return", "<f8"), ("return_sum", "<f8"), ("return_sqsum", "<f8"),
                       ("arps_sum", "<f8"), ("len_sum", "<u8"), ("len_sqsum", "<u8"), ("episodes", "<u4"), ("successes", "<u4"),
                       ("in_success", "<u4"), ("reserved", "<u4")])

STATS_DTYPE = np.dtype([("active_steps", "<u8"), ("episodes", "<u4"), ("successes", "<u4"), ("return_sum", "<f8"),
                        ("last_return", "<f4"), ("last_length", "<u4")])


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


SWEEP_KEYS = ("learning_rate", "gamma", "lambd", "epsilon_start", "epsilon_end", "epsilon_decay")


def sweep_settings(scenario, sweep) -> List[dict]:
    """The settings of a hyper-parameter sweep with every key of SWEEP_KEYS present: keys a setting leaves out come from
    `scenario`. learning_rate None is 1 / visits, as in the scenario. Raises ValueError on anything malformed."""
    if isinstance(sweep, dict) or not hasattr(sweep, "__len__") or len(sweep) == 0:
        raise ValueError("sweep must be a non-empty list of dicts")
    if scenario.shared_q:
        raise ValueError("a sweep needs per-instance tables: the instances of a shared table share one learner")
    out = []
    for j, setting in enumerate(sweep):
        if not isinstance(setting, dict):
            raise ValueError(f"sweep[{j}] is not a dict")
        unknown = set(setting) - set(SWEEP_KEYS)
        if unknown:
            raise ValueError(f"sweep[{j}] has unknown keys {sorted(unknown)}; allowed: {SWEEP_KEYS}")
        s = {k: setting.get(k, getattr(scenario, k)) for k in SWEEP_KEYS}
        for k in SWEEP_KEYS:
            if s[k] is None and k == "learning_rate":
                continue
            if isinstance(s[k], bool) or not isinstance(s[k], (int, float)):
                raise ValueError(f"sweep[{j}][{k!r}] must be a number")
            s[k] = float(s[k])
        if s["learning_rate"] is not None and s["learning_rate"] < 0:
            raise ValueError(f"sweep[{j}]: learning_rate must be >= 0 or None")
        if scenario.use_rsh and s["gamma"] != float(scenario.gamma):
            # the shaping potentials are built from the scenario's gamma (RewardMachine.add_reward_shaping)
            raise ValueError(f"sweep[{j}]: reward shaping takes the scenario's gamma; a setting cannot change it")
        out.append(s)
    return out


class Engine:
    def __init__(self, compiled: Compiled, n_instances: int, device="cuda:0", track_visits: bool = False,
                 with_stats: bool = True, qlambda_sparse: bool = False, host_control: bool = False, sweep=None,
                 sweep_group: Optional[int] = None):
        """host_control: keep the small per-slot control state (slot words, epsilon, running return) in page-locked HOST
        memory instead of device memory. Page-locked memory is device-accessible under unified addressing, so the kernels
        read / write it in place and a host driver (the one-instance reference-shaped classes in envs.py) touches it through
        numpy views without any copy. Meant for small N; large batches keep it in HBM.
        qlambda_sparse: Q(lambda) only — keep the traces as per-agent lists of live entries (sparse-exact, see
        include/rlrm_b200.h) instead of the dense e table. Same results bit for bit, far less memory traffic; the fused
        `train` path only (the call-by-call `update` needs the dense table). Call `sync_tables()` before reading `q`.
        sweep: a hyper-parameter sweep, a list of dicts with keys among SWEEP_KEYS (missing keys come from the scenario).
        Setting g applies to the sweep_group instances with global ids [g * sweep_group, (g + 1) * sweep_group), global id =
        compiled instance_offset + local index; sweep_group defaults to n_instances // len(sweep), which must then divide
        evenly. Every instance behaves bit for bit as in an engine built with its setting (rlrm_set_sweep)."""
        self.L = load()
        if not torch.cuda.is_available():
            raise RuntimeError("multiagent-rl-rm_b200 needs a CUDA device (no CPU fallback)")
        self.c = compiled
        self.cfg = compiled.config
        self.device = torch.device(device)
        self.N, self.A, self.S = int(n_instances), compiled.n_agents, compiled.state_space
        self.sweep = self.sweep_group = None
        if sweep is not None:
            self.sweep = sweep_settings(compiled.scenario, sweep)
            if sweep_group is None:
                if self.N % len(self.sweep):
                    raise ValueError("n_instances must be a multiple of len(sweep) (or pass sweep_group)")
                sweep_group = self.N // len(self.sweep)
            self.sweep_group = int(sweep_group)
            if self.sweep_group <= 0:
                raise ValueError("sweep_group must be positive")
            if int(self.cfg.instance_offset) + self.N > len(self.sweep) * self.sweep_group:
                raise ValueError("the sweep's settings do not cover every instance of this engine")
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self._dev_index = dev_index
        self._tables = compiled.tables_struct()
        h = C.c_void_p()
        check(self.L.rlrm_create(C.byref(self.cfg), C.byref(self._tables), dev_index, C.byref(h)))
        self.h = h
        if self.sweep is not None:
            sets = (abi.Hyper * len(self.sweep))(*[abi.Hyper(-1.0 if s["learning_rate"] is None else s["learning_rate"], s["gamma"],
                                                             s["lambd"], s["epsilon_end"], s["epsilon_decay"]) for s in self.sweep])
            check(self.L.rlrm_set_sweep(self.h, sets, len(self.sweep), self.sweep_group))
        n_slots = self.N * self.A
        n_tab = self.A if self.cfg.shared_q else n_slots
        tab_shape = (n_tab, self.S, 4)
        if self.cfg.per_agent_rm:  # the tables of one instance are concatenated in agent order, S_a = W*H*nQ_a rows each
            self.agent_rows = list(compiled.agent_rows)
            tab_shape = (1 if self.cfg.shared_q else self.N, sum(self.agent_rows), 4)
        d = self.device
        self.table_dtype = torch.float64 if self.cfg.table_dtype == abi.TABLE_F64 else torch.float32
        self.host_control = bool(host_control)
        cd = "cpu" if self.host_control else d  # where the control state lives
        pin = (lambda t: t.pin_memory()) if self.host_control else (lambda t: t)
        self.slot = pin(torch.zeros(n_slots, dtype=torch.int64, device=cd))
        self.epsilon = pin(torch.full((n_slots,), float(self.cfg.epsilon_start), dtype=torch.float64, device=cd))
        self.q = torch.full(tab_shape, float(compiled.scenario.q_init), dtype=self.table_dtype, device=d)
        self.sparse = bool(qlambda_sparse) and self.cfg.algo == abi.ALGO_QLAMBDA
        self.e = torch.zeros(tab_shape, dtype=self.table_dtype, device=d) if (self.cfg.algo == abi.ALGO_QLAMBDA and not self.sparse) else None
        self.tr_cap = 0
        self.tr_pos = self.tr_idx = self.tr_eq = self.tr_len = self.tr_work = None
        if self.sparse:
            if self.S * 4 > 65535:
                raise ValueError("sparse Q(lambda) traces need S*4 <= 65535")
            self.tr_cap = ((int(self.cfg.max_steps) + 1 + 31) // 32) * 32
            self.tr_pos = torch.zeros((n_slots, self.S * 4), dtype=torch.int16, device=d)
            self.tr_idx = torch.zeros((n_slots, self.tr_cap), dtype=torch.int16, device=d)
            self.tr_eq = torch.zeros((n_slots, self.tr_cap, 2), dtype=self.table_dtype, device=d)  # (trace, q value) pairs
            self.tr_len = torch.zeros(n_slots, dtype=torch.int32, device=d)
            self.tr_work = torch.zeros(n_slots, dtype=torch.int64, device=d)
        if self.sweep is not None:  # epsilon starts per setting; the kernels carry it per slot from here on
            g = (int(self.cfg.instance_offset) + torch.arange(self.N)) // self.sweep_group
            eps0 = torch.tensor([s["epsilon_start"] for s in self.sweep], dtype=torch.float64)[g].repeat_interleave(self.A)
            self.epsilon.copy_(eps0)
        lr_none = any(s["learning_rate"] is None for s in self.sweep) if self.sweep is not None else self.cfg.learning_rate < 0
        need_visits = track_visits or lr_none
        self.visits = torch.zeros(tab_shape, dtype=torch.int32, device=d) if need_visits else None
        self.ep_return = pin(torch.zeros(n_slots, dtype=torch.float64, device=cd))
        self.stats = torch.zeros((n_slots, 32), dtype=torch.uint8, device=d) if with_stats else None
        shared = bool(self.cfg.shared_q)
        self.acc_sum = torch.zeros(tab_shape, dtype=torch.int64, device=d) if shared else None
        self.acc_cnt = torch.zeros(tab_shape, dtype=torch.int32, device=d) if shared else None
        self.acc_last = torch.zeros(tab_shape, dtype=torch.float32, device=d) if shared else None
        self.state = abi.State(self.N, _ptr(self.slot), _ptr(self.epsilon), _ptr(self.q), _ptr(self.e), _ptr(self.visits),
                               _ptr(self.ep_return), _ptr(self.stats), _ptr(self.acc_sum), _ptr(self.acc_cnt), _ptr(self.acc_last),
                               _ptr(self.tr_pos), _ptr(self.tr_idx), _ptr(self.tr_eq), _ptr(self.tr_len),
                               _ptr(self.tr_work), self.tr_cap, 0)
        self.t = 0  # lockstep iteration counter (Philox counter word)
        self._it_record = self._it_reward = None
        self._hio = None
        self._ctl_dirty = True

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.L.rlrm_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -- helpers -------------------------------------------------------------------------------
    def _stream(self):
        """torch's current stream on this device as a raw cudaStream_t (one C call; the Stream object is not built). Every launch
        of this engine except step_host asks for it, which is how step_host (own stream) learns that it has to wait for them."""
        self._ctl_dirty = True
        return torch._C._cuda_getCurrentRawStream(self._dev_index)

    def set_learner(self, learning_rate, gamma, lambd=0.0):
        check(self.L.rlrm_set_learner(self.h, -1.0 if learning_rate is None else float(learning_rate), float(gamma), float(lambd)))

    def sync(self):
        """Wait for the work queued on the current stream (rlrm_stream_sync)."""
        check(self.L.rlrm_stream_sync(self.h, self._stream()))

    @property
    def launches(self) -> int:
        return int(self.L.rlrm_launch_count(self.h))

    # -- C ABI calls -----------------------------------------------------------------------------
    def reset(self, mask: Optional[torch.Tensor] = None):
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        check(self.L.rlrm_reset_at(self.h, C.byref(self.state), _ptr(mask), self.t, self._stream()))

    def select_action(self, t: Optional[int] = None, draws: Optional[torch.Tensor] = None, best: bool = False) -> torch.Tensor:
        out = torch.empty(self.N * self.A, dtype=torch.uint8, device=self.device)
        if draws is not None:
            draws = draws.to(device=self.device).contiguous()
        check(self.L.rlrm_select_action(self.h, C.byref(self.state), _ptr(draws), self.t if t is None else t, int(best),
                                        _ptr(out), self._stream()))
        return out.view(self.N, self.A)

    def new_record(self) -> Dict[str, torch.Tensor]:
        """Step-record arrays (rlrm_step_out_t) carved out of ONE allocation; rlrm_step writes every element of every field."""
        n = self.N * self.A
        fields = sorted(abi.STEP_OUT_FIELDS.items(), key=lambda kv: -_TORCH_DT[kv[1]].itemsize)  # widest first keeps alignment
        pad = (-n) % 8
        buf = torch.empty(sum((n + pad) * _TORCH_DT[v].itemsize for _k, v in fields), dtype=torch.uint8, device=self.device)
        rec, off = {}, 0
        for k, v in fields:
            size = n * _TORCH_DT[v].itemsize
            rec[k] = buf[off:off + size].view(_TORCH_DT[v])
            off += (n + pad) * _TORCH_DT[v].itemsize
        self._record_buffer = buf  # lets a caller that wants every field on the host fetch them with one copy
        return {k: rec[k] for k in abi.STEP_OUT_FIELDS}

    def step(self, actions: torch.Tensor, t: Optional[int] = None, draws: Optional[torch.Tensor] = None, with_rm: bool = True,
             rec: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        if draws is not None:
            draws = draws.to(device=self.device).contiguous()
        rec = rec or self.new_record()
        so = abi.StepOut(*[_ptr(rec[k]) for k in abi.STEP_OUT_FIELDS])
        check(self.L.rlrm_step(self.h, C.byref(self.state), _ptr(actions), _ptr(draws), self.t if t is None else t,
                               int(with_rm), C.byref(so), self._stream()))
        return rec

    def rm_step(self, q: torch.Tensor, cell: torch.Tensor, agent: int = 0):
        """RewardMachine.step on explicit (state index, cell) pairs, on agent `agent`'s machine."""
        q = q.to(device=self.device, dtype=torch.uint8).contiguous().clone()
        cell = cell.to(device=self.device, dtype=torch.int16).contiguous()
        ev = torch.empty_like(q)
        r = torch.empty(q.numel(), dtype=torch.float64, device=self.device)
        check(self.L.rlrm_rm_step_agent(self.h, int(agent), q.numel(), _ptr(q), _ptr(cell), _ptr(ev), _ptr(r), self._stream()))
        return q, ev, r

    def mdp(self, agent: int, sub_actions, rm_terminal: bool = True):
        """Product MDP of agent `agent` in one launch (rlrm_mdp; RMEnvironmentWrapper.get_mdp, rm_environment_wrapper.py:185-283).
        sub_actions: [4][n_sub] action indices (4 = wait). Returns numpy (next_state [S,4,n_sub] i32, reward f64, done u8,
        terminal [S] u8)."""
        import numpy as np

        sub = np.ascontiguousarray(sub_actions, dtype=np.uint8)
        if sub.ndim != 2 or sub.shape[0] != 4:
            raise ValueError("sub_actions must be [4][n_sub]")
        n_sub = sub.shape[1]
        S = self.agent_rows[agent] if self.cfg.per_agent_rm else self.S
        nxt = torch.empty((S, 4, n_sub), dtype=torch.int32, device=self.device)
        rew = torch.empty((S, 4, n_sub), dtype=torch.float64, device=self.device)
        done = torch.empty((S, 4, n_sub), dtype=torch.uint8, device=self.device)
        term = torch.empty(S, dtype=torch.uint8, device=self.device)
        check(self.L.rlrm_mdp(self.h, int(agent), n_sub, sub.ctypes.data, int(rm_terminal), _ptr(nxt), _ptr(rew), _ptr(done),
                              _ptr(term), self._stream()))
        return nxt.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), term.cpu().numpy()

    def agent_table(self, a: int) -> torch.Tensor:
        """learner.q_table of agent a for every instance: [N, S_a, 4] (shared learner: [S_a, 4])."""
        self.sync_tables()
        if self.cfg.per_agent_rm:
            lo = sum(self.agent_rows[:a])
            t = self.q[:, lo:lo + self.agent_rows[a], :]
            return t[0] if self.cfg.shared_q else t
        return self.q.view(self.A, self.S, 4)[a] if self.cfg.shared_q else self.q.view(self.N, self.A, self.S, 4)[:, a]

    def update(self, obs_cell: torch.Tensor, actions: torch.Tensor, term_arg: torch.Tensor, rec: Dict[str, torch.Tensor]):
        obs_cell = obs_cell.to(device=self.device, dtype=torch.int16).contiguous()
        actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        term_arg = term_arg.to(device=self.device, dtype=torch.uint8).contiguous()
        so = abi.StepOut(*[_ptr(rec[k]) for k in abi.STEP_OUT_FIELDS])
        check(self.L.rlrm_update(self.h, C.byref(self.state), _ptr(obs_cell), _ptr(actions), _ptr(term_arg), C.byref(so),
                                 self._stream()))

    def train(self, n_iters: int, learn: bool = True, trace: bool = False, t0: Optional[int] = None):
        """n_iters fused lockstep iterations (select -> env/RM step -> update -> auto reset)."""
        t0 = self.t if t0 is None else t0
        tr = torch.zeros((n_iters, self.N * self.A), dtype=torch.int32, device=self.device) if trace else None
        check(self.L.rlrm_train(self.h, C.byref(self.state), t0, n_iters, int(learn), _ptr(tr), self._stream()))
        self.t = t0 + n_iters
        return tr

    def iterate(self, learn: bool = True, record: Optional[torch.Tensor] = None, reward: Optional[torch.Tensor] = None,
                want_reward: bool = True, sync: bool = True):
        """ONE lockstep iteration of the driver loop in one launch (rlrm_iterate): select -> rm_env.step -> update -> reset of
        the finished instances, reporting what rm_env.step returned: `record` int32 [N*A] (packed: bits 0-2 action, 3-5
        executed action, 6-15 new cell, 16-20 new RM state, 21 terminated, 22 truncated, 23 active step) and `reward`
        float64 [N*A]. By default both are page-locked HOST tensors owned by the engine that the kernel writes in place:
        after the stream synchronisation (`sync=True`) the host reads them without a copy. Bit-identical to train(1)."""
        n = self.N * self.A
        if record is None:
            if self._it_record is None:
                self._it_record = torch.zeros(n, dtype=torch.int32).pin_memory()
                self._it_reward = torch.zeros(n, dtype=torch.float64).pin_memory()
            record = self._it_record
            if want_reward and reward is None and not self.cfg.shared_q:  # the shared learner's launch has no per-step reward output
                reward = self._it_reward
        check(self.L.rlrm_iterate(self.h, C.byref(self.state), self.t, int(learn), _ptr(record), _ptr(reward), self._stream()))
        self.t += 1
        if sync:
            self.sync()
        return record, reward

    @staticmethod
    def unpack_record(record: torch.Tensor) -> Dict[str, torch.Tensor]:
        """Fields of the packed step record of :meth:`iterate` / the trace of :meth:`train`."""
        r = record
        return {"action": r & 7, "executed": (r >> 3) & 7, "cell": (r >> 6) & 0x3FF, "q": (r >> 16) & 0x1F,
                "terminated": ((r >> 21) & 1).bool(), "truncated": ((r >> 22) & 1).bool(), "active": ((r >> 23) & 1).bool()}

    # -- one-instance host bridge (envs.py): everything a step needs lives in ONE page-locked block --------------------
    def _host_io(self):
        if self._hio is None:
            n, nq = self.N * self.A, max(1, int(self.cfg.n_qrm_states))
            sizes = [("actions", "uint8", n), ("draws", "uint32", n * 4)] + [(k, v, n) for k, v in abi.STEP_OUT_FIELDS.items()] + \
                    [("cf_q", "uint8", n * nq), ("cf_r", "float64", n * nq)]
            sizes.sort(key=lambda kv: -np.dtype(kv[1]).itemsize)  # widest first keeps every field aligned
            total = sum(-(-np.dtype(dt).itemsize * cnt // 16) * 16 for _k, dt, cnt in sizes)
            buf = torch.zeros(total, dtype=torch.uint8).pin_memory()
            host = buf.numpy()
            views, ptrs, off = {}, {}, 0
            for k, dt, cnt in sizes:
                nbytes = np.dtype(dt).itemsize * cnt
                views[k] = host[off:off + nbytes].view(dt)
                ptrs[k] = buf.data_ptr() + off
                off += -(-nbytes // 16) * 16
            so = abi.StepOut(*[ptrs[k] for k in abi.STEP_OUT_FIELDS], None, None)
            so_cf = abi.StepOut(*[ptrs[k] for k in abi.STEP_OUT_FIELDS], ptrs["cf_q"], ptrs["cf_r"])
            self._hio = {"buf": buf, "v": views, "p": ptrs, "so": so, "so_cf": so_cf, "n_qrm": nq, "so_ref": C.byref(so), "so_cf_ref": C.byref(so_cf),
                         "stream": torch.cuda.Stream(device=self.device)}
            self._state_ref = C.byref(self.state)
        return self._hio

    def step_host(self, actions, draws=None, with_rm: bool = True, counterfactuals: bool = False):
        """rlrm_step driven from the host with no copies (needs host_control=True): `actions` (N*A ints) and `draws`
        (N*A*4 32-bit words, or None) are written into the page-locked block, the kernel reads them and writes the step
        record — plus, when `counterfactuals`, the QRM lookups on the new position (cf_q / cf_r, [N*A][n_qrm]) — in place;
        one launch, one synchronisation. Returns numpy views of the record, valid until the next call."""
        if not self.host_control:
            raise RuntimeError("step_host needs an Engine built with host_control=True")
        io = self._hio or self._host_io()
        io["v"]["actions"][:] = actions
        if draws is not None and draws is not True:  # True: the caller wrote the words into io["v"]["draws"] itself
            io["v"]["draws"][:] = draws
        # the step touches nothing but this engine's page-locked control block, so it runs on a stream of its own: it does not
        # queue behind the learners' update launches on torch's current stream, and the synchronisation waits for it alone
        stream = io["stream"].cuda_stream
        if self._ctl_dirty:  # another call of this engine (reset, select, update, ...) went to torch's current stream: finish it first
            check(self.L.rlrm_stream_sync(self.h, torch._C._cuda_getCurrentRawStream(self._dev_index)))
            self._ctl_dirty = False
        check(self.L.rlrm_step(self.h, self._state_ref, io["p"]["actions"], io["p"]["draws"] if draws is not None else None, 0,
                               int(with_rm), io["so_cf_ref"] if counterfactuals else io["so_ref"], stream))
        check(self.L.rlrm_stream_sync(self.h, stream))
        return io["v"]

    def train_host(self, n_iters: int, host_stats: torch.Tensor, host_slot: Optional[torch.Tensor] = None,
                   host_epsilon: Optional[torch.Tensor] = None, learn: bool = True, t0: Optional[int] = None):
        """End-to-end call on HOST (pinned) buffers: H2D control state, fused iterations, D2H statistics, sync."""
        t0 = self.t if t0 is None else t0
        check(self.L.rlrm_train_host(self.h, C.byref(self.state), t0, n_iters, int(learn), _ptr(host_slot),
                                     _ptr(host_epsilon), _ptr(host_stats), self._stream()))
        self.t = t0 + n_iters

    def sync_tables(self, with_traces: bool = False):
        """Sparse Q(lambda): write the listed (live-trace) q values back into `q` so it can be read; returns the dense
        e table when `with_traces`. No-op for every other configuration."""
        if not self.sparse:
            return self.e if with_traces else None
        e_dense = torch.zeros_like(self.q) if with_traces else None
        check(self.L.rlrm_qlambda_materialize(self.h, C.byref(self.state), _ptr(e_dense), self._stream()))
        return e_dense

    def evaluate(self, n_episodes: int, gamma: float, optimal_steps: float = 1.0, t0: Optional[int] = None,
                 max_iters: Optional[int] = None):
        """Batched greedy evaluation (rlrm_evaluate): every instance plays `n_episodes` episodes with its own tables,
        select_action(best=True), no update. Works on a copy of the environment state, like the reference's
        copy.deepcopy(env) (evaluation_metrics.py:45). Returns a numpy record array [N*A] of rlrm_eval_t."""
        self.sync_tables()
        ev = np.zeros(self.N * self.A, dtype=EVAL_DTYPE)
        ev["cum_gamma"] = 1.0
        ev_dev = torch.from_numpy(ev.view(np.uint8).reshape(-1, EVAL_DTYPE.itemsize).copy()).to(self.device)
        slot = self.slot.clone()
        eps = self.epsilon.clone()
        # e = NULL: the copy's traces are never read by a greedy rollout, and the training traces must not be wiped
        st = abi.State(self.N, _ptr(slot), _ptr(eps), _ptr(self.q), None, None, None, None, None, None, None)
        check(self.L.rlrm_reset_at(self.h, C.byref(st), None, self.t if t0 is None else t0, self._stream()))  # env_test.reset(...)
        n_iters = max_iters or n_episodes * (int(self.cfg.max_steps) + 1)
        check(self.L.rlrm_evaluate(self.h, C.byref(st), _ptr(ev_dev), self.t if t0 is None else t0, n_iters, n_episodes,
                                   float(gamma), float(optimal_steps), self._stream()))
        return ev_dev.cpu().numpy().view(EVAL_DTYPE).reshape(-1)

    # -- views ---------------------------------------------------------------------------------
    def slots_numpy(self):
        s = self.slot.cpu().numpy().view(np.uint64).reshape(self.N, self.A)
        g = lambda sh, m: ((s >> np.uint64(sh)) & np.uint64(m)).astype(np.int32)  # noqa: E731
        return {"cell": g(abi.SLOT_CELL_SHIFT, 0xFFFF), "agent_steps": g(abi.SLOT_STEPS_SHIFT, 0xFFFF),
                "timestep": g(abi.SLOT_TIME_SHIFT, 0xFFFF), "q": g(abi.SLOT_RMSTATE_SHIFT, 0xFF),
                "flags": g(abi.SLOT_FLAGS_SHIFT, 0xFF)}

    def stats_numpy(self):
        return self.stats.cpu().numpy().view(STATS_DTYPE).reshape(-1)

    def group_stats(self) -> Dict[str, torch.Tensor]:
        """Per-setting totals of the finished episodes' statistics, reduced on the device: tensors [len(sweep)] (a uniform
        engine is one group) of `episodes`, `successes`, `active_steps` (int64) and `return_sum` (float64). Settings with no
        instance on this engine (a shard of a sweep) read zero. One learning curve per setting is a series of these."""
        H, k = (len(self.sweep), self.sweep_group) if self.sweep is not None else (1, self.N)
        off = int(self.cfg.instance_offset) if self.sweep is not None else 0
        b = self.stats
        u32 = b.view(torch.int32).to(torch.int64) & 0xFFFFFFFF
        fields = {"episodes": u32[:, 2], "successes": u32[:, 3], "active_steps": b.view(torch.int64)[:, 0],
                  "return_sum": b.view(torch.float64)[:, 2]}
        lead = off % k  # the engine's instances cover groups g0 .. g0 + m - 1, the first and last possibly in part
        g0 = off // k
        m = (lead + self.N + k - 1) // k
        out = {}
        for name, v in fields.items():
            per_inst = v.view(self.N, self.A).sum(dim=1)
            padded = torch.zeros(m * k, dtype=per_inst.dtype, device=per_inst.device)
            padded[lead:lead + self.N] = per_inst
            tot = torch.zeros(H, dtype=per_inst.dtype, device=per_inst.device)
            tot[g0:g0 + m] = padded.view(m, k).sum(dim=1)
            out[name] = tot
        return out

    def total_active_steps(self) -> int:
        """Active agent-steps so far = env.agent_steps of every finished episode (stats.active_steps) + the running
        episodes' agent_steps (slot words), reduced on the device."""
        finished = self.stats.view(torch.int64)[:, 0].sum()
        running = ((self.slot >> abi.SLOT_STEPS_SHIFT) & 0xFFFF).sum()
        return int((finished + running).item())

    # -- checkpoint / resume -----------------------------------------------------------------------
    _STATE_TENSORS = ("slot", "epsilon", "q", "e", "visits", "ep_return", "stats", "acc_sum", "acc_cnt", "acc_last",
                      "tr_pos", "tr_idx", "tr_eq", "tr_len", "tr_work")

    def state_dict(self) -> Dict[str, object]:
        """Everything a run needs to continue bit-identically: the device arrays of rlrm_state_t (CPU copies) and the lockstep
        iteration counter (the Philox counter word). The reference only pickles learner objects (office_main.py:1611-1613,
        1922-1925; see learners.QLearning.__getstate__ for that format); a batch of instances resumes from this instead."""
        out = {k: getattr(self, k).cpu() for k in self._STATE_TENSORS if getattr(self, k) is not None}
        out.update({"t": int(self.t), "n_instances": self.N, "n_agents": self.A, "state_space": self.S, "sparse": self.sparse,
                    "sweep": None if self.sweep is None else [dict(s) for s in self.sweep], "sweep_group": self.sweep_group})
        return out

    def load_state_dict(self, state: Dict[str, object]) -> None:
        if (state["n_instances"], state["n_agents"], state["state_space"], state["sparse"]) != (self.N, self.A, self.S, self.sparse):
            raise ValueError("checkpoint was taken from a differently shaped engine")
        if (state.get("sweep"), state.get("sweep_group")) != (self.sweep, self.sweep_group):
            raise ValueError("checkpoint was taken from an engine with a different hyper-parameter sweep")
        for k in self._STATE_TENSORS:
            mine = getattr(self, k)
            if (mine is None) != (k not in state):
                raise ValueError(f"checkpoint and engine disagree on state array {k!r}")
            if mine is not None:
                mine.copy_(state[k])  # in place: the C-ABI state struct keeps pointing at the same device memory
        self.t = int(state["t"])

    # -- the driver loop, call by call (reference API granularity) ----------------------------------
    def iterate_unfused(self, learn: bool = True, draws: Optional[torch.Tensor] = None, auto_reset: bool = True):
        """One lockstep iteration through the separate entry points, in the reference drivers' order
        (frozen_lake_main.py:345-376 / office_main.py:1709-1749): select for every agent -> wrapper step -> update for
        every agent -> reset of the instances whose episode ended. Bit-identical to one iteration of :meth:`train`."""
        if self.sparse:
            raise RuntimeError("the call-by-call path needs dense Q(lambda) traces: build the Engine with qlambda_sparse=False")
        fl_driver = self.cfg.driver == abi.DRIVER_FROZEN_LAKE_MAIN
        cell_before = (self.slot & 0xFFFF).to(torch.int16)
        first = ((self.slot >> abi.SLOT_FLAGS_SHIFT) & abi.FLAG_FIRST) != 0
        actions = self.select_action(self.t, draws, best=not learn)
        rec = self.step(actions, self.t, draws)
        if learn:
            obs = torch.where(first, rec["cell"], cell_before) if fl_driver else cell_before
            term_arg = (rec["term"] | rec["trunc"]) if fl_driver else rec["term"]
            self.update(obs, actions.reshape(-1), term_arg, rec)
        term = rec["term"].view(self.N, self.A).bool()
        trunc = rec["trunc"].view(self.N, self.A).bool()
        over = term.all(dim=1) | trunc.all(dim=1)
        self.t += 1  # the reset below starts episodes whose first step is iteration t + 1 (keys the random start positions)
        if auto_reset:
            self.reset(over)
        return actions, rec, over
