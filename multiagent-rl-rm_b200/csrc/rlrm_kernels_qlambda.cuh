// rlrm_kernels_qlambda.cuh: Q(lambda) fused kernels, dense-faithful and sparse-exact — part of the single translation unit csrc/rlrm_b200.cu (see its header comment).
#pragma once
#include "rlrm_kernels_api.cuh"
#include "rlrm_kernels_train.cuh"

// PA = agents carry different reward machines: the warp's agent gets its own view of the parameters (a private copy); with
// PA = false the parameter block stays in the constant bank
// SWEEP: the block's instance takes its group's learner settings
template <int ENV, typename T, bool PA, bool SWEEP>
__global__ void __launch_bounds__(256) train_qlambda_kernel(KP p_in, DState st, unsigned long long t0, int n_iters, int learn,
                                                           unsigned* trace, double* reward_out, Sweep sw) {
  typedef RT<T> R;
  typedef typename R::row_t row_t;
  KP p_view, p_sw;  // p_sw: a sweep handle's learner settings, read only where they are used (ph; see train_ql_fast_kernel)
  if (PA) p_view = p_in;
  const KP& p = PA ? p_view : p_in;
  const KP& ph = SWEEP ? p_sw : p;
  Tab tb = stage_tables(p_in);
  __shared__ int sh_term[RLRM_MAX_AGENTS], sh_trunc[RLRM_MAX_AGENTS];
  const long long i = blockIdx.x;
  const int a = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long k = i * p_in.A + a;
  if (PA) agent_view(p_in, p_view, tb, a);  // this warp's agent has its own machine: nQ, final state, table size
  if (SWEEP) {
    p_sw = p;
    apply_sweep(p_sw, sw, i);
  }
  Slot s = unpack_slot(st.slot[k]);
  double eps = st.epsilon[k];
  double ep_ret = st.ep_return ? st.ep_return[k] : 0.0;
  const size_t base = table_base(p_in, i, a);
  T* Q = tab<T>(st.q) + base;
  T* E = tab<T>(st.e) + base;
  unsigned* V = st.visits ? st.visits + base : nullptr;  // QLearningLambda counts visits on every update (qlearning_lambda.py:44)
  unsigned long long active_steps = 0;
  unsigned episodes = 0, successes = 0, last_length = 0;
  float last_return = 0.f;
  bool had_episode = false;
  rlrm_stats_t z;
  if (st.stats) z = st.stats[k];
  double return_sum_add = st.stats ? z.return_sum : 0.0;
  unsigned long long explore_thr = explore_threshold(eps);

  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    unsigned w[4];
    RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
    __syncwarp();
    const row_t row = load_row<T>(Q, s.cell * p.nQ + s.rm);
    const int action = select_action(row, explore_thr, w, learn == 0, p.n_actions);
    const unsigned before = s.cell;
    const bool first = (s.flags & RLRM_FLAG_FIRST) != 0;
    Rec r;
    agent_step<ENV>(p, tb, s, action, w[3], true, r);  // all 32 lanes compute the same scalars
    if (learn) {
      const unsigned obs = (p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? r.cell : before;
      const bool term_arg = p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (r.term || r.trunc) : r.term;
      // warp-cooperative dense sweep (the __syncthreads inside qlambda_sweep is replaced by __syncwarp here)
      const unsigned sidx = obs * p.nQ + r.prev_q, snidx = r.cell * p.nQ + r.q;
      const row_t nrow = load_row<T>(Q, snidx);
      const T qsa = Q[sidx * 4 + action];
      __syncwarp();
      const double best = term_arg ? 0.0 : (double)row_max(nrow);
      const T td = R::sub(R::cvt(__dadd_rn(r.reward, __dmul_rn(ph.h.gamma, best))), qsa);
      const T c = R::mul(R::lr(ph), td);
      const unsigned hot = sidx * 4 + action;
      // learning_rate=None: lr = 1 / visits[s, a] is an np.float64, so lr * td and (lr * td) * e_table are float64 and the
      // in-place add happens in float64 before the cast back to float32 (qlearning_lambda.py:44-49, 63)
      const bool lr_none = ph.h.lr < 0.0;
      unsigned vis = 0;
      if (V) {
        vis = V[hot] + 1;
        __syncwarp();
        if (lane == 0) V[hot] = vis;
      }
      const double c64 = lr_none ? __dmul_rn(__ddiv_rn(1.0, (double)vis), (double)td) : 0.0;
      row_t* Q4 = reinterpret_cast<row_t*>(Q);
      row_t* E4 = reinterpret_cast<row_t*>(E);
      for (long long j = lane; j < p.S4 / 4; j += 32) sweep_row<T>(ph, Q4, E4, j, hot, c, c64, lr_none, term_arg);
      __syncwarp();
    }
    ep_ret = __dadd_rn(ep_ret, r.reward);
    if (trace && lane == 0)
      trace[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = (unsigned)action | (r.executed << 3) | (r.cell << 6) | (r.q << 16) |
                                                           ((unsigned)r.term << 21) | ((unsigned)r.trunc << 22) |
                                                           ((unsigned)r.stepped << 23);
    if (reward_out && lane == 0) reward_out[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = r.reward;
    if (lane == 0) {
      sh_term[a] = r.term;
      sh_trunc[a] = r.trunc;
    }
    __syncthreads();
    bool all_term = true, all_trunc = true;
    for (int b = 0; b < p.A; b++) {
      all_term = all_term && sh_term[b];
      all_trunc = all_trunc && sh_trunc[b];
    }
    __syncthreads();
    if (all_term || all_trunc) {
      episodes++;
      active_steps += s.steps;  // env.agent_steps[agent] of the finished episode
      successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
      last_return = __double2float_rn(ep_ret);
      return_sum_add = __dadd_rn(return_sum_add, ep_ret);
      last_length = s.time;
      had_episode = true;
      ep_ret = 0.0;
      reset_slot(ph, tb, i, a, t + 1, s, eps);
      explore_thr = explore_threshold(eps);
      // reset_e_table (ma_office.py:101-102)
      row_t* E4 = reinterpret_cast<row_t*>(E);
      for (long long j = lane; j < p.S4 / 4; j += 32) E4[j] = R::zero_row();
      __syncwarp();
    }
  }
  if (lane == 0) {
    st.slot[k] = pack_slot(s);
    st.epsilon[k] = eps;
    if (st.ep_return) st.ep_return[k] = ep_ret;
    if (st.stats) {
      z.active_steps += active_steps;
      z.episodes += episodes;
      z.successes += successes;
      z.return_sum = return_sum_add;
      if (had_episode) {
        z.last_return = last_return;
        z.last_length = last_length;
      }
      st.stats[k] = z;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Q(lambda), sparse-exact traces: one warp per instance, one lane group per agent. Only entries with a live trace are
// touched; each agent's live entries sit in a list of (trace, current q value) pairs (a write-back cache over the
// table), so one update step reads/writes the list once, 8 bytes per entry. Bit-identical to the dense sweep of
// QLearningLambda.update (qlearning_lambda.py:33-84) up to the sign of zero: unlisted entries have e == 0 and receive +0.
// ------------------------------------------------------------------------------------------------
template <typename T>
struct TraceList {
  unsigned short* pos;         // [S*4]
  unsigned short* idx;         // [cap]
  typename RT<T>::pair_t* eq;  // [cap] (trace, current q value)
};
template <typename T>
__device__ __forceinline__ typename RT<T>::pair_t* pairs(float2* p) { return reinterpret_cast<typename RT<T>::pair_t*>(p); }

// current value of table entry j: the listed copy when the entry has a live trace, else the table
template <typename T>
__device__ __forceinline__ T trace_lookup(const T* Q, const TraceList<T>& L, unsigned j) {
  const unsigned pz = L.pos[j];
  return pz ? L.eq[pz - 1].y : Q[j];
}

// write the listed values back and forget the list (traces wiped: reset_e_table / e_table.fill(0))
template <typename T>
__device__ __forceinline__ void trace_flush(T* Q, const TraceList<T>& L, unsigned len, int lane, int stride = 32) {
  for (unsigned j = lane; j < len; j += stride) {
    const unsigned id = L.idx[j];
    Q[id] = L.eq[j].y;
    L.pos[id] = 0;
  }
}

// One lane GROUP per agent (LG = p.qls_lg lanes: 8, or 4 with more than four agents), the groups of an instance adjacent,
// 32 / (LG * G) instances per warp — four agents' lists per warp whatever the agent count. The scalar part of a step
// (Philox, epsilon-greedy, env / RM step, TD error) is computed per lane for the lane's own agent — redundantly inside a
// group, but once per warp-instruction for all agents of the instance — and each group sweeps its own agent's list. The
// previous one-warp-per-agent layout spent ~550 warp-instructions per agent-step at 79 % issue utilisation (ncu,
// profiles/r01_sparse_qlambda_ncu.csv): the lists stay L1-resident for the n_iters of a launch, so the kernel is bound by
// instruction issue, not by HBM. Episode-over detection is two warp ballots; no shared memory, no block barrier.
#define QLS_BLOCK 128
#ifndef RLRM_QLS_LG_DEFAULT
#define RLRM_QLS_LG_DEFAULT 8  // lanes per agent (capped at 32 / G): four lists per warp. Measured (profiles/r02c/r02c_qls_lanes_per_agent.json,
                               // config 4's scenario with 1 / 2 / 4 agents): 1 agent 32 -> 8 lanes 1.82e9 -> 3.81e9, 2 agents 16 -> 8 lanes 3.05e9 -> 3.95e9;
                               // 4 lanes halve the rate everywhere (the visited entry's lookup needs a second round, a sweep waits for the longest of 8 lists)
#endif
template <int ENV, typename T, bool PA, bool SWEEP>
__global__ void __launch_bounds__(QLS_BLOCK) train_qlambda_sparse_kernel(KP p_in, DState st, unsigned long long t0, int n_iters, int learn,
                                                                        unsigned* trace, double* reward_out, Sweep sw) {
  typedef RT<T> R;
  typedef typename R::row_t row_t;
  typedef typename R::pair_t pair_t;
  KP p_view, p_sw;  // p_sw: a sweep handle's learner settings, read only where they are used (ph; see train_ql_fast_kernel)
  if (PA) p_view = p_in;
  const KP& p = PA ? p_view : p_in;
  const KP& ph = SWEEP ? p_sw : p;
  Tab tb = stage_tables(p_in);
  // lanes per agent LG (p.qls_lg: 4 .. 32 / G) -> lanes per instance LI = LG * G -> 32 / LI instances per warp
  const unsigned FULL = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const int LG = p_in.qls_lg, LI = LG << p_in.g_shift;
  const long long warp = (long long)blockIdx.x * (QLS_BLOCK / 32) + (threadIdx.x >> 5);
  const long long i_first = warp * (32 / LI);
  if (i_first >= st.N) return;  // whole warps leave; nothing below synchronises across warps
  const long long i_raw = i_first + lane / LI;
  const bool inst_ok = i_raw < st.N;
  const long long i = inst_ok ? i_raw : st.N - 1;  // lanes past the last instance idle on valid addresses
  const int a = (lane & (LI - 1)) / LG;  // this lane's agent (slot a >= A idles when A is not a power of two)
  const int gl = lane & (LG - 1);        // lane within the agent's group
  const bool valid = inst_ok && a < p.A;
  const unsigned inst_mask = (LI == 32 ? FULL : ((1u << LI) - 1u)) << (lane & ~(LI - 1));  // the lanes of this lane's instance
  const long long k = i * p_in.A + (valid ? a : 0);
  if (PA) agent_view(p_in, p_view, tb, valid ? a : 0);  // this lane group's agent has its own machine
  if (SWEEP) {
    p_sw = p;
    apply_sweep(p_sw, sw, i);
  }  // i is clamped to the launch's instances
  Slot s = {0, 0, 0, 0, 0};
  double eps = 0.0, ep_ret = 0.0, return_sum = 0.0;
  T* Q = tab<T>(st.q) + table_base(p_in, i, valid ? a : 0);
  unsigned* V = st.visits ? st.visits + table_base(p_in, i, valid ? a : 0) : nullptr;
  TraceList<T> L;
  L.pos = st.tr_pos + (size_t)k * (size_t)p_in.S4;  // list arrays are strided by the LARGEST table (per-agent machines)
  L.idx = st.tr_idx + (size_t)k * (size_t)st.tr_cap;
  L.eq = pairs<T>(st.tr_eq) + (size_t)k * (size_t)st.tr_cap;
  unsigned len = 0;
  rlrm_stats_t z;
  if (valid) {
    s = unpack_slot(st.slot[k]);
    eps = st.epsilon[k];
    if (st.ep_return) ep_ret = st.ep_return[k];
    len = st.tr_len[k];
    if (st.stats) {
      z = st.stats[k];
      return_sum = z.return_sum;
    }
  }
  unsigned long long work = 0, active_steps = 0;
  unsigned episodes = 0, successes = 0, last_length = 0;
  float last_return = 0.f;
  bool had_episode = false;
  unsigned long long explore_thr = explore_threshold(eps);

  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    unsigned w[4];
    RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
    __syncwarp();
    // Q row of the current state: group lanes 0..3 fetch one action value each
    const unsigned rbase = (s.cell * p.nQ + s.rm) * 4;
    const T mine = (valid && gl < 4) ? trace_lookup<T>(Q, L, rbase + gl) : (T)0;
    row_t row;
    row.x = __shfl_sync(FULL, mine, 0, LG);
    row.y = __shfl_sync(FULL, mine, 1, LG);
    row.z = __shfl_sync(FULL, mine, 2, LG);
    row.w = __shfl_sync(FULL, mine, 3, LG);
    const int action = select_action(row, explore_thr, w, learn == 0, p.n_actions);
    const unsigned before = s.cell;
    const bool first = (s.flags & RLRM_FLAG_FIRST) != 0;
    Rec r;
    agent_step<ENV>(p, tb, s, action, w[3], true, r);  // every lane of a group computes its agent's scalars
    bool wipe = false;
    if (learn) {
      const unsigned obs = (p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? r.cell : before;
      const bool term_arg = p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (r.term || r.trunc) : r.term;
      const unsigned hot = (obs * p.nQ + r.prev_q) * 4 + action, nbase = (r.cell * p.nQ + r.q) * 4;
      // group lanes 0..3: next-state row; lane 4 (groups of 8+) or lane 0 in a second round (groups of 4): Q[s,a] together
      // with its list position (0 = no live trace yet), which also tells the sweep which entry is the visited one
      T got = (T)0;
      unsigned pz = 0;
      if (valid && gl < 4) {
        got = trace_lookup<T>(Q, L, nbase + gl);
      } else if (valid && gl == 4) {
        pz = L.pos[hot];
        got = pz ? L.eq[pz - 1].y : Q[hot];
      }
      const T n0 = __shfl_sync(FULL, got, 0, LG), n1 = __shfl_sync(FULL, got, 1, LG);
      const T n2 = __shfl_sync(FULL, got, 2, LG), n3 = __shfl_sync(FULL, got, 3, LG);
      T qsa;
      unsigned hotpos;
      if (LG > 4) {
        qsa = __shfl_sync(FULL, got, 4, LG);
        hotpos = __shfl_sync(FULL, pz, 4, LG);
      } else {
        T h = (T)0;
        if (valid && gl == 0) {
          pz = L.pos[hot];
          h = pz ? L.eq[pz - 1].y : Q[hot];
        }
        qsa = __shfl_sync(FULL, h, 0, LG);
        hotpos = __shfl_sync(FULL, gl == 0 ? pz : 0u, 0, LG);
      }
      row_t nrow;
      nrow.x = n0; nrow.y = n1; nrow.z = n2; nrow.w = n3;
      const double best = term_arg ? 0.0 : (double)row_max(nrow);
      const T td = R::sub(R::cvt(__dadd_rn(r.reward, __dmul_rn(ph.h.gamma, best))), qsa);
      const T c = R::mul(R::lr(ph), td);
      const bool lr_none = ph.h.lr < 0.0;  // lr = 1 / visits: float64 arithmetic, see train_qlambda_kernel
      unsigned vis = 0;
      if (V && valid) {
        vis = V[hot] + 1;
      }
      __syncwarp();
      if (V && valid && gl == 0) V[hot] = vis;
      const double c64 = lr_none ? __dmul_rn(__ddiv_rn(1.0, (double)(vis ? vis : 1u)), (double)td) : 0.0;
      for (unsigned j = gl; j < len; j += LG) {  // one pass over the agent's live entries (len = 0 on idle lanes)
        pair_t eq = L.eq[j];
        if (j + 1 == hotpos) eq.x = (T)1;  // replacing trace on the visited entry
        eq.y = lr_none ? R::cvt(__dadd_rn((double)eq.y, __dmul_rn(c64, (double)eq.x))) : R::add(eq.y, R::mul(c, eq.x));
        eq.x = term_arg ? (T)0 : R::mul(eq.x, R::decay(ph));
        L.eq[j] = eq;
      }
      work += len;
      if (valid && hotpos == 0u) {  // first visit since the last wipe: the table value (qsa) is current
        if (gl == 0) {
          L.idx[len] = (unsigned short)hot;
          const T q_new = lr_none ? R::cvt(__dadd_rn((double)qsa, __dmul_rn(c64, 1.0))) : R::add(qsa, R::mul(c, (T)1));
          L.eq[len] = R::make_pair(term_arg ? (T)0 : R::mul((T)1, R::decay(ph)), q_new);
          L.pos[hot] = (unsigned short)(len + 1);
        }
        len++;
      }
      wipe = valid && term_arg;  // e_table.fill(0): nothing is live any more
    }
    ep_ret = __dadd_rn(ep_ret, r.reward);
    if (trace && valid && gl == 0)
      trace[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = (unsigned)action | (r.executed << 3) | (r.cell << 6) | (r.q << 16) |
                                                           ((unsigned)r.term << 21) | ((unsigned)r.trunc << 22) |
                                                           ((unsigned)r.stepped << 23);
    if (reward_out && valid && gl == 0) reward_out[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = r.reward;
    // episode over <=> every agent of the instance terminated, or every agent truncated (idle lanes vote yes)
    const unsigned bt = __ballot_sync(FULL, !valid || r.term), bc = __ballot_sync(FULL, !valid || r.trunc);
    const bool over = ((bt & inst_mask) == inst_mask) || ((bc & inst_mask) == inst_mask);
    if (valid && over) {
      episodes++;
      active_steps += s.steps;
      successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
      last_return = __double2float_rn(ep_ret);
      return_sum = __dadd_rn(return_sum, ep_ret);
      last_length = s.time;
      had_episode = true;
      ep_ret = 0.0;
      reset_slot(ph, tb, i, a, t + 1, s, eps);
      explore_thr = explore_threshold(eps);
      wipe = true;  // reset_e_table (ma_office.py:101-102)
    }
    __syncwarp();
    trace_flush<T>(Q, L, wipe ? len : 0u, gl, LG);
    if (wipe) len = 0;
    __syncwarp();
  }
  if (valid && gl == 0) {
    st.slot[k] = pack_slot(s);
    st.epsilon[k] = eps;
    st.tr_len[k] = len;
    if (st.tr_work) st.tr_work[k] += work;
    if (st.ep_return) st.ep_return[k] = ep_ret;
    if (st.stats) {
      z.active_steps += active_steps;
      z.episodes += episodes;
      z.successes += successes;
      z.return_sum = return_sum;
      if (had_episode) {
        z.last_return = last_return;
        z.last_length = last_length;
      }
      st.stats[k] = z;
    }
  }
}

// sparse Q(lambda): listed values -> table (lists stay live); optionally scatter the traces into a dense buffer
template <typename T>
__global__ void __launch_bounds__(256) qlambda_materialize_kernel(KP p, DState st, T* e_dense) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= st.N * p.A) return;
  T* Q = tab<T>(st.q) + table_base(p, warp / p.A, (int)(warp % p.A));
  const unsigned short* idx = st.tr_idx + (size_t)warp * (size_t)st.tr_cap;
  const typename RT<T>::pair_t* leq = pairs<T>(st.tr_eq) + (size_t)warp * (size_t)st.tr_cap;
  const unsigned len = st.tr_len[warp];
  for (unsigned j = lane; j < len; j += 32) {
    const typename RT<T>::pair_t eq = leq[j];
    Q[idx[j]] = eq.y;
    if (e_dense) e_dense[table_base(p, warp / p.A, (int)(warp % p.A)) + idx[j]] = eq.x;
  }
}

// sparse Q(lambda): reset_e_table for the masked instances = flush + forget the lists
template <typename T>
__global__ void __launch_bounds__(256) qlambda_sparse_reset_kernel(KP p, DState st, const unsigned char* mask) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= st.N * p.A) return;
  if (mask && !mask[warp / p.A]) return;
  TraceList<T> L;
  L.pos = st.tr_pos + (size_t)warp * (size_t)p.S4;
  L.idx = st.tr_idx + (size_t)warp * (size_t)st.tr_cap;
  L.eq = pairs<T>(st.tr_eq) + (size_t)warp * (size_t)st.tr_cap;
  trace_flush<T>(tab<T>(st.q) + table_base(p, warp / p.A, (int)(warp % p.A)), L, st.tr_len[warp], lane);
  __syncwarp();
  if (lane == 0) st.tr_len[warp] = 0;
}

