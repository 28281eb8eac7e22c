// rlrm_kernels_api.cuh: call-by-call kernels (reset / select / step / rm_step / update), also the trace-injection parity path — part of the single translation unit csrc/rlrm_b200.cu (see its header comment).
#pragma once
#include "rlrm_device.cuh"

// ------------------------------------------------------------------------------------------------
// unfused kernels (the reference's call-by-call API; also the parity path with injected draws)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) reset_kernel(KP p, DState st, const unsigned char* mask, unsigned long long t, Sweep sw) {
  Tab tb = stage_tables(p);
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= st.N * p.A) return;
  const long long i = k / p.A;
  const int a = (int)(k - i * p.A);
  if (mask && !mask[i]) return;
  if (sw.hyp) apply_sweep(p, sw, i);  // the epsilon decay of the instance's group
  Slot s;
  double eps = st.epsilon[k];
  reset_slot(p, tb, i, a, t, s, eps);
  st.slot[k] = pack_slot(s);
  st.epsilon[k] = eps;
  if (st.ep_return) st.ep_return[k] = 0.0;
}

// Q(lambda): reset_e_table for the masked instances (ma_frozen_lake.py:80-81 ; ma_office.py:101-102)
template <typename T>
__global__ void __launch_bounds__(256) clear_traces_kernel(KP p, DState st, const unsigned char* mask) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // one row (4 entries) of one instance's tables
  const long long per_inst = (p.per_agent ? p.sum4 : (long long)p.A * p.S4) / 4;
  if (g >= st.N * per_inst) return;
  if (mask && !mask[g / per_inst]) return;
  reinterpret_cast<typename RT<T>::row_t*>(st.e)[g] = RT<T>::zero_row();
}

template <bool PA, typename T, bool SOFTMAX>  // SOFTMAX: softmax exploration with beta = 1 / temperature (see train_kernel)
__global__ void __launch_bounds__(256) select_kernel(KP p_in, DState st, const unsigned* draws, unsigned long long t, int best,
                                                    unsigned char* actions_out, double beta) {
  KP p = p_in;
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= st.N * p.A) return;
  const long long i = k / p.A;
  const int a = (int)(k - i * p.A);
  if (PA) p.nQ = p_in.a_nQ[a];
  const Slot s = unpack_slot(st.slot[k]);
  const T* Q = tab<T>(st.q) + table_base(p_in, i, a);
  const typename RT<T>::row_t row = load_row<T>(Q, s.cell * p.nQ + s.rm);
  unsigned w[4];
  if (draws) {
    const uint4 d = reinterpret_cast<const uint4*>(draws)[k];
    w[0] = d.x; w[1] = d.y; w[2] = d.z; w[3] = d.w;
  } else {
    RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
  }
  actions_out[k] = (unsigned char)(SOFTMAX ? select_softmax(row, w[1], beta, best != 0, p.n_actions)
                                           : select_action(row, explore_threshold(st.epsilon[k]), w, best != 0, p.n_actions));
}

__device__ __forceinline__ void store_rec(const DOut& o, long long k, const Rec& r) {
  if (o.prev_cell) o.prev_cell[k] = (unsigned short)r.prev_cell;
  if (o.cell) o.cell[k] = (unsigned short)r.cell;
  if (o.prev_q) o.prev_q[k] = (unsigned char)r.prev_q;
  if (o.q) o.q[k] = (unsigned char)r.q;
  if (o.event) o.event[k] = (unsigned char)r.event;
  if (o.executed) o.executed[k] = (unsigned char)r.executed;
  if (o.renv) o.renv[k] = r.renv;
  if (o.rq) o.rq[k] = r.rq;
  if (o.reward) o.reward[k] = r.reward;
  if (o.env_term) o.env_term[k] = r.env_term;
  if (o.rm_term) o.rm_term[k] = r.rm_term;
  if (o.term) o.term[k] = r.term;
  if (o.trunc) o.trunc[k] = r.trunc;
}

template <int ENV, bool PA>
__global__ void __launch_bounds__(256) step_kernel(KP p_in, DState st, const unsigned char* actions, const unsigned* draws,
                                                  unsigned long long t, int with_rm, DOut out) {
  KP p = p_in;
  Tab tb = stage_tables(p_in);
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= st.N * p.A) return;
  const long long i = k / p.A;
  const int a = (int)(k - i * p.A);
  if (PA) agent_view(p_in, p, tb, a);
  Slot s = unpack_slot(st.slot[k]);
  unsigned w3 = 0;
  if (p.stochastic) {
    if (draws) {
      w3 = draws[k * 4 + 3];
    } else {
      unsigned w[4];
      RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
      w3 = w[3];
    }
  }
  Rec r;
  agent_step<ENV, -1, true>(p, tb, s, min((int)actions[k], RLRM_ACTION_WAIT), w3, with_rm != 0, r);
  st.slot[k] = pack_slot(s);
  store_rec(out, k, r);
  if (out.cf_q || out.cf_r) {  // counterfactual RM lookups on the new position (rm_environment_wrapper.py:144-153)
    const int col = r.event == RLRM_EVENT_NONE ? p.nEv : (int)r.event;
    const int stride = p_in.n_qrm;  // row stride = the maximum over agents
    for (int j = 0; j < p.n_qrm; j++) {
      const unsigned u = tb.qrm_states[j];
      const unsigned d = tb.delta[u * (p.nEv + 1) + col];
      if (out.cf_q) out.cf_q[k * stride + j] = (unsigned char)(d == RLRM_NO_TRANSITION ? u : d);
      if (out.cf_r) out.cf_r[k * stride + j] = d == RLRM_NO_TRANSITION ? 0.0 : tb.rcf[u * (p.nEv + 1) + col];
    }
  }
}

// RMEnvironmentWrapper.get_mdp (rm_environment_wrapper.py:185-283): every (encoded state, nominal action, sub-action) of one
// agent's product MDP in one launch. The reference does reset(seed) + set_state + one step with env.stochastic = False per
// triple; here each thread builds the freshly-reset slot (active, no failure, agent_steps = timestep = 0) at its (cell, RM
// state) and runs the same agent_step the training kernels use, executing the sub-action as is.
struct MdpSub {
  unsigned char a[16];  // [nominal action][sub-action index]
};
template <int ENV>
__global__ void __launch_bounds__(256) mdp_kernel(KP p_in, int agent, int n_sub, MdpSub sub, int rm_terminal, int* next_state,
                                                 double* reward, unsigned char* done, unsigned char* terminal) {
  KP p = p_in;
  Tab tb = stage_tables(p_in);
  if (p_in.per_agent) agent_view(p_in, p, tb, agent);
  const long long n = (long long)p.ncell * p.nQ * 4 * n_sub;
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int j = (int)(k % n_sub);
  const int a = (int)((k / n_sub) & 3);
  const int enc = (int)(k / (4 * n_sub));
  const unsigned cell = enc / p.nQ, q = enc - cell * p.nQ;
  // is_terminal_state_mdp (ma_frozen_lake.py:321-335, ma_office.py:411-432): hazard first, then the RM's final state
  int kind = 0;
  double term_reward = 0.0;
  if ((tb.cell_flags[cell] & 1) && (ENV == RLRM_ENV_FROZEN_LAKE || p.terminate_on_plants)) {
    kind = 1;
    term_reward = p.hole_penalty;
  } else if (rm_terminal && p.rm_final >= 0 && (int)q == p.rm_final) {
    kind = 2;
  }
  if (a == 0 && j == 0) terminal[enc] = (unsigned char)kind;
  if (kind) {  // self-loop (rm_environment_wrapper.py:232-236)
    next_state[k] = enc;
    reward[k] = term_reward;
    done[k] = 1;
    return;
  }
  Slot s;
  s.cell = cell;
  s.steps = 0;
  s.time = 0;
  s.rm = q;
  s.flags = RLRM_FLAG_ACTIVE;
  Rec r;
  agent_step<ENV, 0, true>(p, tb, s, min((int)sub.a[a * 4 + j], RLRM_ACTION_WAIT), 0u, true, r);
  next_state[k] = (int)(r.cell * p.nQ + r.q);
  reward[k] = r.reward;
  done[k] = (r.term || r.trunc) ? 1 : 0;
}

// Value iteration over a product MDP held as padded outcome arrays (mdp_vi.value_iteration, environments/utils_envs/mdp_vi.py:9-60,
// consumes RMEnvironmentWrapper.get_mdp's P[s][a] = [(prob, s', reward, done), ...]). One thread per state and sweep:
// Q[s][a] = sum_j prob * (reward + gamma * V[s'] * !done) in outcome order, V'[s] = max_a Q[s][a]. The reference sweeps the
// states in place (Gauss-Seidel); a parallel sweep reads the previous V (Jacobi): same fixed point and same stopping rule,
// different iterates — results agree to the tolerance the stopping rule implies, not bit for bit (tests/test_mdp.py).
__global__ void __launch_bounds__(256) vi_sweep_kernel(long long S, int n_out, const double* prob, const int* next_state,
                                                      const double* reward, const unsigned char* done, double gamma, int delta_rel,
                                                      const double* v_in, double* v_out, double* Q, int* policy,
                                                      unsigned long long* delta_bits) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double cdelta = 0.0;
  if (s < S) {
    double best = 0.0;
    int arg = 0;
    for (int a = 0; a < 4; a++) {
      double q = 0.0;
      const size_t base = ((size_t)s * 4 + a) * (size_t)n_out;
      for (int j = 0; j < n_out; j++) {
        const double pr = prob[base + j];
        if (pr == 0.0) continue;  // padding
        const double future = done[base + j] ? 0.0 : __dmul_rn(gamma, v_in[next_state[base + j]]);
        q = __dadd_rn(q, __dmul_rn(pr, __dadd_rn(reward[base + j], future)));
      }
      Q[s * 4 + a] = q;
      if (a == 0 || q > best) {
        best = q;
        arg = a;
      }
    }
    v_out[s] = best;
    policy[s] = arg;
    const double diff = fabs(best - v_in[s]);
    cdelta = delta_rel ? diff / (fabs(best) > 1e-12 ? fabs(best) : 1.0) : diff;
  }
  // block maximum, then one atomic per block; non-negative doubles order like their bit patterns
  for (int o = 16; o > 0; o >>= 1) cdelta = fmax(cdelta, __shfl_xor_sync(0xFFFFFFFFu, cdelta, o));
  __shared__ double wmax[8];
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = cdelta;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = wmax[0];
    for (int w = 1; w < 8; w++) m = fmax(m, wmax[w]);
    atomicMax(delta_bits, (unsigned long long)__double_as_longlong(m));
  }
}

// RewardMachine.step on explicit (state, position) pairs (reward_machine.py:45-59)
__global__ void __launch_bounds__(256) rm_step_kernel(KP p_in, int agent, long long n, unsigned char* q, const unsigned short* cell,
                                                     unsigned char* event_out, double* reward_out) {
  KP p = p_in;
  Tab tb = stage_tables(p_in);
  if (p_in.per_agent) agent_view(p_in, p, tb, agent);  // the reward machine of agent `agent`
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const unsigned ev = tb.label[min((unsigned)cell[k], (unsigned)p.ncell - 1u)];  // caller memory: clamp what indexes a table
  const int col = ev == RLRM_EVENT_NONE ? p.nEv : (int)ev;
  const unsigned cur = min((unsigned)q[k], (unsigned)p.nQ - 1u);
  const unsigned d = tb.delta[cur * (p.nEv + 1) + col];
  double r = 0.0;
  if (d != RLRM_NO_TRANSITION) {
    r = tb.rq[cur * (p.nEv + 1) + col];
    q[k] = (unsigned char)d;
  }
  if (event_out) event_out[k] = (unsigned char)ev;
  if (reward_out) reward_out[k] = r;
}

template <int ALGO, bool PA, typename T>
__global__ void __launch_bounds__(256) update_kernel(KP p_in, DState st, const unsigned short* obs_cell, const unsigned char* actions,
                                                    const unsigned char* term_arg, DOut o, Sweep sw) {
  KP p = p_in;
  Tab tb = stage_tables(p_in);
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= st.N * p.A) return;
  const long long i = k / p.A;
  const int a = (int)(k - i * p.A);
  if (PA) agent_view(p_in, p, tb, a);
  if (sw.hyp) apply_sweep(p, sw, i);
  // the record and the arguments are caller memory: clamp every index that addresses a table
  const unsigned cmax = (unsigned)p.ncell - 1u, qmax = (unsigned)p.nQ - 1u;
  Rec r;
  r.prev_cell = min((unsigned)o.prev_cell[k], cmax); r.cell = min((unsigned)o.cell[k], cmax);
  r.prev_q = min((unsigned)o.prev_q[k], qmax); r.q = min((unsigned)o.q[k], qmax);
  r.event = o.event[k] == RLRM_EVENT_NONE ? (unsigned)RLRM_EVENT_NONE : min((unsigned)o.event[k], (unsigned)max(p.nEv, 1) - 1u);
  r.env_term = o.env_term[k] != 0; r.renv = o.renv[k]; r.reward = o.reward[k];
  const size_t base = table_base(p_in, i, a);
  agent_update<ALGO, T>(p, tb, tab<T>(st.q) + base, st.visits ? st.visits + base : nullptr, min((unsigned)obs_cell[k], cmax),
                     min((int)actions[k], RLRM_N_ACTIONS - 1), term_arg[k] != 0, r, make_acc(p, st, base));
}

// QLearningLambda.update (qlearning_lambda.py:33-84), dense sweep exactly as written: one block per (instance, agent).
// q += (lr*td) * e ; e = terminated ? 0 : e * (gamma*lambda), with e[s,a] replaced by 1 first.
// one row (4 entries) of the dense sweep: q += c * e (float64 when lr = 1/visits), then e = terminated ? 0 : e * (gamma*lambda)
template <typename T>
__device__ __forceinline__ void sweep_row(const KP& p, typename RT<T>::row_t* Q4, typename RT<T>::row_t* E4, long long j, unsigned hot, T c,
                                          double c64, bool lr_none, bool terminated) {
  typedef RT<T> R;
  typename R::row_t e = E4[j], q = Q4[j];
  if ((unsigned)j == (hot >> 2)) set_component(e, hot & 3, (T)1);  // replacing trace
  if (lr_none) {
    q.x = R::cvt(__dadd_rn((double)q.x, __dmul_rn(c64, (double)e.x)));
    q.y = R::cvt(__dadd_rn((double)q.y, __dmul_rn(c64, (double)e.y)));
    q.z = R::cvt(__dadd_rn((double)q.z, __dmul_rn(c64, (double)e.z)));
    q.w = R::cvt(__dadd_rn((double)q.w, __dmul_rn(c64, (double)e.w)));
  } else {
    q.x = R::add(q.x, R::mul(c, e.x));
    q.y = R::add(q.y, R::mul(c, e.y));
    q.z = R::add(q.z, R::mul(c, e.z));
    q.w = R::add(q.w, R::mul(c, e.w));
  }
  if (terminated) {
    e = R::zero_row();
  } else {  // next_action defaults to argmax Q[s'] => greedy => decay (qlearning_lambda.py:71-81)
    const T d = R::decay(p);
    e.x = R::mul(e.x, d);
    e.y = R::mul(e.y, d);
    e.z = R::mul(e.z, d);
    e.w = R::mul(e.w, d);
  }
  Q4[j] = q;
  E4[j] = e;
}

template <typename T>
__device__ __forceinline__ void qlambda_sweep(const KP& p, T* Q, T* E, unsigned s, int a, double reward, unsigned sn,
                                              bool terminated, int tid, int nthreads, unsigned visits_now) {
  typedef RT<T> R;
  typedef typename R::row_t row_t;
  // every thread reads the two scalars before anyone writes
  const row_t nrow = load_row<T>(Q, sn);
  const T qsa = Q[s * 4 + a];
  __syncthreads();
  const double best = terminated ? 0.0 : (double)row_max(nrow);
  const T td = R::sub(R::cvt(__dadd_rn(reward, __dmul_rn(p.h.gamma, best))), qsa);
  const T c = R::mul(R::lr(p), td);
  const bool lr_none = p.h.lr < 0.0;  // lr = 1 / visits[s, a] (np.float64): the add happens in float64 (qlearning_lambda.py:44-49, 63)
  const double c64 = lr_none ? __dmul_rn(__ddiv_rn(1.0, (double)(visits_now ? visits_now : 1u)), (double)td) : 0.0;
  const unsigned hot = s * 4 + a;
  row_t* Q4 = reinterpret_cast<row_t*>(Q);
  row_t* E4 = reinterpret_cast<row_t*>(E);
  for (long long j = tid; j < p.S4 / 4; j += nthreads) sweep_row<T>(p, Q4, E4, j, hot, c, c64, lr_none, terminated);
}

template <typename T>
__global__ void __launch_bounds__(256) update_qlambda_kernel(KP p_in, DState st, const unsigned short* obs_cell,
                                                            const unsigned char* actions, const unsigned char* term_arg, DOut o, Sweep sw) {
  KP p = p_in;
  const long long k = blockIdx.x;
  const long long i = k / p.A;
  const int a = (int)(k - i * p.A);
  const size_t base = table_base(p_in, i, a);
  if (p_in.per_agent) {  // agent a's machine: its own state count and table size
    p.nQ = p_in.a_nQ[a];
    p.S4 = (long long)p_in.ncell * p.nQ * 4;
  }
  if (sw.hyp) apply_sweep(p, sw, i);
  // caller memory: clamp what indexes a table
  const unsigned cmax = (unsigned)p.ncell - 1u, qmax = (unsigned)p.nQ - 1u;
  const unsigned s_idx = min((unsigned)obs_cell[k], cmax) * p.nQ + min((unsigned)o.prev_q[k], qmax);
  const unsigned sn_idx = min((unsigned)o.cell[k], cmax) * p.nQ + min((unsigned)o.q[k], qmax);
  const int action = min((int)actions[k], RLRM_N_ACTIONS - 1);
  unsigned vis = 0;
  if (st.visits) {  // every thread reads the old count, then one writes the new one
    vis = st.visits[base + (size_t)s_idx * 4 + action] + 1;
    __syncthreads();
    if (threadIdx.x == 0) st.visits[base + (size_t)s_idx * 4 + action] = vis;
  }
  qlambda_sweep<T>(p, tab<T>(st.q) + base, tab<T>(st.e) + base, s_idx, action, o.reward[k], sn_idx, term_arg[k] != 0, threadIdx.x, blockDim.x, vis);
}


// QLearning.update's inner update_q (qlearning.py:70-79) / QLearningLambda.update (qlearning_lambda.py:33-84) applied to a LIST
// of experiences on one (instance, agent) table, in list order, in one launch: the QRM counterfactual loop of
// QLearning.update (qlearning.py:82-106) hands its experiences over as one list instead of one launch per experience.
// Q-learning / QRM: thread 0 applies them one after the other (each update may read what the previous one wrote);
// Q(lambda): the whole block sweeps the table once per experience.
struct SelArgs {  // the input half of rlrm_select_req_t, passed by value (read on the host at call time)
  unsigned state, best;
  double epsilon;
  unsigned draws[4];
  unsigned seq;
};
template <typename T, bool SOFTMAX>  // SOFTMAX: the selection is softmax exploration with beta = 1 / temperature (see train_kernel)
__global__ void __launch_bounds__(256) update_list_kernel(KP p, DState st, long long slot, int n, const rlrm_experience_t* ex,
                                                         rlrm_select_req_t* sel, SelArgs sa, Sweep sw, double beta) {
  const long long i = slot / p.A;
  const int a = (int)(slot - i * p.A);
  KP pl = p;  // the slot's learner settings (a sweep handle's group); p itself stays in the constant bank
  if (sw.hyp) apply_sweep(pl, sw, i);
  const size_t base = table_base(p, i, a);
  const unsigned rows = (unsigned)p.ncell * (unsigned)(p.per_agent ? p.a_nQ[a] : p.nQ);
  T* Q = tab<T>(st.q) + base;
  unsigned* V = st.visits ? st.visits + base : nullptr;
  if (p.algo == RLRM_ALGO_QLAMBDA) {
    KP pa = pl;
    pa.S4 = (long long)rows * 4;
    T* E = tab<T>(st.e) + base;
    for (int j = 0; j < n; j++) {
      const unsigned s = min(ex[j].s, rows - 1u), sn = min(ex[j].sn, rows - 1u);  // caller memory: clamp what indexes a table
      const int act = min((int)ex[j].action, RLRM_N_ACTIONS - 1);
      unsigned vis = 0;
      if (V) {  // every thread reads the old count, then one writes the new one
        vis = V[(size_t)s * 4 + act] + 1;
        __syncthreads();
        if (threadIdx.x == 0) V[(size_t)s * 4 + act] = vis;
      }
      qlambda_sweep<T>(pa, Q, E, s, act, ex[j].reward, sn, ex[j].terminated != 0, threadIdx.x, blockDim.x, vis);
      __syncthreads();
    }
  } else if (threadIdx.x == 0) {
    const Acc none = {nullptr, nullptr, nullptr, false, nullptr};
    for (int j = 0; j < n; j++)
      update_q<T>(pl, Q, V, min(ex[j].s, rows - 1u), min((int)ex[j].action, RLRM_N_ACTIONS - 1), ex[j].reward, min(ex[j].sn, rows - 1u),
                  ex[j].terminated != 0, none);
  }
  // rlrm_update_list_select: the next selection on the updated table (thread 0 is also the thread that wrote the QL / QRM
  // updates; the Q(lambda) sweeps ended with a block barrier)
  if (sel && threadIdx.x == 0) {
    const unsigned w[4] = {sa.draws[0], sa.draws[1], sa.draws[2], sa.draws[3]};
    const typename RT<T>::row_t row = load_row<T>(Q, min(sa.state, rows - 1u));
    *reinterpret_cast<volatile unsigned*>(&sel->action) =
        (unsigned)(SOFTMAX ? select_softmax(row, w[1], beta, sa.best != 0, p.n_actions)
                           : select_action(row, explore_threshold(sa.epsilon), w, sa.best != 0, p.n_actions));
    __threadfence_system();
    *reinterpret_cast<volatile unsigned*>(&sel->done_seq) = sa.seq;
  }
}

// Shared learner, inter-GPU merge (include/rlrm_b200.h "Shared learner"): q <- (g_0 + g_1 + ... + g_{world-1}) / world with the
// replicas added in RANK ORDER, so every rank computes the same bits whatever the collective that gathered them did.
__global__ void __launch_bounds__(256) merge_replicas_kernel(const float* gathered, int world, long long n, float* q) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  float acc = gathered[j];
  for (int r = 1; r < world; r++) acc = __fadd_rn(acc, gathered[(size_t)r * (size_t)n + j]);
  q[j] = __fdiv_rn(acc, (float)world);
}

// MEASUREMENT AID (bench.py's roofline block; not on the hot path): what the memory system delivers for the ACCESS PATTERN of the
// per-instance-table kernels — independent gathers of random, aligned 16 / 32 / 64-byte blocks spread over a resident table,
// optionally each followed by a 4-byte store into the block (the Q-learning write-back). Every thread keeps UNROLL independent
// gathers in flight (far more memory-level parallelism than a serial agent chain has), so the result is the pattern's ceiling.
template <int VEC>  // 16-byte vectors per block
__global__ void __launch_bounds__(256) probe_gather_kernel(uint4* tab, unsigned long long n_blocks, int per_thread, unsigned seed, int write,
                                                          unsigned* sink) {
  constexpr int UNROLL = 8;
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long x = (tid + 1) * 0x9E3779B97F4A7C15ull ^ ((unsigned long long)seed << 32);
  unsigned acc = 0;
  for (int k = 0; k < per_thread; k += UNROLL) {
    unsigned long long idx[UNROLL];
#pragma unroll
    for (int j = 0; j < UNROLL; j++) {
      x ^= x << 13; x ^= x >> 7; x ^= x << 17;  // xorshift64
      idx[j] = __umul64hi(x, n_blocks);
    }
    uint4 v[UNROLL][VEC];
#pragma unroll
    for (int j = 0; j < UNROLL; j++)
#pragma unroll
      for (int c = 0; c < VEC; c++) v[j][c] = tab[idx[j] * VEC + c];
#pragma unroll
    for (int j = 0; j < UNROLL; j++) {
#pragma unroll
      for (int c = 0; c < VEC; c++) acc += v[j][c].x ^ v[j][c].y ^ v[j][c].z ^ v[j][c].w;
      if (write) reinterpret_cast<unsigned*>(tab + idx[j] * VEC)[(acc >> 3) & (4 * VEC - 1)] = v[j][0].x;  // rewrites a value it just read: contents stay valid floats
    }
  }
  if (acc == 0x12345678u) sink[0] = acc;  // keeps the loads alive
}
