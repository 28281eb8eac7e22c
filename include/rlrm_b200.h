/*
 * rlrm_b200.h — C ABI of the B200-native lockstep hot path of multiagent-rl-rm
 * (grid-world transition -> event label -> Reward Machine transition -> tabular Q / QRM / Q(lambda) update)
 * over large batches of independent environment instances.
 *
 * The reference (Alee08/multiagent-rl-rm v0.3.0) is pure Python and has no FFI layer; each entry point
 * below names the reference Python interface it replaces (R/ = multiagent_rlrm/ in the reference tree).
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C, plain pointers and sizes; no torch / C++ types in any signature
 *   - every pointer inside rlrm_state_t / rlrm_step_out_t is a DEVICE pointer owned by the caller
 *     (the Python host layer allocates them as torch tensors); the library never frees them
 *   - rlrm_tables_t holds HOST pointers; rlrm_create copies those small tables to the device once
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream)
 *   - all functions return 0 on success, <0 on error (rlrm_last_error() gives the message); they never throw
 *   - there is no CPU fallback: without a CUDA device rlrm_create fails with RLRM_ERR_CUDA
 *
 * Indexing
 *   instance i in [0,N), agent a in [0,A), slot = i*A + a
 *   cell = y*W + x                                     (R/environments/frozen_lake/state_encoder_frozen_lake.py:32)
 *   enc  = cell*nQ + q                                 (same file :35; office: state_encoder_office.py:23-24)
 *   Q[slot][enc][action] fp32, action order 0 up, 1 down, 2 left, 3 right
 *                                                      (R/environments/frozen_lake/action_encoder_frozen_lake.py:14-17)
 */
#ifndef RLRM_B200_H
#define RLRM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RLRM_ABI_VERSION 2

#define RLRM_MAX_AGENTS 8      /* agents per instance (lane group = next power of two) */
#define RLRM_MAX_CELLS 1024    /* W*H */
#define RLRM_MAX_RM_STATES 32
#define RLRM_MAX_EVENTS 63     /* distinct detector positions; column nEv of delta is the "None" event */
#define RLRM_N_ACTIONS 4
#define RLRM_ACTION_WAIT 4
#define RLRM_EVENT_NONE 255    /* label value: position is not in the event detector's set */
#define RLRM_NO_TRANSITION 255 /* delta value: (q, event) not in RewardMachine.transitions */

/* error codes */
#define RLRM_OK 0
#define RLRM_ERR_ARG (-1)
#define RLRM_ERR_CUDA (-2)
#define RLRM_ERR_UNSUPPORTED (-3)

/* environments: R/environments/frozen_lake/ma_frozen_lake.py, R/environments/office_world/ma_office.py */
#define RLRM_ENV_FROZEN_LAKE 0
#define RLRM_ENV_OFFICE_WORLD 1

/* learners: R/learning_algorithms/qlearning.py (use_qrm False/True), qlearning_lambda.py */
#define RLRM_ALGO_QL 0
#define RLRM_ALGO_QRM 1
#define RLRM_ALGO_QLAMBDA 2

/* table arithmetic type. The reference keeps q_table / e_table / visits in float64 (np.zeros default: qlearning.py:26-29,
 * qlearning_lambda.py:26-30). RLRM_TABLE_F64 is that arithmetic, bit for bit; RLRM_TABLE_F32 is what NumPy computes once the
 * tables are cast to float32 (half the HBM bytes; the specialised kernels exist for this type only). */
#define RLRM_TABLE_F32 0
#define RLRM_TABLE_F64 1

/* episode-loop semantics: R/environments/frozen_lake/frozen_lake_main.py:336-376,
 * R/environments/office_world/office_main.py:1696-1749 */
#define RLRM_DRIVER_FROZEN_LAKE_MAIN 0
#define RLRM_DRIVER_OFFICE_MAIN 1

/* rlrm_state_t.slot packing: one 64-bit word per (instance, agent) */
#define RLRM_SLOT_CELL_SHIFT 0       /* 16 bits: y*W + x */
#define RLRM_SLOT_STEPS_SHIFT 16     /* 16 bits: env.agent_steps[agent] */
#define RLRM_SLOT_TIME_SHIFT 32      /* 16 bits: env.timestep (replicated in every agent of the instance) */
#define RLRM_SLOT_RMSTATE_SHIFT 48   /*  8 bits: RewardMachine.current_state as index */
#define RLRM_SLOT_FLAGS_SHIFT 56     /*  8 bits: RLRM_FLAG_* */
#define RLRM_FLAG_ACTIVE 1u          /* env.active_agents[agent] */
#define RLRM_FLAG_FAIL 2u            /* env.agent_fail[agent] */
#define RLRM_FLAG_DONE 4u            /* last wrapper `terminations[agent]` */
#define RLRM_FLAG_TRUNC 8u           /* last `truncations[agent]` */
#define RLRM_FLAG_FIRST 16u          /* no step since reset: the FrozenLake driver's `states` still alias agent.state */

typedef struct rlrm_config {
  int32_t abi_version;  /* RLRM_ABI_VERSION */
  int32_t env_kind;     /* RLRM_ENV_* */
  int32_t driver;       /* RLRM_DRIVER_* */
  int32_t algo;         /* RLRM_ALGO_* */
  int32_t width, height;
  int32_t n_agents;     /* A */
  int32_t n_rm_states;  /* nQ = RewardMachine.numbers_state() (reward_machine.py:130-138) */
  int32_t n_events;     /* nEv = number of detector positions with an event id */
  int32_t rm_final;     /* index of RewardMachine.get_final_state() (reward_machine.py:152-163), -1 if none */
  int32_t n_qrm_states; /* len(get_all_states()[:-1]) (rm_environment_wrapper.py:144) */
  int32_t max_steps;    /* 1000: `> 1000` tests in ma_frozen_lake.py:202 / ma_office.py:254 */
  /* dynamics */
  int32_t stochastic;          /* env.frozen_lake_stochastic / env.stochastic */
  int32_t slip_n;              /* outcomes per intended action (3 or 4); 1 when deterministic */
  uint64_t slip_thr[3];        /* draw k (u32) falls in outcome j = #{T in slip_thr[0..slip_n-2] : k >= T};
                                  T = ceil(cdf_j * 2^32) of numpy Generator.choice(p=...) */
  uint8_t slip_outcome[4][4];  /* [intended action][j] -> executed action (0..3) or RLRM_ACTION_WAIT */
  int32_t terminate_on_plants; /* office only (ma_office.py:217) */
  int32_t terminate_hit_walls; /* office only (ma_office.py:322) */
  double hole_penalty;         /* env.penalty_amount (ma_frozen_lake.py:185) / env.plants_penalty_value (ma_office.py:219) */
  double wall_penalty;         /* env.wall_penalty_value (ma_office.py:324); 0 for FrozenLake */
  /* learner (qlearning.py:9-39, qlearning_lambda.py:6-31) */
  double learning_rate;        /* < 0: None => 1/visits (needs rlrm_state_t.visits) */
  double gamma;
  double lambd;
  double epsilon_start, epsilon_end, epsilon_decay;
  int32_t decay_on_reset;      /* 1: env.reset() calls learn_done_episode() (isinstance QLearning; false for Q(lambda)) */
  int32_t shared_q;            /* 0: one table per (instance, agent); 1: one per agent index shared by all instances */
  /* randomness: Philox4x32-10, key = (seed_lo, seed_hi), counter = (t_lo, t_hi, instance_offset + i, a) */
  uint32_t seed_lo, seed_hi;
  uint32_t instance_offset;    /* global id of local instance 0 (multi-GPU sharding keeps draws independent of G) */
  /* Agents with different reward machines (frozen_lake_main.py --rm-spec-a1 / --rm-spec-a2). per_agent_rm = 1: n_rm_states
   * and n_qrm_states are the MAXIMA over the agents (= the row strides of the tables below), every table of rlrm_tables_t
   * that depends on the machine has one section per agent, label included:
   *   label [A][W*H], delta / rq / rcf [A][nQmax][nEv+1], qrm_states [A][nQmax], phi [A][2][nQmax]
   * and agent a uses its own nQ_a for the state encoding, so its table holds W*H*agent_n_rm_states[a] rows; the tables of one
   * instance are concatenated in agent order: Q offset of (i, a) = (i * sum_b S_b + sum_{b<a} S_b) * 4. */
  int32_t per_agent_rm;
  int32_t agent_n_rm_states[RLRM_MAX_AGENTS];
  int32_t agent_rm_final[RLRM_MAX_AGENTS];
  int32_t agent_n_qrm[RLRM_MAX_AGENTS];
  int32_t random_starts;       /* env.random_start_positions (ma_frozen_lake.py:63-64, 156-172): on every reset the agents are
                                  placed on distinct free cells. Sampling (this repo's injection-consistent scheme): partial
                                  Fisher-Yates over tables.free_cells, pick k uses word (k & 3) of
                                  philox(counter = (T_lo, ~T_hi, instance, 0x80000000 | k >> 2)), j = k + ((w * (F - k)) >> 32),
                                  T = iteration index of the new episode's first step */
  int32_t n_free_cells;        /* F */
  int32_t use_rsh;             /* QLearning.use_rsh: potential-based shaping R' = R + gamma*Phi(q') - Phi(q) (qlearning.py:51-66, 93-105) */
  int32_t n_actions;           /* 1..4 usable actions (exploration draws (w1*n_actions)>>32); tables are always 4 wide */
  int32_t reserved;            /* testing switches (paths that must agree bit for bit): bit 0 forces the generic kernels, bit 1 forces the
                                  shared learner's two-launches-per-iteration path instead of the persistent cooperative kernel, bit 2
                                  forces its thread-block-cluster variant (tables partitioned over distributed shared memory) even
                                  when the tables fit in one SM */
  int32_t table_dtype;         /* RLRM_TABLE_F32 / RLRM_TABLE_F64: element type of rlrm_state_t.q / e / tr_eq */
} rlrm_config_t;

/* host pointers; copied at rlrm_create */
typedef struct rlrm_tables {
  const uint16_t* next_cell;  /* [W*H][4] cell reached by action a, == cell when blocked (bounds, office walls)
                                 (ma_frozen_lake.py:224-242; ma_office.py:269-289 + config_office.py:12-39) */
  const uint8_t* cell_flags;  /* [W*H] bit0: hole (FrozenLake) / plant (OfficeWorld) */
  const uint8_t* label;       /* [W*H] event id of the position, RLRM_EVENT_NONE otherwise (detect_event.py:18-33) */
  const uint8_t* delta;       /* [nQ][nEv+1] next RM state index, RLRM_NO_TRANSITION = stay, reward 0 (reward_machine.py:45-59) */
  const double* rq;           /* [nQ][nEv+1] transition reward * wrapper.reward_modifier (rm_environment_wrapper.py:65-69) */
  const double* rcf;          /* [nQ][nEv+1] transition reward for QRM counterfactuals (unscaled, :150-153) */
  const uint8_t* qrm_states;  /* [n_qrm_states] RM state indices, in get_all_states()[:-1] order */
  const uint16_t* start_cell; /* [A] agent.initial_position */
  const uint16_t* free_cells; /* [F] cells that are not holes, enumerated x-major (for x: for y) as ma_frozen_lake.py:163-168; may be NULL
                                 when random_starts == 0 */
  const double* phi;          /* [2][nQ] RewardMachine.potentials (reward_machine.py:197-237); NULL = no shaping.
                                 row 0: Phi of the state with index i — used by the QRM counterfactual loop, which maps
                                        indices back to labels (qlearning.py:100-104);
                                 row 1: potentials.get(i, 0) with the INTEGER i as dict key — what the plain-QL branch
                                        evaluates, because AgentRL.update_policy hands it indices (agent_rl.py:158-172,
                                        qlearning.py:60-65): all zeros unless the RM's state labels are integers */
} rlrm_tables_t;

/* per-(instance, agent) episode statistics, 32 bytes */
typedef struct rlrm_stats {
  uint64_t active_steps;  /* sum of env.agent_steps over FINISHED episodes; add the slot's current agent_steps for the
                             running total of active agent-steps (the headline unit) */
  uint32_t episodes;      /* episodes finished */
  uint32_t successes;     /* episodes that ended with the RM in its final state */
  double return_sum;      /* sum over finished episodes of the undiscounted episode return */
  float last_return;      /* return of the last finished episode */
  uint32_t last_length;   /* env.timestep at the end of the last finished episode */
} rlrm_stats_t;

/* per-(instance, agent) greedy-evaluation bookkeeping, 72 bytes (rlrm_evaluate) */
typedef struct rlrm_eval {
  double cum_gamma;      /* running gamma^t of the current episode (starts at 1) */
  double disc_return;    /* running sum of cum_gamma * reward until the agent succeeds */
  double return_sum;     /* over finished episodes: sum of disc_return, its squares, and of (disc_return/steps)/optimal_steps */
  double return_sqsum;
  double arps_sum;
  uint64_t len_sum;      /* over SUCCESSFUL episodes: sum of episode lengths and of their squares */
  uint64_t len_sqsum;
  uint32_t episodes;     /* evaluation episodes finished */
  uint32_t successes;    /* episodes in which this agent reached the final RM state */
  uint32_t in_success;   /* the agent already succeeded in the current episode */
  uint32_t reserved;
} rlrm_eval_t;

/* device pointers, caller-owned */
typedef struct rlrm_state {
  int64_t n_instances;  /* N (local to this GPU) */
  uint64_t* slot;       /* [N*A] packed env + RM state, see RLRM_SLOT_* */
  double* epsilon;      /* [N*A] learner.epsilon */
  void* q;              /* [N*A*S*4] (shared_q: [A*S*4]) learner.q_table, S = W*H*nQ; float (RLRM_TABLE_F32) or double
                           (RLRM_TABLE_F64). Must be 32-byte aligned (cudaMalloc and torch allocations are): rows are read with
                           16- and 32-byte vector loads. e: same alignment; visits: 16-byte aligned. */
  void* e;              /* Q(lambda) only: learner.e_table, same shape and element type as q; else NULL */
  uint32_t* visits;     /* optional [same shape as q]: learner.visits; required when learning_rate < 0 */
  double* ep_return;    /* [N*A] running (undiscounted) return of the current episode */
  rlrm_stats_t* stats;  /* [N*A] or NULL */
  /* shared_q only (one table per agent index, every instance on this GPU learns into it): per-iteration proposal
   * accumulators, each [A*S*4], zero-initialised by the caller. See "shared learner" below. */
  int64_t* acc_sum;     /* sum of round(new_value * 2^20) over the instances that updated the entry this iteration */
  int32_t* acc_cnt;     /* number of such instances */
  float* acc_last;      /* the new value itself (used verbatim when acc_cnt == 1) */
  /* Q(lambda) sparse-exact traces (optional; give these INSTEAD of `e`). The reference sweeps the whole table every step
   * (q += lr*td*e ; e *= gamma*lambda, qlearning_lambda.py:63,81); entries whose trace is 0 receive +0, so only the
   * entries with a live trace need touching. Each (instance, agent) keeps a list of its live entries holding the trace
   * AND the current q value (the table copy of a listed entry is stale until the list is flushed, which happens when
   * the traces are wiped: terminated update or reset). Results equal the dense sweep bit for bit (up to the sign of
   * zero). rlrm_qlambda_materialize writes the listed values back so `q` can be read. Needs S*4 <= 65535. */
  uint16_t* tr_pos;     /* [N*A][S*4] 0 = entry not listed, else list position + 1 */
  uint16_t* tr_idx;     /* [N*A][tr_cap] listed entry index = enc*4 + action */
  void* tr_eq;          /* [N*A][tr_cap][2] its (trace, current q value), interleaved (element type of q): one 8-byte
                           (float) or 16-byte (double) access per entry */
  uint32_t* tr_len;     /* [N*A] list length */
  uint64_t* tr_work;    /* [N*A] or NULL: sum over update steps of the list length swept (bench: mean live traces) */
  int32_t tr_cap;       /* list capacity; must be >= max_steps + 1 (one new entry per step, wiped every episode) */
  int32_t tr_reserved;
} rlrm_state_t;

/* device pointers, caller-owned, each [N*A]; any may be NULL (not written) */
typedef struct rlrm_step_out {
  uint16_t* prev_cell;  /* infos[agent]["prev_s"] as cell index */
  uint16_t* cell;       /* observations[agent] / infos["s"] */
  uint8_t* prev_q;      /* infos["prev_q"] as index */
  uint8_t* q;           /* infos["q"] as index */
  uint8_t* event;       /* event id detected on the new position, RLRM_EVENT_NONE if none */
  uint8_t* executed;    /* action actually executed after slip / wall (0..3, RLRM_ACTION_WAIT), 5 = agent skipped */
  double* renv;         /* infos["Renv"] */
  double* rq;           /* infos["RQ"] */
  double* reward;       /* rewards[agent] = Renv + RQ */
  uint8_t* env_term;    /* infos["env_terminated"] */
  uint8_t* rm_term;     /* infos["rm_terminated"] */
  uint8_t* term;        /* terminations[agent] */
  uint8_t* trunc;       /* truncations[agent] */
  /* optional, rlrm_step only: the hypothetical Reward-Machine transitions _get_qrm_experiences evaluates on the NEW position
   * (rm_environment_wrapper.py:144-153), for every state u of get_all_states()[:-1] in that order (tables.qrm_states):
   * [N*A][n_qrm_states] next RM state index (u itself when (u, event) has no transition) and its reward (0 then; unscaled
   * by reward_modifier, as the reference). Rows of agents with fewer states (per_agent_rm) are padded. */
  uint8_t* cf_q;
  double* cf_r;
} rlrm_step_out_t;

typedef struct rlrm_handle rlrm_handle_t;

/* library / device */
int rlrm_abi_version(void);
const char* rlrm_last_error(void);
int rlrm_device_count(void);

/* Builds the device-side constant block for one configuration on CUDA device `device`.
 * Replaces object construction in frozen_lake_main.py:200-295 / office_main.py:400-717 (env, RM, encoder, learner). */
int rlrm_create(const rlrm_config_t* cfg, const rlrm_tables_t* tables, int device, rlrm_handle_t** out);
int rlrm_destroy(rlrm_handle_t* h);
/* learner hyper-parameters may be changed between calls (the reference mutates attributes in place) */
int rlrm_set_learner(rlrm_handle_t* h, double learning_rate, double gamma, double lambd);

/* Hyper-parameter sweep: one learner setting for every contiguous group of group_size instances. Instance i (global id
 * cfg.instance_offset + i, the id the random draws are keyed on) trains with sets[(instance_offset + i) / group_size] and behaves
 * bit for bit as instance i of a handle created with that setting. epsilon_start is not here: epsilon is per slot state.
 * n_sets == 0 clears the sweep. RLRM_ERR_UNSUPPORTED on a shared_q handle; RLRM_ERR_ARG for group_size <= 0, and at launch for
 * a setting with learning_rate < 0 (None) without state.visits or for instances not covered by n_sets * group_size.
 * rlrm_set_learner fails on a handle with a sweep. */
typedef struct rlrm_hyper {
  double learning_rate; /* < 0: None (1 / visits) */
  double gamma, lambd, epsilon_end, epsilon_decay;
} rlrm_hyper_t;
int rlrm_set_sweep(rlrm_handle_t* h, const rlrm_hyper_t* sets, int32_t n_sets, int64_t group_size);

/* Exploration of the selections rlrm_train, rlrm_iterate, rlrm_select_action and rlrm_update_list_select make (best == 0 /
 * learn != 0; greedy evaluation stays the first argmax). RLRM_EXPLORE_EPSILON_GREEDY (the default) is QLearning.choose_action.
 * RLRM_EXPLORE_SOFTMAX with temperature tau > 0 and beta = 1.0 / tau (double) selects, for one slot with row Q[0..n-1],
 * n = cfg.n_actions, Q float or double as the table is:
 *   1. m = max Q[0..n-1]; d_a = ((double)Q[a] - (double)m) * beta; w_a = E(d_a), so d_a <= 0 and E(0) = 1.0;
 *   2. C_j = C_{j-1} + w_j in action order (C_0 = w_0), total = C_{n-1};
 *   3. T_j = (uint64_t)ceil(C_j / total * 2^32) for j < n - 1; action = #{ j < n - 1 : w1 >= T_j }
 * with every operation a round-to-nearest double operation (no contraction) and w1 the second word of the iteration's Philox
 * draw (rlrm_select_action's draws[4k + 1]; w3 keeps its slip role, w0 and w2 are unused). E(x), x <= 0, is a fixed operation
 * sequence (rlrm_exp in the sources): +0 below ln(2^-1075); k = rint(x * log2e); r = fma(-k, ln2_hi, x), r = fma(-k, ln2_lo, r);
 * the degree-14 Taylor polynomial of exp(r) by Horner's rule with fma; times 2^k built from its bits (2^(k+54), then 2^-54, when
 * k < -1021).
 * The constants are in csrc/rlrm_device.cuh and, restated, in tests/softmax_oracle.c. It is within 2 ULP of a correctly rounded exp.
 * Actions whose weight underflows to 0 are never chosen. epsilon is still carried and decayed per slot, but not read.
 * RLRM_ERR_ARG for an unknown kind, or a softmax temperature that is not finite, not > 0 or whose reciprocal overflows;
 * RLRM_ERR_UNSUPPORTED on a shared_q handle. Softmax launches take the generic training kernel (or the Q(lambda) kernels);
 * kind = RLRM_EXPLORE_EPSILON_GREEDY restores the epsilon-greedy handle exactly, specialised kernels included. */
#define RLRM_EXPLORE_EPSILON_GREEDY 0
#define RLRM_EXPLORE_SOFTMAX 1
int rlrm_set_exploration(rlrm_handle_t* h, int32_t kind, double temperature);

/* RMEnvironmentWrapper.reset (rm_environment_wrapper.py:28-41) -> env.reset (ma_frozen_lake.py:43-94,
 * ma_office.py:77-120): positions, RM state, counters, epsilon decay, Q(lambda) trace wipe.
 * mask: device uint8 [N] selecting instances, or NULL for all. */
int rlrm_reset(rlrm_handle_t* h, const rlrm_state_t* st, const uint8_t* mask, void* stream);
/* Same with the iteration index `t` of the next step, which keys the random start positions (cfg.random_starts);
 * rlrm_reset is rlrm_reset_at with t = 0. The fused kernels use t + 1 of the iteration that ended the episode. */
int rlrm_reset_at(rlrm_handle_t* h, const rlrm_state_t* st, const uint8_t* mask, uint64_t t, void* stream);

/* AgentRL.select_action (agent_rl.py:80-106) -> QLearning.choose_action (qlearning.py:112-143).
 * draws: device uint32 [N*A*4] injected Philox words (w0 explore, w1 random action, w2 tie-break, w3 slip)
 * or NULL to generate them in-kernel for lockstep iteration t. best != 0: argmax, no randomness. */
int rlrm_select_action(rlrm_handle_t* h, const rlrm_state_t* st, const uint32_t* draws, uint64_t t, int best,
                       uint8_t* actions_out, void* stream);

/* RMEnvironmentWrapper.step (rm_environment_wrapper.py:43-107): env.step (ma_frozen_lake.py:96-154 /
 * ma_office.py:122-202) + RewardMachine.step (reward_machine.py:45-59) per agent + reward / termination merge.
 * actions: device uint8 [N*A], 0..3 or RLRM_ACTION_WAIT (env.wait_action; larger values are treated as wait).
 * with_rm == 0 runs the bare env.step (RM state is read for FrozenLake's rm_done test but not advanced).
 * Robustness contract of the call-by-call entry points: indices read from caller memory (actions, cells, RM states,
 * step records) are clamped to the table they address, so garbage in gives garbage out but never an out-of-bounds
 * access; slot words are only ever produced by rlrm_reset / rlrm_step / rlrm_train and are trusted. */
int rlrm_step(rlrm_handle_t* h, const rlrm_state_t* st, const uint8_t* actions, const uint32_t* draws, uint64_t t,
              int with_rm, const rlrm_step_out_t* out, void* stream);

/* RewardMachine.step (reward_machine.py:45-59) on explicit positions: q[N*A] in/out, cell[N*A] in, reward[N*A] out */
int rlrm_rm_step(rlrm_handle_t* h, int64_t n_slots, uint8_t* q, const uint16_t* cell, uint8_t* event_out,
                 double* reward_out, void* stream);
/* Same on the reward machine of agent `agent` (per_agent_rm configurations; rlrm_rm_step uses agent 0's machine). */
int rlrm_rm_step_agent(rlrm_handle_t* h, int agent, int64_t n_slots, uint8_t* q, const uint16_t* cell, uint8_t* event_out,
                       double* reward_out, void* stream);

/* RMEnvironmentWrapper.get_mdp (rm_environment_wrapper.py:185-283): the product MDP of agent `agent` (grid cell x RM
 * state), every (encoded state s, nominal action a, sub-action j) in one launch. The reference builds it with
 * reset(seed) + env.set_state + one step per triple with env.stochastic forced to False, so each sub-action is executed
 * as is (a blocked OfficeWorld move still becomes "wait" + wall penalty, ma_office.py:311-325).
 * sub_actions: HOST uint8 [4][n_sub], the sub-action lists of get_action_distribution (ma_frozen_lake.py:337-351,
 * ma_office.py:434-453) as action indices, RLRM_ACTION_WAIT allowed; n_sub in 1..4.
 * rm_terminal: treat "RM state == final state" as terminal (is_terminal_state_mdp, ma_office.py:424-428).
 * Outputs, device, index (s*4 + a)*n_sub + j with S = width*height*n_rm_states(agent):
 *   next_state int32 (encoded), reward f64 (env + RM reward * reward_modifier), done u8 (terminated or truncated);
 *   terminal u8 [S]: 0 = not terminal, 1 = hazard cell (hole / terminating plant), 2 = RM final state. Terminal states
 *   self-loop with the terminal reward (hole / plant penalty, or 0) in every (a, j) entry. */
int rlrm_mdp(rlrm_handle_t* h, int agent, int n_sub, const uint8_t* sub_actions, int rm_terminal, int32_t* next_state,
             double* reward, uint8_t* done, uint8_t* terminal, void* stream);

/* mdp_vi.value_iteration (environments/utils_envs/mdp_vi.py:9-60) on the transition model get_mdp / rlrm_mdp produce, as padded
 * outcome arrays (device): prob / next_state / reward / done are [n_states][4][n_outcomes], outcome order = list order of
 * P[s][a], unused slots have prob 0. V starts at 0; a sweep sets Q[s][a] = sum prob * (reward + gamma * V[s'] * !done) and
 * V[s] = max_a Q[s][a]; sweeps repeat until max_s |V_new[s] - V_old[s]| (divided by max(|V_new[s]|, 1e-12 -> 1) when
 * delta_rel) < theta. The reference updates V in place while sweeping (Gauss-Seidel), this kernel sweeps all states in
 * parallel from the previous V (Jacobi): same fixed point and stopping rule, so V agrees within 2*theta*gamma/(1-gamma), not
 * bit for bit; policy[s] = first argmax of the final Q[s]. Outputs (device): V f64 [n_states], Q f64 [n_states][4], policy
 * int32 [n_states]. work: device scratch of n_states + 1 doubles. sweeps_out (host, may be NULL) = sweeps performed.
 * Needs no handle (the model is self-contained): `device` is the CUDA device the arrays live on. Synchronous (one 8-byte
 * read-back per sweep). RLRM_ERR_UNSUPPORTED when max_sweeps is reached. */
int rlrm_value_iteration(int device, int64_t n_states, int n_outcomes, const double* prob, const int32_t* next_state,
                         const double* reward, const uint8_t* done, double gamma, double theta, int delta_rel, int max_sweeps,
                         double* V, double* Q, int32_t* policy, double* work, int32_t* sweeps_out, void* stream);

/* AgentRL.update_policy (agent_rl.py:117-192) -> QLearning.update (qlearning.py:41-110, incl. the QRM
 * counterfactual loop fed by rm_environment_wrapper.py:122-183) or QLearningLambda.update (qlearning_lambda.py:33-84).
 * obs_cell: device uint16 [N*A], the `state` argument the driver passes (previous observation);
 * term_arg: device uint8 [N*A], the `terminated` argument the driver passes. `out` is the record rlrm_step wrote. */
int rlrm_update(rlrm_handle_t* h, const rlrm_state_t* st, const uint16_t* obs_cell, const uint8_t* actions,
                const uint8_t* term_arg, const rlrm_step_out_t* out, void* stream);

/* Shared learner (cfg.shared_q = 1; BASELINE config 5). The reference has no shared learner, so the merge rule is
 * specified here: iterations are synchronous. Within one lockstep iteration every instance selects and computes its
 * update_q result ("proposal") against the SAME table snapshot; afterwards each touched entry becomes the mean of its
 * proposals: Q[s,a] = proposal if one instance proposed, else (float)((double)acc_sum / acc_cnt * 2^-20). Sums are
 * integers, so the result does not depend on thread order or on how instances are spread over blocks/GPUs.
 * With a single instance this is exactly the per-instance learner (for reward machines whose counterfactual updates
 * do not read each other's writes, e.g. chains). rlrm_train runs all n_iters iterations of this mode in ONE persistent
 * cooperative launch (tables and proposal accumulators in shared memory, one grid barrier per iteration; tables too large for
 * one SM's 227 KB are partitioned over the distributed shared memory of a thread-block cluster of 2 / 4 / 8 blocks); with a
 * trace buffer, learn = 0 or tables beyond 8 x 227 KB it falls back to two launches per iteration.
 * Visit counts (state.visits) of a shared table are shared too: each entry counts every proposal made to it, by all
 * instances, in every iteration.
 * Inter-GPU merging (every K iterations) is the caller's step: average the replicas of `q` (dist.merge_replicas gathers
 * them over NCCL and sums in rank order, so the result does not depend on the collective's reduction order). */

/* One launch = n_iters lockstep iterations of the driver loop (select for all agents -> wrapper step -> update for
 * all agents -> per-instance auto reset when the episode ends), state in registers, Philox draws for iterations
 * t0 .. t0+n_iters-1. Replaces the while-loop body of frozen_lake_main.py:345-376 / office_main.py:1709-1749.
 * trace (optional, device): uint32 [n_iters][N*A] packed per-iteration record for replay through the oracle:
 *   bits 0-2 action, 3-5 executed, 6-15 cell after, 16-20 rm state after, 21 term, 22 trunc, 23 active-step. */
int rlrm_train(rlrm_handle_t* h, const rlrm_state_t* st, uint64_t t0, int32_t n_iters, int32_t learn,
               uint32_t* trace, void* stream);

/* ONE lockstep iteration of the driver loop, at the reference's call granularity but in a single launch: select_action for
 * every agent -> rm_env.step -> update_policy for every agent -> rm_env.reset of the instances whose episode ended (the
 * while-loop body of frozen_lake_main.py:345-376 / office_main.py:1709-1749). It is rlrm_train with n_iters = 1 that also
 * reports what rm_env.step returned for this iteration:
 *   record [N*A] uint32, the packed step record described at rlrm_train (action, executed action, new cell, new RM state,
 *          terminated, truncated, active-step);
 *   reward [N*A] double, rewards[agent] = Renv + RQ (rm_environment_wrapper.py:85), or NULL.
 * Both may point to page-locked HOST memory (cudaHostAlloc / torch pin_memory: device-accessible under unified addressing):
 * the kernel then writes the record straight into the caller's buffer and a host loop costs one launch + one stream
 * synchronisation per iteration. Results are bit-identical to the same iteration of rlrm_train. */
int rlrm_iterate(rlrm_handle_t* h, const rlrm_state_t* st, uint64_t t, int32_t learn, uint32_t* record, double* reward,
                 void* stream);

/* One entry of QLearning.update's counterfactual list (qlearning.py:82-106; the tuples built by
 * rm_environment_wrapper.py:155-173) or one plain update (qlearning.py:108 / qlearning_lambda.py:33-84). 24 bytes. */
typedef struct rlrm_experience {
  uint32_t s;          /* encoded state  (enc = cell*nQ + q) */
  uint32_t sn;         /* encoded next state */
  uint8_t action;      /* 0..3 */
  uint8_t terminated;  /* the `terminated` / `_done` flag */
  uint8_t pad[6];
  double reward;
} rlrm_experience_t;
/* update_q (qlearning.py:70-79) / QLearningLambda.update applied to `n` experiences on the table of slot `slot` (= i*A + a),
 * in list order, in one launch. `experiences` is device-accessible memory (device or page-locked host). */
int rlrm_update_list(rlrm_handle_t* h, const rlrm_state_t* st, int64_t slot, int32_t n, const rlrm_experience_t* experiences,
                     void* stream);

/* The same list update FOLLOWED, in the same launch, by the selection a driver loop makes next on that table
 * (frozen_lake_main.py:345-367: update_policy(.., next_state, ..) of iteration t, then select_action(next_state) of iteration
 * t + 1): QLearning.choose_action (qlearning.py:112-143) on encoded state `sel->state` with `sel->epsilon` and the four injected
 * words `sel->draws` (w0 explore, w1 random action, w2 tie-break; best != 0: argmax). `sel` is PAGE-LOCKED HOST memory: its
 * input fields are read by the host at call time (so the caller may overwrite them for the next request as soon as the call
 * returns), the kernel writes `sel->action`, then `sel->done_seq = seq` behind a system-scope fence, so the host can read the
 * result without a stream synchronisation once done_seq == seq. The table is not modified by the selection; a caller that ends
 * up selecting on another state / epsilon simply ignores the answer. n may be 0 (selection only). 48 bytes. */
typedef struct rlrm_select_req {
  uint32_t state;     /* encoded state (enc = cell*nQ + q) to select in */
  uint32_t best;      /* != 0: first argmax, no randomness */
  double epsilon;
  uint32_t draws[4];
  uint32_t seq;       /* in: any value that differs from the previous request's */
  uint32_t action;    /* out: 0..3 */
  uint32_t done_seq;  /* out: = seq once `action` is valid */
  uint32_t pad;
} rlrm_select_req_t;
int rlrm_update_list_select(rlrm_handle_t* h, const rlrm_state_t* st, int64_t slot, int32_t n, const rlrm_experience_t* experiences,
                            rlrm_select_req_t* sel, void* stream);

/* Shared learner, inter-GPU merge: q[j] = (gathered[0][j] + gathered[1][j] + ... + gathered[world-1][j]) / world for j < n,
 * added in rank order (float32, round to nearest), so every rank gets the same bits whatever collective produced
 * `gathered` ([world][n] floats, device; e.g. the output of one NCCL all-gather of the replicas). */
int rlrm_merge_replicas(rlrm_handle_t* h, const float* gathered, int32_t world, int64_t n, float* q, void* stream);

/* cudaStreamSynchronize for hosts without a CUDA runtime binding of their own (ctypes / cgo / JNI callers). */
int rlrm_stream_sync(rlrm_handle_t* h, void* stream);

/* Same call with HOST buffers (the end-to-end path). host_slot / host_epsilon ([N*A], in/out, may be NULL): the
 * environment / RM state and epsilon to resume from are uploaded before the launch and the updated values are
 * downloaded after it; host_stats ([N*A], out, may be NULL) receives the statistics block. The stream is synchronised
 * before returning. All copies are inside this call and therefore inside any end-to-end timing of it. */
int rlrm_train_host(rlrm_handle_t* h, const rlrm_state_t* st, uint64_t t0, int32_t n_iters, int32_t learn,
                    uint64_t* host_slot, double* host_epsilon, rlrm_stats_t* host_stats, void* stream);

/* Greedy policy evaluation = test_policy_optima (R/environments/utils_envs/evaluation_metrics.py:23-190): the driver
 * loop with select_action(best=True), no update, no epsilon decay; per agent and episode the discounted return
 * sum(gamma^t * reward) until the agent succeeds, success = terminated with the RM in its final state, episode length.
 * Runs n_iters lockstep iterations; an instance stops starting new episodes once it finished n_episodes.
 * `ev` is a device array [N*A], zero-initialised with cum_gamma = 1 by the caller. The caller passes a COPY of the
 * environment state (slot) — the reference evaluates on copy.deepcopy(env) — while q is read-only here. */
int rlrm_evaluate(rlrm_handle_t* h, const rlrm_state_t* st, rlrm_eval_t* ev, uint64_t t0, int32_t n_iters, int32_t n_episodes,
                  double gamma, double optimal_steps, void* stream);

/* Sparse Q(lambda) only: write every listed q value back into `q` (lists stay live) and, when e_dense is non-NULL
 * (device, [N*A*S*4], zeroed by the caller), scatter the traces into it — the dense view of learner.q_table / e_table. */
int rlrm_qlambda_materialize(rlrm_handle_t* h, const rlrm_state_t* st, void* e_dense, void* stream);

/* MEASUREMENT AID, not part of the path (bench.py's roofline block): launches `n_gathers` (rounded up to 64 per thread) independent
 * gathers of random aligned `block_bytes` (16 / 32 / 64) blocks of the device buffer `table` (64-byte aligned), eight in flight per
 * thread, each optionally followed by a 4-byte store into the block that rewrites a value just read (`write` != 0). Timed by the
 * caller with CUDA events it gives the ceiling of the memory system for the access pattern of the per-instance-table kernels, which
 * the streaming copy peak does not describe. `sink`: 4 writable device bytes. Needs no handle. */
int rlrm_probe_random_gather(int device, void* table, int64_t table_bytes, int32_t block_bytes, int64_t n_gathers, int32_t write,
                             void* sink, void* stream);

/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
int64_t rlrm_launch_count(const rlrm_handle_t* h);

#ifdef __cplusplus
}
#endif
#endif /* RLRM_B200_H */
