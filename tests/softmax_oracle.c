/*
 * TEST INFRASTRUCTURE — CPU oracle of softmax exploration (rlrm_set_exploration; the rule is stated in include/rlrm_b200.h).
 * Not part of the product path; tests/softmax_oracle.py builds and loads it.
 *
 * This translation unit includes the C oracle (oracle/rlrm_oracle.c) unchanged and adds:
 *   softmax_exp          rlrm_exp of csrc/rlrm_device.cuh, restated operation for operation;
 *   softmax_thresholds   T_j = ceil(C_j / C_{n-1} * 2^32) of one row;
 *   softmax_select_action / softmax_train
 *                        oracle_select_action / oracle_train with the softmax selection in place of the epsilon-greedy one:
 *                        the same env / RM step, update, reset and statistics of the oracle (its static functions), one
 *                        selection per (iteration, instance, agent) on w1 of the same Philox draw.
 * Build with -ffp-contract=off (every operation below then rounds once, as the device's _rn intrinsics do) and
 * -DORACLE_REAL=float or double, as the oracle.
 */
#include "../oracle/rlrm_oracle.c"

double softmax_exp(double x) { /* x <= 0 */
  if (x < -0x1.74910d52d3052p+9) return 0.0; /* below ln(2^-1075): exp(x) rounds to +0 */
  double k = rint(x * 0x1.71547652b82fep+0); /* log2(e) */
  double r = fma(-k, 0x1.62e42fefa39efp-1, x); /* ln2, high part */
  r = fma(-k, 0x1.abc9e3b39803fp-56, r);       /* ln2, low part */
  double p = 0x1.93974a8c07c9dp-37;            /* 1/14!, 1/13!, ..., 1/2!, 1, 1 */
  p = fma(p, r, 0x1.6124613a86d09p-33);
  p = fma(p, r, 0x1.1eed8eff8d898p-29);
  p = fma(p, r, 0x1.ae64567f544e4p-26);
  p = fma(p, r, 0x1.27e4fb7789f5cp-22);
  p = fma(p, r, 0x1.71de3a556c734p-19);
  p = fma(p, r, 0x1.a01a01a01a01ap-16);
  p = fma(p, r, 0x1.a01a01a01a01ap-13);
  p = fma(p, r, 0x1.6c16c16c16c17p-10);
  p = fma(p, r, 0x1.1111111111111p-7);
  p = fma(p, r, 0x1.5555555555555p-5);
  p = fma(p, r, 0x1.5555555555555p-3);
  p = fma(p, r, 0x1.0p-1);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  int ki = (int)k; /* -1075 .. 0 */
  double scale;
  uint64_t bits;
  if (ki < -1021) { /* subnormal range: scale by 2^(k+54) exactly, then round once at the multiplication by 2^-54 */
    bits = (uint64_t)(ki + 54 + 1023) << 52;
    memcpy(&scale, &bits, 8);
    return p * scale * 0x1.0p-54;
  }
  bits = (uint64_t)(ki + 1023) << 52;
  memcpy(&scale, &bits, 8);
  return p * scale;
}

void softmax_exp_array(int64_t n, const double* x, double* out) {
  for (int64_t j = 0; j < n; j++) out[j] = softmax_exp(x[j]);
}

/* thresholds T_j, j < n - 1, of a row of n action values with beta = 1 / temperature; returns n - 1 */
int softmax_thresholds(const real* row, int n, double beta, uint64_t* thr) {
  double m = (double)row[0], c[RLRM_N_ACTIONS], total = 0.0;
  for (int j = 1; j < n; j++) if ((double)row[j] > m) m = (double)row[j];
  for (int j = 0; j < n; j++) { total += softmax_exp(((double)row[j] - m) * beta); c[j] = total; }
  for (int j = 0; j + 1 < n; j++) thr[j] = (uint64_t)ceil(c[j] / total * 4294967296.0);
  return n - 1;
}

static int select_softmax(const rlrm_config_t* cfg, const real* row, const uint32_t w[4], int best, double beta) {
  if (best) return select_one(cfg, row, 0.0, w, 1); /* greedy evaluation: the first argmax */
  uint64_t thr[RLRM_N_ACTIONS];
  int action = 0;
  for (int j = 0, n = softmax_thresholds(row, cfg->n_actions, beta, thr); j < n; j++) action += (uint64_t)w[1] >= thr[j];
  return action;
}

static const real* current_row(const rlrm_config_t* cfg, const rlrm_tables_t* tb, const rlrm_state_t* st, int64_t i, int a) {
  slot_t s = unpack(st->slot[(size_t)i * cfg->n_agents + a]);
  return (const real*)st->q + table_base(cfg, i, a) + ((size_t)s.cell * agent_rm(cfg, tb, a).nQ + s.rm) * 4;
}

int softmax_select_action(const rlrm_config_t* cfg, const rlrm_tables_t* tb, const rlrm_state_t* st, const uint32_t* draws,
                          uint64_t t, int best, double beta, uint8_t* actions_out) {
  for (int64_t i = 0; i < st->n_instances; i++)
    for (int a = 0; a < cfg->n_agents; a++) {
      uint32_t w[4];
      get_draws(cfg, draws, t, i, a, w);
      actions_out[(size_t)i * cfg->n_agents + a] = (uint8_t)select_softmax(cfg, current_row(cfg, tb, st, i, a), w, best, beta);
    }
  return 0;
}

/* train_iteration of the oracle (the driver loop, frozen_lake_main.py:345-376 ; office_main.py:1709-1749) with the softmax
 * selection; everything after the selection is the oracle's own code */
static void softmax_iteration(const rlrm_config_t* cfg, const rlrm_tables_t* tb, const rlrm_state_t* st, int64_t i, uint64_t t,
                              int32_t it, int32_t learn, uint32_t* trace, double beta) {
  int A = cfg->n_agents;
  rec_t rec[RLRM_MAX_AGENTS];
  uint8_t act[RLRM_MAX_AGENTS];
  uint32_t before[RLRM_MAX_AGENTS];
  int first = 0;
  for (int a = 0; a < A; a++) { /* every agent selects, finished ones included */
    slot_t s = unpack(st->slot[(size_t)i * A + a]);
    before[a] = s.cell;
    first = (s.flags & RLRM_FLAG_FIRST) != 0;
    uint32_t w[4];
    get_draws(cfg, NULL, t, i, a, w);
    act[a] = (uint8_t)select_softmax(cfg, current_row(cfg, tb, st, i, a), w, !learn, beta);
  }
  step_instance(cfg, tb, st, i, act, NULL, t, 1, rec);
  int all_term = 1, all_trunc = 1;
  for (int a = 0; a < A; a++) {
    size_t k = (size_t)i * A + a;
    uint32_t obs = (cfg->driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? rec[a].cell : before[a];
    int term_arg = cfg->driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (rec[a].term || rec[a].trunc) : rec[a].term;
    if (learn) update_slot(cfg, tb, st, i, a, obs, act[a], term_arg, &rec[a]);
    all_term &= (int)rec[a].term; all_trunc &= (int)rec[a].trunc;
    if (st->ep_return) st->ep_return[k] += rec[a].reward;
    if (trace)
      trace[(size_t)it * st->n_instances * A + k] = (uint32_t)act[a] | (rec[a].executed << 3) | (rec[a].cell << 6) |
          (rec[a].q << 16) | (rec[a].term << 21) | (rec[a].trunc << 22) | (rec[a].stepped << 23);
  }
  clear_first(cfg, st, i);
  if (all_term || all_trunc) {
    for (int a = 0; a < A; a++) {
      size_t k = (size_t)i * A + a;
      if (st->stats) {
        slot_t s = unpack(st->slot[k]);
        rlrm_stats_t* z = &st->stats[k];
        z->episodes++;
        z->active_steps += s.steps;
        { int fin = agent_rm(cfg, tb, a).final; z->successes += (fin >= 0 && (int)s.rm == fin); }
        double ret = st->ep_return ? st->ep_return[k] : 0.0;
        z->last_return = (float)ret;
        z->return_sum += ret;
        z->last_length = s.time;
      }
    }
    reset_instance_at(cfg, tb, st, i, t + 1);
  }
}

/* oracle_train with softmax exploration; per-instance tables only (softmax is unsupported on a shared table) */
int softmax_train(const rlrm_config_t* cfg, const rlrm_tables_t* tb, const rlrm_state_t* st, uint64_t t0, int32_t n_iters,
                  int32_t learn, uint32_t* trace, double beta) {
  if (cfg->shared_q) return RLRM_ERR_UNSUPPORTED;
  for (int64_t i = 0; i < st->n_instances; i++)
    for (int32_t it = 0; it < n_iters; it++) softmax_iteration(cfg, tb, st, i, t0 + (uint64_t)it, it, learn, trace, beta);
  return 0;
}
