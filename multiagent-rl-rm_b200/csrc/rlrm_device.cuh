// rlrm_device.cuh: parameter blocks, shared-memory tables, Philox, and the per-agent device functions
// (select / env + RM step / Q updates / reset) shared by every kernel — part of the single translation unit csrc/rlrm_b200.cu (see its header comment).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rlrm_b200.h"

// ------------------------------------------------------------------------------------------------
// kernel parameter block (passed by value)
// ------------------------------------------------------------------------------------------------
// Learner hyper-parameters and the constants derived from them on the host (fill_learner). Every kernel reads them as KP::h;
// a sweep handle (rlrm_set_sweep) owns a device array of them, one per setting, which apply_sweep loads into a kernel's copy.
struct Hyp {
  double lr, gamma, eps_end, eps_decay;
  float lr_f, one_minus_lr_f, gamma_f, trace_decay_f;  // (float)lr, (float)(1-lr), (float)gamma, (float)(gamma*lambda)
  double one_minus_lr, trace_decay;                    // 1 - lr and gamma*lambda as doubles (float64 tables)
};
// The settings of a sweep handle: instance i (global id instance_offset + i) trains with hyp[(instance_offset + i) / group].
// Passed as the LAST kernel argument, so the parameter offsets of everything before it are those of a uniform launch.
struct Sweep {
  const Hyp* hyp;  // null: uniform handle
  long long group;
};

struct KP {
  int env_kind, driver, algo;
  int A, G, g_shift;  // agents, lane-group size (power of two >= A), log2(G)
  int nQ, nEv, rm_final, n_qrm, max_steps, ncell;
  int stochastic, slip_n;
  int slip_cnt;              // thresholds below 2^32 (a threshold of 2^32 can never be reached by a 32-bit draw)
  unsigned slip_thr32[3];
  unsigned long long slip_thr[3];
  unsigned char slip_outcome[16];
  unsigned long long slip_nib;  // slip_outcome as 16 nibbles: outcome of (intended a, threshold index k) at bits 4*(4a+k)
  int terminate_on_plants, terminate_hit_walls;
  double hole_penalty, wall_penalty;
  Hyp h;  // same place and layout as the fields it groups, so uniform kernels address the constant bank as before
  int decay_on_reset, shared_q, use_rsh, random_starts, n_free;
  int shared_balanced;  // shared_train_kernel: contiguous equal chunks per block (1) or grid-stride (0)
  int qls_lg;           // train_qlambda_sparse_kernel: lanes per agent (power of two, 4 .. 32 / G)
  // agents with different reward machines (rlrm_config_t.per_agent_rm): per-agent scalars and table strides
  int per_agent, a_nQ[RLRM_MAX_AGENTS], a_final[RLRM_MAX_AGENTS], a_nqrm[RLRM_MAX_AGENTS];
  long long a_prefix4[RLRM_MAX_AGENTS], sum4;  // float offset of agent a's table inside one instance, floats per instance
  int nd;                                       // nQmax * (nEv + 1): one agent's delta / rq / rcf section
  int phi_row;                                  // nQmax: row stride of phi ([2][nQmax] per machine)
  unsigned seed_lo, seed_hi, instance_offset, n_actions;
  unsigned rk[20];  // Philox round keys: rk[2r] = seed_lo + r*0x9E3779B9, rk[2r+1] = seed_hi + r*0xBB67AE85
  long long S4;  // W*H*nQ*4 floats per table
  // table blob in global memory and section offsets (bytes) inside it / inside the shared-memory copy
  const unsigned char* blob;
  int blob_bytes;
  int off_next, off_flags, off_label, off_delta, off_rq, off_rcf, off_qrm, off_start, off_phi, off_free;
  int off_q4cell, off_q4rec, off_q4rew;  // train_qrm4_kernel's precomputed step records (see that kernel), empty otherwise
};

struct Tab {
  const unsigned short* next_cell;
  const unsigned char* cell_flags;
  const unsigned char* label;
  const unsigned char* delta;
  const double* rq;
  const double* rcf;
  const unsigned char* qrm_states;
  const unsigned short* start_cell;
  const unsigned short* free_cells;
  const double* phi;
};

struct DState {  // rlrm_state_t by value
  long long N;
  unsigned long long* slot;
  double* epsilon;
  float* q;  // learner.q_table; holds doubles when the handle was created with table_dtype = RLRM_TABLE_F64 (tab<T>() below)
  float* e;
  unsigned* visits;
  double* ep_return;
  rlrm_stats_t* stats;
  long long* acc_sum;  // shared learner accumulators (include/rlrm_b200.h "Shared learner"), null otherwise
  int* acc_cnt;
  float* acc_last;
  unsigned short* tr_pos;  // Q(lambda) sparse-exact traces (include/rlrm_b200.h), null otherwise
  unsigned short* tr_idx;
  float2* tr_eq;  // (trace, current q value) of each listed entry (double2 for float64 tables)
  unsigned* tr_len;
  unsigned long long* tr_work;
  int tr_cap;
};

struct Acc {  // accumulators of one agent's shared table, or nulls
  long long* sum;
  int* cnt;
  float* last;
  bool smem;  // the accumulators live in shared memory (shared_propose_kernel)
  const float* rmax;  // optional: max over actions of every table row as of the start of the iteration (proposals do not
                      // touch Q until apply_shared_kernel, so it stays valid for the whole launch); null = read the row
};

struct DOut {  // rlrm_step_out_t by value
  unsigned short *prev_cell, *cell;
  unsigned char *prev_q, *q, *event, *executed;
  double *renv, *rq, *reward;
  unsigned char *env_term, *rm_term, *term, *trunc;
  unsigned char* cf_q;
  double* cf_r;
};

extern __shared__ __align__(16) unsigned char smem_raw[];

__device__ __forceinline__ Tab stage_tables(const KP& p) {
  // cooperative 16-byte copy of the (<= ~45 KB, typically 1-3 KB) table blob into shared memory
  const uint4* src = reinterpret_cast<const uint4*>(p.blob);
  uint4* dst = reinterpret_cast<uint4*>(smem_raw);
  for (int k = threadIdx.x; k < p.blob_bytes / 16; k += blockDim.x) dst[k] = __ldg(src + k);
  __syncthreads();
  Tab t;
  t.next_cell = reinterpret_cast<const unsigned short*>(smem_raw + p.off_next);
  t.cell_flags = smem_raw + p.off_flags;
  t.label = smem_raw + p.off_label;
  t.delta = smem_raw + p.off_delta;
  t.rq = reinterpret_cast<const double*>(smem_raw + p.off_rq);
  t.rcf = reinterpret_cast<const double*>(smem_raw + p.off_rcf);
  t.qrm_states = smem_raw + p.off_qrm;
  t.start_cell = reinterpret_cast<const unsigned short*>(smem_raw + p.off_start);
  t.phi = reinterpret_cast<const double*>(smem_raw + p.off_phi);
  t.free_cells = reinterpret_cast<const unsigned short*>(smem_raw + p.off_free);
  return t;
}

// ------------------------------------------------------------------------------------------------
// table arithmetic type. The reference keeps q_table / e_table in float64 (np.zeros default, qlearning.py:26-29,
// qlearning_lambda.py:26-30); RT<double> is that arithmetic. RT<float> is what NumPy computes when the tables are cast to
// float32 (NEP 50: weak Python scalars are rounded to the table dtype first, every operation rounds separately — hence the
// explicit _rn intrinsics, which also keep the compiler from contracting a*b+c into an FMA).
// ------------------------------------------------------------------------------------------------
struct __align__(32) double4r {
  double x, y, z, w;
};
template <typename T>
struct RT;
template <>
struct RT<float> {
  typedef float4 row_t;
  typedef float2 pair_t;
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float cvt(double x) { return __double2float_rn(x); }
  static __device__ __forceinline__ bool same_bits(float a, float b) { return __float_as_uint(a) == __float_as_uint(b); }
  static __device__ __forceinline__ float lr(const KP& p) { return p.h.lr_f; }
  static __device__ __forceinline__ float one_minus_lr(const KP& p) { return p.h.one_minus_lr_f; }
  static __device__ __forceinline__ float gamma(const KP& p) { return p.h.gamma_f; }
  static __device__ __forceinline__ float decay(const KP& p) { return p.h.trace_decay_f; }
  static __device__ __forceinline__ row_t zero_row() { return make_float4(0.f, 0.f, 0.f, 0.f); }
  static __device__ __forceinline__ pair_t make_pair(float a, float b) { return make_float2(a, b); }
};
template <>
struct RT<double> {
  typedef double4r row_t;
  typedef double2 pair_t;
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double cvt(double x) { return x; }
  static __device__ __forceinline__ bool same_bits(double a, double b) { return __double_as_longlong(a) == __double_as_longlong(b); }
  static __device__ __forceinline__ double lr(const KP& p) { return p.h.lr; }
  static __device__ __forceinline__ double one_minus_lr(const KP& p) { return p.h.one_minus_lr; }
  static __device__ __forceinline__ double gamma(const KP& p) { return p.h.gamma; }
  static __device__ __forceinline__ double decay(const KP& p) { return p.h.trace_decay; }
  static __device__ __forceinline__ row_t zero_row() { return double4r{0.0, 0.0, 0.0, 0.0}; }
  static __device__ __forceinline__ pair_t make_pair(double a, double b) { return make_double2(a, b); }
};
template <typename T>
__device__ __forceinline__ T* tab(float* p) { return reinterpret_cast<T*>(p); }  // typed view of a DState table pointer
template <typename T>
__device__ __forceinline__ typename RT<T>::row_t load_row(const T* Q, size_t row) {
  return *reinterpret_cast<const typename RT<T>::row_t*>(Q + row * 4);
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Random123): counter (t_lo, t_hi, instance, agent), key (seed_lo, seed_hi)
// ------------------------------------------------------------------------------------------------
// The 10 round keys (k0 + r*W0, k1 + r*W1) depend only on the seed: they are precomputed on the host into KP::rk so every
// round is two wide multiplies and two three-input XORs whose key operand comes straight from the constant bank.
#define RLRM_PHILOX(c0, c1, c2, c3, p, w) philox4x32_10_rk(c0, c1, c2, c3, (p).rk, w)
__device__ __forceinline__ void philox4x32_10_rk(unsigned c0, unsigned c1, unsigned c2, unsigned c3, const unsigned (&rk)[20],
                                                 unsigned w[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
    const unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ rk[2 * r], n2 = (unsigned)(p0 >> 32) ^ c3 ^ rk[2 * r + 1];
    c1 = (unsigned)p1;
    c3 = (unsigned)p0;
    c0 = n0;
    c2 = n2;
  }
  w[0] = c0; w[1] = c1; w[2] = c2; w[3] = c3;
}

// ------------------------------------------------------------------------------------------------
// per-agent pieces
// ------------------------------------------------------------------------------------------------
struct Slot {
  unsigned cell, steps, time, rm, flags;
};
__device__ __forceinline__ Slot unpack_slot(unsigned long long w) {
  Slot s;
  s.cell = (unsigned)(w >> RLRM_SLOT_CELL_SHIFT) & 0xFFFFu;
  s.steps = (unsigned)(w >> RLRM_SLOT_STEPS_SHIFT) & 0xFFFFu;
  s.time = (unsigned)(w >> RLRM_SLOT_TIME_SHIFT) & 0xFFFFu;
  s.rm = (unsigned)(w >> RLRM_SLOT_RMSTATE_SHIFT) & 0xFFu;
  s.flags = (unsigned)(w >> RLRM_SLOT_FLAGS_SHIFT) & 0xFFu;
  return s;
}
__device__ __forceinline__ unsigned long long pack_slot(const Slot& s) {
  return ((unsigned long long)s.cell << RLRM_SLOT_CELL_SHIFT) | ((unsigned long long)s.steps << RLRM_SLOT_STEPS_SHIFT) |
         ((unsigned long long)s.time << RLRM_SLOT_TIME_SHIFT) | ((unsigned long long)s.rm << RLRM_SLOT_RMSTATE_SHIFT) |
         ((unsigned long long)s.flags << RLRM_SLOT_FLAGS_SHIFT);
}

// explore iff w0 / 2^32 < epsilon  <=>  w0 < ceil(epsilon * 2^32)   (w0 integer; the scaling by 2^32 is exact)
__device__ __forceinline__ unsigned long long explore_threshold(double eps) {
  if (!(eps > 0.0)) return 0ull;
  if (eps >= 1.0) return 1ull << 32;
  return (unsigned long long)ceil(eps * 4294967296.0);
}

// QLearning.choose_action / choose_action_greedy (qlearning.py:112-143)
template <typename R>
__device__ __forceinline__ int select_action(const R& row, unsigned long long explore_thr, const unsigned w[4], bool best,
                                             unsigned n_actions) {
  // np.argmax: first maximum
  int va = 0;
  auto m = row.x;
  if (row.y > m) { m = row.y; va = 1; }
  if (row.z > m) { m = row.z; va = 2; }
  if (row.w > m) { m = row.w; va = 3; }
  if (best) return va;
  if ((unsigned long long)w[0] < explore_thr) return (int)__umulhi(w[1], n_actions);  // rng.choice(range(A))
  const int e0 = row.x == m, e1 = row.y == m, e2 = row.z == m, e3 = row.w == m;
  const int n = e0 + e1 + e2 + e3;
  if (n == 1) return va;
  const int pick = (int)__umulhi(w[2], (unsigned)n);  // rng.choice(maxs): the pick-th maximal index
  // rank of each maximal index among the maxima
  const int r1 = e0, r2 = e0 + e1, r3 = e0 + e1 + e2;
  int a = va;
  if (e1 && r1 == pick) a = 1;
  if (e2 && r2 == pick) a = 2;
  if (e3 && r3 == pick) a = 3;
  if (e0 && pick == 0) a = 0;
  return a;
}

// Softmax exploration (rlrm_set_exploration; the rule is stated in include/rlrm_b200.h). rlrm_exp is a fixed sequence of IEEE-754
// double operations for x <= 0 that the CPU oracle restates operation for operation (tests/softmax_oracle.c), so both sides get the
// same bits: Cody-Waite reduction x = k*ln2 + r with |r| <= ln2/2, the degree-14 Taylor polynomial of exp(r) by Horner's rule with
// FMA, and a scaling by 2^k built from its bit pattern (in two steps below 2^-1021, so that a subnormal result is rounded once).
__device__ __forceinline__ double rlrm_exp(double x) {
  if (x < -0x1.74910d52d3052p+9) return 0.0;  // below ln(2^-1075): exp(x) rounds to +0
  const double k = rint(__dmul_rn(x, 0x1.71547652b82fep+0));  // log2(e)
  double r = __fma_rn(-k, 0x1.62e42fefa39efp-1, x);            // ln2, high part
  r = __fma_rn(-k, 0x1.abc9e3b39803fp-56, r);                  // ln2, low part
  double p = 0x1.93974a8c07c9dp-37;                            // 1/14!, 1/13!, ..., 1/2!, 1, 1
  p = __fma_rn(p, r, 0x1.6124613a86d09p-33);
  p = __fma_rn(p, r, 0x1.1eed8eff8d898p-29);
  p = __fma_rn(p, r, 0x1.ae64567f544e4p-26);
  p = __fma_rn(p, r, 0x1.27e4fb7789f5cp-22);
  p = __fma_rn(p, r, 0x1.71de3a556c734p-19);
  p = __fma_rn(p, r, 0x1.a01a01a01a01ap-16);
  p = __fma_rn(p, r, 0x1.a01a01a01a01ap-13);
  p = __fma_rn(p, r, 0x1.6c16c16c16c17p-10);
  p = __fma_rn(p, r, 0x1.1111111111111p-7);
  p = __fma_rn(p, r, 0x1.5555555555555p-5);
  p = __fma_rn(p, r, 0x1.5555555555555p-3);
  p = __fma_rn(p, r, 0x1.0p-1);
  p = __fma_rn(p, r, 1.0);
  p = __fma_rn(p, r, 1.0);
  const int ki = (int)k;  // -1075 .. 0
  if (ki < -1021) return __dmul_rn(__dmul_rn(p, __longlong_as_double((long long)(ki + 54 + 1023) << 52)), 0x1.0p-54);
  return __dmul_rn(p, __longlong_as_double((long long)(ki + 1023) << 52));
}

// Softmax selection on the row's first n_actions entries with beta = 1 / temperature: weights w_a = rlrm_exp((Q[a] - max) * beta),
// cumulative sums C_j in action order, thresholds T_j = ceil(C_j / C_{n-1} * 2^32), action = #{j < n-1 : w1 >= T_j}. Zero
// weights give empty intervals. best: the first argmax, exactly as select_action.
template <typename R>
__device__ __forceinline__ int select_softmax(const R& row, unsigned w1, double beta, bool best, unsigned n_actions) {
  if (best) {
    const unsigned w[4] = {0u, 0u, 0u, 0u};
    return select_action(row, 0ull, w, true, n_actions);
  }
  const double q[4] = {(double)row.x, (double)row.y, (double)row.z, (double)row.w};
  double m = q[0];
#pragma unroll
  for (int j = 1; j < 4; j++)
    if ((unsigned)j < n_actions && q[j] > m) m = q[j];
  double c[4], total = 0.0;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    if ((unsigned)j < n_actions) total = __dadd_rn(total, rlrm_exp(__dmul_rn(__dsub_rn(q[j], m), beta)));
    c[j] = total;
  }
  int action = 0;
#pragma unroll
  for (int j = 0; j < 3; j++)
    if ((unsigned)j + 1u < n_actions)
      action += (unsigned long long)w1 >= (unsigned long long)ceil(__dmul_rn(__ddiv_rn(c[j], total), 4294967296.0));
  return action;
}

__device__ __forceinline__ int slip_outcome(const KP& p, int intended, unsigned k) {
  int idx = 0;
#pragma unroll
  for (int j = 0; j < 3; j++) idx += (j < p.slip_cnt) && (k >= p.slip_thr32[j]);
  return p.slip_outcome[intended * 4 + idx];
}

struct Rec {
  unsigned prev_cell, cell, prev_q, q, event, executed;
  bool env_term, rm_term, term, trunc, stepped;
  double renv, rq, reward;
};

// env.step + check_terminations + RewardMachine.step + wrapper merge for ONE agent. Every quantity an agent needs is
// its own (the shared env.timestep is replicated per agent), so lanes never exchange data here.
// WAIT_OK: the caller may pass RLRM_ACTION_WAIT itself (env.wait_action through the call-by-call API and the "wait"
// sub-action of get_mdp); the fused kernels only ever select 0..3 and skip the test.
// PRE: the move-table row of the current cell (`nrow`, four u16 targets) and the slip threshold index (`sidx`) were fetched /
// computed BEFORE the action was selected, so that action -> executed action -> new cell is pure ALU work (two shifts) instead
// of a dependent constant-bank lookup followed by a dependent shared-memory lookup: the new cell is what the Q-block load after a
// move waits for, i.e. this chain sits on the per-iteration critical path of the fused kernels.
struct PreStep {
  unsigned long long nrow;
  unsigned sidx;
};
// Index into KP::slip_nib. rlrm_create pads the thresholds past slip_cnt with 0xFFFFFFFF and the nibble of index 3 with the
// outcome of index slip_cnt, so no slip_cnt test is needed: only k = 0xFFFFFFFF reaches a padded threshold, and then all three.
__device__ __forceinline__ unsigned slip_index(const KP& p, unsigned k) {
  return (unsigned)(k >= p.slip_thr32[0]) + (unsigned)(k >= p.slip_thr32[1]) + (unsigned)(k >= p.slip_thr32[2]);
}
__device__ __forceinline__ PreStep pre_step(const KP& p, const Tab& tb, unsigned cell, unsigned w3, bool stochastic) {
  PreStep ps;
  ps.nrow = *reinterpret_cast<const unsigned long long*>(tb.next_cell + cell * 4);
  ps.sidx = stochastic ? slip_index(p, w3) : 0u;
  return ps;
}
template <int ENV, int STOCH = -1, bool WAIT_OK = false, bool PRE = false>  // STOCH: -1 = read p.stochastic at run time, 0/1 = compile-time
__device__ __forceinline__ void agent_step(const KP& p, const Tab& tb, Slot& s, int action, unsigned w3, bool with_rm, Rec& r,
                                           PreStep ps = PreStep{0ull, 0u}) {
  const bool stochastic = STOCH < 0 ? (p.stochastic != 0) : (STOCH != 0);
  // (plain expressions, not lambdas: a by-reference closure over `p` makes the kernels' private copy of the parameter block
  // address-taken and sends all 656 bytes of it to local memory — +13 us on every one-iteration launch of rlrm_iterate)
#define RLRM_NEXT_OF(ex) (PRE ? ((unsigned)(ps.nrow >> ((ex) * 16)) & 0xFFFFu) : (unsigned)tb.next_cell[s.cell * 4 + (ex)])
#define RLRM_SLIP_OF(a) (PRE ? (int)((unsigned)(p.slip_nib >> (((a) * 4 + (int)ps.sidx) * 4)) & 0xFu) : slip_outcome(p, (a), w3))
  r.prev_cell = s.cell;
  r.executed = 5;
  r.stepped = false;
  r.renv = 0.0;
  r.rq = 0.0;
  const bool active = (s.flags & RLRM_FLAG_ACTIVE) != 0;
  if (ENV == RLRM_ENV_FROZEN_LAKE) {
    const bool rm_done = p.rm_final >= 0 && (int)s.rm == p.rm_final;  // ma_frozen_lake.py:107-115
    if (active && !rm_done) {
      int ex = action;
      if (stochastic && (!WAIT_OK || action != RLRM_ACTION_WAIT)) ex = RLRM_SLIP_OF(action);
      if (ex != RLRM_ACTION_WAIT) s.cell = RLRM_NEXT_OF(ex);
      if (tb.cell_flags[s.cell] & 1) {  // holes_in_the_ice
        s.flags |= RLRM_FLAG_FAIL;
        r.renv = p.hole_penalty;
      }
      s.steps++;
      r.executed = ex;
      r.stepped = true;
    }
  } else {
    if (active) {  // ma_office.py:143-186
      int ex = action;
      double wall_pen = 0.0;
      // is_wall_collision("wait") is False (ma_office.py:299-300)
      if ((!WAIT_OK || action != RLRM_ACTION_WAIT) && RLRM_NEXT_OF(action) == s.cell) {  // apply_wall_penalty: blocked -> "wait", no slip draw
        if (p.terminate_hit_walls) s.flags |= RLRM_FLAG_FAIL;
        wall_pen = p.wall_penalty;
        ex = RLRM_ACTION_WAIT;
      }
      if (stochastic && ex != RLRM_ACTION_WAIT) ex = RLRM_SLIP_OF(ex);
      if (ex != RLRM_ACTION_WAIT) s.cell = RLRM_NEXT_OF(ex);
      double plant = 0.0;
      if (tb.cell_flags[s.cell] & 1) {  // plants_in_the_office
        if (p.terminate_on_plants) s.flags |= RLRM_FLAG_FAIL;
        plant = p.hole_penalty;
      }
      r.renv = __dadd_rn(wall_pen, plant);
      s.steps++;
      r.executed = ex;
      r.stepped = true;
    }
  }
  r.cell = s.cell;
  s.time++;
  const bool fail = (s.flags & RLRM_FLAG_FAIL) != 0;
  if (ENV == RLRM_ENV_FROZEN_LAKE) {  // ma_frozen_lake.py:189-215 (RM state as of BEFORE this step's RM update)
    r.trunc = ((int)s.steps > p.max_steps) || ((int)s.time > p.max_steps);
    r.env_term = r.trunc || (p.rm_final >= 0 && (int)s.rm == p.rm_final) || fail;
    if (r.env_term) s.flags &= ~RLRM_FLAG_ACTIVE;
  } else {  // ma_office.py:240-257
    r.trunc = (int)s.time > p.max_steps;
    r.env_term = fail;
    if (r.env_term || r.trunc) s.flags &= ~RLRM_FLAG_ACTIVE;
  }
  // rm_environment_wrapper.py:57-107
  r.prev_q = s.rm;
  r.event = tb.label[s.cell];
  r.rm_term = false;
  if (with_rm) {
    const int col = r.event == RLRM_EVENT_NONE ? p.nEv : (int)r.event;
    const unsigned d = tb.delta[s.rm * (p.nEv + 1) + col];
    if (d != RLRM_NO_TRANSITION) {
      r.rq = tb.rq[s.rm * (p.nEv + 1) + col];
      s.rm = d;
    }
    r.rm_term = p.rm_final >= 0 && (int)s.rm == p.rm_final;
  }
  r.q = s.rm;
  r.reward = __dadd_rn(r.renv, r.rq);
  r.term = r.env_term || r.rm_term;
  s.flags &= ~(RLRM_FLAG_DONE | RLRM_FLAG_TRUNC | RLRM_FLAG_FIRST);
  if (r.term) s.flags |= RLRM_FLAG_DONE;
  if (r.trunc) s.flags |= RLRM_FLAG_TRUNC;
#undef RLRM_NEXT_OF
#undef RLRM_SLIP_OF
}

template <typename R, typename T>
__device__ __forceinline__ void set_component(R& v, unsigned c, T x) {
  if (c == 0) v.x = x;
  else if (c == 1) v.y = x;
  else if (c == 2) v.z = x;
  else v.w = x;
}

template <typename R>
__device__ __forceinline__ auto get_component(const R& v, unsigned c) -> decltype(v.x) {
  return c == 0 ? v.x : (c == 1 ? v.y : (c == 2 ? v.z : v.w));
}

__device__ __forceinline__ float row_max(const float4& v) { return fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)); }
__device__ __forceinline__ double row_max(const double4r& v) { return fmax(fmax(v.x, v.y), fmax(v.z, v.w)); }

// update_q (qlearning.py:70-79) in the float32 arithmetic numpy performs on a float32 table: weak Python scalars are
// rounded to float32 first, every operation rounds separately (no FMA contraction).
template <typename T>
__device__ __forceinline__ void update_q(const KP& p, T* Q, unsigned* V, unsigned s, int a, double r, unsigned sn, bool terminated,
                                         const Acc& acc) {
  typedef RT<T> R;
  const T cur = Q[s * 4 + a];
  T mx;
  if (sizeof(T) == 4 && acc.rmax) mx = (T)acc.rmax[sn];
  else mx = row_max(load_row<T>(Q, sn));
  const T mf = R::mul(terminated ? (T)0 : (T)1, mx);
  const T inner = R::add(R::cvt(r), R::mul(R::gamma(p), mf));
  T out;
  if (p.h.lr < 0.0) {  // lr = 1/visits is an np.float64: the outer expression is evaluated in double
    const unsigned v = V[s * 4 + a] + 1;
    V[s * 4 + a] = v;
    const double lr = __ddiv_rn(1.0, (double)v);
    out = R::cvt(__dadd_rn(__dmul_rn(__dsub_rn(1.0, lr), (double)cur), __dmul_rn(lr, (double)inner)));
  } else {
    if (V) {  // a shared table's counts are shared by every instance: count each proposal atomically
      if (acc.sum) atomicAdd(V + s * 4 + a, 1u);
      else V[s * 4 + a] += 1;
    }
    out = R::add(R::mul(R::one_minus_lr(p), cur), R::mul(R::lr(p), inner));
  }
  if (sizeof(T) == 4 && acc.sum) {  // shared learner (float32 tables only): propose; apply_shared_kernel turns the proposals of this iteration into their mean
    const float outf = (float)out;
    const unsigned long long v = (unsigned long long)__float2ll_rn(__fmul_rn(outf, 1048576.0f));
    if (acc.smem) {
      // shared memory has no native 64-bit add (the compiler emits a CAS spin loop, which collapses when many lanes propose
      // to the same entry): add the low word, derive the carry from the value the atomic returns, add the high word. Each
      // 32-bit add is atomic and addition commutes, so the 64-bit sum is exact in any order.
      unsigned* w = reinterpret_cast<unsigned*>(acc.sum + s * 4 + a);
      const unsigned lo = (unsigned)v, hi = (unsigned)(v >> 32);
      const unsigned old = atomicAdd(w, lo);
      const unsigned up = hi + ((old + lo) < old ? 1u : 0u);
      if (up) atomicAdd(w + 1, up);
    } else {
      atomicAdd(reinterpret_cast<unsigned long long*>(acc.sum + s * 4 + a), v);
    }
    atomicAdd(acc.cnt + s * 4 + a, 1);
    acc.last[s * 4 + a] = outf;
  } else {
    Q[s * 4 + a] = out;
  }
}

// QL / QRM update of one agent (agent_rl.py:117-192 -> qlearning.py:41-110; QRM experiences rm_environment_wrapper.py:122-183)
template <int ALGO, typename T>
__device__ __forceinline__ void agent_update(const KP& p, const Tab& tb, T* Q, unsigned* V, unsigned obs_cell, int action,
                                             bool term_arg, const Rec& r, const Acc& acc) {
  if (ALGO == RLRM_ALGO_QRM) {
    const int col = r.event == RLRM_EVENT_NONE ? p.nEv : (int)r.event;
    for (int j = 0; j < p.n_qrm; j++) {
      const unsigned u = tb.qrm_states[j];
      const unsigned d = tb.delta[u * (p.nEv + 1) + col];
      const unsigned un = d == RLRM_NO_TRANSITION ? u : d;
      const double ru = d == RLRM_NO_TRANSITION ? 0.0 : tb.rcf[u * (p.nEv + 1) + col];
      const bool done = r.env_term || (p.rm_final >= 0 && (int)un == p.rm_final);
      double rew = __dadd_rn(r.renv, ru);
      if (p.use_rsh) rew = __dadd_rn(rew, __dsub_rn(__dmul_rn(p.h.gamma, tb.phi[un]), tb.phi[u]));  // qlearning.py:93-105
      update_q(p, Q, V, r.prev_cell * p.nQ + u, action, rew, r.cell * p.nQ + un, done, acc);
    }
  } else {
    double rew = r.reward;
    if (p.use_rsh) rew = __dadd_rn(rew, __dsub_rn(__dmul_rn(p.h.gamma, tb.phi[p.phi_row + r.q]), tb.phi[p.phi_row + r.prev_q]));  // qlearning.py:51-66
    update_q(p, Q, V, obs_cell * p.nQ + r.prev_q, action, rew, r.cell * p.nQ + r.q, term_arg, acc);
  }
}

// _sample_start_positions (ma_frozen_lake.py:156-172): agent a's start cell = entry a of a Fisher-Yates shuffle of the free
// cells driven by Philox words keyed on (T, instance) — see rlrm_config_t.random_starts. Every agent replays steps 0..a.
__device__ __forceinline__ unsigned sample_start(const KP& p, const Tab& tb, long long i, int a, unsigned long long T) {
  unsigned pos[RLRM_MAX_AGENTS], val[RLRM_MAX_AGENTS];
  unsigned w[4] = {0, 0, 0, 0}, out = 0;
  for (int k = 0; k <= a; k++) {
    if ((k & 3) == 0)
      RLRM_PHILOX((unsigned)T, ~(unsigned)(T >> 32), p.instance_offset + (unsigned)i, 0x80000000u | (unsigned)(k >> 2), p, w);
    const unsigned wk = (k & 3) == 0 ? w[0] : ((k & 3) == 1 ? w[1] : ((k & 3) == 2 ? w[2] : w[3]));
    const unsigned j = (unsigned)k + __umulhi(wk, (unsigned)(p.n_free - k));
    unsigned vk = tb.free_cells[k], vj = tb.free_cells[j];
    for (int m = 0; m < k; m++) {
      if (pos[m] == (unsigned)k) vk = val[m];
      if (pos[m] == j) vj = val[m];
    }
    out = vj;
    pos[k] = j;
    val[k] = vk;
  }
  return out;
}

// env.reset for one agent; T = iteration index of the new episode's first step (keys the random start positions)
template <bool RANDOM_STARTS = true>  // false: the caller guarantees cfg.random_starts == 0 (keeps the sampler out of hot kernels)
__device__ __forceinline__ void reset_slot(const KP& p, const Tab& tb, long long i, int a, unsigned long long T, Slot& s, double& eps) {
  s.cell = (RANDOM_STARTS && p.random_starts) ? sample_start(p, tb, i, a, T) : tb.start_cell[a];
  s.steps = 0;
  s.time = 0;
  s.rm = 0;  // the initial RM state has index 0 (reward_machine.py:32-36)
  s.flags = RLRM_FLAG_ACTIVE | RLRM_FLAG_FIRST;
  if (p.decay_on_reset) eps = fmax(p.h.eps_end, __dmul_rn(eps, p.h.eps_decay));  // learn_done_episode (qlearning.py:153-155)
}

__device__ __forceinline__ size_t table_base(const KP& p, long long i, int a) {
  if (p.per_agent) return (size_t)((p.shared_q ? 0ll : i * p.sum4) + p.a_prefix4[a]);
  return (size_t)(p.shared_q ? (long long)a : i * p.A + a) * (size_t)p.S4;
}

// Per-agent reward machines: turn the uniform parameter block / table pointers into agent a's own (nQ, final state, number
// of counterfactual states, table sections). Called only from kernels instantiated with PA = true; `p` must be the kernel's
// private copy of the parameter block, so with PA = false nothing here exists and the parameters stay in the constant bank.
__device__ __forceinline__ void agent_view(const KP& p_in, KP& p, Tab& tb, int a) {
  p.nQ = p_in.a_nQ[a];
  p.rm_final = p_in.a_final[a];
  p.n_qrm = p_in.a_nqrm[a];
  p.S4 = (long long)p_in.ncell * p.nQ * 4;
  tb.label += (size_t)a * p_in.ncell;
  tb.delta += (size_t)a * p_in.nd;
  tb.rq += (size_t)a * p_in.nd;
  tb.rcf += (size_t)a * p_in.nd;
  tb.qrm_states += (size_t)a * p_in.nQ;
  tb.phi += (size_t)a * 2 * p_in.nQ;
}
// Sweep handles: the learner settings of instance i's group replace the uniform ones in a copy `p` of the parameter block (one
// 64-byte load at kernel entry). `i` must be an instance of the launch. Kernels instantiated with SWEEP = false never call it,
// so their parameter block stays in the constant bank; the unfused entry points call it when sw.hyp is set.
__device__ __forceinline__ void apply_sweep(KP& p, const Sweep& sw, long long i) {
  p.h = sw.hyp[((long long)p.instance_offset + i) / sw.group];
}
__device__ __forceinline__ Acc make_acc(const KP& p, const DState& st, size_t base) {
  Acc acc = {nullptr, nullptr, nullptr, false, nullptr};
  if (p.shared_q && st.acc_sum) {
    acc.sum = st.acc_sum + base;
    acc.cnt = st.acc_cnt + base;
    acc.last = st.acc_last + base;
  }
  return acc;
}

