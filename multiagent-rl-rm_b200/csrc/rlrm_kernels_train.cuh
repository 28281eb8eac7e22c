// rlrm_kernels_train.cuh: fused persistent training kernels (generic train_kernel and the QRM nQ=4 fast path) — part of the single translation unit csrc/rlrm_b200.cu (see its header comment).
#pragma once
#include "rlrm_device.cuh"

// ------------------------------------------------------------------------------------------------
// fused persistent kernel: n_iters lockstep iterations, state in registers
// ------------------------------------------------------------------------------------------------
#define TRAIN_BLOCK 128
#ifndef QLF_MINB
#define QLF_MINB 8
#endif
// RLRM_PRESTEP(ENV): the specialised kernels fetch the current cell's move-table row and the slip index before the selection
// (agent_step<.., PRE = true>, see rlrm_device.cuh) so that action -> new cell is ALU-only. Measured A/B (profiles/r02c/
// r02c_prestep_ab.txt): OfficeWorld, where the chain is blocked-check -> slip -> move, gains 0.3-1.4 %; FrozenLake LOSES 0.2-1.5 %
// (config 3 headline 4.125e10 -> 4.065e10), so it is on for OfficeWorld only. -DRLRM_PRESTEP_ALL=0/1 forces it off / on.
// train_qrm4_kernel has its own table-driven step and does not use it (see there).
#ifdef RLRM_PRESTEP_ALL
#define RLRM_PRESTEP(ENV) (RLRM_PRESTEP_ALL != 0)
#else
#define RLRM_PRESTEP(ENV) ((ENV) == RLRM_ENV_OFFICE_WORLD)
#endif

// T = table arithmetic type (float: float32 tables; double: the reference's native float64 tables, see RT<T>)
// SWEEP: the handle carries per-group learner settings (rlrm_set_sweep); every fused kernel takes the flag the same way
template <int ENV, int ALGO, bool PA, typename T, bool SWEEP>
__global__ void __launch_bounds__(TRAIN_BLOCK, sizeof(T) == 4 ? 7 : 5) train_kernel(KP p_in, DState st, unsigned long long t0, int n_iters, int learn,
                                                           unsigned* trace, double* reward_out, Sweep sw) {
  typedef RT<T> R;
  typedef typename R::row_t row_t;
  KP p = p_in;
  Tab tb = stage_tables(p_in);
  // SWEEP: the instance's learner settings go into a separate copy read only where they are used (ph). The parameter block
  // (with PA, the per-agent view) is indexed dynamically (slip outcomes) and would move to local memory as a whole if it were written.
  KP p_sw;
  if (SWEEP) p_sw = p;
  const KP& ph = SWEEP ? p_sw : p;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = tid >> p.g_shift;
  const int a = (int)(tid & (p.G - 1));
  const bool valid = (i < st.N) && (a < p.A);
  const long long k = i * p.A + a;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned group_mask = (p.G == 32 ? 0xFFFFFFFFu : ((1u << p.G) - 1u)) << (lane & ~(unsigned)(p.G - 1));

  Slot s = {0, 0, 0, 0, 0};
  double eps = 0.0, ep_ret = 0.0;
  T* Q = nullptr;
  unsigned* V = nullptr;
  Acc acc = {nullptr, nullptr, nullptr, false, nullptr};
  unsigned long long active_steps = 0;
  unsigned episodes = 0, successes = 0, last_length = 0;
  double return_sum = 0.0;
  float last_return = 0.f;
  if (valid) {
    s = unpack_slot(st.slot[k]);
    eps = st.epsilon[k];
    if (st.ep_return) ep_ret = st.ep_return[k];
    if (st.stats) return_sum = st.stats[k].return_sum;
    if (PA) agent_view(p_in, p, tb, a);
    if (SWEEP) {
      p_sw = p;  // after the per-agent view
      apply_sweep(p_sw, sw, i);
    }
    const size_t base = table_base(p_in, i, a);
    Q = tab<T>(st.q) + base;
    V = st.visits ? st.visits + base : nullptr;
    acc = make_acc(p, st, base);
  }
  unsigned long long explore_thr = explore_threshold(eps);
  bool had_episode = false;
  // plain QL with a private table, fixed learning rate and no visit counts: carry the current row across iterations
  const bool carry = (ALGO == RLRM_ALGO_QL) && !V && !acc.sum && ph.h.lr >= 0.0;
  row_t row = R::zero_row();
  unsigned row_idx = 0xFFFFFFFFu;

  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    bool term = true, trunc = true;
    Rec r;
    int action = 0;
    if (valid) {
      unsigned w[4];
      RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
      // every agent selects on every iteration, finished ones included (frozen_lake_main.py:350-352)
      const unsigned cur_idx = s.cell * p.nQ + s.rm;
      if (cur_idx != row_idx) {  // plain QL carries the row of its current state in registers (1-entry cache of Q)
        row = load_row<T>(Q, cur_idx);
        row_idx = carry ? cur_idx : 0xFFFFFFFFu;
      }
      action = select_action(row, explore_thr, w, learn == 0, p.n_actions);
      const unsigned before = s.cell;
      const bool first = (s.flags & RLRM_FLAG_FIRST) != 0;
      agent_step<ENV>(p, tb, s, action, w[3], true, r);
      if (learn) {
        // FrozenLake driver: on an episode's first iteration `states` still aliases agent.state, so update_policy
        // receives the NEW position as `state` (frozen_lake_main.py:337,359 ; office_main.py:1700 deep-copies)
        const unsigned obs = (p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? r.cell : before;
        const bool term_arg = p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (r.term || r.trunc) : r.term;
        if (ALGO == RLRM_ALGO_QL && carry) {
          // update_q (qlearning.py:70-79) against the carried row: normally Q[s] is the carried row and only Q[s'] is loaded
          const unsigned sidx = obs * p.nQ + r.prev_q, snidx = r.cell * p.nQ + r.q;
          row_t nrow = (snidx == row_idx) ? row : load_row<T>(Q, snidx);
          const T cur = (sidx == row_idx) ? get_component(row, action)
                                               : ((sidx == snidx) ? get_component(nrow, action) : Q[(size_t)sidx * 4 + action]);
          double rew = r.reward;
          if (p.use_rsh) rew = __dadd_rn(rew, __dsub_rn(__dmul_rn(ph.h.gamma, tb.phi[p.phi_row + r.q]), tb.phi[p.phi_row + r.prev_q]));
          const T mf = R::mul(term_arg ? (T)0 : (T)1, row_max(nrow));
          const T inner = R::add(R::cvt(rew), R::mul(R::gamma(ph), mf));
          const T out = R::add(R::mul(R::one_minus_lr(ph), cur), R::mul(R::lr(ph), inner));
          if (!R::same_bits(out, cur)) Q[(size_t)sidx * 4 + action] = out;
          if (sidx == row_idx) set_component(row, action, out);
          if (snidx != row_idx) {  // the next state's row becomes the carried one
            if (sidx == snidx) set_component(nrow, action, out);
            row = nrow;
            row_idx = snidx;
          }
        } else {
          agent_update<ALGO, T>(ph, tb, Q, V, obs, action, term_arg, r, acc);
        }
      }
      term = r.term;
      trunc = r.trunc;
      ep_ret = __dadd_rn(ep_ret, r.reward);
      if (trace)
        trace[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = (unsigned)action | (r.executed << 3) | (r.cell << 6) | (r.q << 16) |
                                                             ((unsigned)r.term << 21) | ((unsigned)r.trunc << 22) |
                                                             ((unsigned)r.stepped << 23);
      if (reward_out) reward_out[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = r.reward;  // rewards[agent] of rm_env.step
    }
    // episode over when all agents terminated, or all truncated (frozen_lake_main.py:345,375 ; office_main.py:1748)
    const unsigned bt = __ballot_sync(0xFFFFFFFFu, term), bc = __ballot_sync(0xFFFFFFFFu, trunc);
    const bool over = ((bt & group_mask) == group_mask) || ((bc & group_mask) == group_mask);
    if (valid && over) {
      episodes++;
      active_steps += s.steps;  // env.agent_steps[agent] of the finished episode
      successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
      last_return = __double2float_rn(ep_ret);
      return_sum = __dadd_rn(return_sum, ep_ret);
      last_length = s.time;
      had_episode = true;
      ep_ret = 0.0;
      reset_slot(ph, tb, i, a, t + 1, s, eps);  // next episode starts with rm_env.reset (frozen_lake_main.py:337)
      explore_thr = explore_threshold(eps);
    }
  }
  if (valid) {
    st.slot[k] = pack_slot(s);
    st.epsilon[k] = eps;
    if (st.ep_return) st.ep_return[k] = ep_ret;
    if (st.stats) {
      rlrm_stats_t z = st.stats[k];
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

// ------------------------------------------------------------------------------------------------
// fast path: QRM with nQ == 4 (BASELINE configs 1/3/5). The 64-byte cell block Q[cell, 0..3, 0..3] lives in registers
// between iterations: it is fetched with two 256-bit loads only when the agent changes cell, the counterfactual
// updates run on registers, and the new values go back as scalar stores. Requires
// qrm_states == [0, 1, 2] (so a static unroll over rows is the reference's update order), per-instance
// tables, fixed learning rate, no visit counts; anything else takes train_kernel.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sel4(float a, float b, float c, float d, unsigned k) {
  const float lo = (k & 1u) ? b : a, hi = (k & 1u) ? d : c;
  return (k & 2u) ? hi : lo;
}
// 32-bit shared-memory loads from the staged table blob: train_qrm4_kernel keeps the blob's shared-window address in one
// register and adds section offsets from the parameter block, instead of carrying (or rebuilding) generic table pointers.
__device__ __forceinline__ unsigned smem_addr() { return (unsigned)__cvta_generic_to_shared(smem_raw); }
__device__ __forceinline__ unsigned lds_u16(unsigned a) {
  unsigned short v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ double lds_f64(unsigned a) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint4 lds_v4(unsigned a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
// B = the 64-byte block at `blk` if `take`, else unchanged: two predicated 256-bit loads, no branch
__device__ __forceinline__ void load_block4_if(const float* blk, bool take, float B[16]) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %17, 0;\n\t"
      "@p ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%16];\n\t"
      "@p ld.global.v8.f32 {%8,%9,%10,%11,%12,%13,%14,%15}, [%16+32];\n\t}"
      : "+f"(B[0]), "+f"(B[1]), "+f"(B[2]), "+f"(B[3]), "+f"(B[4]), "+f"(B[5]), "+f"(B[6]), "+f"(B[7]), "+f"(B[8]), "+f"(B[9]),
        "+f"(B[10]), "+f"(B[11]), "+f"(B[12]), "+f"(B[13]), "+f"(B[14]), "+f"(B[15])
      : "l"(blk), "r"((unsigned)take)
      : "memory");
}
// i * A + a of the calling thread from fresh special-register reads: a kernel that needs the slot index only before and after
// its loop recomputes it rather than holding two registers across the loop (a spill at the register cap)
__device__ __forceinline__ long long epilogue_slot(const KP& p) {
  unsigned tx, bx;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tx));
  asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(bx));
  const long long tid = (long long)bx * TRAIN_BLOCK + tx;
  return (tid >> p.g_shift) * p.A + (int)(tid & (p.G - 1));
}
__device__ __forceinline__ float max4(const float* v) { return fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])); }

// STOCH / LEARN / TRACE are compile-time copies of p.stochastic / learn / (trace != nullptr): the loop body is latency- and
// issue-bound, so runtime flag tests and their constant-bank loads are specialised away. n_qrm is 3 on this path.
// MINB = resident blocks per SM the register allocation is sized for: 7 (72 registers) when the whole batch fits in 28 warps
// per SM anyway (BASELINE config 3: 131,072 threads on 148 SMs), 8 (64 registers) when there are more threads than that and
// the extra resident warps pay (config 5).
//
// The env + reward-machine step reads rlrm_create's qrm4 sections (KP::off_q4cell / off_q4rec / off_q4rew) instead of
// label / cell_flags / delta / rq / rcf. For a cell, q4cell holds its event column times the number of env-reward classes
// (2 for FrozenLake: 0 or the hole penalty; 4 for OfficeWorld: 0, wall, plant, wall + plant) and the hole / plant flag in
// bit 15. Column and class select one 16-byte record: the three counterfactual rewards (float)(renv + rcf[u][col]) (rcf
// counts 0 without a transition) already rounded to float32, and a word with the counterfactual next states un(u) (2 bits
// each), "un(u) is final" (bits 6..8) and the next RM state of every current state (2 bits each from bit 12). q4rew holds the
// step reward renv + rq[rm][col] per (record, current state). Host double addition and (float) are the kernel's __dadd_rn
// and __double2float_rn, so every stored value is bit-identical to evaluating the tables here; the only float64 operation
// left in the loop is the episode-return sum.
//
// Loop shape: an iteration is three regions. (1) select, step, issue the (predicated) fetch of the next cell's block, then
// the work that does not read it: the Philox words of iteration t+1 and the slip threshold index (the counter depends on t
// alone and random starts are excluded, so an episode reset in between changes nothing) and the episode-return sum. (2) The
// episode-end reduction, a warp-wide shuffle outside the per-slot branches. (3) The counterfactual updates, which read the
// block. ptxas does not move instructions across these region boundaries, so the draws sit between the fetch and the first
// instruction that waits for it in every instantiation; within one region it would schedule them after the updates where
// registers are short (the 72-register MINB 7 case). The same-cell patches of the block are selects. Every Q store of
// iteration t precedes the fetch of t+1 in program order: an agent that steps back into the cell it just left must read
// what it wrote.
template <int ENV, bool STOCH, bool LEARN, bool TRACE, int MINB, bool SWEEP>
__global__ void __launch_bounds__(TRAIN_BLOCK, MINB) train_qrm4_kernel(KP p, DState st, unsigned long long t0, int n_iters,
                                                                unsigned* trace, Sweep sw) {
  Tab tb = stage_tables(p);
  const unsigned sm = smem_addr();
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = tid >> p.g_shift;
  const int a = (int)(tid & (p.G - 1));
  const bool valid = (i < st.N) && (a < p.A);
  const long long k = i * p.A + a;
  const unsigned n_cls = ENV == RLRM_ENV_FROZEN_LAKE ? 2u : 4u;  // env-reward classes per event column

  Slot s = {0, 0, 0, 0, 0};
  double eps = 0.0, ep_ret = 0.0, return_sum = 0.0;
  // first cell block of this slot's table, counted in 64-byte blocks: 32 bits suffice, as 2^32 blocks are 256 GiB
  unsigned qblk = 0u;
#define RLRM_Q4_BLOCK(cell) (st.q + (size_t)(qblk + (cell)) * 16)
  unsigned long long active_steps = 0;
  unsigned episodes = 0, successes = 0, last_length = 0;
  float last_return = 0.f;
  float B[16];  // carried cell block Q[cell, rm state, action]
#pragma unroll
  for (int j = 0; j < 16; j++) B[j] = 0.f;
  unsigned w[4] = {0u, 0u, 0u, 0u}, sidx = 0u;  // Philox words and slip threshold index of the coming iteration
  if (valid) {
    // nothing here indexes the parameter block dynamically: the written settings stay in registers, the rest in the constant bank
    if (SWEEP) apply_sweep(p, sw, i);
    s = unpack_slot(st.slot[k]);
    eps = st.epsilon[k];
    if (st.ep_return) ep_ret = st.ep_return[k];
    if (st.stats) return_sum = st.stats[k].return_sum;
    qblk = (unsigned)k * (unsigned)p.ncell;  // table_base(p, i, a) / 16 on this path
    load_block4_if(RLRM_Q4_BLOCK(s.cell), true, B);
    RLRM_PHILOX((unsigned)t0, (unsigned)(t0 >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
    if (STOCH) sidx = slip_index(p, w[3]);
  }
  unsigned long long explore_thr = explore_threshold(eps);
  bool had_episode = false;

  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    bool term = true, trunc = true;
    // what the counterfactual updates take from the step
    int action = 0;
    unsigned before = 0u;
    bool env_term = false, moved = false;
    uint4 rec = make_uint4(0u, 0u, 0u, 0u);
    float cur[3] = {0.f, 0.f, 0.f};
    if (valid) {
      float4 row;
      row.x = sel4(B[0], B[4], B[8], B[12], s.rm);
      row.y = sel4(B[1], B[5], B[9], B[13], s.rm);
      row.z = sel4(B[2], B[6], B[10], B[14], s.rm);
      row.w = sel4(B[3], B[7], B[11], B[15], s.rm);
      action = select_action(row, explore_thr, w, !LEARN, p.n_actions);
      // env.step + check_terminations (agent_step<ENV, STOCH>, table-driven; slip outcomes from KP::slip_nib)
#define RLRM_Q4_SLIP(x) ((unsigned)(p.slip_nib >> (((x) * 4 + sidx) * 4)) & 0xFu)
#define RLRM_Q4_NEXT(x) lds_u16(sm + p.off_next + (s.cell * 4 + (x)) * 2)
      before = s.cell;
      const bool active = (s.flags & RLRM_FLAG_ACTIVE) != 0;
      bool stepped;
      unsigned ex, cls, crec;
      if (ENV == RLRM_ENV_FROZEN_LAKE) {
        const bool rm_done = (int)s.rm == p.rm_final;  // ma_frozen_lake.py:107-115 (rm_final < 0 never matches)
        stepped = active && !rm_done;
        ex = STOCH ? RLRM_Q4_SLIP((unsigned)action) : (unsigned)action;
        const unsigned nc = RLRM_Q4_NEXT(ex & 3u);
        if (stepped && ex != RLRM_ACTION_WAIT) s.cell = nc;
        crec = lds_u16(sm + p.off_q4cell + s.cell * 2);
        const bool hole = stepped && (crec & 0x8000u);
        if (hole) s.flags |= RLRM_FLAG_FAIL;
        cls = hole ? 1u : 0u;
        s.steps += stepped ? 1u : 0u;
        s.time++;
        trunc = ((int)s.steps > p.max_steps) || ((int)s.time > p.max_steps);
        env_term = trunc || rm_done || (s.flags & RLRM_FLAG_FAIL);
        if (env_term) s.flags &= ~RLRM_FLAG_ACTIVE;
      } else {
        stepped = active;
        // the wall test and the move both follow from the action alone: two independent table loads
        const unsigned slipped = STOCH ? RLRM_Q4_SLIP((unsigned)action) : (unsigned)action;
        const unsigned nb = RLRM_Q4_NEXT((unsigned)action), nc = RLRM_Q4_NEXT(slipped & 3u);
        const bool blocked = active && nb == s.cell;  // apply_wall_penalty: "wait", no slip draw
        if (blocked && p.terminate_hit_walls) s.flags |= RLRM_FLAG_FAIL;
        ex = blocked ? (unsigned)RLRM_ACTION_WAIT : slipped;
        if (active && ex != RLRM_ACTION_WAIT) s.cell = nc;
        crec = lds_u16(sm + p.off_q4cell + s.cell * 2);
        const bool plant = active && (crec & 0x8000u);
        if (plant && p.terminate_on_plants) s.flags |= RLRM_FLAG_FAIL;
        cls = (blocked ? 1u : 0u) | (plant ? 2u : 0u);
        s.steps += active ? 1u : 0u;
        s.time++;
        trunc = (int)s.time > p.max_steps;
        env_term = (s.flags & RLRM_FLAG_FAIL) != 0;
        if (env_term || trunc) s.flags &= ~RLRM_FLAG_ACTIVE;
      }
#undef RLRM_Q4_SLIP
#undef RLRM_Q4_NEXT
      // RewardMachine.step + wrapper merge (rm_environment_wrapper.py:57-107) and the counterfactual inputs, one record
      const unsigned ri = (crec & 0x7FFFu) + cls;
      rec = lds_v4(sm + p.off_q4rec + ri * 16);
      const double reward = lds_f64(sm + p.off_q4rew + (ri * 4 + s.rm) * 8);
      s.rm = (rec.w >> (12 + 2 * s.rm)) & 3u;
      term = env_term || (int)s.rm == p.rm_final;
      s.flags &= ~(RLRM_FLAG_DONE | RLRM_FLAG_TRUNC | RLRM_FLAG_FIRST);
      if (term) s.flags |= RLRM_FLAG_DONE;
      if (trunc) s.flags |= RLRM_FLAG_TRUNC;
      if (TRACE)
        trace[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = (unsigned)action | ((stepped ? ex : 5u) << 3) | (s.cell << 6) |
                                                             (s.rm << 16) | ((unsigned)term << 21) | ((unsigned)trunc << 22) |
                                                             ((unsigned)stepped << 23);

      moved = s.cell != before;
      // values the updates overwrite, read before the carried block is replaced
#pragma unroll
      for (int u = 0; u < 3; u++) cur[u] = sel4(B[4 * u], B[4 * u + 1], B[4 * u + 2], B[4 * u + 3], (unsigned)action);
      load_block4_if(RLRM_Q4_BLOCK(s.cell), moved, B);  // the carried block becomes the NEXT cell's block
      // the next iteration's draws, independent of the block in flight
      {
        const unsigned long long tn = t + 1ull;
        RLRM_PHILOX((unsigned)tn, (unsigned)(tn >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
        if (STOCH) sidx = slip_index(p, w[3]);
      }
      ep_ret = __dadd_rn(ep_ret, reward);
    }
    // episode over <=> every agent of the instance terminated, or every agent truncated: AND-reduce the two flags (packed in
    // one word) over the instance's lane group with a fixed xor butterfly; a step at a distance of G or more is masked off
    unsigned flags2 = (term ? 1u : 0u) | (trunc ? 2u : 0u);
#pragma unroll
    for (int o = 1; o < RLRM_MAX_AGENTS; o <<= 1) flags2 &= __shfl_xor_sync(0xFFFFFFFFu, flags2, o) | (o < p.G ? 0u : 3u);
    const bool over = flags2 != 0u;
    if (LEARN && valid) {
      // QRM counterfactual experiences (rm_environment_wrapper.py:122-183) applied by update_q (qlearning.py:70-106),
      // in get_all_states()[:-1] order == row order 0..n_qrm-1 on this path. The next state's row maximum comes from
      // the carried block: a different block when the agent moved, else the live one including earlier updates.
      float bmax[4];
#pragma unroll
      for (int r = 0; r < 4; r++) bmax[r] = max4(B + 4 * r);
      float* dst = RLRM_Q4_BLOCK(before) + action;  // infos["prev_s"] is the position before the move
      const float cf[3] = {__uint_as_float(rec.x), __uint_as_float(rec.y), __uint_as_float(rec.z)};
#pragma unroll
      for (int u = 0; u < 3; u++) {
        const unsigned un = (rec.w >> (2 * u)) & 3u;
        const bool done = env_term || ((rec.w >> (6 + u)) & 1u);
        const float mx = sel4(bmax[0], bmax[1], bmax[2], bmax[3], un);
        const float mf = __fmul_rn(done ? 0.0f : 1.0f, mx);
        const float inner = __fadd_rn(cf[u], __fmul_rn(p.h.gamma_f, mf));
        const float nv = __fadd_rn(__fmul_rn(p.h.one_minus_lr_f, cur[u]), __fmul_rn(p.h.lr_f, inner));
        if (__float_as_uint(nv) != __float_as_uint(cur[u])) dst[4 * u] = nv;  // a bit-identical value needs no store
        // same cell: the carried block is the one just written
#pragma unroll
        for (int c = 0; c < 4; c++) B[4 * u + c] = (!moved && c == action) ? nv : B[4 * u + c];
        if (u < 2) bmax[u] = max4(B + 4 * u);
      }
    }
    if (valid && over) {
      episodes++;
      active_steps += s.steps;  // env.agent_steps[agent] of the finished episode
      successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
      last_return = __double2float_rn(ep_ret);
      return_sum = __dadd_rn(return_sum, ep_ret);
      last_length = s.time;
      had_episode = true;
      ep_ret = 0.0;
      reset_slot<false>(p, tb, i, a, t + 1, s, eps);
      explore_thr = explore_threshold(eps);
      load_block4_if(RLRM_Q4_BLOCK(s.cell), true, B);
    }
  }
#undef RLRM_Q4_BLOCK
  if (valid) {
    const long long ko = epilogue_slot(p);
    st.slot[ko] = pack_slot(s);
    st.epsilon[ko] = eps;
    if (st.ep_return) st.ep_return[ko] = ep_ret;
    if (st.stats) {
      rlrm_stats_t z = st.stats[ko];
      z.active_steps += active_steps;
      z.episodes += episodes;
      z.successes += successes;
      z.return_sum = return_sum;
      if (had_episode) {
        z.last_return = last_return;
        z.last_length = last_length;
      }
      st.stats[ko] = z;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fast path: QRM with NQ = 3 or 5 reward-machine states (OfficeWorld's built-in tasks exp0-exp4). Same scheme as
// train_qrm4_kernel — the cell block Q[cell, 0..NQ-1, 0..3] lives in registers between iterations, it is re-fetched (NQ 16-byte
// loads) only when the agent changes cell, the NQ-1 counterfactual updates run on registers in get_all_states()[:-1] order and
// go back as scalar stores — with the state count as a template parameter. Requires qrm_states == [0 .. NQ-2].
// ------------------------------------------------------------------------------------------------
template <int NQ>
__device__ __forceinline__ float sel_state(const float* v, int stride, unsigned k) {  // v[k * stride], k < NQ, without indexing
  float r = v[0];
#pragma unroll
  for (int j = 1; j < NQ; j++) r = (k == (unsigned)j) ? v[j * stride] : r;
  return r;
}
template <int NQ>
__device__ __forceinline__ void load_block_n(const float* Q, unsigned cell, float* B, float* bmax) {
  const float4* src = reinterpret_cast<const float4*>(Q + (size_t)cell * (NQ * 4));
#pragma unroll
  for (int r = 0; r < NQ; r++) {
    const float4 v = src[r];
    B[4 * r] = v.x;
    B[4 * r + 1] = v.y;
    B[4 * r + 2] = v.z;
    B[4 * r + 3] = v.w;
    bmax[r] = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
  }
}

template <int ENV, int NQ, bool STOCH, bool LEARN, bool TRACE, bool SWEEP>
__global__ void __launch_bounds__(TRAIN_BLOCK, 7) train_qrmn_kernel(KP p, DState st, unsigned long long t0, int n_iters, unsigned* trace,
                                                                   Sweep sw) {
  Tab tb = stage_tables(p);
  // SWEEP: the instance's learner settings go into a separate copy read only where they are used (ph). The parameter block
  // itself is indexed dynamically (slip outcomes) and would move to local memory as a whole if it were written.
  KP p_sw;
  if (SWEEP) p_sw = p;
  const KP& ph = SWEEP ? p_sw : p;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = tid >> p.g_shift;
  const int a = (int)(tid & (p.G - 1));
  const bool valid = (i < st.N) && (a < p.A);
  const long long k = i * p.A + a;

  Slot s = {0, 0, 0, 0, 0};
  double eps = 0.0, ep_ret = 0.0, return_sum = 0.0;
  float* Q = st.q;
  unsigned long long active_steps = 0;
  unsigned episodes = 0, successes = 0, last_length = 0;
  float last_return = 0.f;
  float B[NQ * 4], bmax[NQ];  // carried cell block Q[cell, rm state, action] and its row maxima
#pragma unroll
  for (int j = 0; j < NQ * 4; j++) B[j] = 0.f;
#pragma unroll
  for (int j = 0; j < NQ; j++) bmax[j] = 0.f;
  if (valid) {
    if (SWEEP) apply_sweep(p_sw, sw, i);
    s = unpack_slot(st.slot[k]);
    eps = st.epsilon[k];
    if (st.ep_return) ep_ret = st.ep_return[k];
    if (st.stats) return_sum = st.stats[k].return_sum;
    Q = st.q + table_base(p, i, a);
    load_block_n<NQ>(Q, s.cell, B, bmax);
  }
  unsigned long long explore_thr = explore_threshold(eps);
  bool had_episode = false;

  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    bool term = true, trunc = true;
    if (valid) {
      unsigned w[4];
      RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
      const PreStep ps = RLRM_PRESTEP(ENV) ? pre_step(p, tb, s.cell, w[3], STOCH) : PreStep{0ull, 0u};
      float4 row;
      row.x = sel_state<NQ>(B + 0, 4, s.rm);
      row.y = sel_state<NQ>(B + 1, 4, s.rm);
      row.z = sel_state<NQ>(B + 2, 4, s.rm);
      row.w = sel_state<NQ>(B + 3, 4, s.rm);
      const int action = select_action(row, explore_thr, w, !LEARN, p.n_actions);
      const unsigned before = s.cell;
      Rec r;
      agent_step<ENV, STOCH, false, RLRM_PRESTEP(ENV)>(p, tb, s, action, w[3], true, r, ps);
      const bool moved = r.cell != before;
      float cur[NQ - 1];  // values the updates overwrite, read before the carried block is replaced
#pragma unroll
      for (int u = 0; u < NQ - 1; u++) cur[u] = sel4(B[4 * u], B[4 * u + 1], B[4 * u + 2], B[4 * u + 3], (unsigned)action);
      if (moved) load_block_n<NQ>(Q, r.cell, B, bmax);  // the carried block becomes the NEXT cell's block
      if (LEARN) {
        const int col = r.event == RLRM_EVENT_NONE ? p.nEv : (int)r.event;
        float* dst = Q + (size_t)before * (NQ * 4) + action;  // infos["prev_s"] is the position before the move
#pragma unroll
        for (int u = 0; u < NQ - 1; u++) {
          const unsigned d = tb.delta[u * (p.nEv + 1) + col];
          const unsigned un = d == RLRM_NO_TRANSITION ? (unsigned)u : d;
          const double ru = d == RLRM_NO_TRANSITION ? 0.0 : tb.rcf[u * (p.nEv + 1) + col];
          const bool done = r.env_term || (p.rm_final >= 0 && (int)un == p.rm_final);
          const float mx = sel_state<NQ>(bmax, 1, un);
          const float mf = __fmul_rn(done ? 0.0f : 1.0f, mx);
          const float inner = __fadd_rn(__double2float_rn(__dadd_rn(r.renv, ru)), __fmul_rn(ph.h.gamma_f, mf));
          const float nv = __fadd_rn(__fmul_rn(ph.h.one_minus_lr_f, cur[u]), __fmul_rn(ph.h.lr_f, inner));
          if (__float_as_uint(nv) != __float_as_uint(cur[u])) dst[4 * u] = nv;  // a bit-identical value needs no store
          if (!moved) {  // same cell: the carried block is the one just written
#pragma unroll
            for (int c = 0; c < 4; c++) B[4 * u + c] = (c == action) ? nv : B[4 * u + c];
            bmax[u] = fmaxf(fmaxf(B[4 * u], B[4 * u + 1]), fmaxf(B[4 * u + 2], B[4 * u + 3]));
          }
        }
      }
      term = r.term;
      trunc = r.trunc;
      ep_ret = __dadd_rn(ep_ret, r.reward);
      if (TRACE)
        trace[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = (unsigned)action | (r.executed << 3) | (r.cell << 6) | (r.q << 16) |
                                                             ((unsigned)r.term << 21) | ((unsigned)r.trunc << 22) |
                                                             ((unsigned)r.stepped << 23);
    }
    unsigned flags2 = (term ? 1u : 0u) | (trunc ? 2u : 0u);
    for (int o = 1; o < p.G; o <<= 1) flags2 &= __shfl_xor_sync(0xFFFFFFFFu, flags2, o);
    const bool over = flags2 != 0u;
    if (valid && over) {
      episodes++;
      active_steps += s.steps;
      successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
      last_return = __double2float_rn(ep_ret);
      return_sum = __dadd_rn(return_sum, ep_ret);
      last_length = s.time;
      had_episode = true;
      ep_ret = 0.0;
      reset_slot<false>(ph, tb, i, a, t + 1, s, eps);
      explore_thr = explore_threshold(eps);
      load_block_n<NQ>(Q, s.cell, B, bmax);
    }
  }
  if (valid) {
    st.slot[k] = pack_slot(s);
    st.epsilon[k] = eps;
    if (st.ep_return) st.ep_return[k] = ep_ret;
    if (st.stats) {
      rlrm_stats_t z = st.stats[k];
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

// ------------------------------------------------------------------------------------------------
// fast path: QRM with MORE than five reward-machine states (OfficeWorld exp5 / exp6: 9 / 10 states, BASELINE config 4's
// 12-state machine with the QRM learner). The generic kernel issues, per counterfactual state, a dependent load -> update ->
// store chain on global memory (ncu: 81 % of the warp time on the long scoreboard, issue slots 22 % busy). Here the cell block
// Q[cell, 0..nQ-1, 0..3] of the agent's current cell lives in SHARED memory (16*nQ bytes per thread, laid out [row][thread]
// so that every access is a conflict-free 16-byte one): it is (re)fetched with one cp.async per row — all rows in flight at
// once, no registers — only when the agent changes cell; selection and the row maxima of the counterfactual targets are LDS;
// the new values go back to global memory as scalar stores and, when the agent stayed in its cell, into the shared block.
// A register-carried block (train_qrmn_kernel) would need 4*nQ + nQ registers; shared memory also makes the dynamic row
// index free, so qrm_states may be any permutation (the 12-state chain's index map is lexicographic: q10 < q2).
// NU = compile-time bound on the number of counterfactual states (the values they overwrite are read into registers before
// the block is replaced). Supports shaping and random starts; per-agent machines / lr=None / shared tables stay generic.
// Also THE specialised QRM kernel of the float64 table mode (T = double, any 2..16 states incl. BASELINE config 3's four): a row is
// then two 16-byte chunks (8 cp.async per move for nQ = 4); config 3 on float64 tables: 1.45e10 (generic kernel) -> 2.27e10.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }
// the nQ rows of one cell block: global -> shared. QRMB_FETCH = 0 (default): one cp.async per row — all rows in flight, no
// registers; the data lands in shared memory per global sector (14 wavefronts per row, profiles/r02b). QRMB_FETCH = NB > 0:
// batches of NB 16-byte loads through registers + conflict-free 16-byte shared stores (4 wavefronts per row). Measured on
// exp6 / chain-12: cp.async 1.55e10 / 1.11e10; NB = 2: 1.31e10 / 0.93e10; NB = 4: 0.96e10 / 0.75e10 (one global latency per
// batch and, from NB = 3 on, spills under the 72-register budget) — the wavefronts cp.async wastes cost less than latency.
#ifndef QRMB_FETCH
#define QRMB_FETCH 0
#endif
#ifndef QRMB_MINB_F64
#define QRMB_MINB_F64 7
#endif
#define QRMB_MINB(T) (sizeof(T) == 4 ? 7 : QRMB_MINB_F64)  // resident blocks per SM the register allocation is sized for
// TMA = true: the cell block is fetched by ONE bulk copy per thread (cp.async.bulk, the TMA engine: no LSU / shared-memory wavefronts
// for the fetch) into a per-thread contiguous slot, completion through a per-thread mbarrier with expect_tx. The slot stride is the
// block size rounded up to 16 (mod 32) bytes, so that eight consecutive lanes' 16-byte accesses to one chunk index cover all 32
// banks. A bulk copy issues from the uniform datapath (per-lane copies become an ELECT / R2UR / UBLKCP loop, ~9 instructions per
// lane) and goes past the L1, so it only pays for LARGE blocks: measured +13.5 % at 192 bytes (12 states, float32), -8 % at 160,
// -50 % at 128 (profiles/r02c/r02c_tma_fetch_ab.txt, r02c_tma_dense.txt); the host picks it from 192 bytes on (RLRM_QRMB_TMA=0/1
// overrides). TMA = false: one cp.async per 16-byte chunk into the [chunk][thread] layout.
__host__ __device__ __forceinline__ int qrmb_slot_bytes(int block_bytes) { return ((block_bytes + 31) & ~31) | 16; }
__device__ __forceinline__ void fetch_cell_block_tma(uint4* blk, const void* src, int bytes, unsigned bar, unsigned& phase) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(blk);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // this thread's earlier generic accesses to the slot come first
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
  unsigned ok = 0;
  while (!ok)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(bar), "r"(phase) : "memory");
  phase ^= 1u;
}
__device__ __forceinline__ void fetch_cell_block(uint4* blk, const void* src_, int n_chunks) {  // n_chunks 16-byte pieces: nQ rows of float4, 2 * nQ of double4r
  const uint4* src = reinterpret_cast<const uint4*>(src_);
#if QRMB_FETCH == 0
  for (int c = 0; c < n_chunks; c++) cp_async16(blk + c * TRAIN_BLOCK, src + c);
  cp_async_wait_all();
#else
  constexpr int NB = QRMB_FETCH;  // chunks per batch
  for (int r0 = 0; r0 < n_chunks; r0 += NB) {
    uint4 v[NB];
#pragma unroll
    for (int k = 0; k < NB; k++)
      if (r0 + k < n_chunks) v[k] = src[r0 + k];
#pragma unroll
    for (int k = 0; k < NB; k++)
      if (r0 + k < n_chunks) blk[(r0 + k) * TRAIN_BLOCK] = v[k];
  }
#endif
}
// one table row of the shared-memory cell block: a float4 is one 16-byte chunk, a double4r two (chunk c of this thread lives at
// blk[c * TRAIN_BLOCK], so a warp's access to one chunk index is 32 consecutive 16-byte words: conflict-free)
template <typename T>
__device__ __forceinline__ T sel4t(T a, T b, T c, T d, unsigned k) {
  const T lo = (k & 1u) ? b : a, hi = (k & 1u) ? d : c;
  return (k & 2u) ? hi : lo;
}
template <typename T, int CS>  // CS: distance (in 16-byte units) between consecutive chunks of one thread
struct BlkRow;
template <int CS>
struct BlkRow<float, CS> {
  static constexpr int CH = 1;
  static __device__ __forceinline__ float4 load(const uint4* blk, unsigned r) { return *reinterpret_cast<const float4*>(blk + r * CS); }
  static __device__ __forceinline__ void set(uint4* blk, unsigned r, int a, float v) { reinterpret_cast<float*>(blk + r * CS)[a] = v; }
  static __device__ __forceinline__ float get(const uint4* blk, unsigned r, int a) {  // one element: the whole row is one 16-byte access anyway
    const float4 v = load(blk, r);
    return sel4t<float>(v.x, v.y, v.z, v.w, (unsigned)a);
  }
};
template <int CS>
struct BlkRow<double, CS> {
  static constexpr int CH = 2;
  static __device__ __forceinline__ double4r load(const uint4* blk, unsigned r) {
    const double2 lo = *reinterpret_cast<const double2*>(blk + (2 * r) * CS), hi = *reinterpret_cast<const double2*>(blk + (2 * r + 1) * CS);
    return double4r{lo.x, lo.y, hi.x, hi.y};
  }
  static __device__ __forceinline__ void set(uint4* blk, unsigned r, int a, double v) {
    reinterpret_cast<double*>(blk + (2 * r + ((unsigned)a >> 1)) * CS)[a & 1] = v;
  }
  static __device__ __forceinline__ double get(const uint4* blk, unsigned r, int a) {  // one 8-byte access instead of the row's two 16-byte ones
    return reinterpret_cast<const double*>(blk + (2 * r + ((unsigned)a >> 1)) * CS)[a & 1];
  }
};

// T = table type: float, or double for the reference's native float64 tables (a row is then two 16-byte chunks; BASELINE config 3's
// four-state machine in float64 takes this kernel too: 128 bytes of block per thread)
template <int ENV, int NU, typename T, bool TMA, bool SWEEP>
__global__ void __launch_bounds__(TRAIN_BLOCK, QRMB_MINB(T)) train_qrm_block_kernel(KP p, DState st, unsigned long long t0, int n_iters, int learn,
                                                                                unsigned* trace, Sweep sw) {
  typedef RT<T> R;
  typedef BlkRow<T, TMA ? 1 : TRAIN_BLOCK> BR;
  typedef typename R::row_t row_t;
  Tab tb = stage_tables(p);
  // SWEEP: the instance's learner settings go into a separate copy read only where they are used (ph). The parameter block
  // itself is indexed dynamically (slip outcomes) and would move to local memory as a whole if it were written.
  KP p_sw;
  if (SWEEP) p_sw = p;
  const KP& ph = SWEEP ? p_sw : p;
  unsigned char* area = smem_raw + ((p.blob_bytes + 15) & ~15);
  unsigned bar = 0, phase = 0;
  uint4* blk;
  if constexpr (TMA) {  // [TRAIN_BLOCK] mbarriers, then [TRAIN_BLOCK] per-thread slots
    bar = (unsigned)__cvta_generic_to_shared(area + threadIdx.x * 8);
    blk = reinterpret_cast<uint4*>(area + TRAIN_BLOCK * 8 + (size_t)threadIdx.x * qrmb_slot_bytes(p.nQ * 4 * (int)sizeof(T)));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
  } else {
    blk = reinterpret_cast<uint4*>(area) + threadIdx.x;  // 16-byte chunk c of this thread: blk[c * TRAIN_BLOCK]
  }
  const int blk_bytes = p.nQ * 4 * (int)sizeof(T);
  // (a macro, not a by-reference lambda: see the note in agent_step)
#define QRMB_FETCH_BLOCK(src)                                                         \
  do {                                                                               \
    if constexpr (TMA) fetch_cell_block_tma(blk, (src), blk_bytes, bar, phase);      \
    else fetch_cell_block(blk, (src), blk_bytes / 16);                               \
  } while (0)
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = tid >> p.g_shift;
  const int a = (int)(tid & (p.G - 1));
  const bool valid = (i < st.N) && (a < p.A);
  const long long k = i * p.A + a;
  const int nQ = p.nQ, nE1 = p.nEv + 1;

  Slot s = {0, 0, 0, 0, 0};
  double eps = 0.0, ep_ret = 0.0, return_sum = 0.0;
  T* Q = tab<T>(st.q);
  unsigned long long active_steps = 0;
  unsigned episodes = 0, successes = 0, last_length = 0;
  float last_return = 0.f;
  if (valid) {
    if (SWEEP) apply_sweep(p_sw, sw, i);
    s = unpack_slot(st.slot[k]);
    eps = st.epsilon[k];
    if (st.ep_return) ep_ret = st.ep_return[k];
    if (st.stats) return_sum = st.stats[k].return_sum;
    Q = tab<T>(st.q) + table_base(p, i, a);
    QRMB_FETCH_BLOCK(Q + (size_t)s.cell * (size_t)(nQ * 4));
  }
  unsigned long long explore_thr = explore_threshold(eps);
  bool had_episode = false;

  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    bool term = true, trunc = true;
    if (valid) {
      unsigned w[4];
      RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
      const PreStep ps = RLRM_PRESTEP(ENV) ? pre_step(p, tb, s.cell, w[3], p.stochastic != 0) : PreStep{0ull, 0u};
      const row_t row = BR::load(blk, s.rm);
      const int action = select_action(row, explore_thr, w, learn == 0, p.n_actions);
      const unsigned before = s.cell;
      Rec r;
      agent_step<ENV, -1, false, RLRM_PRESTEP(ENV)>(p, tb, s, action, w[3], true, r, ps);
      const bool moved = r.cell != before;
      if (learn) {
        T cur[NU];  // values the updates overwrite, read before the block is replaced
#pragma unroll
        for (int j = 0; j < NU; j++) cur[j] = BR::get(blk, j < p.n_qrm ? tb.qrm_states[j] : 0, action);
        if (moved) QRMB_FETCH_BLOCK(Q + (size_t)r.cell * (size_t)(nQ * 4));  // the shared block becomes the NEXT cell's block
        // QRM counterfactual experiences (rm_environment_wrapper.py:122-183) applied by update_q (qlearning.py:70-106) in
        // get_all_states()[:-1] order. The next state's row maximum comes from the shared block: the new cell's block when
        // the agent moved, else the live one including this step's earlier updates.
        const int col = r.event == RLRM_EVENT_NONE ? p.nEv : (int)r.event;
        T* dst = Q + (size_t)before * (size_t)(nQ * 4) + action;  // infos["prev_s"] is the position before the move
#pragma unroll
        for (int j = 0; j < NU; j++) {
          if (j < p.n_qrm) {
            const unsigned u = tb.qrm_states[j];
            const unsigned d = tb.delta[u * nE1 + col];
            const unsigned un = d == RLRM_NO_TRANSITION ? u : d;
            const double ru = d == RLRM_NO_TRANSITION ? 0.0 : tb.rcf[u * nE1 + col];
            const bool done = r.env_term || (p.rm_final >= 0 && (int)un == p.rm_final);
            double rew = __dadd_rn(r.renv, ru);
            if (p.use_rsh) rew = __dadd_rn(rew, __dsub_rn(__dmul_rn(ph.h.gamma, tb.phi[un]), tb.phi[u]));  // qlearning.py:93-105
            const T mf = R::mul(done ? (T)0 : (T)1, row_max(BR::load(blk, un)));
            const T inner = R::add(R::cvt(rew), R::mul(R::gamma(ph), mf));
            const T nv = R::add(R::mul(R::one_minus_lr(ph), cur[j]), R::mul(R::lr(ph), inner));
            if (!R::same_bits(nv, cur[j])) dst[4 * u] = nv;  // a bit-identical value needs no store
            if (!moved) BR::set(blk, u, action, nv);  // same cell: the shared block is the one just written
          }
        }
      } else if (moved) {
        QRMB_FETCH_BLOCK(Q + (size_t)r.cell * (size_t)(nQ * 4));
      }
      term = r.term;
      trunc = r.trunc;
      ep_ret = __dadd_rn(ep_ret, r.reward);
      if (trace)
        trace[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = (unsigned)action | (r.executed << 3) | (r.cell << 6) | (r.q << 16) |
                                                             ((unsigned)r.term << 21) | ((unsigned)r.trunc << 22) |
                                                             ((unsigned)r.stepped << 23);
    }
    unsigned flags2 = (term ? 1u : 0u) | (trunc ? 2u : 0u);
    for (int o = 1; o < p.G; o <<= 1) flags2 &= __shfl_xor_sync(0xFFFFFFFFu, flags2, o);
    const bool over = flags2 != 0u;
    if (valid && over) {
      episodes++;
      active_steps += s.steps;
      successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
      last_return = __double2float_rn(ep_ret);
      return_sum = __dadd_rn(return_sum, ep_ret);
      last_length = s.time;
      had_episode = true;
      ep_ret = 0.0;
      const unsigned old_cell = s.cell;
      reset_slot(ph, tb, i, a, t + 1, s, eps);
      explore_thr = explore_threshold(eps);
      if (s.cell != old_cell) QRMB_FETCH_BLOCK(Q + (size_t)s.cell * (size_t)(nQ * 4));
    }
  }
  if (valid) {
    st.slot[k] = pack_slot(s);
    st.epsilon[k] = eps;
    if (st.ep_return) st.ep_return[k] = ep_ret;
    if (st.stats) {
      rlrm_stats_t z = st.stats[k];
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

#undef QRMB_FETCH_BLOCK

// ------------------------------------------------------------------------------------------------
// fast path: plain Q-learning with a private table per (instance, agent), fixed learning rate, no visit counts, no shaping
// (BASELINE config 3's `use_qrm=0, lr=0.1` variant). Same algorithm as train_kernel's row-carry branch — the row of the
// agent's current state stays in registers, one 16-byte load of Q[s'] and at most one 4-byte store per step — with the
// run-time switches (stochastic / learn / trace / per-agent views / random starts / shared accumulators) compiled out.
// ------------------------------------------------------------------------------------------------
template <int ENV, bool STOCH, bool LEARN, bool TRACE, bool SWEEP>
__global__ void __launch_bounds__(TRAIN_BLOCK, QLF_MINB) train_ql_fast_kernel(KP p, DState st, unsigned long long t0, int n_iters,
                                                                   unsigned* trace, Sweep sw) {
  Tab tb = stage_tables(p);
  // SWEEP: the instance's learner settings go into a separate copy read only where they are used (ph). The parameter block
  // itself is indexed dynamically (slip outcomes) and would move to local memory as a whole if it were written.
  KP p_sw;
  if (SWEEP) p_sw = p;
  const KP& ph = SWEEP ? p_sw : p;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = tid >> p.g_shift;
  const int a = (int)(tid & (p.G - 1));
  const bool valid = (i < st.N) && (a < p.A);
  const long long k = i * p.A + a;

  Slot s = {0, 0, 0, 0, 0};
  double eps = 0.0, ep_ret = 0.0, return_sum = 0.0;
  float* Q = st.q;
  unsigned long long active_steps = 0;
  unsigned episodes = 0, successes = 0, last_length = 0;
  float last_return = 0.f;
  float4 row = make_float4(0.f, 0.f, 0.f, 0.f);  // Q[row_idx, :], the 1-entry register cache of the table
  unsigned row_idx = 0;
  if (valid) {
    if (SWEEP) apply_sweep(p_sw, sw, i);
    s = unpack_slot(st.slot[k]);
    eps = st.epsilon[k];
    if (st.ep_return) ep_ret = st.ep_return[k];
    if (st.stats) return_sum = st.stats[k].return_sum;
    Q = st.q + table_base(p, i, a);
    row_idx = s.cell * p.nQ + s.rm;
    row = *reinterpret_cast<const float4*>(Q + (size_t)row_idx * 4);
  }
  unsigned long long explore_thr = explore_threshold(eps);
  bool had_episode = false;

  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    bool term = true, trunc = true;
    if (valid) {
      unsigned w[4];
      RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
      const PreStep ps = RLRM_PRESTEP(ENV) ? pre_step(p, tb, s.cell, w[3], STOCH) : PreStep{0ull, 0u};
      const int action = select_action(row, explore_thr, w, !LEARN, p.n_actions);  // row_idx == enc(current state) here
      const unsigned before = s.cell;
      const bool first = (s.flags & RLRM_FLAG_FIRST) != 0;
      Rec r;
      agent_step<ENV, STOCH, false, RLRM_PRESTEP(ENV)>(p, tb, s, action, w[3], true, r, ps);
      const unsigned snidx = r.cell * p.nQ + r.q;
      float4 nrow = row;
      if (snidx != row_idx) nrow = *reinterpret_cast<const float4*>(Q + (size_t)snidx * 4);
      if (LEARN) {
        // update_q (qlearning.py:70-79). `state` is the previous observation, except on an episode's first iteration under
        // the FrozenLake driver where it aliases the new position (frozen_lake_main.py:337,359)
        const unsigned obs = (p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? r.cell : before;
        const bool term_arg = p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (r.term || r.trunc) : r.term;
        const unsigned sidx = obs * p.nQ + r.prev_q;
        // branch-free component picks: lanes of a warp hold different actions, a switch would serialise them
        const float row_a = sel4(row.x, row.y, row.z, row.w, (unsigned)action);
        const float nrow_a = sel4(nrow.x, nrow.y, nrow.z, nrow.w, (unsigned)action);
        float cur = (sidx == row_idx) ? row_a : nrow_a;
        if (sidx != row_idx && sidx != snidx) cur = Q[(size_t)sidx * 4 + action];  // only the aliased first iteration gets here
        const float mf = __fmul_rn(term_arg ? 0.0f : 1.0f, row_max(nrow));
        const float inner = __fadd_rn(__double2float_rn(r.reward), __fmul_rn(ph.h.gamma_f, mf));
        const float out = __fadd_rn(__fmul_rn(ph.h.one_minus_lr_f, cur), __fmul_rn(ph.h.lr_f, inner));
        if (__float_as_uint(out) != __float_as_uint(cur)) Q[(size_t)sidx * 4 + action] = out;
        const bool same = sidx == snidx;  // the updated entry belongs to the row carried into the next iteration
        nrow.x = (same && action == 0) ? out : nrow.x;
        nrow.y = (same && action == 1) ? out : nrow.y;
        nrow.z = (same && action == 2) ? out : nrow.z;
        nrow.w = (same && action == 3) ? out : nrow.w;
      }
      row = nrow;  // the next state's row is the one the next selection reads
      row_idx = snidx;
      term = r.term;
      trunc = r.trunc;
      ep_ret = __dadd_rn(ep_ret, r.reward);
      if (TRACE)
        trace[(size_t)it * (size_t)(st.N * p.A) + (size_t)k] = (unsigned)action | (r.executed << 3) | (r.cell << 6) | (r.q << 16) |
                                                             ((unsigned)r.term << 21) | ((unsigned)r.trunc << 22) |
                                                             ((unsigned)r.stepped << 23);
    }
    unsigned flags2 = (term ? 1u : 0u) | (trunc ? 2u : 0u);
    for (int o = 1; o < p.G; o <<= 1) flags2 &= __shfl_xor_sync(0xFFFFFFFFu, flags2, o);
    const bool over = flags2 != 0u;
    if (valid && over) {
      episodes++;
      active_steps += s.steps;  // env.agent_steps[agent] of the finished episode
      successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
      last_return = __double2float_rn(ep_ret);
      return_sum = __dadd_rn(return_sum, ep_ret);
      last_length = s.time;
      had_episode = true;
      ep_ret = 0.0;
      reset_slot<false>(ph, tb, i, a, t + 1, s, eps);
      explore_thr = explore_threshold(eps);
      row_idx = s.cell * p.nQ + s.rm;
      row = *reinterpret_cast<const float4*>(Q + (size_t)row_idx * 4);
    }
  }
  if (valid) {
    st.slot[k] = pack_slot(s);
    st.epsilon[k] = eps;
    if (st.ep_return) st.ep_return[k] = ep_ret;
    if (st.stats) {
      rlrm_stats_t z = st.stats[k];
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

// Q(lambda) fused: one block per instance, one warp per agent; the dense trace sweep is cooperative over the warp.
