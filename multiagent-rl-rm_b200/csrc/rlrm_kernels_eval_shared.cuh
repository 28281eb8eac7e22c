// rlrm_kernels_eval_shared.cuh: greedy evaluation and the shared-learner kernels — part of the single translation unit csrc/rlrm_b200.cu (see its header comment).
#pragma once
#include <cooperative_groups.h>

#include "rlrm_kernels_train.cuh"

// ------------------------------------------------------------------------------------------------
// greedy evaluation (test_policy_optima, evaluation_metrics.py:23-190): the driver loop with best=True and no update
// ------------------------------------------------------------------------------------------------
template <int ENV, bool PA, typename T>
__global__ void __launch_bounds__(TRAIN_BLOCK) eval_kernel(KP p_in, DState st, rlrm_eval_t* evs, unsigned long long t0, int n_iters,
                                                          int n_episodes, double gamma, double optimal_steps) {
  KP p = p_in;
  Tab tb = stage_tables(p_in);
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = tid >> p.g_shift;
  const int a = (int)(tid & (p.G - 1));
  const bool valid = (i < st.N) && (a < p.A);
  const long long k = i * p.A + a;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned group_mask = (p.G == 32 ? 0xFFFFFFFFu : ((1u << p.G) - 1u)) << (lane & ~(unsigned)(p.G - 1));
  Slot s = {0, 0, 0, 0, 0};
  rlrm_eval_t e;
  memset(&e, 0, sizeof(e));
  const T* Q = tab<T>(st.q);
  if (valid) {
    s = unpack_slot(st.slot[k]);
    e = evs[k];
    if (PA) agent_view(p_in, p, tb, a);
    Q = tab<T>(st.q) + table_base(p_in, i, a);
  }
  const unsigned w0[4] = {0, 0, 0, 0};
  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    bool term = true, trunc = true;
    const bool running = valid && (int)e.episodes < n_episodes;  // all agents of an instance finish episodes together
    if (running) {
      const typename RT<T>::row_t row = load_row<T>(Q, s.cell * p.nQ + s.rm);
      const int action = select_action(row, 0ull, w0, true, p.n_actions);
      unsigned w3 = 0;
      if (p.stochastic) {
        unsigned w[4];
        RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
        w3 = w[3];
      }
      Rec r;
      agent_step<ENV>(p, tb, s, action, w3, true, r);
      if (!e.in_success) {
        e.disc_return = __dadd_rn(e.disc_return, __dmul_rn(e.cum_gamma, r.reward));
        if (r.term && p.rm_final >= 0 && (int)r.q == p.rm_final) {
          e.successes++;
          e.in_success = 1;
        }
      }
      e.cum_gamma = __dmul_rn(e.cum_gamma, gamma);
      term = r.term;
      trunc = r.trunc;
    }
    const unsigned bt = __ballot_sync(0xFFFFFFFFu, term), bc = __ballot_sync(0xFFFFFFFFu, trunc);
    const bool over = ((bt & group_mask) == group_mask) || ((bc & group_mask) == group_mask);
    if (running && over) {
      const unsigned long long len = s.time;
      e.episodes++;
      e.return_sum = __dadd_rn(e.return_sum, e.disc_return);
      e.return_sqsum = __dadd_rn(e.return_sqsum, __dmul_rn(e.disc_return, e.disc_return));
      if (e.in_success) {
        e.len_sum += len;
        e.len_sqsum += len * len;
      }
      if (len > 0) e.arps_sum = __dadd_rn(e.arps_sum, __ddiv_rn(__ddiv_rn(e.disc_return, (double)len), optimal_steps));
      e.cum_gamma = 1.0;
      e.disc_return = 0.0;
      e.in_success = 0;
      double eps_unused = 0.0;
      KP q = p;
      q.decay_on_reset = 0;  // evaluation runs on a copy of the env: the training epsilon is not touched
      reset_slot(q, tb, i, a, t + 1, s, eps_unused);
    }
  }
  if (valid) {
    st.slot[k] = pack_slot(s);
    evs[k] = e;
  }
}

// ------------------------------------------------------------------------------------------------
// shared learner, fast path: ONE lockstep iteration over all instances by persistent blocks. The per-agent shared
// tables (A*S*4 floats, 25.6 KB for config 5) and the proposal accumulators live in SHARED memory: Q reads are LDS,
// proposals are shared-memory atomics, and each block flushes its non-empty accumulators to the global ones once.
// Integer sums make the result independent of the block/thread order (include/rlrm_b200.h "Shared learner").
// Slot state is streamed from HBM (8 B in + 8 B out per slot); statistics are only touched when an episode ends.
// ------------------------------------------------------------------------------------------------
#define SHARED_BLOCK 1024

template <int ENV, int ALGO>
__global__ void __launch_bounds__(SHARED_BLOCK, 1) shared_propose_kernel(KP p, DState st, unsigned long long t, int learn,
                                                                        unsigned* trace) {
  Tab tb = stage_tables(p);
  const int n_ent = p.A * (int)p.S4;
  float* Qs = reinterpret_cast<float*>(smem_raw + p.blob_bytes);
  unsigned long long* s_sum = reinterpret_cast<unsigned long long*>(Qs + n_ent);
  int* s_cnt = reinterpret_cast<int*>(s_sum + n_ent);
  float* s_last = reinterpret_cast<float*>(s_cnt + n_ent);
  float* s_rmax = s_last + n_ent;  // [n_ent / 4] max over actions of every row: one 4-byte read per counterfactual instead of 16
  for (int j = threadIdx.x; j < n_ent / 4; j += blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(st.q) + j);
    reinterpret_cast<float4*>(Qs)[j] = v;
    s_rmax[j] = row_max(v);
  }
  for (int j = threadIdx.x; j < n_ent; j += blockDim.x) {
    s_sum[j] = 0ull;
    s_cnt[j] = 0;
  }
  __syncthreads();

  const unsigned lane = threadIdx.x & 31u;
  const unsigned group_mask = (p.G == 32 ? 0xFFFFFFFFu : ((1u << p.G) - 1u)) << (lane & ~(unsigned)(p.G - 1));
  const long long total = st.N << p.g_shift;
  for (long long b0 = (long long)blockIdx.x * blockDim.x; b0 < total; b0 += (long long)gridDim.x * blockDim.x) {
    const long long tid = b0 + threadIdx.x;
    const long long i = tid >> p.g_shift;
    const int a = (int)(tid & (p.G - 1));
    const bool valid = (i < st.N) && (a < p.A);
    const long long k = i * p.A + a;
    bool term = true, trunc = true;
    Slot s = {0, 0, 0, 0, 0};
    double eps = 0.0;
    Rec r;
    r.reward = 0.0;
    if (valid) {
      s = unpack_slot(st.slot[k]);
      eps = st.epsilon[k];
      unsigned w[4];
      RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
      float* Q = Qs + (size_t)a * (size_t)p.S4;
      const float4 row = *reinterpret_cast<const float4*>(Q + (size_t)(s.cell * p.nQ + s.rm) * 4);
      const int action = select_action(row, explore_threshold(eps), w, learn == 0, p.n_actions);
      const unsigned before = s.cell;
      const bool first = (s.flags & RLRM_FLAG_FIRST) != 0;
      agent_step<ENV>(p, tb, s, action, w[3], true, r);
      if (learn) {
        const unsigned obs = (p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? r.cell : before;
        const bool term_arg = p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (r.term || r.trunc) : r.term;
        Acc acc = {reinterpret_cast<long long*>(s_sum) + (size_t)a * (size_t)p.S4, s_cnt + (size_t)a * (size_t)p.S4,
                   s_last + (size_t)a * (size_t)p.S4, true, s_rmax + (size_t)a * (size_t)(p.S4 / 4)};
        agent_update<ALGO, float>(p, tb, Q, nullptr, obs, action, term_arg, r, acc);
      }
      term = r.term;
      trunc = r.trunc;
      if (r.reward != 0.0 && st.ep_return) st.ep_return[k] = __dadd_rn(st.ep_return[k], r.reward);
      if (trace)
        trace[k] = (unsigned)action | (r.executed << 3) | (r.cell << 6) | (r.q << 16) | ((unsigned)r.term << 21) |
                   ((unsigned)r.trunc << 22) | ((unsigned)r.stepped << 23);
    }
    const unsigned bt = __ballot_sync(0xFFFFFFFFu, term), bc = __ballot_sync(0xFFFFFFFFu, trunc);
    const bool over = ((bt & group_mask) == group_mask) || ((bc & group_mask) == group_mask);
    if (valid) {
      if (over) {
        const double ret = st.ep_return ? st.ep_return[k] : 0.0;
        if (st.stats) {
          rlrm_stats_t z = st.stats[k];
          z.episodes++;
          z.active_steps += s.steps;
          z.successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
          z.last_return = __double2float_rn(ret);
          z.return_sum = __dadd_rn(z.return_sum, ret);
          z.last_length = s.time;
          st.stats[k] = z;
        }
        if (st.ep_return) st.ep_return[k] = 0.0;
        reset_slot(p, tb, i, a, t + 1, s, eps);
        st.epsilon[k] = eps;
      }
      st.slot[k] = pack_slot(s);
    }
  }
  __syncthreads();
  if (learn) {
    for (int j = threadIdx.x; j < n_ent; j += blockDim.x) {
      const int c = s_cnt[j];
      if (c) {
        atomicAdd(st.acc_cnt + j, c);
        atomicAdd(reinterpret_cast<unsigned long long*>(st.acc_sum) + j, s_sum[j]);
        st.acc_last[j] = s_last[j];  // only read back when the GLOBAL count is 1, i.e. exactly one block wrote it
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// shared learner, persistent path: n_iters synchronous lockstep iterations in ONE cooperative launch (one block per SM). The
// per-agent tables stay in shared memory for the whole launch; per iteration every block proposes into its shared-memory
// accumulators, flushes the non-empty ones into a GLOBAL accumulator set with integer atomics, the grid synchronises ONCE,
// and every block then folds the global sums into its own table copy (apply_shared_kernel's arithmetic, evaluated redundantly
// by all blocks from the same integers => identical copies). Three global accumulator sets are used round-robin: set
// it % 3 is filled in iteration it, read after that iteration's grid barrier, and cleared during iteration it + 1's read phase —
// its next fill (it + 3) is separated from the clearing by the barrier of it + 2, so one barrier per iteration suffices.
// Replaces 2 launches per iteration (shared_propose_kernel + apply_shared_kernel); results are bit-identical to them.
// ------------------------------------------------------------------------------------------------
template <int ENV, int ALGO>
__global__ void __launch_bounds__(SHARED_BLOCK, 1) shared_train_kernel(KP p, DState st, unsigned long long t0, int n_iters,
                                                                      unsigned long long* g_sum, int* g_cnt, float* g_last) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  Tab tb = stage_tables(p);
  const int n_ent = p.A * (int)p.S4;
  float* Qs = reinterpret_cast<float*>(smem_raw + p.blob_bytes);
  unsigned long long* s_sum = reinterpret_cast<unsigned long long*>(Qs + n_ent);
  int* s_cnt = reinterpret_cast<int*>(s_sum + n_ent);
  float* s_last = reinterpret_cast<float*>(s_cnt + n_ent);
  float* s_rmax = s_last + n_ent;
  for (int j = threadIdx.x; j < n_ent / 4; j += blockDim.x) {
    const float4 v = __ldcg(reinterpret_cast<const float4*>(st.q) + j);
    reinterpret_cast<float4*>(Qs)[j] = v;
    s_rmax[j] = row_max(v);
  }
  for (int j = threadIdx.x; j < n_ent; j += blockDim.x) {
    s_sum[j] = 0ull;
    s_cnt[j] = 0;
  }
  __syncthreads();

  const unsigned lane = threadIdx.x & 31u;
  const unsigned group_mask = (p.G == 32 ? 0xFFFFFFFFu : ((1u << p.G) - 1u)) << (lane & ~(unsigned)(p.G - 1));
  const long long total = st.N << p.g_shift;
  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    // ---- propose: same per-slot code as shared_propose_kernel ----
    // the slot word / epsilon of the NEXT slot this thread handles are fetched while the current one is processed (the
    // streamed state is the only HBM traffic of this kernel; unprefetched, its latency was the top stall: ncu source page)
    // slots -> blocks: either one contiguous, warp-aligned chunk per block walked with a block-wide stride (equal work per
    // block) or the classic grid-stride walk; p.shared_balanced picks (measured, see DESIGN.md)
    const long long chunk = (((total + gridDim.x - 1) / gridDim.x) + 31) & ~31ll;
    const long long stride = p.shared_balanced ? (long long)blockDim.x : (long long)gridDim.x * blockDim.x;
    const long long lo = p.shared_balanced ? (long long)blockIdx.x * chunk : (long long)blockIdx.x * blockDim.x;
    const long long hi = p.shared_balanced ? ((lo + chunk < total) ? lo + chunk : total) : total;
    unsigned long long w_next = 0ull;
    double eps_next = 0.0;
    {
      const long long tid = lo + threadIdx.x;
      const long long i = tid >> p.g_shift;
      const int a = (int)(tid & (p.G - 1));
      if (tid < hi && i < st.N && a < p.A) {
        w_next = st.slot[i * p.A + a];
        eps_next = st.epsilon[i * p.A + a];
      }
    }
    for (long long b0 = lo; b0 < hi; b0 += stride) {
      const long long tid = b0 + threadIdx.x;
      const long long i = tid >> p.g_shift;
      const int a = (int)(tid & (p.G - 1));
      const bool valid = (tid < hi) && (i < st.N) && (a < p.A);
      const long long k = i * p.A + a;
      bool term = true, trunc = true;
      Slot s = {0, 0, 0, 0, 0};
      double eps = 0.0;
      Rec r;
      r.reward = 0.0;
      const unsigned long long w_cur = w_next;
      const double eps_cur = eps_next;
      {
        const long long tn = tid + stride, in = tn >> p.g_shift;
        const int an = (int)(tn & (p.G - 1));
        if (tn < hi && in < st.N && an < p.A) {
          w_next = st.slot[in * p.A + an];
          eps_next = st.epsilon[in * p.A + an];
        }
      }
      if (valid) {
        s = unpack_slot(w_cur);
        eps = eps_cur;
        unsigned w[4];
        RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
        float* Q = Qs + (size_t)a * (size_t)p.S4;
        const float4 row = *reinterpret_cast<const float4*>(Q + (size_t)(s.cell * p.nQ + s.rm) * 4);
        const int action = select_action(row, explore_threshold(eps), w, false, p.n_actions);
        const unsigned before = s.cell;
        const bool first = (s.flags & RLRM_FLAG_FIRST) != 0;
        agent_step<ENV>(p, tb, s, action, w[3], true, r);
        const unsigned obs = (p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? r.cell : before;
        const bool term_arg = p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (r.term || r.trunc) : r.term;
        Acc acc = {reinterpret_cast<long long*>(s_sum) + (size_t)a * (size_t)p.S4, s_cnt + (size_t)a * (size_t)p.S4,
                   s_last + (size_t)a * (size_t)p.S4, true, s_rmax + (size_t)a * (size_t)(p.S4 / 4)};
        agent_update<ALGO, float>(p, tb, Q, nullptr, obs, action, term_arg, r, acc);
        term = r.term;
        trunc = r.trunc;
        if (r.reward != 0.0 && st.ep_return) st.ep_return[k] = __dadd_rn(st.ep_return[k], r.reward);
      }
      const unsigned bt = __ballot_sync(0xFFFFFFFFu, term), bc = __ballot_sync(0xFFFFFFFFu, trunc);
      const bool over = ((bt & group_mask) == group_mask) || ((bc & group_mask) == group_mask);
      if (valid) {
        if (over) {
          const double ret = st.ep_return ? st.ep_return[k] : 0.0;
          if (st.stats) {
            rlrm_stats_t z = st.stats[k];
            z.episodes++;
            z.active_steps += s.steps;
            z.successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
            z.last_return = __double2float_rn(ret);
            z.return_sum = __dadd_rn(z.return_sum, ret);
            z.last_length = s.time;
            st.stats[k] = z;
          }
          if (st.ep_return) st.ep_return[k] = 0.0;
          reset_slot(p, tb, i, a, t + 1, s, eps);
          st.epsilon[k] = eps;
        }
        st.slot[k] = pack_slot(s);
      }
    }
    __syncthreads();
    // ---- flush this block's proposals into global accumulator set `it % 3` (integer atomics: order-independent). All three
    // phases below work on whole table rows (4 entries, one 16-byte access per array) so that a thread's few rows are
    // independent vector accesses instead of a chain of dependent scalar ones ----
    const size_t cur = (size_t)(it % 3) * (size_t)n_ent, prev = (size_t)((it + 2) % 3) * (size_t)n_ent;
    for (int j = threadIdx.x; j < n_ent / 4; j += blockDim.x) {
      const int4 c = reinterpret_cast<const int4*>(s_cnt)[j];
      if (c.x | c.y | c.z | c.w) {
        const int cc[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int e = 0; e < 4; e++)
          if (cc[e]) {
            atomicAdd(g_cnt + cur + 4 * j + e, cc[e]);
            atomicAdd(g_sum + cur + 4 * j + e, s_sum[4 * j + e]);
            g_last[cur + 4 * j + e] = s_last[4 * j + e];  // only read back when the GLOBAL count is 1, i.e. exactly one block wrote it
            s_sum[4 * j + e] = 0ull;
          }
        reinterpret_cast<int4*>(s_cnt)[j] = make_int4(0, 0, 0, 0);
      }
    }
    grid.sync();
    // ---- apply: fold the global sums into this block's table copy (apply_shared_kernel's arithmetic) and refresh the row maxima ----
    for (int j = threadIdx.x; j < n_ent / 4; j += blockDim.x) {
      const int4 c = __ldcg(reinterpret_cast<const int4*>(g_cnt + cur) + j);
      if (c.x | c.y | c.z | c.w) {
        const int cc[4] = {c.x, c.y, c.z, c.w};
        const float4 last = __ldcg(reinterpret_cast<const float4*>(g_last + cur) + j);
        const ulonglong2 s01 = __ldcg(reinterpret_cast<const ulonglong2*>(g_sum + cur) + 2 * j);
        const ulonglong2 s23 = __ldcg(reinterpret_cast<const ulonglong2*>(g_sum + cur) + 2 * j + 1);
        const float ll[4] = {last.x, last.y, last.z, last.w};
        const unsigned long long ss[4] = {s01.x, s01.y, s23.x, s23.y};
        float4 q = reinterpret_cast<const float4*>(Qs)[j];
        float qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 4; e++) {
          if (cc[e] == 1) qq[e] = ll[e];
          else if (cc[e] > 1) qq[e] = __double2float_rn(__dmul_rn(__ddiv_rn((double)(long long)ss[e], (double)cc[e]), 9.5367431640625e-07));
        }
        q = make_float4(qq[0], qq[1], qq[2], qq[3]);
        reinterpret_cast<float4*>(Qs)[j] = q;
        s_rmax[j] = row_max(q);
      }
    }
    // the set filled in the PREVIOUS iteration has been read by every block (before this iteration's barrier): clear it
    if (it > 0)
      for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_ent / 4; j += (long long)gridDim.x * blockDim.x) {
        reinterpret_cast<int4*>(g_cnt + prev)[j] = make_int4(0, 0, 0, 0);
        reinterpret_cast<ulonglong2*>(g_sum + prev)[2 * j] = make_ulonglong2(0ull, 0ull);
        reinterpret_cast<ulonglong2*>(g_sum + prev)[2 * j + 1] = make_ulonglong2(0ull, 0ull);
      }
    __syncthreads();
  }
  // leave the tables in global memory and every accumulator set clean
  grid.sync();
  if (blockIdx.x == 0)
    for (int j = threadIdx.x; j < n_ent / 4; j += blockDim.x) reinterpret_cast<float4*>(st.q)[j] = reinterpret_cast<const float4*>(Qs)[j];
  if (n_iters > 0) {
    const size_t last = (size_t)((n_iters - 1) % 3) * (size_t)n_ent;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_ent; j += (long long)gridDim.x * blockDim.x) {
      g_cnt[last + j] = 0;
      g_sum[last + j] = 0ull;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// shared learner, persistent path for tables that do NOT fit in one SM's shared memory (21 bytes per entry: e.g. the 12-state
// OfficeWorld machine with four agents, 20,736 entries = 435 KB): the same algorithm as shared_train_kernel with the table rows,
// row maxima and proposal accumulators PARTITIONED over the CL thread blocks of a cluster — row R lives in block (R mod CL) at
// local row R / CL — and reached through distributed shared memory (cluster.map_shared_rank: remote LDS / atomics over the
// SM-to-SM network, ~215 cycles). Every cluster holds one complete copy; a block flushes / folds only the rows it owns, so the
// per-iteration reduction work is split CL ways. Barriers per iteration: cluster (proposals of all peers are in) -> grid (global
// sums complete) -> cluster (folded values visible to the peers). Launched cooperatively with a cluster dimension.
// ------------------------------------------------------------------------------------------------
template <int ENV, int ALGO, int CL>
__global__ void __launch_bounds__(SHARED_BLOCK, 1) shared_train_cluster_kernel(KP p, DState st, unsigned long long t0, int n_iters,
                                                                              unsigned long long* g_sum, int* g_cnt, float* g_last) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  cg::cluster_group cluster = cg::this_cluster();
  constexpr unsigned LOG = CL == 2 ? 1 : (CL == 4 ? 2 : 3);
  const unsigned rank = cluster.block_rank();
  Tab tb = stage_tables(p);
  const int n_ent = p.A * (int)p.S4;
  const int rows = n_ent / 4, rows_loc = (rows + CL - 1) / CL;
  float* Qs = reinterpret_cast<float*>(smem_raw + ((p.blob_bytes + 15) & ~15));                 // [rows_loc][4]
  unsigned long long* s_sum = reinterpret_cast<unsigned long long*>(Qs + rows_loc * 4);          // [rows_loc][4]
  int* s_cnt = reinterpret_cast<int*>(s_sum + rows_loc * 4);
  float* s_last = reinterpret_cast<float*>(s_cnt + rows_loc * 4);
  float* s_rmax = s_last + rows_loc * 4;                                                         // [rows_loc]
  for (int lr = threadIdx.x; lr < rows_loc; lr += blockDim.x) {
    const int R = lr * CL + (int)rank;
    const float4 v = R < rows ? __ldcg(reinterpret_cast<const float4*>(st.q) + R) : make_float4(0.f, 0.f, 0.f, 0.f);
    reinterpret_cast<float4*>(Qs)[lr] = v;
    s_rmax[lr] = row_max(v);
    reinterpret_cast<int4*>(s_cnt)[lr] = make_int4(0, 0, 0, 0);
    reinterpret_cast<ulonglong2*>(s_sum)[2 * lr] = make_ulonglong2(0ull, 0ull);
    reinterpret_cast<ulonglong2*>(s_sum)[2 * lr + 1] = make_ulonglong2(0ull, 0ull);
  }
  cluster.sync();

  // row R of a partitioned array whose local part starts at `base` (elements per row: `per`)
#define CL_ROW(base, R, per) cluster.map_shared_rank((base) + (size_t)((R) >> LOG) * (per), (R) & (CL - 1))
  const unsigned lane = threadIdx.x & 31u;
  const unsigned group_mask = (p.G == 32 ? 0xFFFFFFFFu : ((1u << p.G) - 1u)) << (lane & ~(unsigned)(p.G - 1));
  const long long total = st.N << p.g_shift;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const unsigned rows_per_agent = (unsigned)(p.S4 / 4);
  for (int it = 0; it < n_iters; it++) {
    const unsigned long long t = t0 + (unsigned long long)it;
    for (long long b0 = (long long)blockIdx.x * blockDim.x; b0 < total; b0 += stride) {
      const long long tid = b0 + threadIdx.x;
      const long long i = tid >> p.g_shift;
      const int a = (int)(tid & (p.G - 1));
      const bool valid = (i < st.N) && (a < p.A);
      const long long k = i * p.A + a;
      bool term = true, trunc = true;
      Slot s = {0, 0, 0, 0, 0};
      double eps = 0.0;
      Rec r;
      r.reward = 0.0;
      if (valid) {
        s = unpack_slot(st.slot[k]);
        eps = st.epsilon[k];
        unsigned w[4];
        RLRM_PHILOX((unsigned)t, (unsigned)(t >> 32), p.instance_offset + (unsigned)i, (unsigned)a, p, w);
        const unsigned R0 = (unsigned)a * rows_per_agent;  // first row of agent a's table
        const float4 row = *reinterpret_cast<const float4*>(CL_ROW(Qs, R0 + s.cell * p.nQ + s.rm, 4));
        const int action = select_action(row, explore_threshold(eps), w, false, p.n_actions);
        const unsigned before = s.cell;
        const bool first = (s.flags & RLRM_FLAG_FIRST) != 0;
        agent_step<ENV>(p, tb, s, action, w[3], true, r);
        // update_q as a proposal (rlrm_device.cuh update_q, shared-memory branch) on partitioned rows
        auto propose = [&](unsigned Rs, double rew, unsigned Rsn, bool terminated) {
          const float cur = CL_ROW(Qs, Rs, 4)[action];
          const float mx = *CL_ROW(s_rmax, Rsn, 1);
          const float mf = __fmul_rn(terminated ? 0.0f : 1.0f, mx);
          const float inner = __fadd_rn(__double2float_rn(rew), __fmul_rn(p.h.gamma_f, mf));
          const float out = __fadd_rn(__fmul_rn(p.h.one_minus_lr_f, cur), __fmul_rn(p.h.lr_f, inner));
          const unsigned long long v = (unsigned long long)__float2ll_rn(__fmul_rn(out, 1048576.0f));
          unsigned* wsum = reinterpret_cast<unsigned*>(CL_ROW(s_sum, Rs, 4) + action);
          const unsigned lo = (unsigned)v, hi = (unsigned)(v >> 32);
          const unsigned old = atomicAdd(wsum, lo);
          const unsigned up = hi + ((old + lo) < old ? 1u : 0u);
          if (up) atomicAdd(wsum + 1, up);
          atomicAdd(CL_ROW(s_cnt, Rs, 4) + action, 1);
          CL_ROW(s_last, Rs, 4)[action] = out;
        };
        if (ALGO == RLRM_ALGO_QRM) {
          const int col = r.event == RLRM_EVENT_NONE ? p.nEv : (int)r.event;
          for (int j = 0; j < p.n_qrm; j++) {
            const unsigned u = tb.qrm_states[j];
            const unsigned d = tb.delta[u * (p.nEv + 1) + col];
            const unsigned un = d == RLRM_NO_TRANSITION ? u : d;
            const double ru = d == RLRM_NO_TRANSITION ? 0.0 : tb.rcf[u * (p.nEv + 1) + col];
            const bool done = r.env_term || (p.rm_final >= 0 && (int)un == p.rm_final);
            double rew = __dadd_rn(r.renv, ru);
            if (p.use_rsh) rew = __dadd_rn(rew, __dsub_rn(__dmul_rn(p.h.gamma, tb.phi[un]), tb.phi[u]));
            propose(R0 + r.prev_cell * p.nQ + u, rew, R0 + r.cell * p.nQ + un, done);
          }
        } else {
          const unsigned obs = (p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN && first) ? r.cell : before;
          const bool term_arg = p.driver == RLRM_DRIVER_FROZEN_LAKE_MAIN ? (r.term || r.trunc) : r.term;
          double rew = r.reward;
          if (p.use_rsh) rew = __dadd_rn(rew, __dsub_rn(__dmul_rn(p.h.gamma, tb.phi[p.phi_row + r.q]), tb.phi[p.phi_row + r.prev_q]));
          propose(R0 + obs * p.nQ + r.prev_q, rew, R0 + r.cell * p.nQ + r.q, term_arg);
        }
        term = r.term;
        trunc = r.trunc;
        if (r.reward != 0.0 && st.ep_return) st.ep_return[k] = __dadd_rn(st.ep_return[k], r.reward);
      }
      const unsigned bt = __ballot_sync(0xFFFFFFFFu, term), bc = __ballot_sync(0xFFFFFFFFu, trunc);
      const bool over = ((bt & group_mask) == group_mask) || ((bc & group_mask) == group_mask);
      if (valid) {
        if (over) {
          const double ret = st.ep_return ? st.ep_return[k] : 0.0;
          if (st.stats) {
            rlrm_stats_t z = st.stats[k];
            z.episodes++;
            z.active_steps += s.steps;
            z.successes += (p.rm_final >= 0 && (int)s.rm == p.rm_final) ? 1u : 0u;
            z.last_return = __double2float_rn(ret);
            z.return_sum = __dadd_rn(z.return_sum, ret);
            z.last_length = s.time;
            st.stats[k] = z;
          }
          if (st.ep_return) st.ep_return[k] = 0.0;
          reset_slot(p, tb, i, a, t + 1, s, eps);
          st.epsilon[k] = eps;
        }
        st.slot[k] = pack_slot(s);
      }
    }
    cluster.sync();  // every peer's proposals for the rows this block owns are in
    const size_t cur = (size_t)(it % 3) * (size_t)n_ent, prev = (size_t)((it + 2) % 3) * (size_t)n_ent;
    for (int lr = threadIdx.x; lr < rows_loc; lr += blockDim.x) {
      const int4 c = reinterpret_cast<const int4*>(s_cnt)[lr];
      if (c.x | c.y | c.z | c.w) {
        const size_t R = (size_t)lr * CL + rank;
        const int cc[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int e = 0; e < 4; e++)
          if (cc[e]) {
            atomicAdd(g_cnt + cur + 4 * R + e, cc[e]);
            atomicAdd(g_sum + cur + 4 * R + e, s_sum[4 * lr + e]);
            g_last[cur + 4 * R + e] = s_last[4 * lr + e];
            s_sum[4 * lr + e] = 0ull;
          }
        reinterpret_cast<int4*>(s_cnt)[lr] = make_int4(0, 0, 0, 0);
      }
    }
    grid.sync();
    for (int lr = threadIdx.x; lr < rows_loc; lr += blockDim.x) {
      const size_t R = (size_t)lr * CL + rank;
      if (R >= (size_t)rows) continue;
      const int4 c = __ldcg(reinterpret_cast<const int4*>(g_cnt + cur) + R);
      if (c.x | c.y | c.z | c.w) {
        const int cc[4] = {c.x, c.y, c.z, c.w};
        const float4 last = __ldcg(reinterpret_cast<const float4*>(g_last + cur) + R);
        const ulonglong2 s01 = __ldcg(reinterpret_cast<const ulonglong2*>(g_sum + cur) + 2 * R);
        const ulonglong2 s23 = __ldcg(reinterpret_cast<const ulonglong2*>(g_sum + cur) + 2 * R + 1);
        const float ll[4] = {last.x, last.y, last.z, last.w};
        const unsigned long long ss[4] = {s01.x, s01.y, s23.x, s23.y};
        float4 q = reinterpret_cast<const float4*>(Qs)[lr];
        float qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 4; e++) {
          if (cc[e] == 1) qq[e] = ll[e];
          else if (cc[e] > 1) qq[e] = __double2float_rn(__dmul_rn(__ddiv_rn((double)(long long)ss[e], (double)cc[e]), 9.5367431640625e-07));
        }
        q = make_float4(qq[0], qq[1], qq[2], qq[3]);
        reinterpret_cast<float4*>(Qs)[lr] = q;
        s_rmax[lr] = row_max(q);
      }
    }
    if (it > 0)
      for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_ent / 4; j += (long long)gridDim.x * blockDim.x) {
        reinterpret_cast<int4*>(g_cnt + prev)[j] = make_int4(0, 0, 0, 0);
        reinterpret_cast<ulonglong2*>(g_sum + prev)[2 * j] = make_ulonglong2(0ull, 0ull);
        reinterpret_cast<ulonglong2*>(g_sum + prev)[2 * j + 1] = make_ulonglong2(0ull, 0ull);
      }
    cluster.sync();  // the folded values of this block's rows are visible to its peers before they select / propose again
  }
#undef CL_ROW
  grid.sync();
  if (blockIdx.x < CL)  // the first cluster writes the tables back: every block its own rows
    for (int lr = threadIdx.x; lr < rows_loc; lr += blockDim.x) {
      const int R = lr * CL + (int)rank;
      if (R < rows) reinterpret_cast<float4*>(st.q)[R] = reinterpret_cast<const float4*>(Qs)[lr];
    }
  if (n_iters > 0) {
    const size_t last = (size_t)((n_iters - 1) % 3) * (size_t)n_ent;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_ent; j += (long long)gridDim.x * blockDim.x) {
      g_cnt[last + j] = 0;
      g_sum[last + j] = 0ull;
    }
  }
  cluster.sync();  // no block leaves while a peer could still address its shared memory
}

// shared learner: every touched entry becomes the mean of this iteration's proposals; accumulators are cleared
__global__ void __launch_bounds__(256) apply_shared_kernel(KP p, DState st) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= (p.per_agent ? p.sum4 : (long long)p.A * p.S4)) return;
  const int c = st.acc_cnt[j];
  if (c == 0) return;
  if (c == 1) st.q[j] = st.acc_last[j];
  else st.q[j] = __double2float_rn(__dmul_rn(__ddiv_rn((double)st.acc_sum[j], (double)c), 9.5367431640625e-07));
  st.acc_cnt[j] = 0;
  st.acc_sum[j] = 0;
}

