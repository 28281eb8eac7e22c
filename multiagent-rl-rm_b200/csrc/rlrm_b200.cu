// rlrm_b200.cu — hand-written CUDA (sm_100a) for the lockstep hot path of multiagent-rl-rm and its C ABI
// (include/rlrm_b200.h). One thread per (environment instance, agent); the map / label / Reward-Machine tables are
// staged once per block in shared memory; Q rows are 16-byte vector gathers/scatters on per-instance tables in HBM;
// randomness is Philox4x32-10 on (iteration, instance, agent) counters; per-instance episode termination is a warp
// ballot / xor-shuffle reduction over the instance's lane group. No tensor cores (nothing here is a contraction), no CPU
// fallback. This file is the single translation unit: device code lives in the rlrm_*.cuh headers next to it, the C ABI
// (handle, argument checks, launches) below.
//
// Reference semantics restated per function (R/ = /root/reference/multiagent_rlrm/):
//   env.step      R/environments/frozen_lake/ma_frozen_lake.py:96-154,189-215 ; office_world/ma_office.py:122-257
//   RM step       R/multi_agent/reward_machine.py:45-59
//   wrapper       R/multi_agent/wrappers/rm_environment_wrapper.py:43-107,122-183
//   select        R/learning_algorithms/qlearning.py:112-143
//   update        R/learning_algorithms/qlearning.py:70-110 ; qlearning_lambda.py:33-84
//   driver loops  R/environments/frozen_lake/frozen_lake_main.py:336-376 ; office_world/office_main.py:1696-1749
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/rlrm_b200.h"
#include "rlrm_device.cuh"
#include "rlrm_kernels_api.cuh"
#include "rlrm_kernels_train.cuh"
#include "rlrm_kernels_qlambda.cuh"
#include "rlrm_kernels_eval_shared.cuh"

// ------------------------------------------------------------------------------------------------
// host side: handle + C ABI
// ------------------------------------------------------------------------------------------------
struct rlrm_handle {
  KP kp;
  rlrm_config_t cfg;
  int device;
  unsigned char* d_blob;
  int smem_bytes;
  long long launches;
  int qrm4_fast;  // train_qrm4_kernel is applicable (see its header comment)
  int ql_fast;    // train_ql_fast_kernel is applicable (see its header comment)
  int qrmn_fast;  // train_qrmn_kernel<NQ = 3 or 5> is applicable (see its header comment)
  int qrmb_tma;   // train_qrm_block_kernel fetches the cell block with per-thread bulk copies (blocks of 192 bytes and more)
  int qrmb_fast;  // train_qrm_block_kernel is applicable (QRM, any state order, 6..16 RM states; see its header comment)
  int qrmb_smem;  // its dynamic shared memory: table blob + 16*nQ bytes per thread
  int shared_fast;       // shared_propose_kernel is applicable (tables + accumulators fit in shared memory)
  int shared_smem_bytes;
  unsigned char* d_coop;  // shared learner, persistent path: three global accumulator sets (sum i64 | count i32 | last f32), zeroed
  int coop_ok;            // cooperative launch is supported and the kernel attributes were set
  int shared_cluster;     // tables partitioned over a thread-block cluster of this many blocks (shared_train_cluster_kernel), 0 = not used
  int shared_cluster_smem;
  int num_sms;
  cudaStream_t pipe_stream[2];  // rlrm_train_host: copy-in / copy-out streams of the chunk pipeline (created on first use)
  cudaEvent_t pipe_event[3 * 8];
  int pipe_ready;
  int f64;        // float64 tables (cfg.table_dtype == RLRM_TABLE_F64): generic kernels instantiated on double
  int max_smem;   // cudaDevAttrMaxSharedMemoryPerBlockOptin of the device
  Hyp* d_sweep;   // rlrm_set_sweep: one Hyp per setting (device), null = uniform handle
  int n_sweep;
  long long sweep_group;
  int sweep_lr_none;  // some setting has learning_rate = None (needs state.visits)
};

// run STMT with T = float or double, whichever table type the handle was created for
#define RLRM_BY_T(h, ...)   \
  do {                      \
    if ((h)->f64) {         \
      typedef double T;     \
      __VA_ARGS__;          \
    } else {                \
      typedef float T;      \
      __VA_ARGS__;          \
    }                       \
  } while (0)

static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, const char* detail = "") {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}
#define CUDA_TRY(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) return fail(RLRM_ERR_CUDA, #expr ": %s", cudaGetErrorString(_e)); \
  } while (0)

static int align16(int x) { return (x + 15) & ~15; }

extern "C" int rlrm_abi_version(void) { return RLRM_ABI_VERSION; }
extern "C" const char* rlrm_last_error(void) { return g_err; }
extern "C" int rlrm_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

// the one place the learner constants are derived: the handle's uniform settings and every setting of a sweep
static void fill_learner(Hyp& hp, double lr, double gamma, double lambd, double eps_end, double eps_decay) {
  hp.lr = lr;
  hp.gamma = gamma;
  hp.eps_end = eps_end;
  hp.eps_decay = eps_decay;
  hp.lr_f = (float)lr;
  hp.one_minus_lr_f = (float)(1.0 - lr);
  hp.gamma_f = (float)gamma;
  hp.trace_decay_f = (float)(gamma * lambd);
  hp.one_minus_lr = 1.0 - lr;
  hp.trace_decay = gamma * lambd;
}
static Sweep sweep_of(const rlrm_handle* h) { return Sweep{h->d_sweep, h->sweep_group}; }

// Table CONTENTS are indices the kernels follow without bounds checks: reject anything out of range here, on the host.
static int validate_tables(const rlrm_config_t* cfg, const rlrm_tables_t* tb) {
  const int ncell = cfg->width * cfg->height, nQ = cfg->n_rm_states, nEv = cfg->n_events;
  const int sec = cfg->per_agent_rm ? cfg->n_agents : 1;
  for (int j = 0; j < ncell * 4; j++)
    if (tb->next_cell[j] >= ncell) return fail(RLRM_ERR_ARG, "tables.next_cell holds a cell index >= width*height");
  for (int a = 0; a < cfg->n_agents; a++)
    if (tb->start_cell[a] >= ncell) return fail(RLRM_ERR_ARG, "tables.start_cell holds a cell index >= width*height");
  for (int j = 0; j < ncell * sec; j++)
    if (tb->label[j] != RLRM_EVENT_NONE && tb->label[j] >= nEv) return fail(RLRM_ERR_ARG, "tables.label holds an event id >= n_events");
  for (int j = 0; j < nQ * (nEv + 1) * sec; j++)
    if (tb->delta[j] != RLRM_NO_TRANSITION && tb->delta[j] >= nQ) return fail(RLRM_ERR_ARG, "tables.delta holds a state index >= n_rm_states");
  if (cfg->rm_final >= nQ) return fail(RLRM_ERR_ARG, "rm_final >= n_rm_states");
  if (cfg->n_qrm_states > 0) {
    if (!tb->qrm_states) return fail(RLRM_ERR_ARG, "n_qrm_states > 0 needs tables.qrm_states");
    for (int s = 0; s < sec; s++) {
      const int n = cfg->per_agent_rm ? cfg->agent_n_qrm[s] : cfg->n_qrm_states;
      const int lim = cfg->per_agent_rm ? cfg->agent_n_rm_states[s] : nQ;
      for (int j = 0; j < n && j < nQ; j++)
        if (tb->qrm_states[(cfg->per_agent_rm ? s * nQ : 0) + j] >= lim) return fail(RLRM_ERR_ARG, "tables.qrm_states holds a state index out of range");
    }
  }
  if (cfg->random_starts)
    for (int j = 0; j < cfg->n_free_cells; j++)
      if (tb->free_cells[j] >= ncell) return fail(RLRM_ERR_ARG, "tables.free_cells holds a cell index >= width*height");
  for (int a = 0; a < 4; a++)
    for (int j = 0; j < 4; j++)
      if (cfg->slip_outcome[a][j] > RLRM_ACTION_WAIT) return fail(RLRM_ERR_ARG, "slip_outcome holds an action > RLRM_ACTION_WAIT");
  if (cfg->per_agent_rm)
    for (int a = 0; a < cfg->n_agents; a++) {
      if (cfg->agent_n_rm_states[a] < 1 || cfg->agent_n_rm_states[a] > nQ || cfg->agent_n_qrm[a] < 0 || cfg->agent_n_qrm[a] > nQ ||
          cfg->agent_rm_final[a] >= cfg->agent_n_rm_states[a])
        return fail(RLRM_ERR_ARG, "per-agent reward machine sizes out of range");
    }
  if (cfg->max_steps < 0 || cfg->max_steps > 65534) return fail(RLRM_ERR_ARG, "max_steps must be in 0..65534 (16-bit step counters)");
  return RLRM_OK;
}

// shared_train_cluster_kernel: attributes + cooperative cluster launch
template <int ENV, int ALGO, int CL>
static cudaError_t cluster_kernel_setup(int max_smem) {
  return cudaFuncSetAttribute(shared_train_cluster_kernel<ENV, ALGO, CL>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
}
template <int ENV, int ALGO, int CL>
static cudaError_t cluster_kernel_launch(const rlrm_handle* h, const KP& kp, const DState& d, unsigned long long t0, int n_iters, long long want_blocks,
                                         unsigned long long* g_sum, int* g_cnt, float* g_last, cudaStream_t s) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attrs[2];
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = CL; attrs[0].val.clusterDim.y = 1; attrs[0].val.clusterDim.z = 1;
  attrs[1].id = cudaLaunchAttributeCooperative;
  attrs[1].val.cooperative = 1;
  cfg.blockDim = dim3(SHARED_BLOCK);
  cfg.dynamicSmemBytes = (size_t)h->shared_cluster_smem;
  cfg.stream = s;
  cfg.attrs = attrs;
  cfg.numAttrs = 2;
  cfg.gridDim = dim3(CL);
  int max_clusters = 0;  // clusters that can be co-resident (a cooperative launch needs the whole grid resident)
  cudaError_t e = cudaOccupancyMaxActiveClusters(&max_clusters, shared_train_cluster_kernel<ENV, ALGO, CL>, &cfg);
  if (e != cudaSuccess) return e;
  if (max_clusters < 1) return cudaErrorLaunchOutOfResources;
  long long clusters = (want_blocks + CL - 1) / CL;
  if (clusters > max_clusters) clusters = max_clusters;
  if (clusters < 1) clusters = 1;
  cfg.gridDim = dim3((unsigned)(clusters * CL));
  return cudaLaunchKernelEx(&cfg, shared_train_cluster_kernel<ENV, ALGO, CL>, kp, d, t0, n_iters, g_sum, g_cnt, g_last);
}
#define RLRM_CLUSTER_DISPATCH(FN, ...)                                                                                        \
  (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE                                                                                    \
       ? (h->kp.algo == RLRM_ALGO_QRM ? RLRM_CLUSTER_CL(FN, RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QRM, __VA_ARGS__)                \
                                      : RLRM_CLUSTER_CL(FN, RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QL, __VA_ARGS__))                 \
       : (h->kp.algo == RLRM_ALGO_QRM ? RLRM_CLUSTER_CL(FN, RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QRM, __VA_ARGS__)               \
                                      : RLRM_CLUSTER_CL(FN, RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QL, __VA_ARGS__)))
#define RLRM_CLUSTER_CL(FN, ENV, ALGO, ...) \
  (h->shared_cluster == 2 ? FN<ENV, ALGO, 2>(__VA_ARGS__) : (h->shared_cluster == 4 ? FN<ENV, ALGO, 4>(__VA_ARGS__) : FN<ENV, ALGO, 8>(__VA_ARGS__)))

extern "C" int rlrm_create(const rlrm_config_t* cfg, const rlrm_tables_t* tb, int device, rlrm_handle_t** out) {
  if (!cfg || !tb || !out) return fail(RLRM_ERR_ARG, "null argument");
  if (cfg->abi_version != RLRM_ABI_VERSION) return fail(RLRM_ERR_ARG, "abi_version mismatch");
  const int ncell = cfg->width * cfg->height;
  if (ncell <= 0 || ncell > RLRM_MAX_CELLS) return fail(RLRM_ERR_ARG, "width*height out of range");
  if (cfg->n_agents < 1 || cfg->n_agents > RLRM_MAX_AGENTS) return fail(RLRM_ERR_ARG, "n_agents out of range");
  if (cfg->n_rm_states < 1 || cfg->n_rm_states > RLRM_MAX_RM_STATES) return fail(RLRM_ERR_ARG, "n_rm_states out of range");
  if (cfg->n_events < 0 || cfg->n_events > RLRM_MAX_EVENTS) return fail(RLRM_ERR_ARG, "n_events out of range");
  if (cfg->n_qrm_states < 0 || cfg->n_qrm_states > RLRM_MAX_RM_STATES) return fail(RLRM_ERR_ARG, "n_qrm_states out of range");
  if (cfg->slip_n < 1 || cfg->slip_n > 4) return fail(RLRM_ERR_ARG, "slip_n out of range");
  if (cfg->n_actions < 1 || cfg->n_actions > RLRM_N_ACTIONS) return fail(RLRM_ERR_ARG, "n_actions out of range");
  if (cfg->random_starts && (!tb || !tb->free_cells || cfg->n_free_cells < cfg->n_agents || cfg->n_free_cells > ncell))
    return fail(RLRM_ERR_ARG, "random_starts needs tables.free_cells with n_agents <= n_free_cells <= width*height");
  if (cfg->algo < 0 || cfg->algo > RLRM_ALGO_QLAMBDA) return fail(RLRM_ERR_ARG, "unknown algo");
  if (cfg->env_kind != RLRM_ENV_FROZEN_LAKE && cfg->env_kind != RLRM_ENV_OFFICE_WORLD) return fail(RLRM_ERR_ARG, "unknown env_kind");
  if (cfg->algo == RLRM_ALGO_QLAMBDA && cfg->shared_q) return fail(RLRM_ERR_UNSUPPORTED, "Q(lambda) with a shared table is not supported");
  if (cfg->table_dtype != RLRM_TABLE_F32 && cfg->table_dtype != RLRM_TABLE_F64) return fail(RLRM_ERR_ARG, "unknown table_dtype");
  if (cfg->table_dtype == RLRM_TABLE_F64 && cfg->shared_q)
    return fail(RLRM_ERR_UNSUPPORTED, "the shared learner is specified on float32 tables (fixed-point proposal sums of float32 values)");
  if (!tb->next_cell || !tb->cell_flags || !tb->label || !tb->delta || !tb->rq || !tb->rcf || !tb->start_cell)
    return fail(RLRM_ERR_ARG, "null table");
  if (int rc = validate_tables(cfg, tb)) return rc;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(RLRM_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(RLRM_ERR_ARG, "device out of range");
  CUDA_TRY(cudaSetDevice(device));

  rlrm_handle* h = new (std::nothrow) rlrm_handle();
  if (!h) return fail(RLRM_ERR_ARG, "out of host memory");
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg;
  if (getenv("RLRM_FORCE_GENERIC")) h->cfg.reserved |= 1;  // measurement switch: generic kernels only (same as reserved bit 0)
  h->device = device;
  h->f64 = cfg->table_dtype == RLRM_TABLE_F64;
  KP& kp = h->kp;
  kp.env_kind = cfg->env_kind; kp.driver = cfg->driver; kp.algo = cfg->algo;
  kp.A = cfg->n_agents;
  kp.G = 1; kp.g_shift = 0;
  while (kp.G < kp.A) { kp.G <<= 1; kp.g_shift++; }
  kp.nQ = cfg->n_rm_states; kp.nEv = cfg->n_events; kp.rm_final = cfg->rm_final; kp.n_qrm = cfg->n_qrm_states;
  kp.max_steps = cfg->max_steps; kp.ncell = ncell;
  kp.stochastic = cfg->stochastic; kp.slip_n = cfg->slip_n;
  for (int j = 0; j < 3; j++) kp.slip_thr[j] = cfg->slip_thr[j];
  kp.slip_cnt = 0;
  for (int j = 0; j + 1 < cfg->slip_n && j < 3; j++) {
    if (cfg->slip_thr[j] > 0xFFFFFFFFull) break;  // cumulative thresholds are non-decreasing
    kp.slip_thr32[j] = (unsigned)cfg->slip_thr[j];
    kp.slip_cnt = j + 1;
  }
  for (int j = kp.slip_cnt; j < 3; j++) kp.slip_thr32[j] = 0xFFFFFFFFu;  // padding for slip_index (see there)
  for (int a = 0; a < 4; a++)
    for (int j = 0; j < 4; j++) kp.slip_outcome[a * 4 + j] = cfg->slip_outcome[a][j];
  kp.slip_nib = 0ull;
  for (int k = 0; k < 16; k++) {
    // slip_index returns 3 for a draw of 0xFFFFFFFF whatever slip_cnt is; that draw selects outcome slip_cnt
    const int src = (k & 3) == 3 ? (k & ~3) + kp.slip_cnt : k;
    kp.slip_nib |= (unsigned long long)(kp.slip_outcome[src] & 0xF) << (4 * k);
  }
  kp.terminate_on_plants = cfg->terminate_on_plants; kp.terminate_hit_walls = cfg->terminate_hit_walls;
  kp.hole_penalty = cfg->hole_penalty; kp.wall_penalty = cfg->wall_penalty;
  fill_learner(kp.h, cfg->learning_rate, cfg->gamma, cfg->lambd, cfg->epsilon_end, cfg->epsilon_decay);
  kp.decay_on_reset = cfg->decay_on_reset; kp.shared_q = cfg->shared_q;
  {
    const char* e = getenv("RLRM_SHARED_BALANCED");  // tuning switch, see shared_train_kernel
    kp.shared_balanced = e ? atoi(e) : 0;
  }
  {  // sparse Q(lambda): lanes per agent (see train_qlambda_sparse_kernel); RLRM_QLS_LG overrides the default for A/B runs
    const int lg_max = 32 >> kp.g_shift;
    int lg = RLRM_QLS_LG_DEFAULT < lg_max ? RLRM_QLS_LG_DEFAULT : lg_max;
    const char* e = getenv("RLRM_QLS_LG");
    if (e && (atoi(e) == 4 || atoi(e) == 8 || atoi(e) == 16 || atoi(e) == 32)) lg = atoi(e) < lg_max ? atoi(e) : lg_max;
    kp.qls_lg = lg < 4 ? 4 : lg;
  }
  kp.use_rsh = (cfg->use_rsh && tb->phi) ? 1 : 0;
  kp.per_agent = cfg->per_agent_rm ? 1 : 0;
  kp.nd = kp.nQ * (kp.nEv + 1);
  kp.phi_row = kp.nQ;
  kp.sum4 = 0;
  for (int a = 0; a < kp.A; a++) {
    kp.a_nQ[a] = kp.per_agent ? cfg->agent_n_rm_states[a] : kp.nQ;
    kp.a_final[a] = kp.per_agent ? cfg->agent_rm_final[a] : kp.rm_final;
    kp.a_nqrm[a] = kp.per_agent ? cfg->agent_n_qrm[a] : kp.n_qrm;
    kp.a_prefix4[a] = kp.sum4;
    kp.sum4 += (long long)ncell * kp.a_nQ[a] * 4;
  }
  kp.random_starts = cfg->random_starts ? 1 : 0;
  kp.n_free = cfg->n_free_cells;
  kp.seed_lo = cfg->seed_lo; kp.seed_hi = cfg->seed_hi; kp.instance_offset = cfg->instance_offset;
  kp.n_actions = (unsigned)cfg->n_actions;
  for (int r = 0; r < 10; r++) {
    kp.rk[2 * r] = cfg->seed_lo + (unsigned)r * 0x9E3779B9u;
    kp.rk[2 * r + 1] = cfg->seed_hi + (unsigned)r * 0xBB67AE85u;
  }
  kp.S4 = (long long)ncell * kp.nQ * 4;

  const bool f32 = !h->f64;  // the specialised kernels exist for float32 tables
  h->qrm4_fast = (f32 && kp.algo == RLRM_ALGO_QRM && kp.nQ == 4 && kp.n_qrm == 3 && !kp.shared_q && !kp.use_rsh && !kp.random_starts && !kp.per_agent && cfg->learning_rate >= 0.0 &&
                  !(h->cfg.reserved & 1));
  for (int j = 0; j < kp.n_qrm; j++)
    if (!tb->qrm_states || tb->qrm_states[j] != j) h->qrm4_fast = 0;

  // pack the tables into one 16-byte aligned blob
  const int sec = kp.per_agent ? kp.A : 1;  // machine-dependent tables have one section per agent
  const int nd = kp.nQ * (kp.nEv + 1) * sec;
  const int q4_cls = kp.env_kind == RLRM_ENV_FROZEN_LAKE ? 2 : 4;  // train_qrm4_kernel: env-reward classes per event column
  const int q4_rec = h->qrm4_fast ? (kp.nEv + 1) * q4_cls : 0;
  int off = 0;
  kp.off_phi = off; off = align16(off + sec * 2 * RLRM_MAX_RM_STATES * 8);
  kp.off_rq = off; off = align16(off + nd * 8);
  kp.off_rcf = off; off = align16(off + nd * 8);
  kp.off_next = off; off = align16(off + ncell * 4 * 2);
  kp.off_start = off; off = align16(off + RLRM_MAX_AGENTS * 2);
  kp.off_flags = off; off = align16(off + ncell);
  kp.off_label = off; off = align16(off + ncell * sec);
  kp.off_delta = off; off = align16(off + nd);
  kp.off_qrm = off; off = align16(off + RLRM_MAX_RM_STATES * sec);
  kp.off_free = off; off = align16(off + (kp.random_starts ? kp.n_free : 0) * 2);
  kp.off_q4cell = off; off = align16(off + (q4_rec ? ncell : 0) * 2);
  kp.off_q4rec = off; off = align16(off + q4_rec * 16);
  kp.off_q4rew = off; off = align16(off + q4_rec * 4 * 8);
  kp.blob_bytes = off;
  if (off > 48 * 1024) {  // every kernel stages the blob in (non-opt-in) dynamic shared memory
    delete h;
    return fail(RLRM_ERR_UNSUPPORTED, "the table blob exceeds 48 KB of shared memory (too many per-agent reward-machine sections x states x events)");
  }
  unsigned char* host = new (std::nothrow) unsigned char[off];
  if (!host) { delete h; return fail(RLRM_ERR_ARG, "out of host memory"); }
  memset(host, 0, off);
  if (tb->phi) memcpy(host + kp.off_phi, tb->phi, (size_t)sec * kp.nQ * 2 * 8);
  memcpy(host + kp.off_rq, tb->rq, (size_t)nd * 8);
  memcpy(host + kp.off_rcf, tb->rcf, (size_t)nd * 8);
  memcpy(host + kp.off_next, tb->next_cell, (size_t)ncell * 8);
  memcpy(host + kp.off_start, tb->start_cell, (size_t)kp.A * 2);
  memcpy(host + kp.off_flags, tb->cell_flags, ncell);
  memcpy(host + kp.off_label, tb->label, (size_t)ncell * sec);
  memcpy(host + kp.off_delta, tb->delta, nd);
  if (kp.n_qrm > 0 && tb->qrm_states) memcpy(host + kp.off_qrm, tb->qrm_states, kp.per_agent ? (size_t)kp.nQ * sec : (size_t)kp.n_qrm);
  if (kp.random_starts) memcpy(host + kp.off_free, tb->free_cells, (size_t)kp.n_free * 2);
  if (q4_rec) {  // train_qrm4_kernel's step records; the layout is described at that kernel
    const int ncol = kp.nEv + 1;
    uint16_t* q4cell = reinterpret_cast<uint16_t*>(host + kp.off_q4cell);
    for (int c = 0; c < ncell; c++) {
      const int col = tb->label[c] == RLRM_EVENT_NONE ? kp.nEv : tb->label[c];
      q4cell[c] = (uint16_t)(col * q4_cls) | (uint16_t)((tb->cell_flags[c] & 1) << 15);
    }
    for (int col = 0; col < ncol; col++)
      for (int cls = 0; cls < q4_cls; cls++) {
        // renv as the kernels form it: FrozenLake r.renv = hole_penalty; OfficeWorld __dadd_rn(wall_pen, plant)
        const double renv = kp.env_kind == RLRM_ENV_FROZEN_LAKE ? (cls ? kp.hole_penalty : 0.0)
                                                                 : (cls & 1 ? kp.wall_penalty : 0.0) + (cls & 2 ? kp.hole_penalty : 0.0);
        const int ri = col * q4_cls + cls;
        float cf[3];
        uint32_t meta = 0;
        for (int u = 0; u < 3; u++) {
          const unsigned d = tb->delta[u * ncol + col];
          const unsigned un = d == RLRM_NO_TRANSITION ? (unsigned)u : d;
          cf[u] = (float)(renv + (d == RLRM_NO_TRANSITION ? 0.0 : tb->rcf[u * ncol + col]));
          meta |= un << (2 * u);
          if (kp.rm_final >= 0 && (int)un == kp.rm_final) meta |= 1u << (6 + u);
        }
        double* rew = reinterpret_cast<double*>(host + kp.off_q4rew) + ri * 4;
        for (int q = 0; q < 4; q++) {
          const unsigned d = tb->delta[q * ncol + col];
          meta |= (d == RLRM_NO_TRANSITION ? (unsigned)q : d) << (12 + 2 * q);
          rew[q] = renv + (d == RLRM_NO_TRANSITION ? 0.0 : tb->rq[q * ncol + col]);
        }
        unsigned char* r = host + kp.off_q4rec + ri * 16;
        memcpy(r, cf, 12);
        memcpy(r + 12, &meta, 4);
      }
  }
  cudaError_t e = cudaMalloc(&h->d_blob, off);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_blob, host, off, cudaMemcpyHostToDevice);
  delete[] host;
  if (e != cudaSuccess) { delete h; return fail(RLRM_ERR_CUDA, "table upload: %s", cudaGetErrorString(e)); }
  kp.blob = h->d_blob;
  h->smem_bytes = off;
  h->qrmn_fast = (f32 && kp.algo == RLRM_ALGO_QRM && (kp.nQ == 3 || kp.nQ == 5) && kp.n_qrm == kp.nQ - 1 && !kp.shared_q && !kp.use_rsh &&
                  !kp.random_starts && !kp.per_agent && cfg->learning_rate >= 0.0 && !(h->cfg.reserved & 1));
  for (int j = 0; j < kp.n_qrm; j++)
    if (!tb->qrm_states || tb->qrm_states[j] != j) h->qrmn_fast = 0;
  h->ql_fast = (f32 && kp.algo == RLRM_ALGO_QL && !kp.shared_q && !kp.use_rsh && !kp.random_starts && !kp.per_agent && cfg->learning_rate >= 0.0 &&
                !(h->cfg.reserved & 1));
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device);
  cudaDeviceGetAttribute(&h->max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  {  // cell-block fetch through per-thread bulk copies (TMA) from 192-byte blocks on: measured, see train_qrm_block_kernel
    const int block_bytes = kp.nQ * (h->f64 ? 32 : 16);
    h->qrmb_tma = block_bytes >= 192;
    const char* e = getenv("RLRM_QRMB_TMA");  // measurement switch
    if (e) h->qrmb_tma = atoi(e) != 0;
    h->qrmb_smem = h->qrmb_tma ? align16(off) + TRAIN_BLOCK * 8 + TRAIN_BLOCK * qrmb_slot_bytes(block_bytes) : align16(off) + block_bytes * TRAIN_BLOCK;
  }
  // float64 tables: the block kernel is the one specialised QRM kernel (the register-carried ones are float32-only)
  h->qrmb_fast = (kp.algo == RLRM_ALGO_QRM && !h->qrm4_fast && !h->qrmn_fast && kp.nQ >= 2 && kp.nQ <= 16 && kp.n_qrm >= 1 && kp.n_qrm <= 15 &&
                  !kp.shared_q && !kp.per_agent && cfg->learning_rate >= 0.0 && h->qrmb_smem <= h->max_smem && !(h->cfg.reserved & 1));
  if (h->qrmb_fast) {  // opt in to the device maximum (per function, only ever raised)
    cudaError_t e2 = cudaSuccess;
#define RLRM_OPTIN(K) if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem)
#define RLRM_OPTIN_T(T, M, SW)                                                                                                                             \
    RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_FROZEN_LAKE, 3, T, M, SW>)); RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_OFFICE_WORLD, 3, T, M, SW>));          \
    RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_FROZEN_LAKE, 7, T, M, SW>)); RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_FROZEN_LAKE, 11, T, M, SW>));         \
    RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_FROZEN_LAKE, 15, T, M, SW>)); RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_OFFICE_WORLD, 7, T, M, SW>));        \
    RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_OFFICE_WORLD, 11, T, M, SW>)); RLRM_OPTIN((train_qrm_block_kernel<RLRM_ENV_OFFICE_WORLD, 15, T, M, SW>))
#define RLRM_OPTIN_TS(T, M) RLRM_OPTIN_T(T, M, false); RLRM_OPTIN_T(T, M, true)  /* uniform and sweep instantiations */
    if (h->f64) { if (h->qrmb_tma) { RLRM_OPTIN_TS(double, true); } else { RLRM_OPTIN_TS(double, false); } }
    else { if (h->qrmb_tma) { RLRM_OPTIN_TS(float, true); } else { RLRM_OPTIN_TS(float, false); } }
#undef RLRM_OPTIN_TS
#undef RLRM_OPTIN_T
#undef RLRM_OPTIN
    if (e2 != cudaSuccess) h->qrmb_fast = 0;
  }
  {
    const long long n_ent = (long long)kp.A * kp.S4;
    const long long need = (long long)off + n_ent * 21;  // Q 4 B + sum 8 B + count 4 B + last 4 B per entry + row max 4 B per 4 entries
    h->shared_smem_bytes = (int)need;
    h->shared_fast = (kp.shared_q && !kp.per_agent && kp.algo != RLRM_ALGO_QLAMBDA && cfg->learning_rate >= 0.0 && need <= 227 * 1024 &&
                      !(h->cfg.reserved & 1));
    if (need > h->max_smem) h->shared_fast = 0;
    if (h->shared_fast) {
      // opt every instantiation in to the DEVICE maximum: the attribute is per function, not per handle, so a later handle
      // with a smaller table must never lower it under an earlier, larger one
      cudaError_t e1 = cudaFuncSetAttribute(shared_propose_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QRM>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(shared_propose_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QL>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(shared_propose_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QRM>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(shared_propose_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QL>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e1 != cudaSuccess) h->shared_fast = 0;
    }
    if (h->shared_fast) {  // persistent cooperative path
      int coop = 0;
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
      cudaError_t e3 = coop ? cudaSuccess : cudaErrorNotSupported;
      if (e3 == cudaSuccess) e3 = cudaFuncSetAttribute(shared_train_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QRM>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e3 == cudaSuccess) e3 = cudaFuncSetAttribute(shared_train_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QL>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e3 == cudaSuccess) e3 = cudaFuncSetAttribute(shared_train_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QRM>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e3 == cudaSuccess) e3 = cudaFuncSetAttribute(shared_train_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QL>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem);
      if (e3 == cudaSuccess) e3 = cudaMalloc(&h->d_coop, (size_t)3 * n_ent * 16);
      if (e3 == cudaSuccess) e3 = cudaMemset(h->d_coop, 0, (size_t)3 * n_ent * 16);
      h->coop_ok = e3 == cudaSuccess;
      cudaGetLastError();
    }
    // tables too large for one SM (or bit 2 of `reserved`: testing): partition them over a thread-block cluster
    const bool cluster_ok = kp.shared_q && !kp.per_agent && kp.algo != RLRM_ALGO_QLAMBDA && cfg->learning_rate >= 0.0 && !h->f64 && !(h->cfg.reserved & 1);
    int cl_min = 2;
    {
      const char* e = getenv("RLRM_SHARED_CLUSTER");  // tuning switch: force the cluster kernel with at least this many blocks per cluster
      if (e && atoi(e) >= 2) { cl_min = atoi(e) >= 8 ? 8 : (atoi(e) >= 4 ? 4 : 2); h->cfg.reserved |= 4; }
    }
    if (cluster_ok && (!h->shared_fast || (h->cfg.reserved & 4))) {
      int coop = 0;
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
      const long long rows = n_ent / 4;
      for (int cl = cl_min; cl <= 8 && coop && !h->shared_cluster; cl *= 2) {
        const long long smem = align16(off) + ((rows + cl - 1) / cl) * 84;  // per row: Q 16 + sums 32 + counts 16 + last 16 + row max 4
        if (smem <= h->max_smem) {
          h->shared_cluster = cl;
          h->shared_cluster_smem = (int)smem;
        }
      }
      if (h->shared_cluster) {
        cudaError_t e4 = RLRM_CLUSTER_DISPATCH(cluster_kernel_setup, h->max_smem);
        if (e4 == cudaSuccess && !h->d_coop) {
          e4 = cudaMalloc(&h->d_coop, (size_t)3 * n_ent * 16);
          if (e4 == cudaSuccess) e4 = cudaMemset(h->d_coop, 0, (size_t)3 * n_ent * 16);
        }
        if (e4 != cudaSuccess) h->shared_cluster = 0;
        cudaGetLastError();
      }
    }
  }
  *out = h;
  return RLRM_OK;
}

extern "C" int rlrm_destroy(rlrm_handle_t* h) {
  if (!h) return RLRM_OK;
  cudaSetDevice(h->device);
  if (h->d_blob) cudaFree(h->d_blob);
  if (h->d_coop) cudaFree(h->d_coop);
  if (h->d_sweep) cudaFree(h->d_sweep);
  if (h->pipe_ready) {
    for (int k = 0; k < 2; k++) cudaStreamDestroy(h->pipe_stream[k]);
    for (int k = 0; k < 3 * 8; k++) cudaEventDestroy(h->pipe_event[k]);
  }
  delete h;
  return RLRM_OK;
}

extern "C" int rlrm_set_learner(rlrm_handle_t* h, double learning_rate, double gamma, double lambd) {
  if (!h) return fail(RLRM_ERR_ARG, "null handle");
  if (h->d_sweep) return fail(RLRM_ERR_UNSUPPORTED, "rlrm_set_learner on a sweep handle: change the settings with rlrm_set_sweep");
  h->cfg.learning_rate = learning_rate; h->cfg.gamma = gamma; h->cfg.lambd = lambd;
  fill_learner(h->kp.h, learning_rate, gamma, lambd, h->kp.h.eps_end, h->kp.h.eps_decay);
  if (learning_rate < 0.0) h->qrm4_fast = h->ql_fast = h->qrmn_fast = h->qrmb_fast = 0;
  return RLRM_OK;
}

extern "C" int rlrm_set_sweep(rlrm_handle_t* h, const rlrm_hyper_t* sets, int32_t n_sets, int64_t group_size) {
  if (!h) return fail(RLRM_ERR_ARG, "null handle");
  if (n_sets < 0 || (n_sets > 0 && !sets)) return fail(RLRM_ERR_ARG, "rlrm_set_sweep: bad settings list");
  if (n_sets > 0 && h->cfg.shared_q) return fail(RLRM_ERR_UNSUPPORTED, "rlrm_set_sweep: instances of a shared table share one learner");
  if (n_sets > 0 && group_size <= 0) return fail(RLRM_ERR_ARG, "rlrm_set_sweep: group_size must be positive");
  CUDA_TRY(cudaSetDevice(h->device));
  Hyp* d = nullptr;
  int lr_none = 0;
  if (n_sets > 0) {
    Hyp* host = new (std::nothrow) Hyp[n_sets];
    if (!host) return fail(RLRM_ERR_ARG, "out of host memory");
    for (int g = 0; g < n_sets; g++) {
      fill_learner(host[g], sets[g].learning_rate, sets[g].gamma, sets[g].lambd, sets[g].epsilon_end, sets[g].epsilon_decay);
      lr_none |= sets[g].learning_rate < 0.0;
    }
    cudaError_t e = cudaMalloc(&d, (size_t)n_sets * sizeof(Hyp));
    if (e == cudaSuccess) e = cudaMemcpy(d, host, (size_t)n_sets * sizeof(Hyp), cudaMemcpyHostToDevice);
    delete[] host;
    if (e != cudaSuccess) {
      if (d) cudaFree(d);
      return fail(RLRM_ERR_CUDA, "rlrm_set_sweep: upload: %s", cudaGetErrorString(e));
    }
  }
  if (h->d_sweep) {
    CUDA_TRY(cudaDeviceSynchronize());  // launches already queued may still read the old settings
    cudaFree(h->d_sweep);
  }
  h->d_sweep = d;
  h->n_sweep = n_sets;
  h->sweep_group = n_sets > 0 ? group_size : 0;
  h->sweep_lr_none = lr_none;
  return RLRM_OK;
}

extern "C" int64_t rlrm_launch_count(const rlrm_handle_t* h) { return h ? (int64_t)h->launches : 0; }

static DState dstate(const rlrm_state_t* st) {
  DState d;
  d.N = st->n_instances; d.slot = (unsigned long long*)st->slot; d.epsilon = st->epsilon; d.q = (float*)st->q; d.e = (float*)st->e;
  d.visits = st->visits; d.ep_return = st->ep_return; d.stats = st->stats;
  d.acc_sum = (long long*)st->acc_sum; d.acc_cnt = st->acc_cnt; d.acc_last = st->acc_last;
  d.tr_pos = st->tr_pos; d.tr_idx = st->tr_idx; d.tr_eq = (float2*)st->tr_eq; d.tr_len = st->tr_len;
  d.tr_work = (unsigned long long*)st->tr_work; d.tr_cap = st->tr_cap;
  return d;
}
static DOut dout(const rlrm_step_out_t* o) {
  DOut d;
  memset(&d, 0, sizeof(d));
  if (o) {
    d.prev_cell = o->prev_cell; d.cell = o->cell; d.prev_q = o->prev_q; d.q = o->q; d.event = o->event; d.executed = o->executed;
    d.renv = o->renv; d.rq = o->rq; d.reward = o->reward; d.env_term = o->env_term; d.rm_term = o->rm_term; d.term = o->term;
    d.trunc = o->trunc; d.cf_q = o->cf_q; d.cf_r = o->cf_r;
  }
  return d;
}

static int check_state(const rlrm_handle_t* h, const rlrm_state_t* st, bool need_q) {
  if (!h || !st) return fail(RLRM_ERR_ARG, "null handle/state");
  if (st->n_instances <= 0) return fail(RLRM_ERR_ARG, "n_instances must be positive");
  if (!st->slot || !st->epsilon) return fail(RLRM_ERR_ARG, "state.slot / state.epsilon are required");
  if (need_q && !st->q) return fail(RLRM_ERR_ARG, "state.q is required");
  if (need_q && ((uintptr_t)st->q & 31u)) return fail(RLRM_ERR_ARG, "state.q must be 32-byte aligned");
  if (st->e && ((uintptr_t)st->e & (h->f64 ? 31u : 15u))) return fail(RLRM_ERR_ARG, "state.e must be 16-byte (float64 tables: 32-byte) aligned");
  if (need_q && h->cfg.algo == RLRM_ALGO_QLAMBDA && !st->e) {
    if (!st->tr_pos || !st->tr_idx || !st->tr_eq || !st->tr_len)
      return fail(RLRM_ERR_ARG, "Q(lambda) needs state.e (dense traces) or state.tr_* (sparse traces)");
    if (st->tr_cap < h->cfg.max_steps + 1) return fail(RLRM_ERR_ARG, "tr_cap must be >= max_steps + 1");
    if (h->kp.S4 > 65535) return fail(RLRM_ERR_UNSUPPORTED, "sparse traces need S*4 <= 65535");
  }
  if (need_q && (h->d_sweep ? h->sweep_lr_none : h->cfg.learning_rate < 0) && !st->visits)
    return fail(RLRM_ERR_ARG, "learning_rate=None needs state.visits");
  if (h->d_sweep && (long long)h->kp.instance_offset + st->n_instances > (long long)h->n_sweep * h->sweep_group)
    return fail(RLRM_ERR_ARG, "the sweep's settings do not cover instances [instance_offset, instance_offset + n_instances)");
  if (need_q && h->cfg.shared_q && h->cfg.learning_rate < 0) return fail(RLRM_ERR_UNSUPPORTED, "shared table with learning_rate=None");
  if (need_q && h->cfg.shared_q && (!st->acc_sum || !st->acc_cnt || !st->acc_last))
    return fail(RLRM_ERR_ARG, "shared_q needs state.acc_sum / acc_cnt / acc_last");
  return RLRM_OK;
}

#define LAUNCH_CHECK(h)                                                                     \
  do {                                                                                      \
    (h)->launches++;                                                                        \
    cudaError_t _e = cudaGetLastError();                                                    \
    if (_e != cudaSuccess) return fail(RLRM_ERR_CUDA, "kernel launch: %s", cudaGetErrorString(_e)); \
  } while (0)

static unsigned blocks_for(long long n, int block) { return (unsigned)((n + block - 1) / block); }

extern "C" int rlrm_reset_at(rlrm_handle_t* h, const rlrm_state_t* st, const uint8_t* mask, uint64_t t, void* stream);
extern "C" int rlrm_reset(rlrm_handle_t* h, const rlrm_state_t* st, const uint8_t* mask, void* stream) {
  return rlrm_reset_at(h, st, mask, 0, stream);
}

extern "C" int rlrm_reset_at(rlrm_handle_t* h, const rlrm_state_t* st, const uint8_t* mask, uint64_t t, void* stream) {
  int rc = check_state(h, st, false);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const long long n = st->n_instances * h->kp.A;
  reset_kernel<<<blocks_for(n, 256), 256, h->smem_bytes, s>>>(h->kp, dstate(st), mask, t, sweep_of(h));
  LAUNCH_CHECK(h);
  if (h->cfg.algo == RLRM_ALGO_QLAMBDA && st->e) {
    RLRM_BY_T(h, clear_traces_kernel<T><<<blocks_for(st->n_instances * ((h->kp.per_agent ? h->kp.sum4 : (long long)h->kp.A * h->kp.S4) / 4), 256), 256, 0, s>>>(h->kp, dstate(st), mask));
    LAUNCH_CHECK(h);
  } else if (h->cfg.algo == RLRM_ALGO_QLAMBDA && st->tr_pos && st->q) {
    RLRM_BY_T(h, qlambda_sparse_reset_kernel<T><<<blocks_for(n * 32, 256), 256, 0, s>>>(h->kp, dstate(st), mask));
    LAUNCH_CHECK(h);
  }
  return RLRM_OK;
}

extern "C" int rlrm_select_action(rlrm_handle_t* h, const rlrm_state_t* st, const uint32_t* draws, uint64_t t, int best,
                                  uint8_t* actions_out, void* stream) {
  int rc = check_state(h, st, true);
  if (rc) return rc;
  if (!actions_out) return fail(RLRM_ERR_ARG, "actions_out is null");
  CUDA_TRY(cudaSetDevice(h->device));
  const long long n = st->n_instances * h->kp.A;
  if (h->kp.per_agent) RLRM_BY_T(h, select_kernel<true, T><<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(h->kp, dstate(st), draws, t, best, actions_out));
  else RLRM_BY_T(h, select_kernel<false, T><<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(h->kp, dstate(st), draws, t, best, actions_out));
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_step(rlrm_handle_t* h, const rlrm_state_t* st, const uint8_t* actions, const uint32_t* draws, uint64_t t,
                         int with_rm, const rlrm_step_out_t* out, void* stream) {
  int rc = check_state(h, st, false);
  if (rc) return rc;
  if (!actions) return fail(RLRM_ERR_ARG, "actions is null");
  CUDA_TRY(cudaSetDevice(h->device));
  const long long n = st->n_instances * h->kp.A;
  cudaStream_t s = (cudaStream_t)stream;
#define RLRM_STEP(ENV, PA) step_kernel<ENV, PA><<<blocks_for(n, 256), 256, h->smem_bytes, s>>>(h->kp, dstate(st), actions, draws, t, with_rm, dout(out))
  if (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE) {
    if (h->kp.per_agent) RLRM_STEP(RLRM_ENV_FROZEN_LAKE, true); else RLRM_STEP(RLRM_ENV_FROZEN_LAKE, false);
  } else {
    if (h->kp.per_agent) RLRM_STEP(RLRM_ENV_OFFICE_WORLD, true); else RLRM_STEP(RLRM_ENV_OFFICE_WORLD, false);
  }
#undef RLRM_STEP
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_rm_step_agent(rlrm_handle_t* h, int agent, int64_t n_slots, uint8_t* q, const uint16_t* cell, uint8_t* event_out,
                                  double* reward_out, void* stream);
extern "C" int rlrm_rm_step(rlrm_handle_t* h, int64_t n_slots, uint8_t* q, const uint16_t* cell, uint8_t* event_out,
                            double* reward_out, void* stream) {
  return rlrm_rm_step_agent(h, 0, n_slots, q, cell, event_out, reward_out, stream);
}

extern "C" int rlrm_rm_step_agent(rlrm_handle_t* h, int agent, int64_t n_slots, uint8_t* q, const uint16_t* cell, uint8_t* event_out,
                                  double* reward_out, void* stream) {
  if (!h || !q || !cell) return fail(RLRM_ERR_ARG, "null argument");
  if (agent < 0 || agent >= h->kp.A) return fail(RLRM_ERR_ARG, "agent out of range");
  if (n_slots <= 0) return RLRM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  rm_step_kernel<<<blocks_for(n_slots, 256), 256, h->smem_bytes, (cudaStream_t)stream>>>(h->kp, agent, n_slots, q, cell, event_out, reward_out);
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_mdp(rlrm_handle_t* h, int agent, int n_sub, const uint8_t* sub_actions, int rm_terminal, int32_t* next_state,
                        double* reward, uint8_t* done, uint8_t* terminal, void* stream) {
  if (!h || !sub_actions || !next_state || !reward || !done || !terminal) return fail(RLRM_ERR_ARG, "null argument");
  if (agent < 0 || agent >= h->kp.A) return fail(RLRM_ERR_ARG, "agent out of range");
  if (n_sub < 1 || n_sub > 4) return fail(RLRM_ERR_ARG, "n_sub must be 1..4");
  MdpSub sub;
  for (int a = 0; a < 4; a++)
    for (int j = 0; j < 4; j++) {
      const int v = j < n_sub ? sub_actions[a * n_sub + j] : RLRM_ACTION_WAIT;
      if (v > RLRM_ACTION_WAIT) return fail(RLRM_ERR_ARG, "sub-action out of range");
      sub.a[a * 4 + j] = (unsigned char)v;
    }
  CUDA_TRY(cudaSetDevice(h->device));
  const int nQ = h->kp.per_agent ? h->kp.a_nQ[agent] : h->kp.nQ;
  const long long n = (long long)h->kp.ncell * nQ * 4 * n_sub;
  cudaStream_t s = (cudaStream_t)stream;
  if (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE)
    mdp_kernel<RLRM_ENV_FROZEN_LAKE><<<blocks_for(n, 256), 256, h->smem_bytes, s>>>(h->kp, agent, n_sub, sub, rm_terminal, next_state, reward, done, terminal);
  else
    mdp_kernel<RLRM_ENV_OFFICE_WORLD><<<blocks_for(n, 256), 256, h->smem_bytes, s>>>(h->kp, agent, n_sub, sub, rm_terminal, next_state, reward, done, terminal);
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_value_iteration(int device, int64_t n_states, int n_outcomes, const double* prob, const int32_t* next_state,
                                    const double* reward, const uint8_t* done, double gamma, double theta, int delta_rel, int max_sweeps,
                                    double* V, double* Q, int32_t* policy, double* work, int32_t* sweeps_out, void* stream) {
  if (!prob || !next_state || !reward || !done || !V || !Q || !policy || !work) return fail(RLRM_ERR_ARG, "null argument");
  if (n_states <= 0 || n_outcomes < 1) return fail(RLRM_ERR_ARG, "n_states / n_outcomes out of range");
  if (!(theta > 0.0) || max_sweeps < 1) return fail(RLRM_ERR_ARG, "theta must be positive and max_sweeps >= 1");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(RLRM_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(RLRM_ERR_ARG, "device out of range");
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  double* v[2] = {V, work};  // ping-pong; the result is copied back into V at the end if it landed in work
  unsigned long long* d_delta = reinterpret_cast<unsigned long long*>(work + n_states);
  CUDA_TRY(cudaMemsetAsync(V, 0, (size_t)n_states * sizeof(double), s));  // V = 0 (mdp_vi.py:28)
  int cur = 0, sweeps = 0;
  for (;;) {
    CUDA_TRY(cudaMemsetAsync(d_delta, 0, sizeof(unsigned long long), s));
    vi_sweep_kernel<<<blocks_for(n_states, 256), 256, 0, s>>>(n_states, n_outcomes, prob, next_state, reward, done, gamma, delta_rel,
                                                           v[cur], v[cur ^ 1], Q, policy, d_delta);
    CUDA_TRY(cudaGetLastError());
    unsigned long long bits = 0;
    CUDA_TRY(cudaMemcpyAsync(&bits, d_delta, sizeof(bits), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    cur ^= 1;
    sweeps++;
    double delta;
    memcpy(&delta, &bits, sizeof(delta));
    if (delta < theta) break;  // mdp_vi.py:56-57
    if (sweeps >= max_sweeps) {
      if (sweeps_out) *sweeps_out = sweeps;
      return fail(RLRM_ERR_UNSUPPORTED, "value iteration did not converge within max_sweeps");
    }
  }
  if (cur == 1) CUDA_TRY(cudaMemcpyAsync(V, work, (size_t)n_states * sizeof(double), cudaMemcpyDeviceToDevice, s));
  if (sweeps_out) *sweeps_out = sweeps;
  return RLRM_OK;
}

extern "C" int rlrm_update(rlrm_handle_t* h, const rlrm_state_t* st, const uint16_t* obs_cell, const uint8_t* actions,
                           const uint8_t* term_arg, const rlrm_step_out_t* out, void* stream) {
  int rc = check_state(h, st, true);
  if (rc) return rc;
  if (!obs_cell || !actions || !term_arg || !out) return fail(RLRM_ERR_ARG, "null argument");
  if (!out->prev_cell || !out->cell || !out->prev_q || !out->q || !out->event || !out->env_term || !out->renv || !out->reward)
    return fail(RLRM_ERR_ARG, "step record is missing fields the update needs");
  CUDA_TRY(cudaSetDevice(h->device));
  const long long n = st->n_instances * h->kp.A;
  cudaStream_t s = (cudaStream_t)stream;
  if (h->kp.algo == RLRM_ALGO_QLAMBDA && !st->e)
    return fail(RLRM_ERR_UNSUPPORTED, "rlrm_update on Q(lambda) needs dense traces (state.e); sparse traces are for rlrm_train");
  if (h->kp.algo == RLRM_ALGO_QLAMBDA)
    RLRM_BY_T(h, update_qlambda_kernel<T><<<(unsigned)n, 256, 0, s>>>(h->kp, dstate(st), obs_cell, actions, term_arg, dout(out), sweep_of(h)));
#define RLRM_UPD(ALGO, PA) RLRM_BY_T(h, update_kernel<ALGO, PA, T><<<blocks_for(n, 256), 256, h->smem_bytes, s>>>(h->kp, dstate(st), obs_cell, actions, term_arg, dout(out), sweep_of(h)))
  else if (h->kp.algo == RLRM_ALGO_QRM) {
    if (h->kp.per_agent) RLRM_UPD(RLRM_ALGO_QRM, true); else RLRM_UPD(RLRM_ALGO_QRM, false);
  } else {
    if (h->kp.per_agent) RLRM_UPD(RLRM_ALGO_QL, true); else RLRM_UPD(RLRM_ALGO_QL, false);
  }
#undef RLRM_UPD
  LAUNCH_CHECK(h);
  if (h->kp.shared_q) {
    apply_shared_kernel<<<blocks_for(h->kp.per_agent ? h->kp.sum4 : (long long)h->kp.A * h->kp.S4, 256), 256, 0, s>>>(h->kp, dstate(st));
    LAUNCH_CHECK(h);
  }
  return RLRM_OK;
}

// SWEEP: the handle has per-group settings (h->d_sweep); every family takes them in its own kernel, fast paths included
template <int ENV, bool SWEEP>
static void launch_train(rlrm_handle_t* h, const rlrm_state_t* st, uint64_t t0, int n_iters, int learn, uint32_t* trace, cudaStream_t s,
                         double* reward_out = nullptr) {
  const KP& kp = h->kp;
  const Sweep sw = sweep_of(h);
  const bool fast_ok = reward_out == nullptr;  // the per-step reward output exists in the generic kernels only
  if (kp.algo == RLRM_ALGO_QLAMBDA && !st->e) {
    const long long ipw = 32 / (kp.qls_lg << kp.g_shift);  // instances per warp
    const long long qls_warps = (st->n_instances + ipw - 1) / ipw;
    if (kp.per_agent) RLRM_BY_T(h, train_qlambda_sparse_kernel<ENV, T, true, SWEEP><<<blocks_for(qls_warps * 32, QLS_BLOCK), QLS_BLOCK, h->smem_bytes, s>>>(kp, dstate(st), t0, n_iters, learn, trace, reward_out, sw));
    else RLRM_BY_T(h, train_qlambda_sparse_kernel<ENV, T, false, SWEEP><<<blocks_for(qls_warps * 32, QLS_BLOCK), QLS_BLOCK, h->smem_bytes, s>>>(kp, dstate(st), t0, n_iters, learn, trace, reward_out, sw));
  } else if (kp.algo == RLRM_ALGO_QLAMBDA) {
    if (kp.per_agent) RLRM_BY_T(h, train_qlambda_kernel<ENV, T, true, SWEEP><<<(unsigned)st->n_instances, kp.A * 32, h->smem_bytes, s>>>(kp, dstate(st), t0, n_iters, learn, trace, reward_out, sw));
    else RLRM_BY_T(h, train_qlambda_kernel<ENV, T, false, SWEEP><<<(unsigned)st->n_instances, kp.A * 32, h->smem_bytes, s>>>(kp, dstate(st), t0, n_iters, learn, trace, reward_out, sw));
  } else {
    const long long threads = st->n_instances * kp.G;
    const unsigned grid = blocks_for(threads, TRAIN_BLOCK);
#define RLRM_TRAIN(ALGO, PA) RLRM_BY_T(h, train_kernel<ENV, ALGO, PA, T, SWEEP><<<grid, TRAIN_BLOCK, h->smem_bytes, s>>>(kp, dstate(st), t0, n_iters, learn, trace, reward_out, sw))
    if (fast_ok && kp.algo == RLRM_ALGO_QRM && h->qrm4_fast && !st->visits) {
      const DState d = dstate(st);
#define RLRM_QRM4(ST, LE, TR)                                                                                          \
  do {                                                                                                                \
    if (dense_batch) train_qrm4_kernel<ENV, ST, LE, TR, 8, SWEEP><<<grid, TRAIN_BLOCK, h->smem_bytes, s>>>(kp, d, t0, n_iters, trace, sw); \
    else train_qrm4_kernel<ENV, ST, LE, TR, 7, SWEEP><<<grid, TRAIN_BLOCK, h->smem_bytes, s>>>(kp, d, t0, n_iters, trace, sw);   \
  } while (0)
      // more threads than 7 resident blocks per SM hold: take the 64-register instantiation (8 blocks per SM)
      const bool dense_batch = threads > (long long)h->num_sms * 7 * TRAIN_BLOCK;
      const int key = (kp.stochastic ? 4 : 0) | (learn ? 2 : 0) | (trace ? 1 : 0);
      switch (key) {
        case 0: RLRM_QRM4(false, false, false); break;
        case 1: RLRM_QRM4(false, false, true); break;
        case 2: RLRM_QRM4(false, true, false); break;
        case 3: RLRM_QRM4(false, true, true); break;
        case 4: RLRM_QRM4(true, false, false); break;
        case 5: RLRM_QRM4(true, false, true); break;
        case 6: RLRM_QRM4(true, true, false); break;
        default: RLRM_QRM4(true, true, true); break;
      }
#undef RLRM_QRM4
    }
    else if (fast_ok && kp.algo == RLRM_ALGO_QRM && h->qrmn_fast && !st->visits) {
      const DState d = dstate(st);
#define RLRM_QRMN(ST, LE, TR)                                                                                             \
  do {                                                                                                                   \
    if (kp.nQ == 3) train_qrmn_kernel<ENV, 3, ST, LE, TR, SWEEP><<<grid, TRAIN_BLOCK, h->smem_bytes, s>>>(kp, d, t0, n_iters, trace, sw); \
    else train_qrmn_kernel<ENV, 5, ST, LE, TR, SWEEP><<<grid, TRAIN_BLOCK, h->smem_bytes, s>>>(kp, d, t0, n_iters, trace, sw);       \
  } while (0)
      const int key = (kp.stochastic ? 4 : 0) | (learn ? 2 : 0) | (trace ? 1 : 0);
      switch (key) {
        case 0: RLRM_QRMN(false, false, false); break;
        case 1: RLRM_QRMN(false, false, true); break;
        case 2: RLRM_QRMN(false, true, false); break;
        case 3: RLRM_QRMN(false, true, true); break;
        case 4: RLRM_QRMN(true, false, false); break;
        case 5: RLRM_QRMN(true, false, true); break;
        case 6: RLRM_QRMN(true, true, false); break;
        default: RLRM_QRMN(true, true, true); break;
      }
#undef RLRM_QRMN
    }
    else if (fast_ok && kp.algo == RLRM_ALGO_QRM && h->qrmb_fast && !st->visits) {
      const DState d = dstate(st);
#define RLRM_QRMB(M)                                                                                                                       \
  do {                                                                                                                                   \
    if (kp.n_qrm <= 3) RLRM_BY_T(h, train_qrm_block_kernel<ENV, 3, T, M, SWEEP><<<grid, TRAIN_BLOCK, h->qrmb_smem, s>>>(kp, d, t0, n_iters, learn, trace, sw));        \
    else if (kp.n_qrm <= 7) RLRM_BY_T(h, train_qrm_block_kernel<ENV, 7, T, M, SWEEP><<<grid, TRAIN_BLOCK, h->qrmb_smem, s>>>(kp, d, t0, n_iters, learn, trace, sw));   \
    else if (kp.n_qrm <= 11) RLRM_BY_T(h, train_qrm_block_kernel<ENV, 11, T, M, SWEEP><<<grid, TRAIN_BLOCK, h->qrmb_smem, s>>>(kp, d, t0, n_iters, learn, trace, sw)); \
    else RLRM_BY_T(h, train_qrm_block_kernel<ENV, 15, T, M, SWEEP><<<grid, TRAIN_BLOCK, h->qrmb_smem, s>>>(kp, d, t0, n_iters, learn, trace, sw));                     \
  } while (0)
      if (h->qrmb_tma) RLRM_QRMB(true); else RLRM_QRMB(false);
#undef RLRM_QRMB
    }
    else if (fast_ok && kp.algo == RLRM_ALGO_QL && h->ql_fast && !st->visits) {
      const DState d = dstate(st);
#define RLRM_QLF(ST, LE, TR) train_ql_fast_kernel<ENV, ST, LE, TR, SWEEP><<<grid, TRAIN_BLOCK, h->smem_bytes, s>>>(kp, d, t0, n_iters, trace, sw)
      const int key = (kp.stochastic ? 4 : 0) | (learn ? 2 : 0) | (trace ? 1 : 0);
      switch (key) {
        case 0: RLRM_QLF(false, false, false); break;
        case 1: RLRM_QLF(false, false, true); break;
        case 2: RLRM_QLF(false, true, false); break;
        case 3: RLRM_QLF(false, true, true); break;
        case 4: RLRM_QLF(true, false, false); break;
        case 5: RLRM_QLF(true, false, true); break;
        case 6: RLRM_QLF(true, true, false); break;
        default: RLRM_QLF(true, true, true); break;
      }
#undef RLRM_QLF
    }
    else if (kp.algo == RLRM_ALGO_QRM) {
      if (kp.per_agent) RLRM_TRAIN(RLRM_ALGO_QRM, true); else RLRM_TRAIN(RLRM_ALGO_QRM, false);
    } else {
      if (kp.per_agent) RLRM_TRAIN(RLRM_ALGO_QL, true); else RLRM_TRAIN(RLRM_ALGO_QL, false);
    }
#undef RLRM_TRAIN
  }
}

extern "C" int rlrm_train(rlrm_handle_t* h, const rlrm_state_t* st, uint64_t t0, int32_t n_iters, int32_t learn, uint32_t* trace,
                          void* stream) {
  int rc = check_state(h, st, true);
  if (rc) return rc;
  if (n_iters < 0) return fail(RLRM_ERR_ARG, "n_iters < 0");
  if (n_iters == 0) return RLRM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (h->kp.shared_q) {
    // synchronous iterations: one propose launch over all instances + one apply launch per lockstep iteration
    const size_t stride = (size_t)st->n_instances * h->kp.A;
    if (h->shared_fast && h->coop_ok && !st->visits && learn && !trace && !(h->cfg.reserved & 2) && !((h->cfg.reserved & 4) && h->shared_cluster)) {
      // persistent path: all n_iters iterations in one cooperative launch (see shared_train_kernel)
      const long long threads = st->n_instances * h->kp.G;
      long long want = (threads + SHARED_BLOCK - 1) / SHARED_BLOCK;
      const unsigned grid = (unsigned)(want < h->num_sms ? want : h->num_sms);
      KP kp = h->kp;
      DState d = dstate(st);
      unsigned long long tt = t0;
      int ni = n_iters;
      const size_t n_ent = (size_t)kp.A * (size_t)kp.S4;
      unsigned long long* g_sum = reinterpret_cast<unsigned long long*>(h->d_coop);
      int* g_cnt = reinterpret_cast<int*>(h->d_coop + 3 * n_ent * 8);
      float* g_last = reinterpret_cast<float*>(h->d_coop + 3 * n_ent * 12);
      void* args[] = {&kp, &d, &tt, &ni, &g_sum, &g_cnt, &g_last};
      const void* fn;
      if (kp.env_kind == RLRM_ENV_FROZEN_LAKE) fn = kp.algo == RLRM_ALGO_QRM ? (const void*)shared_train_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QRM> : (const void*)shared_train_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QL>;
      else fn = kp.algo == RLRM_ALGO_QRM ? (const void*)shared_train_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QRM> : (const void*)shared_train_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QL>;
      CUDA_TRY(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(SHARED_BLOCK), args, (size_t)h->shared_smem_bytes, s));
      LAUNCH_CHECK(h);
      return RLRM_OK;
    }
    if (h->shared_cluster && !(h->shared_fast && !(h->cfg.reserved & 4)) && !st->visits && learn && !trace && !(h->cfg.reserved & 2)) {
      // persistent path with the tables partitioned over a thread-block cluster (see shared_train_cluster_kernel)
      const long long threads = st->n_instances * h->kp.G;
      const long long want = (threads + SHARED_BLOCK - 1) / SHARED_BLOCK;
      const DState d = dstate(st);
      const size_t n_ent = (size_t)h->kp.A * (size_t)h->kp.S4;
      unsigned long long* g_sum = reinterpret_cast<unsigned long long*>(h->d_coop);
      int* g_cnt = reinterpret_cast<int*>(h->d_coop + 3 * n_ent * 8);
      float* g_last = reinterpret_cast<float*>(h->d_coop + 3 * n_ent * 12);
      CUDA_TRY(RLRM_CLUSTER_DISPATCH(cluster_kernel_launch, h, h->kp, d, (unsigned long long)t0, (int)n_iters, want, g_sum, g_cnt, g_last, s));
      LAUNCH_CHECK(h);
      return RLRM_OK;
    }
    for (int it = 0; it < n_iters; it++) {
      uint32_t* tr = trace ? trace + (size_t)it * stride : nullptr;
      if (h->shared_fast && !st->visits) {
        const long long threads = st->n_instances * h->kp.G;
        long long want = (threads + SHARED_BLOCK - 1) / SHARED_BLOCK;
        const unsigned grid = (unsigned)(want < h->num_sms ? want : h->num_sms);
        const DState d = dstate(st);
        if (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE) {
          if (h->kp.algo == RLRM_ALGO_QRM) shared_propose_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QRM><<<grid, SHARED_BLOCK, h->shared_smem_bytes, s>>>(h->kp, d, t0 + it, learn, tr);
          else shared_propose_kernel<RLRM_ENV_FROZEN_LAKE, RLRM_ALGO_QL><<<grid, SHARED_BLOCK, h->shared_smem_bytes, s>>>(h->kp, d, t0 + it, learn, tr);
        } else {
          if (h->kp.algo == RLRM_ALGO_QRM) shared_propose_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QRM><<<grid, SHARED_BLOCK, h->shared_smem_bytes, s>>>(h->kp, d, t0 + it, learn, tr);
          else shared_propose_kernel<RLRM_ENV_OFFICE_WORLD, RLRM_ALGO_QL><<<grid, SHARED_BLOCK, h->shared_smem_bytes, s>>>(h->kp, d, t0 + it, learn, tr);
        }
      } else if (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE) launch_train<RLRM_ENV_FROZEN_LAKE, false>(h, st, t0 + it, 1, learn, tr, s);
      else launch_train<RLRM_ENV_OFFICE_WORLD, false>(h, st, t0 + it, 1, learn, tr, s);
      LAUNCH_CHECK(h);
      if (learn) {
        apply_shared_kernel<<<blocks_for(h->kp.per_agent ? h->kp.sum4 : (long long)h->kp.A * h->kp.S4, 256), 256, 0, s>>>(h->kp, dstate(st));
        LAUNCH_CHECK(h);
      }
    }
    return RLRM_OK;
  }
  if (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE) {
    if (h->d_sweep) launch_train<RLRM_ENV_FROZEN_LAKE, true>(h, st, t0, n_iters, learn, trace, s);
    else launch_train<RLRM_ENV_FROZEN_LAKE, false>(h, st, t0, n_iters, learn, trace, s);
  } else {
    if (h->d_sweep) launch_train<RLRM_ENV_OFFICE_WORLD, true>(h, st, t0, n_iters, learn, trace, s);
    else launch_train<RLRM_ENV_OFFICE_WORLD, false>(h, st, t0, n_iters, learn, trace, s);
  }
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_evaluate(rlrm_handle_t* h, const rlrm_state_t* st, rlrm_eval_t* ev, uint64_t t0, int32_t n_iters,
                             int32_t n_episodes, double gamma, double optimal_steps, void* stream) {
  int rc = check_state(h, st, false);
  if (rc) return rc;
  if (!st->q || !ev) return fail(RLRM_ERR_ARG, "state.q and ev are required");
  if (n_iters <= 0 || n_episodes <= 0) return RLRM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  const unsigned grid = blocks_for(st->n_instances * h->kp.G, TRAIN_BLOCK);
  cudaStream_t s = (cudaStream_t)stream;
#define RLRM_EVAL(ENV, PA) RLRM_BY_T(h, eval_kernel<ENV, PA, T><<<grid, TRAIN_BLOCK, h->smem_bytes, s>>>(h->kp, dstate(st), ev, t0, n_iters, n_episodes, gamma, optimal_steps))
  if (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE) {
    if (h->kp.per_agent) RLRM_EVAL(RLRM_ENV_FROZEN_LAKE, true); else RLRM_EVAL(RLRM_ENV_FROZEN_LAKE, false);
  } else {
    if (h->kp.per_agent) RLRM_EVAL(RLRM_ENV_OFFICE_WORLD, true); else RLRM_EVAL(RLRM_ENV_OFFICE_WORLD, false);
  }
#undef RLRM_EVAL
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_qlambda_materialize(rlrm_handle_t* h, const rlrm_state_t* st, void* e_dense, void* stream) {
  if (!h || !st) return fail(RLRM_ERR_ARG, "null handle/state");
  if (!st->q || !st->tr_idx || !st->tr_eq || !st->tr_len) return fail(RLRM_ERR_ARG, "no sparse trace state");
  CUDA_TRY(cudaSetDevice(h->device));
  const long long n = st->n_instances * h->kp.A;
  RLRM_BY_T(h, qlambda_materialize_kernel<T><<<blocks_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(h->kp, dstate(st), (T*)e_dense));
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

// rlrm_state_t restricted to instances [start, start + count): every per-slot / per-table array is offset, so a kernel launched
// on the view with kp.instance_offset advanced by `start` computes exactly what the full launch computes for those instances
// (instances never interact and the Philox counters are keyed on the global instance id).
static rlrm_state_t sub_state(const rlrm_handle_t* h, const rlrm_state_t* st, long long start, long long count) {
  rlrm_state_t v = *st;
  const KP& kp = h->kp;
  const size_t slots = (size_t)start * kp.A;
  const size_t ent = kp.per_agent ? (size_t)start * (size_t)kp.sum4 : slots * (size_t)kp.S4;  // table entries before `start`
  const size_t esz = h->f64 ? 8 : 4;
  v.n_instances = count;
  v.slot = st->slot + slots;
  v.epsilon = st->epsilon + slots;
  v.q = (char*)st->q + ent * esz;
  if (st->e) v.e = (char*)st->e + ent * esz;
  if (st->visits) v.visits = st->visits + ent;
  if (st->ep_return) v.ep_return = st->ep_return + slots;
  if (st->stats) v.stats = st->stats + slots;
  if (st->tr_pos) v.tr_pos = st->tr_pos + slots * (size_t)kp.S4;
  if (st->tr_idx) v.tr_idx = st->tr_idx + slots * (size_t)st->tr_cap;
  if (st->tr_eq) v.tr_eq = (char*)st->tr_eq + slots * (size_t)st->tr_cap * 2 * esz;
  if (st->tr_len) v.tr_len = st->tr_len + slots;
  if (st->tr_work) v.tr_work = st->tr_work + slots;
  return v;
}

extern "C" int rlrm_train_host(rlrm_handle_t* h, const rlrm_state_t* st, uint64_t t0, int32_t n_iters, int32_t learn,
                               uint64_t* host_slot, double* host_epsilon, rlrm_stats_t* host_stats, void* stream) {
  int rc = check_state(h, st, true);
  if (rc) return rc;
  if (host_stats && !st->stats) return fail(RLRM_ERR_ARG, "host_stats requested but state.stats is null");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)st->n_instances * h->kp.A;
  const size_t bytes = n * ((host_slot ? 16 : 0) + (host_epsilon ? 16 : 0) + (host_stats ? sizeof(rlrm_stats_t) : 0));
  // Independent instances and enough bytes to matter: split the instance range into chunks and pipeline them over two extra
  // streams — chunk c's upload, chunk c-1's kernel and chunk c-2's download overlap. Results are bit-identical to the
  // single launch (sub_state). The shared learner's iterations are synchronous over ALL instances, so it cannot be chunked.
  // Every chunk must still fill the GPU on its own, otherwise the chunk kernels would run one after the other at a fraction of
  // the occupancy of the single launch: >= 512 Ki slots for the thread-per-agent kernels, >= 64 Ki for the Q(lambda) kernels
  // (a warp per agent / a lane group per agent).
  int chunks = 1;
  if (!h->kp.shared_q && n_iters > 0 && bytes >= (8u << 20)) {
    const size_t fit = n / ((h->kp.algo == RLRM_ALGO_QLAMBDA ? 64u : 512u) * 1024u);
    chunks = fit >= 8 ? 8 : (fit >= 2 ? (int)fit : 1);
  }
  if (chunks == 1) {
    if (host_slot) CUDA_TRY(cudaMemcpyAsync(st->slot, host_slot, n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    if (host_epsilon) CUDA_TRY(cudaMemcpyAsync(st->epsilon, host_epsilon, n * sizeof(double), cudaMemcpyHostToDevice, s));
    rc = rlrm_train(h, st, t0, n_iters, learn, nullptr, stream);
    if (rc) return rc;
    if (host_stats) CUDA_TRY(cudaMemcpyAsync(host_stats, st->stats, n * sizeof(rlrm_stats_t), cudaMemcpyDeviceToHost, s));
    if (host_slot) CUDA_TRY(cudaMemcpyAsync(host_slot, st->slot, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (host_epsilon) CUDA_TRY(cudaMemcpyAsync(host_epsilon, st->epsilon, n * sizeof(double), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return RLRM_OK;
  }
  if (!h->pipe_ready) {
    for (int k = 0; k < 2; k++) CUDA_TRY(cudaStreamCreateWithFlags(&h->pipe_stream[k], cudaStreamNonBlocking));
    for (int k = 0; k < 3 * 8; k++) CUDA_TRY(cudaEventCreateWithFlags(&h->pipe_event[k], cudaEventDisableTiming));
    h->pipe_ready = 1;
  }
  cudaStream_t up = h->pipe_stream[0], down = h->pipe_stream[1];
  cudaEvent_t* ev = h->pipe_event;  // [c]: caller's stream reached this call; [8 + c]: chunk c uploaded; [16 + c]: chunk c computed
  CUDA_TRY(cudaEventRecord(ev[0], s));
  CUDA_TRY(cudaStreamWaitEvent(up, ev[0], 0));  // earlier work of the caller's stream may still use the state arrays
  const unsigned base_offset = h->kp.instance_offset;
  const long long per = (st->n_instances + chunks - 1) / chunks;
  for (int c = 0; c < chunks; c++) {
    const long long start = (long long)c * per, count = (start + per <= st->n_instances) ? per : st->n_instances - start;
    if (count <= 0) break;
    const rlrm_state_t v = sub_state(h, st, start, count);
    const size_t off = (size_t)start * h->kp.A, m = (size_t)count * h->kp.A;
    if (host_slot) CUDA_TRY(cudaMemcpyAsync(v.slot, host_slot + off, m * sizeof(uint64_t), cudaMemcpyHostToDevice, up));
    if (host_epsilon) CUDA_TRY(cudaMemcpyAsync(v.epsilon, host_epsilon + off, m * sizeof(double), cudaMemcpyHostToDevice, up));
    CUDA_TRY(cudaEventRecord(ev[8 + c], up));
    CUDA_TRY(cudaStreamWaitEvent(s, ev[8 + c], 0));
    h->kp.instance_offset = base_offset + (unsigned)start;
    rc = rlrm_train(h, &v, t0, n_iters, learn, nullptr, stream);
    h->kp.instance_offset = base_offset;
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(ev[16 + c], s));
    CUDA_TRY(cudaStreamWaitEvent(down, ev[16 + c], 0));
    if (host_stats) CUDA_TRY(cudaMemcpyAsync(host_stats + off, v.stats, m * sizeof(rlrm_stats_t), cudaMemcpyDeviceToHost, down));
    if (host_slot) CUDA_TRY(cudaMemcpyAsync(host_slot + off, v.slot, m * sizeof(uint64_t), cudaMemcpyDeviceToHost, down));
    if (host_epsilon) CUDA_TRY(cudaMemcpyAsync(host_epsilon + off, v.epsilon, m * sizeof(double), cudaMemcpyDeviceToHost, down));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaStreamSynchronize(down));
  return RLRM_OK;
}

extern "C" int rlrm_iterate(rlrm_handle_t* h, const rlrm_state_t* st, uint64_t t, int32_t learn, uint32_t* record, double* reward,
                            void* stream) {
  int rc = check_state(h, st, true);
  if (rc) return rc;
  if (h->kp.shared_q) {
    if (reward) return fail(RLRM_ERR_UNSUPPORTED, "rlrm_iterate: the per-step reward output is not available with a shared table");
    return rlrm_train(h, st, t, 1, learn, record, stream);
  }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (h->kp.env_kind == RLRM_ENV_FROZEN_LAKE) {
    if (h->d_sweep) launch_train<RLRM_ENV_FROZEN_LAKE, true>(h, st, t, 1, learn, record, s, reward);
    else launch_train<RLRM_ENV_FROZEN_LAKE, false>(h, st, t, 1, learn, record, s, reward);
  } else {
    if (h->d_sweep) launch_train<RLRM_ENV_OFFICE_WORLD, true>(h, st, t, 1, learn, record, s, reward);
    else launch_train<RLRM_ENV_OFFICE_WORLD, false>(h, st, t, 1, learn, record, s, reward);
  }
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

static int update_list_impl(rlrm_handle_t* h, const rlrm_state_t* st, int64_t slot, int32_t n, const rlrm_experience_t* experiences,
                            rlrm_select_req_t* sel, void* stream) {
  int rc = check_state(h, st, true);
  if (rc) return rc;
  if (n < 0 || (n > 0 && !experiences)) return fail(RLRM_ERR_ARG, "rlrm_update_list: bad experience list");
  if (slot < 0 || slot >= st->n_instances * h->kp.A) return fail(RLRM_ERR_ARG, "rlrm_update_list: slot out of range");
  if (h->kp.shared_q) return fail(RLRM_ERR_UNSUPPORTED, "rlrm_update_list on a shared table (proposals need the synchronous iteration of rlrm_train)");
  if (h->kp.algo == RLRM_ALGO_QLAMBDA && !st->e) return fail(RLRM_ERR_UNSUPPORTED, "rlrm_update_list on Q(lambda) needs dense traces (state.e)");
  if (n == 0 && !sel) return RLRM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  SelArgs sa;
  memset(&sa, 0, sizeof(sa));
  if (sel) {  // page-locked host memory: the request is read here, the answer is written by the kernel
    sa.state = sel->state; sa.best = sel->best; sa.epsilon = sel->epsilon; sa.seq = sel->seq;
    for (int j = 0; j < 4; j++) sa.draws[j] = sel->draws[j];
  }
  RLRM_BY_T(h, update_list_kernel<T><<<1, (h->kp.algo == RLRM_ALGO_QLAMBDA && n > 0) ? 256 : 32, 0, (cudaStream_t)stream>>>(h->kp, dstate(st), slot, n, experiences, sel, sa, sweep_of(h)));
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_update_list(rlrm_handle_t* h, const rlrm_state_t* st, int64_t slot, int32_t n, const rlrm_experience_t* experiences,
                                void* stream) {
  return update_list_impl(h, st, slot, n, experiences, nullptr, stream);
}

extern "C" int rlrm_update_list_select(rlrm_handle_t* h, const rlrm_state_t* st, int64_t slot, int32_t n, const rlrm_experience_t* experiences,
                                       rlrm_select_req_t* sel, void* stream) {
  if (!sel) return fail(RLRM_ERR_ARG, "rlrm_update_list_select: null selection request");
  return update_list_impl(h, st, slot, n, experiences, sel, stream);
}

extern "C" int rlrm_merge_replicas(rlrm_handle_t* h, const float* gathered, int32_t world, int64_t n, float* q, void* stream) {
  if (!h || !gathered || !q) return fail(RLRM_ERR_ARG, "null argument");
  if (world < 1 || n <= 0) return fail(RLRM_ERR_ARG, "rlrm_merge_replicas: world / n out of range");
  if (h->f64) return fail(RLRM_ERR_UNSUPPORTED, "the shared learner is specified on float32 tables");
  CUDA_TRY(cudaSetDevice(h->device));
  merge_replicas_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(gathered, world, n, q);
  LAUNCH_CHECK(h);
  return RLRM_OK;
}

extern "C" int rlrm_stream_sync(rlrm_handle_t* h, void* stream) {
  if (!h) return fail(RLRM_ERR_ARG, "null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return RLRM_OK;
}

extern "C" int rlrm_probe_random_gather(int device, void* table, int64_t table_bytes, int32_t block_bytes, int64_t n_gathers, int32_t write,
                                        void* sink, void* stream) {
  if (!table || !sink) return fail(RLRM_ERR_ARG, "null argument");
  if (block_bytes != 16 && block_bytes != 32 && block_bytes != 64) return fail(RLRM_ERR_ARG, "block_bytes must be 16, 32 or 64");
  if (table_bytes < block_bytes || n_gathers < 1 || ((uintptr_t)table & 63u)) return fail(RLRM_ERR_ARG, "table too small / misaligned or n_gathers < 1");
  CUDA_TRY(cudaSetDevice(device));
  const unsigned long long n_blocks = (unsigned long long)table_bytes / (unsigned)block_bytes;
  const int per_thread = 64;
  const long long threads = (n_gathers + per_thread - 1) / per_thread;
  const unsigned grid = blocks_for(threads, 256);
  cudaStream_t s = (cudaStream_t)stream;
  if (block_bytes == 16) probe_gather_kernel<1><<<grid, 256, 0, s>>>((uint4*)table, n_blocks, per_thread, 12345u, write, (unsigned*)sink);
  else if (block_bytes == 32) probe_gather_kernel<2><<<grid, 256, 0, s>>>((uint4*)table, n_blocks, per_thread, 12345u, write, (unsigned*)sink);
  else probe_gather_kernel<4><<<grid, 256, 0, s>>>((uint4*)table, n_blocks, per_thread, 12345u, write, (unsigned*)sink);
  CUDA_TRY(cudaGetLastError());
  return RLRM_OK;
}
