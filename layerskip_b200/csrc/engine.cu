// engine.cu — liblsk: C ABI (include/lsk.h) + host-side orchestration of the sm_100a kernels.
//
// The engine owns: packed weights, the paged KV pool, scratch activations, the device-resident
// generation state, one stream and a cache of CUDA graphs (one per (E, d_req) round shape).
// A speculation round is ONE graph replay and ONE host synchronisation.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <nccl.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <map>
#include <string>
#include <vector>

#include "../../include/lsk.h"
#include "attention.cuh"
#include "common.cuh"
#include "gemm_skinny.cuh"
#include "tp_peer.cuh"
#include "lmhead_tc.cuh"
#include "prefill_tc.cuh"
#include "misc_kernels.cuh"
#include "sampling.cuh"

using namespace lsk;

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CU(expr)                                                                         \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      return fail(LSK_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),  \
                  __FILE__, __LINE__);                                                   \
  } while (0)

#define NC(expr)                                                                         \
  do {                                                                                   \
    ncclResult_t _r = (expr);                                                            \
    if (_r != ncclSuccess)                                                               \
      return fail(LSK_ERR_NCCL, "%s failed: %s (%s:%d)", #expr, ncclGetErrorString(_r),  \
                  __FILE__, __LINE__);                                                   \
  } while (0)

#define TRY(expr)            \
  do {                       \
    int _s = (expr);         \
    if (_s != LSK_OK) return _s; \
  } while (0)

// ---------------------------------------------------------------------------------------------
// engine
// ---------------------------------------------------------------------------------------------
struct LayerWeights {
  __nv_bfloat16* wqkv = nullptr;  // packed [(q_rows + 2 kv_rows), hidden]
  __nv_bfloat16* wo = nullptr;    // packed [hidden, q_rows]
  __nv_bfloat16* wgu = nullptr;   // packed [2 * inter_l, hidden]  (gate/up interleaved by 8)
  __nv_bfloat16* wd = nullptr;    // packed [hidden, inter_l]
  __nv_bfloat16* ln1 = nullptr;
  __nv_bfloat16* ln2 = nullptr;
  // tcgen05 prefill (prefill_tc.cuh): second copy in the canonical K-major tile layout
  unsigned char* wqkv_c = nullptr;
  unsigned char* wo_c = nullptr;
  unsigned char* wgu_c = nullptr;
  unsigned char* wd_c = nullptr;
  unsigned loaded = 0;            // bit per role
};

struct GemmPlan {
  int n_tiles = 0, nsb = 0, K = 0;
};

struct lsk_engine {
  lsk_config cfg{};
  int sm_count = 0;
  // local (tensor-parallel shard) dimensions
  int heads_l = 0, kv_heads_l = 0, q_rows = 0, kv_rows = 0, inter_l = 0, vocab_l = 0,
      vocab_l_pad = 0, vocab_off = 0, group = 0, inter_l_pad = 0;
  int n_pages = 0, max_pos = 0, n_splits = 0;
  int attn_stages = 4;                 // K/V ring depth of the attention kernel (LSK_ATTN_STAGES, 2..4)
  int max_rows = kMaxRows;             // token rows one step can carry (8 when 16 do not fit)
  bool use_pdl = true, use_graph = true, keep_logits = false;

  std::vector<LayerWeights> layers;
  __nv_bfloat16* embed = nullptr;      // [vocab, hidden] natural (replicated)
  __nv_bfloat16* final_norm = nullptr;
  __nv_bfloat16* lm_head = nullptr;    // packed [vocab_l_pad, hidden]
  // opt-in tcgen05 LM head (lmhead_tc.cuh): a second, canonical-layout copy of the head weights
  bool lm_tc = false;
  unsigned char* lm_head_tc = nullptr;   // [lm_tc_tiles][hidden / 64][16 KiB]
  int lm_tc_tiles = 0, lm_tc_grid = 0, lm_tc_stages = 0;
  unsigned globals_loaded = 0;
  // tcgen05 prefill: 128-token passes (on unless LSK_FLAG_NO_PREFILL_TC / LSK_PREFILL_TC=0)
  bool pf_tc = false;
  int pf_stages = 0;
  int kst_h = 0, kst_q = 0, kst_i = 0;          // 64-wide k stages of hidden / q_rows / inter_l
  int pf_t_qkv = 0, pf_t_h = 0, pf_t_gu = 0;     // 128-row tiles of qkv / hidden / gate-up outputs
  float* hidden_p = nullptr;             // [128][hidden] fp32 residual rows of a prompt chunk
  float* tp_buf_p = nullptr;             // [128][hidden] fp32 row-parallel partial sums (TP)
  float* part_p = nullptr;               // [4 k-splits][128][hidden] fp32 partial tiles of the O / down GEMMs
  __nv_bfloat16* q_p = nullptr;          // [128][q_rows]
  unsigned char* xn_c = nullptr;         // canonical activations: RMS-normed rows   [kst_h][16 KiB]
  unsigned char* attn_c = nullptr;       //                        attention output   [kst_q][16 KiB]
  unsigned char* act_c = nullptr;        //                        silu(gate) * up    [kst_i][16 KiB]

  __nv_bfloat16* kpool = nullptr;      // [layer][page][kv_head][64][128]
  __nv_bfloat16* vpool = nullptr;
  size_t pool_layer_elems = 0;
  int* page_table = nullptr;
  float2* rope = nullptr;

  float* hidden = nullptr;             // [16][hidden] fp32 residual-stream rows
  __nv_bfloat16* qbuf = nullptr;       // [16][q_rows]
  __nv_bfloat16* attn_out = nullptr;   // [16][q_rows]
  __nv_bfloat16* act = nullptr;        // [16][inter_l]
  float* tp_buf = nullptr;             // [16][hidden] row-parallel partial sums (TP)
  float* logits = nullptr;             // [16][vocab_l_pad] (optional)
  float* logits_gath = nullptr;        // TP sampling: [tp][16][vocab_l_pad] all-gathered shards
  float* logits_full = nullptr;        // TP sampling: [16][vocab] rows every rank samples from
  float* probs_d = nullptr;            // sampling: [16][vocab] warped draft distributions
  float* probs_v = nullptr;            // sampling: [16][vocab] warped verifier distributions
  float* samp_scratch = nullptr;       // sampling: [vocab] residual weights
  float* cand_val = nullptr;           // [n_cand_max][16]
  int* cand_idx = nullptr;
  float* gath_val = nullptr;           // TP: [tp_size][16]
  int* gath_idx = nullptr;
  float* ban_val = nullptr;            // n-gram ban: [16] arg-max of the banned logits rows (n_cand == 1 layout)
  int* ban_idx = nullptr;
  float* rank_val = nullptr;           // TP: [16]
  int* rank_idx = nullptr;
  int* d_zero = nullptr;
  int* d_prompt = nullptr;             // [max_ctx] prompt ids, then the emitted tokens (n-gram ban history)
  int* d_dbg_ids = nullptr;            // [kMaxRows] ids of lsk_debug_forward_rows (kept out of the history)
  DevState* state = nullptr;
  GenParams* gen_dev = nullptr;
  RoundResult* res_host = nullptr;     // mapped pinned
  RoundResult* res_dev = nullptr;      // device alias of res_host

  GemmPlan p_qkv, p_o, p_gu, p_d, p_lm;
  size_t l2_prefetch_bytes = 0;          // LSK_L2_PREFETCH_MB: head of the NEXT kernel's weights pulled into L2 (A/B: no gain, +11 % traffic -> off)
  const float* cur_cand_val = nullptr;  // candidates of the last enqueued LM head (epilogue's, or the banned rows' arg-max)
  const int* cur_cand_idx = nullptr;
  int cur_n_cand = 0;

  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::map<long long, cudaGraphExec_t> graphs;
  ncclComm_t comm = nullptr;
  // one-shot collectives over peer-mapped HBM (tp_peer.cuh); opt-in, NCCL otherwise
  bool want_peer = false, peer_ok = false;
  unsigned ablate = 0;                   // LSK_ABLATE: timing-only diagnostics, kernel classes NOT launched
  int peer_mode = 1;                     // 1: push kernel after the GEMM; 2: push fused into the GEMM epilogue
  PeerComm peer{};
  void* peer_region = nullptr;           // this rank's peer-visible allocation
  void* peer_opened[kMaxPeers] = {};     // IPC mappings of the other ranks' regions
  int* peer_err_host = nullptr;          // mapped pinned: set by a kernel whose wait timed out

  lsk_generation gen{};
  bool began = false, prefilled = false;
  int host_len = 0;                    // host mirror of the committed KV length
  int seq = 0;
  int64_t launches = 0;
  int64_t capture_launches = 0;        // launches recorded while capturing the current graph
  std::map<long long, int64_t> graph_launches;
  float last_ms = 0.f;
  // per-kernel-class timing (lsk_profile_round): events around every launch, eager mode
  bool profiling = false;
  int cur_class = 0;
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> prof_events;
};

enum { CLS_QKV = 0, CLS_ATTN = 1, CLS_O = 2, CLS_GATEUP = 3, CLS_DOWN = 4, CLS_LMHEAD = 5, CLS_MISC = 6, CLS_COMM = 7, CLS_COUNT = 8 };

static constexpr int kSmemMax = 227 * 1024;

// ---------------------------------------------------------------------------------------------
// launch helper (programmatic dependent launch attribute on every kernel)
// ---------------------------------------------------------------------------------------------
template <typename... KArgs, typename... Args>
static cudaError_t launch(lsk_engine* e, void (*kern)(KArgs...), dim3 grid, dim3 block,
                          size_t smem, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = e->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = e->use_pdl ? 1 : 0;
  e->launches += 1;
  e->capture_launches += 1;
  if (!e->profiling) return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  cudaEventRecord(a, e->stream);
  cudaError_t err = cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
  cudaEventRecord(b, e->stream);
  e->prof_events.push_back({e->cur_class, {a, b}});
  return err;
}

// ---------------------------------------------------------------------------------------------
// GEMM planning / dispatch
// ---------------------------------------------------------------------------------------------
static GemmPlan make_plan(int n_rows, int K, int sm_count) {
  GemmPlan p;
  p.n_tiles = n_rows / 16;
  p.K = K;
  p.nsb = K / 32;
  (void)sm_count;
  return p;
}

// Per-launch schedule: how much of K is resident (activation chunk), how many tiles are
// accumulated side by side, and how deep the TMA ring can be in the remaining shared memory.
struct GemmSched {
  int tpp = 1, n_chunks = 1, kc_sbs = 0, n_stages = 0, grid = 0;
  size_t smem = 0;
  bool ok = false;
};
static GemmSched plan_sched(int NT, int M, int pro, int epi, const GemmPlan& p, int sm_count) {
  constexpr int fixed_ring = 0;
  GemmSched best;
  for (int want = 1; want <= 16; ++want) {
    // RMSNorm prologue: whole rows resident whenever that fits; otherwise (16-row blocks at hidden
    // > 4096) the statistics are computed up front and the rows are normalised chunk by chunk
    if (pro == PRO_RMS && want == 2 && best.ok) break;   // whole rows fit: keep the resident mode
    int kc = (p.nsb + want - 1) / want;
    if (want > 1) kc = (kc + kStageSbs - 1) / kStageSbs * kStageSbs;
    const int n_chunks = (p.nsb + kc - 1) / kc;
    const int tpp = n_chunks > 1 ? kMaxTilesPerPass : 1;
    const GemmScratch L = gemm_scratch_layout(NT, M, kc * 32, tpp, epi);
    const int st_hi = fixed_ring > 0 ? fixed_ring : kMaxStages;
    const int st_lo = fixed_ring > 0 ? fixed_ring : 2;
    for (int st = st_hi; st >= st_lo; --st) {
      if (gemm_smem_total(st, L.total) <= (size_t)kSmemMax) {
        if (!best.ok || st > best.n_stages) {
          best.ok = true; best.tpp = tpp; best.n_chunks = n_chunks; best.kc_sbs = kc;
          best.n_stages = st; best.smem = gemm_smem_total(st, L.total);
        }
        break;
      }
    }
    if (best.ok && (fixed_ring > 0 || best.n_stages >= 5)) break;   // >= 80 KiB in flight per SM
  }
  if (best.ok) {
    const int n_slots = (p.n_tiles + best.tpp - 1) / best.tpp;
    best.grid = n_slots < sm_count ? n_slots : sm_count;
    // Tile quantisation: with g CTAs the kernel lasts ceil(n_slots / g) slot-times.  Among the
    // CTA counts that reach the minimum number of waves, take the SMALLEST one that wastes the
    // fewest slots (e.g. 768 tiles: 128 CTAs x 6 instead of 148 CTAs of which 28 run a 6th tile
    // alone) — the TMA ring lets ~85 % of the SMs saturate HBM (LSK_GRID_EVEN=0 disables).
    static const bool even = !(getenv("LSK_GRID_EVEN") && atoi(getenv("LSK_GRID_EVEN")) == 0);
    if (even && fixed_ring == 0 && n_slots > sm_count) {
      const int waves = (n_slots + sm_count - 1) / sm_count;
      int g = (n_slots + waves - 1) / waves;          // smallest CTA count with that many waves
      const int lo = sm_count * 4 / 5;
      if (g < lo) g = lo;
      best.grid = g;
    }
  }
  return best;
}

template <int NT, int PRO, int EPI>
static int launch_gemm_t(lsk_engine* e, const GemmPlan& p, GemmArgs& a) {
  // the attribute is per DEVICE: one process may drive engines on several GPUs
  static std::atomic<uint64_t> configured{0};
  auto kern = gemm_skinny_kernel<NT, PRO, EPI>;
  int dev = 0;
  CU(cudaGetDevice(&dev));
  const uint64_t bit = 1ull << (dev & 63);
  if (!(configured.load(std::memory_order_relaxed) & bit)) {
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
    configured.fetch_or(bit, std::memory_order_relaxed);
  }
  const GemmSched sc = plan_sched(NT, a.M, PRO, EPI, p, e->sm_count);
  if (!sc.ok)
    return fail(LSK_ERR_INVALID, "skinny GEMM does not fit shared memory (K=%d, NT=%d)", p.K, NT);
  a.n_tiles = p.n_tiles;
  a.nsb = p.nsb;
  a.K = p.K;
  a.tiles_per_pass = sc.tpp;
  a.n_chunks = sc.n_chunks;
  a.kc_sbs = sc.kc_sbs;
  a.n_stages = sc.n_stages;
  a.xs_rows = a.M;
  CU(launch(e, kern, dim3(sc.grid), dim3(kGemmThreads), sc.smem, a));
  return LSK_OK;
}

template <int PRO, int EPI>
static int launch_gemm(lsk_engine* e, const GemmPlan& p, GemmArgs a) {
  const int NT = a.M <= 8 ? 1 : 2;
  if (NT == 1) return launch_gemm_t<1, PRO, EPI>(e, p, a);
  if (plan_sched(2, a.M, PRO, EPI, p, e->sm_count).ok) return launch_gemm_t<2, PRO, EPI>(e, p, a);
  return fail(LSK_ERR_INVALID, "%d token rows need the 16-row kernel, which does not fit next to K=%d "
              "(hidden sizes > 4096 support at most 8 rows, i.e. num_speculations <= 7)", a.M, p.K);
}

// Tensor parallel: x[0..M) += sum over ranks of tp_buf (the fp32 partial of a row-parallel GEMM).
// Peer mode 1 (default, tp_peer.cuh): ONE kernel pushes the partial to every peer over NVLink as
// LL lines (flag inside the data), polls theirs and adds the rank-ordered sum to the residual.
// Peer mode 3: the fence + flag protocol (A/B).  Without peer access: NCCL all-reduce + residual add,
// timed by its own event pair so that `comm` never reads 0.
static int ll_grid(int n2) {
  int g = (n2 + kArThreads - 1) / kArThreads;
  return g < 1 ? 1 : (g > 148 ? 148 : g);      // every CTA resident at once (spin-wait safety)
}
static int emit_allreduce_resid_nccl(lsk_engine* e, float* buf, float* x, int M) {
  const lsk_config& c = e->cfg;
  e->cur_class = CLS_COMM;
  cudaEvent_t ea = nullptr, eb = nullptr;
  if (e->profiling) {
    cudaEventCreate(&ea); cudaEventCreate(&eb);
    cudaEventRecord(ea, e->stream);
  }
  e->launches += 1;
  e->capture_launches += 1;
  NC(ncclAllReduce(buf, buf, (size_t)M * c.hidden, ncclFloat, ncclSum, e->comm, e->stream));
  if (e->profiling) {
    cudaEventRecord(eb, e->stream);
    e->prof_events.push_back({CLS_COMM, {ea, eb}});
  }
  e->cur_class = CLS_MISC;
  CU(launch(e, residual_add_kernel, dim3(8, M), dim3(256), 0, x, c.hidden, (const float*)buf, c.hidden, c.hidden));
  return LSK_OK;
}
static int emit_allreduce_resid(lsk_engine* e, float* x, int M) {
  const lsk_config& c = e->cfg;
  if (e->peer_ok && e->peer_mode == 3) {
    e->cur_class = CLS_COMM;
    const int n4 = M * c.hidden / 4;
    const int grid = (n4 + kArVecPerCta - 1) / kArVecPerCta;      // <= kMaxArCtas (hidden <= 8192)
    CU(launch(e, tp_allreduce_resid_kernel, dim3(grid), dim3(kArThreads), 0, e->peer,
              (const float*)e->tp_buf, x, n4));
    return LSK_OK;
  }
  if (e->peer_ok) {
    e->cur_class = CLS_COMM;
    const int n2 = M * c.hidden / 2;
    CU(launch(e, tp_allreduce_ll_kernel, dim3(ll_grid(n2)), dim3(kArThreads), 0, e->peer,
              (const float*)e->tp_buf, x, n2));
    return LSK_OK;
  }
  return emit_allreduce_resid_nccl(e, e->tp_buf, x, M);
}

// Fused variant (peer_mode 2): the row-parallel GEMM pushes its tiles to every rank from its
// epilogue as LL lines while it is still streaming weights (gemm_skinny_push_kernel); a small
// kernel polls the lines of all ranks and adds the rank-ordered sum to the residual rows.
static int emit_gemm_push_resid(lsk_engine* e, const GemmPlan& p, GemmArgs a, float* x) {
  const lsk_config& c = e->cfg;
  const int NT = a.M <= 8 ? 1 : 2;
  const GemmSched sc = plan_sched(NT, a.M, PRO_BF16, EPI_PUSH, p, e->sm_count);
  if (!sc.ok) return fail(LSK_ERR_INVALID, "skinny GEMM does not fit shared memory (K=%d, NT=%d)", p.K, NT);
  a.n_tiles = p.n_tiles; a.nsb = p.nsb; a.K = p.K;
  a.tiles_per_pass = sc.tpp; a.n_chunks = sc.n_chunks; a.kc_sbs = sc.kc_sbs; a.n_stages = sc.n_stages;
  a.xs_rows = a.M;
  static std::atomic<uint64_t> configured{0};
  int dev = 0;
  CU(cudaGetDevice(&dev));
  const uint64_t bit = 1ull << (dev & 63);
  if (!(configured.load(std::memory_order_relaxed) & bit)) {
    CU(cudaFuncSetAttribute(gemm_skinny_push_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
    CU(cudaFuncSetAttribute(gemm_skinny_push_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
    configured.fetch_or(bit, std::memory_order_relaxed);
  }
  if (NT == 1) CU(launch(e, gemm_skinny_push_kernel<1>, dim3(sc.grid), dim3(kGemmThreads), sc.smem, a, e->peer));
  else CU(launch(e, gemm_skinny_push_kernel<2>, dim3(sc.grid), dim3(kGemmThreads), sc.smem, a, e->peer));
  e->cur_class = CLS_COMM;
  const int n2 = a.M * c.hidden / 2;
  CU(launch(e, tp_finish_ll_kernel, dim3(ll_grid(n2)), dim3(kArThreads), 0, e->peer, x, n2));
  return LSK_OK;
}

// Host-side launch plan of the attention kernel (pure host logic; lsk_plan_attention exposes it):
// split count = engine constant (batch invariance), ring depth as deep as shared memory allows, and a
// shared-memory floor that gives a one-wave grid a whole SM per CTA (profiles/r2_attention_sweep.md).
static int attn_default_splits(int sm_count, int kv_heads_local) {
  return std::max(1, std::min(4, sm_count / std::max(1, kv_heads_local)));
}
struct AttnLaunchPlan {
  AttnSmemPlan sp;
  int stages;
  size_t smem;
  bool ok;
};
static AttnLaunchPlan plan_attention_launch(int head_dim, int group, int M, int kv_heads_local, int n_splits,
                                            int want_stages, int sm_count) {
  AttnLaunchPlan p;
  int st = want_stages;
  while (st > 2 && attn_smem_plan(head_dim, group, M, st).total > (size_t)kSmemMax) --st;
  p.sp = attn_smem_plan(head_dim, group, M, st);
  p.stages = st;
  p.ok = p.sp.total <= (size_t)kSmemMax;
  p.smem = p.sp.total;
  if (kv_heads_local * n_splits <= sm_count && p.smem < (size_t)116 * 1024) p.smem = (size_t)116 * 1024;
  return p;
}

// Attention over the paged cache: the splits of one kv head = one thread-block cluster (DSMEM
// merge); head_dim selects the instantiation, the shared-memory plan depends on (group, M).
template <int HD>
static int launch_attention_t(lsk_engine* e, AttnArgs& a) {
  static std::atomic<uint64_t> configured{0};
  auto kern = attn_cluster_kernel<HD>;
  int dev = 0;
  CU(cudaGetDevice(&dev));
  const uint64_t bit = 1ull << (dev & 63);
  if (!(configured.load(std::memory_order_relaxed) & bit)) {
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
    configured.fetch_or(bit, std::memory_order_relaxed);
  }
  const AttnLaunchPlan lp = plan_attention_launch(HD, a.group, a.M, a.n_kv_heads, a.n_splits, e->attn_stages, e->sm_count);
  const AttnSmemPlan& sp = lp.sp;
  a.n_stages = lp.stages;
  if (!lp.ok)
    return fail(LSK_ERR_INVALID, "attention: %d query rows per kv head do not fit shared memory", a.group * a.M);
  a.rows_pad = (a.group * a.M + 15) / 16 * 16;
  a.merge_off = sp.merge_off; a.part_off = sp.part_off; a.reload_per_rb = sp.reload_per_rb;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(a.n_kv_heads, a.n_splits);
  cfg.blockDim = dim3(kAttnThreads);
  // a grid that fits one wave gets a whole SM per CTA (> half of the SM's shared memory): the
  // CTAs then spread over the SMs instead of sharing a few SMs' load bandwidth
  cfg.dynamicSmemBytes = lp.smem;
  cfg.stream = e->stream;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 1; at[0].val.clusterDim.y = a.n_splits; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = e->use_pdl ? 2 : 1;
  e->launches += 1;
  e->capture_launches += 1;
  if (!e->profiling) {
    CU(cudaLaunchKernelEx(&cfg, kern, a));
  } else {
    cudaEvent_t ea, eb;
    cudaEventCreate(&ea); cudaEventCreate(&eb);
    cudaEventRecord(ea, e->stream);
    cudaError_t err = cudaLaunchKernelEx(&cfg, kern, a);
    cudaEventRecord(eb, e->stream);
    e->prof_events.push_back({e->cur_class, {ea, eb}});
    CU(err);
  }
  return LSK_OK;
}
static int launch_attention(lsk_engine* e, AttnArgs& a, int head_dim) {
  switch (head_dim) {
    case 128: return launch_attention_t<128>(e, a);
    case 64: return launch_attention_t<64>(e, a);
    case 32: return launch_attention_t<32>(e, a);
    default: return fail(LSK_ERR_INVALID, "head_dim %d unsupported (32, 64 or 128)", head_dim);
  }
}

// ---------------------------------------------------------------------------------------------
// one decoder layer on hidden rows [row0, row0 + M) at positions *base_len + pos_off + i
//   (HF LlamaDecoderLayer as called at llama_model_utils.py:193-201,253-261,354-362,375-383)
// ---------------------------------------------------------------------------------------------
static int enqueue_layer(lsk_engine* e, int li, int row0, int M, const int* base_len, int pos_off,
                         const void* after_W = nullptr, size_t after_bytes = 0) {
  const lsk_config& c = e->cfg;
  LayerWeights& L = e->layers[li];
  float* x = e->hidden + (size_t)row0 * c.hidden;
  __nv_bfloat16* kp = e->kpool + (size_t)li * e->pool_layer_elems;
  __nv_bfloat16* vp = e->vpool + (size_t)li * e->pool_layer_elems;
  const bool tp = c.tp_size > 1;
  const size_t h2 = (size_t)c.hidden * 2;
  auto cap = [&](size_t bytes) { return bytes < e->l2_prefetch_bytes ? bytes : e->l2_prefetch_bytes; };

  if (!(e->ablate & (1u << CLS_QKV))) {  // RMSNorm -> QKV -> RoPE -> KV append
    e->cur_class = CLS_QKV;
    GemmArgs a{};
    a.W = reinterpret_cast<const uint4*>(L.wqkv);
    a.M = M;
    a.x_f32 = x; a.x_ld = c.hidden; a.norm_w = L.ln1; a.eps = c.rms_eps;
    a.q_out = e->qbuf; a.q_ld = e->q_rows;
    a.kpool = kp; a.vpool = vp; a.page_table = e->page_table;
    a.base_len = base_len; a.pos_off = pos_off; a.rope = e->rope; a.head_dim = c.head_dim;
    a.q_rows = e->q_rows; a.kv_rows = e->kv_rows; a.n_kv_heads = e->kv_heads_l;
    a.next_W = L.wo; a.next_bytes = e->l2_prefetch_bytes ? (size_t)e->q_rows * h2 : 0;
    TRY((launch_gemm<PRO_RMS, EPI_QKV>(e, e->p_qkv, a)));
  }
  if (!(e->ablate & (1u << CLS_ATTN))) {  // attention over the paged cache
    e->cur_class = CLS_ATTN;
    AttnArgs a{};
    a.q = e->qbuf; a.q_ld = e->q_rows; a.out = e->attn_out; a.out_ld = e->q_rows;
    a.kpool = kp; a.vpool = vp; a.page_table = e->page_table;
    a.base_len = base_len; a.pos_off = pos_off; a.M = M; a.group = e->group;
    a.n_kv_heads = e->kv_heads_l; a.n_splits = e->n_splits;
    a.scale = 1.0f / sqrtf((float)c.head_dim);
    TRY(launch_attention(e, a, c.head_dim));
  }
  if (!(e->ablate & (1u << CLS_O))) {  // O projection (+ residual, or all-reduce then residual under TP)
    e->cur_class = CLS_O;
    GemmArgs a{};
    a.W = reinterpret_cast<const uint4*>(L.wo);
    a.M = M;
    a.x_bf16 = e->attn_out; a.xb_ld = e->q_rows;
    a.next_W = L.wgu; a.next_bytes = cap((size_t)2 * e->inter_l * h2);
    if (!tp) {
      a.out_f32 = x; a.out_ld = c.hidden;
      TRY((launch_gemm<PRO_BF16, EPI_RESID>(e, e->p_o, a)));
    } else if (e->peer_ok && e->peer_mode == 2) {
      TRY(emit_gemm_push_resid(e, e->p_o, a, x));
    } else {
      a.out_f32 = e->tp_buf; a.out_ld = c.hidden;
      TRY((launch_gemm<PRO_BF16, EPI_STORE>(e, e->p_o, a)));
      TRY(emit_allreduce_resid(e, x, M));
    }
  }
  if (!(e->ablate & (1u << CLS_GATEUP))) {  // RMSNorm -> gate/up -> SiLU * up
    e->cur_class = CLS_GATEUP;
    GemmArgs a{};
    a.W = reinterpret_cast<const uint4*>(L.wgu);
    a.M = M;
    a.x_f32 = x; a.x_ld = c.hidden; a.norm_w = L.ln2; a.eps = c.rms_eps;
    a.act = e->act; a.act_ld = e->inter_l_pad;
    a.next_W = L.wd; a.next_bytes = cap((size_t)e->inter_l * h2);
    TRY((launch_gemm<PRO_RMS, EPI_SILU>(e, e->p_gu, a)));
  }
  if (!(e->ablate & (1u << CLS_DOWN))) {  // down projection (+ residual)
    e->cur_class = CLS_DOWN;
    GemmArgs a{};
    a.W = reinterpret_cast<const uint4*>(L.wd);
    a.M = M;
    a.x_bf16 = e->act; a.xb_ld = e->inter_l_pad;
    a.next_W = after_W; a.next_bytes = after_W ? cap(after_bytes) : 0;
    if (!tp) {
      a.out_f32 = x; a.out_ld = c.hidden;
      TRY((launch_gemm<PRO_BF16, EPI_RESID>(e, e->p_d, a)));
    } else if (e->peer_ok && e->peer_mode == 2) {
      TRY(emit_gemm_push_resid(e, e->p_d, a, x));
    } else {
      a.out_f32 = e->tp_buf; a.out_ld = c.hidden;
      TRY((launch_gemm<PRO_BF16, EPI_STORE>(e, e->p_d, a)));
      TRY(emit_allreduce_resid(e, x, M));
    }
  }
  return LSK_OK;
}

// ---------------------------------------------------------------------------------------------
// prompt chunk of m <= 128 tokens at positions c0 .. c0+m-1 through every layer on the tcgen05
// GEMMs (forward_early + forward_remainder of llama_model_utils.py:213-276 / 363-383 on s = T_p)
// ---------------------------------------------------------------------------------------------
template <int EPI>
static int launch_prefill_gemm(lsk_engine* e, PrefillGemmArgs& a) {
  a.n_stages = e->pf_stages;
  const int items = a.n_tiles * (EPI == PF_EPI_STORE && a.k_splits > 1 ? a.k_splits : 1);
  const int grid = items < e->sm_count ? items : e->sm_count;
  CU(launch(e, prefill_gemm_tc_kernel<EPI>, dim3(grid), dim3(kTcThreads), prefill_tc_smem_bytes(a.n_stages), a));
  return LSK_OK;
}

static int enqueue_prefill_chunk(lsk_engine* e, int c0, int m) {
  const lsk_config& c = e->cfg;
  const bool tp = c.tp_size > 1;
  e->cur_class = CLS_MISC;
  CU(launch(e, embed_tokens_kernel, dim3(m), dim3(256), 0, (const __nv_bfloat16*)e->embed, c.hidden,
            (const int*)(e->d_prompt + c0), e->hidden_p, c.hidden));
  // rows of one attention launch: as many as fit its shared-memory plan (multiple of 16)
  int m_attn = 16;
  for (int cand = kPfTokens; cand >= 16; cand -= 16)
    if (attn_smem_plan(c.head_dim, e->group, cand, 2).total <= (size_t)kSmemMax) { m_attn = cand; break; }
  // row-parallel GEMMs (O / down): hidden / 128 feature tiles are too few to keep the SMs streaming
  // -> split K; the partial tiles are summed (fixed order) by the next rms_canon_kernel
  const int ks_o = std::max(1, std::min(std::min(4, e->kst_q), e->sm_count / e->pf_t_h));
  const int ks_d = std::max(1, std::min(std::min(4, e->kst_i), e->sm_count / e->pf_t_h));
  const size_t part_stride = (size_t)kPfTokens * c.hidden;
  // pending row-parallel partials that the next norm kernel has to add to the residual rows
  const float* pend = nullptr;
  int n_pend = 0;
  auto after_row_parallel = [&](int n_splits) -> int {
    if (!tp) { pend = e->part_p; n_pend = n_splits; return LSK_OK; }
    e->cur_class = CLS_COMM;
    CU(launch(e, reduce_partials_kernel, dim3(m), dim3(256), 0, (const float*)e->part_p, n_splits, part_stride,
              c.hidden, c.hidden, e->tp_buf_p));
    e->launches += 1;
    e->capture_launches += 1;
    NC(ncclAllReduce(e->tp_buf_p, e->tp_buf_p, (size_t)m * c.hidden, ncclFloat, ncclSum, e->comm, e->stream));
    pend = e->tp_buf_p; n_pend = 1;
    return LSK_OK;
  };
  for (int li = 0; li < c.n_layers; ++li) {
    LayerWeights& L = e->layers[li];
    __nv_bfloat16* kp = e->kpool + (size_t)li * e->pool_layer_elems;
    __nv_bfloat16* vp = e->vpool + (size_t)li * e->pool_layer_elems;
    e->cur_class = CLS_QKV;
    CU(launch(e, rms_canon_kernel, dim3(m), dim3(256), 0, e->hidden_p, c.hidden, pend, n_pend, part_stride,
              (const __nv_bfloat16*)L.ln1, c.rms_eps, c.hidden, e->xn_c));
    {
      PrefillGemmArgs a{};
      a.W = L.wqkv_c; a.X = e->xn_c; a.n_tiles = e->pf_t_qkv; a.n_rows = e->q_rows + 2 * e->kv_rows;
      a.n_kst = e->kst_h; a.M = m; a.k_splits = 1;
      a.q_out = e->q_p; a.q_ld = e->q_rows; a.kpool = kp; a.vpool = vp; a.page_table = e->page_table;
      a.pos0 = c0; a.rope = e->rope; a.head_dim = c.head_dim;
      a.q_rows = e->q_rows; a.kv_rows = e->kv_rows; a.n_kv_heads = e->kv_heads_l;
      TRY(launch_prefill_gemm<PF_EPI_QKV>(e, a));
    }
    // the prompt pass has no LM head (the reference discards those logits): once the last layer's
    // K/V rows are written nothing downstream is needed
    if (li + 1 == c.n_layers) break;
    e->cur_class = CLS_ATTN;
    for (int r0 = 0; r0 < m; r0 += m_attn) {
      AttnArgs a{};
      a.q = e->q_p + (size_t)r0 * e->q_rows; a.q_ld = e->q_rows;
      // operand rows are addressed by token index inside the 128-row stage: shift by r0 rows
      a.out = reinterpret_cast<__nv_bfloat16*>(e->attn_c + canon_offset(r0, 0)); a.out_canon = 1;
      a.kpool = kp; a.vpool = vp; a.page_table = e->page_table;
      a.base_len = e->d_zero; a.pos_off = c0 + r0; a.M = (m - r0) < m_attn ? (m - r0) : m_attn;
      a.group = e->group; a.n_kv_heads = e->kv_heads_l; a.n_splits = e->n_splits;
      a.scale = 1.0f / sqrtf((float)c.head_dim);
      TRY(launch_attention(e, a, c.head_dim));
    }
    e->cur_class = CLS_O;
    {
      PrefillGemmArgs a{};
      a.W = L.wo_c; a.X = e->attn_c; a.n_tiles = e->pf_t_h; a.n_rows = c.hidden; a.n_kst = e->kst_q; a.M = m;
      a.k_splits = ks_o; a.out_f32 = e->part_p; a.out_ld = c.hidden;
      TRY(launch_prefill_gemm<PF_EPI_STORE>(e, a));
      TRY(after_row_parallel(ks_o));
    }
    e->cur_class = CLS_GATEUP;
    CU(launch(e, rms_canon_kernel, dim3(m), dim3(256), 0, e->hidden_p, c.hidden, pend, n_pend, part_stride,
              (const __nv_bfloat16*)L.ln2, c.rms_eps, c.hidden, e->xn_c));
    {
      PrefillGemmArgs a{};
      a.W = L.wgu_c; a.X = e->xn_c; a.n_tiles = e->pf_t_gu; a.n_rows = 2 * e->inter_l; a.n_kst = e->kst_h; a.M = m;
      a.k_splits = 1; a.act_canon = e->act_c;
      TRY(launch_prefill_gemm<PF_EPI_SILU>(e, a));
    }
    e->cur_class = CLS_DOWN;
    {
      PrefillGemmArgs a{};
      a.W = L.wd_c; a.X = e->act_c; a.n_tiles = e->pf_t_h; a.n_rows = c.hidden; a.n_kst = e->kst_i; a.M = m;
      a.k_splits = ks_d; a.out_f32 = e->part_p; a.out_ld = c.hidden;
      TRY(launch_prefill_gemm<PF_EPI_STORE>(e, a));
      TRY(after_row_parallel(ks_d));
    }
  }
  return LSK_OK;
}

// ---------------------------------------------------------------------------------------------
// small stages
// ---------------------------------------------------------------------------------------------
static int emit_embed(lsk_engine* e, const int* ids, float* rows, int n_rows) {
  const lsk_config& c = e->cfg;
  e->cur_class = CLS_MISC;
  CU(launch(e, embed_tokens_kernel, dim3(n_rows), dim3(256), 0, (const __nv_bfloat16*)e->embed, c.hidden,
            ids, rows, c.hidden));
  return LSK_OK;
}
static const float* cand_val_ptr(lsk_engine* e);
static const int* cand_idx_ptr(lsk_engine* e);
// what the sampling kernels read: the local logits, or under TP the gathered [16][vocab] rows
static const float* samp_logits(lsk_engine* e) { return e->cfg.tp_size > 1 ? e->logits_full : e->logits; }
static int samp_ld(lsk_engine* e) { return e->cfg.tp_size > 1 ? e->cfg.vocab : e->vocab_l_pad; }
static int n_cand(lsk_engine* e);
static int emit_finalize(lsk_engine* e, int slot, float* dst_row) {
  const lsk_config& c = e->cfg;
  e->cur_class = CLS_MISC;
  CU(launch(e, finalize_embed_kernel, dim3(8), dim3(128), 0, cand_val_ptr(e), cand_idx_ptr(e), n_cand(e),
            e->state, slot, (const __nv_bfloat16*)e->embed, c.hidden, dst_row));
  return LSK_OK;
}
// token history (prompt ids + emitted tokens) is kept on the device only when the n-gram ban needs it
static int* hist_ptr(lsk_engine* e) { return e->gen.no_repeat_ngram_size > 0 ? e->d_prompt : nullptr; }
static int emit_accept(lsk_engine* e, int d_spec, int seq) {
  e->cur_class = CLS_MISC;
  CU(launch(e, accept_greedy_kernel, dim3(1), dim3(256), 0, cand_val_ptr(e), cand_idx_ptr(e), n_cand(e), d_spec,
            e->state, (const GenParams*)e->gen_dev, e->res_dev, seq, hist_ptr(e)));
  return LSK_OK;
}
static int emit_ar_commit(lsk_engine* e, int seq) {
  e->cur_class = CLS_MISC;
  CU(launch(e, ar_commit_kernel, dim3(1), dim3(32), 0, cand_val_ptr(e), cand_idx_ptr(e), n_cand(e), e->state,
            e->res_dev, seq, hist_ptr(e)));
  return LSK_OK;
}

// final RMSNorm + LM head on rows [row0, row0+M): arg-max candidates (and optional logits).
// (llama_model_utils.py:204-205, 271-273, 386-387).  Afterwards e->cand_* / n_cand() hold one
// (value, index) per candidate per row.
// With no_repeat_ngram_size > 0 (NoRepeatNGramLogitsProcessor, generator_base.py:77-85) the logits
// are materialised, the tokens that would repeat an n-gram of the sequence so far are set to -inf
// (row r continues prompt ++ output ++ draft[0 .. j0 + r)), and the arg-max is taken from the
// banned rows instead of the LM-head epilogue.
static int enqueue_lm_head(lsk_engine* e, int row0, int M, int j0, const void* after_W = nullptr, size_t after_bytes = 0) {
  const lsk_config& c = e->cfg;
  const bool ban = e->gen.no_repeat_ngram_size > 0;
  e->cur_class = CLS_LMHEAD;
  GemmArgs a{};
  a.W = reinterpret_cast<const uint4*>(e->lm_head);
  a.M = M;
  a.x_f32 = e->hidden + (size_t)row0 * c.hidden; a.x_ld = c.hidden;
  a.norm_w = e->final_norm; a.eps = c.rms_eps;
  a.logits = (e->keep_logits || e->gen.sample || ban) ? e->logits : nullptr; a.logits_ld = e->vocab_l_pad;
  a.n_valid_rows = e->vocab_l; a.vocab_off = e->vocab_off;
  a.part_val = e->cand_val; a.part_idx = e->cand_idx;
  a.next_W = after_W;
  a.next_bytes = after_W ? (after_bytes < e->l2_prefetch_bytes ? after_bytes : e->l2_prefetch_bytes) : 0;
  if (e->lm_tc) {
    if (!(e->ablate & (1u << CLS_LMHEAD))) {
      LmHeadTcArgs t{};
      t.W = e->lm_head_tc; t.n_tiles = e->lm_tc_tiles; t.K = c.hidden; t.M = M; t.n_stages = e->lm_tc_stages;
      t.x_f32 = a.x_f32; t.x_ld = a.x_ld; t.norm_w = a.norm_w; t.eps = a.eps;
      t.logits = a.logits; t.logits_ld = a.logits_ld; t.n_valid_rows = a.n_valid_rows; t.vocab_off = a.vocab_off;
      t.part_val = a.part_val; t.part_idx = a.part_idx;
      CU(launch(e, lmhead_tc_kernel, dim3(e->lm_tc_grid), dim3(kTcThreads),
                lmhead_tc_smem_bytes(c.hidden, e->lm_tc_stages), t));
    }
  } else if (!(e->ablate & (1u << CLS_LMHEAD))) TRY((launch_gemm<PRO_RMS, EPI_LMHEAD>(e, e->p_lm, a)));
  e->cur_class = CLS_MISC;
  const float* cv = e->cand_val;
  const int* ci = e->cand_idx;
  // one candidate per CTA of the launch above.  The even-wave grid of the skinny GEMM can be
  // smaller than min(tiles, SMs); a slot no CTA wrote would hold a stale (0.0, index 0) pair and
  // win every row whose logits are all negative.
  int ncand = e->lm_tc ? e->lm_tc_grid : plan_sched(M <= 8 ? 1 : 2, M, PRO_RMS, EPI_LMHEAD, e->p_lm, e->sm_count).grid;
  if (ban) {
    CU(launch(e, ngram_ban_kernel, dim3(M), dim3(256), 0, e->logits, e->vocab_l_pad, e->vocab_l, e->vocab_off,
              (const int*)e->d_prompt, (const DevState*)e->state, (int)e->gen.no_repeat_ngram_size, j0));
    if (!e->gen.sample) {
      CU(launch(e, argmax_rows_kernel, dim3(M), dim3(1024), 0, (const float*)e->logits, e->vocab_l_pad, e->vocab_l,
                e->vocab_off, e->ban_val, e->ban_idx));
      cv = e->ban_val; ci = e->ban_idx; ncand = 1;
    }
  }
  e->cur_cand_val = cv; e->cur_cand_idx = ci; e->cur_n_cand = ncand;
  if (c.tp_size > 1 && e->gen.sample) {
    // every rank needs the whole distribution: all-gather the vocab shards of the M rows, lay them
    // out as [M][vocab]; all ranks then run the same warp / Philox draw and stay in lockstep
    e->cur_class = CLS_COMM;
    NC(ncclAllGather(e->logits, e->logits_gath, (size_t)M * e->vocab_l_pad, ncclFloat, e->comm, e->stream));
    CU(launch(e, tp_logits_rows_kernel, dim3(32, M), dim3(256), 0, (const float*)e->logits_gath, c.tp_size, M,
              e->vocab_l, e->vocab_l_pad, e->logits_full, c.vocab));
    e->cur_class = CLS_MISC;
  }
  if (c.tp_size > 1 && e->peer_ok) {
    CU(launch(e, tp_gather_best_kernel, dim3(1), dim3(256), 0, e->peer, cv, ci, ncand, M, e->gath_val, e->gath_idx));
  } else if (c.tp_size > 1) {
    CU(launch(e, rank_best_kernel, dim3(1), dim3(256), 0, cv, ci, ncand, M, e->rank_val, e->rank_idx));
    NC(ncclAllGather(e->rank_val, e->gath_val, kMaxRows, ncclFloat, e->comm, e->stream));
    NC(ncclAllGather(e->rank_idx, e->gath_idx, kMaxRows, ncclInt32, e->comm, e->stream));
  }
  return LSK_OK;
}
// candidates of the LAST enqueued LM head (what the following finalize / accept kernel consumes)
static const float* cand_val_ptr(lsk_engine* e) { return e->cfg.tp_size > 1 ? e->gath_val : e->cur_cand_val; }
static const int* cand_idx_ptr(lsk_engine* e) { return e->cfg.tp_size > 1 ? e->gath_idx : e->cur_cand_idx; }
static int n_cand(lsk_engine* e) { return e->cfg.tp_size > 1 ? e->cfg.tp_size : e->cur_n_cand; }

// ---------------------------------------------------------------------------------------------
// round / AR-step command streams
// ---------------------------------------------------------------------------------------------
static int enqueue_round(lsk_engine* e, int E, int d, int seq) {
  const lsk_config& c = e->cfg;
  const int* len = &e->state->len;
  // row 0 <- embedding of the pending token (self_speculation_generator.py:122, input_ids)
  TRY(emit_embed(e, &e->state->tok[0], e->hidden, 1));
  // draft loop (:127-148): step i runs layers [0,E) on row i at position len+i, then the shared
  // head; its arg-max becomes tok[i+1] and is embedded into row i+1.
  const size_t qkv_bytes = (size_t)(e->q_rows + 2 * e->kv_rows) * c.hidden * 2;
  const size_t lm_bytes = (size_t)e->vocab_l_pad * c.hidden * 2;
  auto layer_then = [&](int l, int row0, int M, int pos_off, int stop) -> int {
    // what streams after layer l: the next layer's QKV, or the LM head at the end of a pass
    const void* nw = (l + 1 < stop) ? (const void*)e->layers[l + 1].wqkv : (const void*)e->lm_head;
    const size_t nb = (l + 1 < stop) ? qkv_bytes : lm_bytes;
    return enqueue_layer(e, l, row0, M, len, pos_off, nw, nb);
  };
  for (int i = 0; i < d; ++i) {
    for (int l = 0; l < E; ++l) TRY(layer_then(l, i, 1, i, E));
    TRY(enqueue_lm_head(e, i, 1, i, e->layers[0].wqkv, qkv_bytes));
    e->cur_class = CLS_MISC;
    if (!e->gen.sample) {
      TRY(emit_finalize(e, 1 + i, e->hidden + (size_t)(i + 1) * c.hidden));
    } else {
      // decode_next_token sampling branch (llama_model_utils.py:123-131): keep the warped
      // distribution of draft i (needed by the rejection test), draw tok[i+1], embed it.
      CU(launch(e, warp_and_sample_kernel, dim3(1), dim3(kSampleThreads), 0, samp_logits(e),
                samp_ld(e), c.vocab, (const GenParams*)e->gen_dev, (const DevState*)e->state,
                e->probs_d + (size_t)i * c.vocab, &e->state->tok[1 + i], (int)RNG_DRAFT, i));
      CU(launch(e, embed_tokens_kernel, dim3(1), dim3(256), 0, (const __nv_bfloat16*)e->embed, c.hidden,
                (const int*)&e->state->tok[1 + i], e->hidden + (size_t)(i + 1) * c.hidden, c.hidden));
    }
  }
  // verify (:164-174 -> llama_model_utils.py:280-391): the last drafted token has not been
  // through layers < E yet (:350-362) ...
  for (int l = 0; l < E; ++l) {
    if (l + 1 < E || E < c.n_layers) TRY(enqueue_layer(e, l, d, 1, len, d, e->layers[l + 1].wqkv, qkv_bytes));
    else TRY(enqueue_layer(e, l, d, 1, len, d, e->lm_head, lm_bytes));
  }
  // ... then layers >= E see [exit rows of the draft steps ; that row] = rows 0..d (:363-383)
  for (int l = E; l < c.n_layers; ++l) TRY(layer_then(l, 0, d + 1, 0, c.n_layers));
  TRY(enqueue_lm_head(e, 0, d + 1, 0, e->layers[0].wqkv, qkv_bytes));
  e->cur_class = CLS_MISC;
  if (!e->gen.sample) {
    TRY(emit_accept(e, d, seq));
  } else {
    CU(launch(e, warp_and_sample_kernel, dim3(d + 1), dim3(kSampleThreads), 0, samp_logits(e),
              samp_ld(e), c.vocab, (const GenParams*)e->gen_dev, (const DevState*)e->state,
              e->probs_v, &e->state->verified[0], (int)RNG_VERIFY, 0));
    CU(launch(e, accept_sample_kernel, dim3(1), dim3(kSampleThreads), 0, (const float*)e->probs_d,
              (const float*)e->probs_v, c.vocab, d, e->state, (const GenParams*)e->gen_dev, e->res_dev,
              e->samp_scratch, seq, hist_ptr(e)));
  }
  return LSK_OK;
}

static int enqueue_ar(lsk_engine* e, int n_layers_run, int seq) {
  const lsk_config& c = e->cfg;
  const int* len = &e->state->len;
  TRY(emit_embed(e, &e->state->tok[0], e->hidden, 1));
  const size_t qkv_bytes = (size_t)(e->q_rows + 2 * e->kv_rows) * c.hidden * 2;
  const size_t lm_bytes = (size_t)e->vocab_l_pad * c.hidden * 2;
  for (int l = 0; l < n_layers_run; ++l) {
    if (l + 1 < n_layers_run) TRY(enqueue_layer(e, l, 0, 1, len, 0, e->layers[l + 1].wqkv, qkv_bytes));
    else TRY(enqueue_layer(e, l, 0, 1, len, 0, e->lm_head, lm_bytes));
  }
  TRY(enqueue_lm_head(e, 0, 1, 0, e->layers[0].wqkv, qkv_bytes));
  e->cur_class = CLS_MISC;
  if (!e->gen.sample) {
    TRY(emit_ar_commit(e, seq));
  } else {
    CU(launch(e, warp_and_sample_kernel, dim3(1), dim3(kSampleThreads), 0, samp_logits(e),
              samp_ld(e), c.vocab, (const GenParams*)e->gen_dev, (const DevState*)e->state,
              e->probs_v, &e->state->verified[0], (int)RNG_VERIFY, 0));
    CU(launch(e, ar_commit_sampled_kernel, dim3(1), dim3(32), 0, e->state, e->res_dev, seq, hist_ptr(e)));
  }
  return LSK_OK;
}

// Run `enqueue` either eagerly or as a cached CUDA graph keyed by `key`.  The completion stamp
// (`seq`) is baked into eager launches; graph replays use stamp 0 + an event instead.
template <typename F>
static int run_cached(lsk_engine* e, long long key, F enqueue) {
  CU(cudaEventRecord(e->ev0, e->stream));
  if (!e->use_graph) {
    TRY(enqueue());
  } else {
    auto it = e->graphs.find(key);
    if (it == e->graphs.end()) {
      cudaGraph_t graph = nullptr;
      const int64_t before = e->launches;
      e->capture_launches = 0;
      CU(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
      int st = enqueue();
      cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
      if (st != LSK_OK) { if (graph) cudaGraphDestroy(graph); return st; }
      if (ce != cudaSuccess) return fail(LSK_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(ce));
      cudaGraphExec_t exec = nullptr;
      CU(cudaGraphInstantiate(&exec, graph, 0));
      CU(cudaGraphDestroy(graph));
      e->graph_launches[key] = e->capture_launches;
      e->launches = before;   // captured, not executed
      it = e->graphs.emplace(key, exec).first;
    }
    CU(cudaGraphLaunch(it->second, e->stream));
    e->launches += e->graph_launches[key];
  }
  CU(cudaEventRecord(e->ev1, e->stream));
  CU(cudaEventSynchronize(e->ev1));
  CU(cudaEventElapsedTime(&e->last_ms, e->ev0, e->ev1));
  return LSK_OK;
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int lsk_abi_version(void) { return LSK_ABI_VERSION; }
const char* lsk_last_error(void) { return g_last_error.c_str(); }

static int create_into(lsk_engine* e, const lsk_config& c);

int lsk_create(const lsk_config* cfg, lsk_engine** out) {
  if (!cfg || !out) return fail(LSK_ERR_INVALID, "null argument");
  const lsk_config& c = *cfg;
  if (c.head_dim != 128 && c.head_dim != 64 && c.head_dim != 32)
    return fail(LSK_ERR_INVALID, "head_dim %d unsupported (32, 64 or 128)", c.head_dim);
  if (c.rope_scaling < LSK_ROPE_DEFAULT || c.rope_scaling > LSK_ROPE_LLAMA3)
    return fail(LSK_ERR_INVALID, "rope_scaling %d unknown", c.rope_scaling);
  if (c.rope_scaling != LSK_ROPE_DEFAULT && !(c.rope_factor > 0.f))
    return fail(LSK_ERR_INVALID, "rope scaling needs factor > 0");
  if (c.rope_scaling == LSK_ROPE_LLAMA3 &&
      (!(c.rope_high_freq_factor > c.rope_low_freq_factor) || c.rope_original_max_pos < 1))
    return fail(LSK_ERR_INVALID, "llama3 rope scaling needs high_freq_factor > low_freq_factor and original_max_position_embeddings");
  if (c.tp_size < 1 || c.tp_rank < 0 || c.tp_rank >= c.tp_size) return fail(LSK_ERR_INVALID, "bad tp_rank/tp_size");
  if (c.n_heads % c.tp_size || c.n_kv_heads % c.tp_size || c.n_heads % c.n_kv_heads)
    return fail(LSK_ERR_INVALID, "heads (%d) / kv heads (%d) must divide by tp_size (%d)", c.n_heads, c.n_kv_heads, c.tp_size);
  if (c.inter % (c.tp_size * 8)) return fail(LSK_ERR_INVALID, "intermediate size %d must be a multiple of 8*tp_size", c.inter);
  if (c.hidden % 32 || c.hidden > 8192) return fail(LSK_ERR_INVALID, "hidden %d must be a multiple of 32 and <= 8192", c.hidden);
  if (c.vocab % c.tp_size) return fail(LSK_ERR_INVALID, "vocab must divide by tp_size");
  if (c.n_layers < 1 || c.max_ctx < 2) return fail(LSK_ERR_INVALID, "bad n_layers / max_ctx");

  // everything that can fail half-way runs in create_into(); a failure releases what was built
  lsk_engine* e = new lsk_engine();
  const int st = create_into(e, c);
  if (st != LSK_OK) {
    const std::string why = g_last_error;
    lsk_destroy(e);
    g_last_error = why;
    return st;
  }
  *out = e;
  return LSK_OK;
}

static int create_into(lsk_engine* e, const lsk_config& c) {
  e->cfg = c;
  int dev = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, dev));
  e->use_pdl = !(c.flags & LSK_FLAG_NO_PDL);
  e->use_graph = !(c.flags & LSK_FLAG_NO_GRAPH);
  e->keep_logits = (c.flags & LSK_FLAG_KEEP_LOGITS) != 0;
  // tensor-parallel collectives: one-shot kernels over peer-mapped HBM.  Default 2 = the
  // row-parallel GEMM pushes its tiles to every rank from its own epilogue as LL lines (measured
  // 7B TP=2: 173 tok/s; 1 = separate LL push + reduce kernel 169; 3 = fence + flag protocol 129;
  // 0 = NCCL 134 — profiles/r2_tp2_modes.md).  LSK_FLAG_TP_NCCL forces NCCL from the API.
  {
    const char* env = getenv("LSK_TP_ONESHOT");
    const int mode = env ? atoi(env) : ((c.flags & LSK_FLAG_TP_NCCL) ? 0 : 2);
    e->want_peer = c.tp_size > 1 && mode != 0;
    e->peer_mode = (mode >= 1 && mode <= 3) ? mode : 2;
  }
  if (const char* env = getenv("LSK_ABLATE")) {
    // diagnostics only: the named kernel classes are not launched (results are garbage, the
    // round keeps its shape) so that t(full) - t(ablated) gives a class's cost INSIDE the graph
    static const char* names[] = {"qkv", "attn", "o", "gate_up", "down", "lm_head"};
    std::string list(env);
    for (size_t pos = 0; pos <= list.size();) {            // comma-separated, exact names
      const size_t end = std::min(list.find(',', pos), list.size());
      const std::string tok = list.substr(pos, end - pos);
      for (int i = 0; i < 6; ++i)
        if (tok == names[i]) e->ablate |= 1u << i;
      pos = end + 1;
    }
    if (e->ablate) fprintf(stderr, "[lsk] LSK_ABLATE=%s: kernel classes skipped, outputs are NOT valid\n", env);
  }
  e->heads_l = c.n_heads / c.tp_size;
  e->kv_heads_l = c.n_kv_heads / c.tp_size;
  e->group = c.n_heads / c.n_kv_heads;
  e->q_rows = e->heads_l * c.head_dim;
  e->kv_rows = e->kv_heads_l * c.head_dim;
  e->inter_l = c.inter / c.tp_size;
  e->inter_l_pad = (e->inter_l + 31) / 32 * 32;   // K of the down projection (zero columns beyond inter_l)
  e->vocab_l = c.vocab / c.tp_size;
  e->vocab_l_pad = (e->vocab_l + 15) / 16 * 16;
  e->vocab_off = c.tp_rank * e->vocab_l;
  e->n_pages = (c.max_ctx + kPageTokens - 1) / kPageTokens;
  e->max_pos = e->n_pages * kPageTokens;
  // split-KV factor: a constant of the engine (results are batch-invariant only for a fixed
  // partition).  Measured (profiles/r2_attention_sweep.md): the kernel is bound by per-SM load
  // bandwidth and barrier latency, so the best grid is ONE CTA per SM on as many SMs as possible —
  // splits = floor(SMs / kv heads), at most 4 (7B: 32 heads x 4 splits; an 8-CTA cluster's barrier
  // and 8-way merge cost more than the extra SMs bring: 16 heads x 8 splits ran 23 us against 15).
  e->n_splits = c.attn_splits > 0 ? c.attn_splits : attn_default_splits(e->sm_count, e->kv_heads_l);
  if (const char* env = getenv("LSK_ATTN_SPLITS")) e->n_splits = atoi(env);   // clamped to [1, 8] below
  if (const char* env = getenv("LSK_ATTN_STAGES")) e->attn_stages = atoi(env);
  if (e->attn_stages < 2) e->attn_stages = 2;
  if (e->attn_stages > kAttnMaxStages) e->attn_stages = kAttnMaxStages;
  if (e->n_splits > 8) e->n_splits = 8;
  if (e->n_splits < 1) e->n_splits = 1;

  e->p_qkv = make_plan(e->q_rows + 2 * e->kv_rows, c.hidden, e->sm_count);
  e->p_o = make_plan(c.hidden, e->q_rows, e->sm_count);
  e->p_gu = make_plan(2 * e->inter_l, c.hidden, e->sm_count);
  e->p_d = make_plan(c.hidden, e->inter_l_pad, e->sm_count);
  e->p_lm = make_plan(e->vocab_l_pad, c.hidden, e->sm_count);
  if (const char* env = getenv("LSK_L2_PREFETCH_MB")) e->l2_prefetch_bytes = (size_t)atoi(env) << 20;
  if (getenv("LSK_LMHEAD_TC") && atoi(getenv("LSK_LMHEAD_TC")) != 0) {
    // tcgen05 LM head: needs hidden % 64 == 0 and the 16-token B operand + a >= 3-stage ring in
    // shared memory (hidden <= 5120); otherwise stay on the mma.sync kernel, loudly
    int st = kTcMaxStages;
    while (st >= 3 && lmhead_tc_smem_bytes(c.hidden, st) > (size_t)kSmemMax) --st;
    if (c.hidden % kTcStageK == 0 && st >= 3) {
      e->lm_tc = true;
      e->lm_tc_stages = st;
      e->lm_tc_tiles = (e->vocab_l + kTcTileRows - 1) / kTcTileRows;
      const int waves = (e->lm_tc_tiles + e->sm_count - 1) / e->sm_count;
      e->lm_tc_grid = (e->lm_tc_tiles + waves - 1) / waves;        // even waves
    } else {
      fprintf(stderr, "[lsk] LSK_LMHEAD_TC ignored: hidden %d does not fit the tcgen05 LM head\n", c.hidden);
    }
  }
  e->max_rows = plan_sched(2, kMaxRows, PRO_RMS, EPI_QKV, e->p_qkv, e->sm_count).ok ? kMaxRows : 8;
  {
    const char* env = getenv("LSK_PREFILL_TC");
    e->pf_tc = !(c.flags & LSK_FLAG_NO_PREFILL_TC) && !(env && atoi(env) == 0) && c.hidden % 64 == 0;
    e->pf_stages = kPfMaxStages;
    e->kst_h = c.hidden / 64;
    e->kst_q = (e->q_rows + 63) / 64;
    e->kst_i = (e->inter_l + 63) / 64;
    e->pf_t_qkv = (e->q_rows + 2 * e->kv_rows + 127) / 128;
    e->pf_t_h = (c.hidden + 127) / 128;
    e->pf_t_gu = (2 * e->inter_l + 127) / 128;
  }

  CU(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  CU(cudaEventCreate(&e->ev0));
  CU(cudaEventCreate(&e->ev1));

  auto alloc = [&](void** p, size_t bytes) -> int {
    cudaError_t er = cudaMalloc(p, bytes);
    if (er != cudaSuccess) return fail(LSK_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(er));
    cudaMemsetAsync(*p, 0, bytes, e->stream);
    return LSK_OK;
  };
  const size_t h = c.hidden;
  e->layers.resize(c.n_layers);
  for (auto& L : e->layers) {
    TRY(alloc((void**)&L.wqkv, (size_t)(e->q_rows + 2 * e->kv_rows) * h * 2));
    TRY(alloc((void**)&L.wo, h * e->q_rows * 2));
    TRY(alloc((void**)&L.wgu, (size_t)2 * e->inter_l * h * 2));
    TRY(alloc((void**)&L.wd, h * e->inter_l_pad * 2));
    TRY(alloc((void**)&L.ln1, h * 2));
    TRY(alloc((void**)&L.ln2, h * 2));
    if (e->pf_tc) {
      TRY(alloc((void**)&L.wqkv_c, (size_t)e->pf_t_qkv * e->kst_h * kCanonStageBytes));
      TRY(alloc((void**)&L.wo_c, (size_t)e->pf_t_h * e->kst_q * kCanonStageBytes));
      TRY(alloc((void**)&L.wgu_c, (size_t)e->pf_t_gu * e->kst_h * kCanonStageBytes));
      TRY(alloc((void**)&L.wd_c, (size_t)e->pf_t_h * e->kst_i * kCanonStageBytes));
    }
  }
  if (e->pf_tc) {
    TRY(alloc((void**)&e->hidden_p, (size_t)kPfTokens * h * 4));
    TRY(alloc((void**)&e->tp_buf_p, (size_t)kPfTokens * h * 4));
    TRY(alloc((void**)&e->part_p, (size_t)4 * kPfTokens * h * 4));
    TRY(alloc((void**)&e->q_p, (size_t)kPfTokens * e->q_rows * 2));
    TRY(alloc((void**)&e->xn_c, (size_t)e->kst_h * kCanonStageBytes));
    TRY(alloc((void**)&e->attn_c, (size_t)e->kst_q * kCanonStageBytes));
    TRY(alloc((void**)&e->act_c, (size_t)e->kst_i * kCanonStageBytes));
    CU(cudaFuncSetAttribute(prefill_gemm_tc_kernel<PF_EPI_QKV>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
    CU(cudaFuncSetAttribute(prefill_gemm_tc_kernel<PF_EPI_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
    CU(cudaFuncSetAttribute(prefill_gemm_tc_kernel<PF_EPI_SILU>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
  }
  TRY(alloc((void**)&e->embed, (size_t)c.vocab * h * 2));
  TRY(alloc((void**)&e->final_norm, h * 2));
  TRY(alloc((void**)&e->lm_head, (size_t)e->vocab_l_pad * h * 2));
  if (e->lm_tc) {
    TRY(alloc((void**)&e->lm_head_tc, (size_t)e->lm_tc_tiles * kTcTileRows * h * 2));
    CU(cudaFuncSetAttribute(lmhead_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
  }
  e->pool_layer_elems = (size_t)e->n_pages * e->kv_heads_l * kPageTokens * c.head_dim;
  TRY(alloc((void**)&e->kpool, e->pool_layer_elems * c.n_layers * 2));
  TRY(alloc((void**)&e->vpool, e->pool_layer_elems * c.n_layers * 2));
  TRY(alloc((void**)&e->page_table, (size_t)e->n_pages * 4));
  TRY(alloc((void**)&e->rope, (size_t)e->max_pos * (c.head_dim / 2) * sizeof(float2)));
  TRY(alloc((void**)&e->hidden, (size_t)(kMaxRows + 1) * h * 4));
  TRY(alloc((void**)&e->qbuf, (size_t)kMaxRows * e->q_rows * 2));
  TRY(alloc((void**)&e->attn_out, (size_t)kMaxRows * e->q_rows * 2));
  TRY(alloc((void**)&e->act, (size_t)kMaxRows * e->inter_l_pad * 2));   // pad columns stay zero
  TRY(alloc((void**)&e->tp_buf, (size_t)kMaxRows * h * 4));
  if (e->keep_logits) TRY(alloc((void**)&e->logits, (size_t)kMaxRows * e->vocab_l_pad * 4));
  TRY(alloc((void**)&e->cand_val, (size_t)e->sm_count * kMaxRows * 4));
  TRY(alloc((void**)&e->cand_idx, (size_t)e->sm_count * kMaxRows * 4));
  TRY(alloc((void**)&e->gath_val, (size_t)c.tp_size * kMaxRows * 4));
  TRY(alloc((void**)&e->gath_idx, (size_t)c.tp_size * kMaxRows * 4));
  TRY(alloc((void**)&e->ban_val, kMaxRows * 4));
  TRY(alloc((void**)&e->ban_idx, kMaxRows * 4));
  TRY(alloc((void**)&e->rank_val, kMaxRows * 4));
  TRY(alloc((void**)&e->rank_idx, kMaxRows * 4));
  TRY(alloc((void**)&e->d_zero, 4));
  TRY(alloc((void**)&e->d_prompt, (size_t)e->max_pos * 4));
  TRY(alloc((void**)&e->d_dbg_ids, kMaxRows * 4));
  TRY(alloc((void**)&e->state, sizeof(DevState)));
  TRY(alloc((void**)&e->gen_dev, sizeof(GenParams)));
  CU(cudaHostAlloc((void**)&e->res_host, sizeof(RoundResult), cudaHostAllocMapped));
  memset(e->res_host, 0, sizeof(RoundResult));
  CU(cudaHostGetDevicePointer((void**)&e->res_dev, e->res_host, 0));

  {  // identity page table + RoPE table (fp32 maths as HF: inv_freq, angle and cos/sin in fp32)
    std::vector<int> pt(e->n_pages);
    for (int i = 0; i < e->n_pages; ++i) pt[i] = i;
    CU(cudaMemcpyAsync(e->page_table, pt.data(), pt.size() * 4, cudaMemcpyHostToDevice, e->stream));
    // inv_freq as transformers computes it (modeling_rope_utils.py): default theta^(-2i/d), then the
    // checkpoint's scaling rule; angle and cos/sin in fp32 like LlamaRotaryEmbedding.forward
    const int half = c.head_dim / 2;
    std::vector<float2> tab((size_t)e->max_pos * half);
    for (int d = 0; d < half; ++d) {
      float inv_freq = 1.0f / powf(c.rope_theta, (float)(2 * d) / (float)c.head_dim);
      if (c.rope_scaling == LSK_ROPE_LINEAR) {
        inv_freq /= c.rope_factor;
      } else if (c.rope_scaling == LSK_ROPE_LLAMA3) {
        const float old_len = (float)c.rope_original_max_pos;
        const float low_wavelen = old_len / c.rope_low_freq_factor, high_wavelen = old_len / c.rope_high_freq_factor;
        const float wavelen = 2.0f * (float)M_PI / inv_freq;
        float scaled = wavelen > low_wavelen ? inv_freq / c.rope_factor : inv_freq;
        if (!(wavelen < high_wavelen) && !(wavelen > low_wavelen)) {
          const float smooth = (old_len / wavelen - c.rope_low_freq_factor) /
                               (c.rope_high_freq_factor - c.rope_low_freq_factor);
          scaled = (1.0f - smooth) * scaled / c.rope_factor + smooth * scaled;
        }
        inv_freq = scaled;
      }
      for (int p = 0; p < e->max_pos; ++p) {
        const float ang = (float)p * inv_freq;
        tab[(size_t)p * half + d] = make_float2((float)cos((double)ang), (float)sin((double)ang));
      }
    }
    CU(cudaMemcpyAsync(e->rope, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice, e->stream));
    CU(cudaStreamSynchronize(e->stream));
  }
  return LSK_OK;
}

void lsk_destroy(lsk_engine* e) {
  if (!e) return;
  if (e->stream) cudaStreamSynchronize(e->stream);
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  for (void* p : e->peer_opened) if (p) cudaIpcCloseMemHandle(p);
  if (e->peer_region) cudaFree(e->peer_region);
  if (e->peer_err_host) cudaFreeHost(e->peer_err_host);
  if (e->comm) ncclCommDestroy(e->comm);
  for (auto& L : e->layers) {
    cudaFree(L.wqkv); cudaFree(L.wo); cudaFree(L.wgu); cudaFree(L.wd); cudaFree(L.ln1); cudaFree(L.ln2);
    cudaFree(L.wqkv_c); cudaFree(L.wo_c); cudaFree(L.wgu_c); cudaFree(L.wd_c);
  }
  {
    void* pf[] = {e->hidden_p, e->tp_buf_p, e->part_p, e->q_p, e->xn_c, e->attn_c, e->act_c};
    for (void* p : pf) if (p) cudaFree(p);
  }
  void* ptrs[] = {e->embed, e->final_norm, e->lm_head, e->lm_head_tc, e->kpool, e->vpool, e->page_table, e->rope,
                  e->hidden, e->qbuf, e->attn_out, e->act, e->tp_buf, e->logits, e->logits_gath, e->logits_full, e->probs_d, e->probs_v, e->samp_scratch, e->cand_val,
                  e->cand_idx, e->gath_val, e->gath_idx, e->ban_val, e->ban_idx, e->rank_val, e->rank_idx,
                  e->d_zero, e->d_prompt, e->d_dbg_ids, e->state, e->gen_dev};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (e->res_host) cudaFreeHost(e->res_host);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  if (e->stream) cudaStreamDestroy(e->stream);
  cudaGetLastError();   // a half-built engine may have left a sticky-free error behind
  delete e;
}

int lsk_comm_unique_id(uint8_t id_out[128]) {
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  ncclUniqueId id;
  NC(ncclGetUniqueId(&id));
  memcpy(id_out, &id, 128);
  return LSK_OK;
}

// Map every rank's peer region into this process (CUDA IPC; the handles travel over the engine's
// own NCCL communicator) and switch the TP collectives to the one-shot kernels of tp_peer.cuh.
static int peer_setup(lsk_engine* e) {
  const int tp = e->cfg.tp_size, rank = e->cfg.tp_rank;
  if (tp > kMaxPeers) return fail(LSK_ERR_INVALID, "one-shot collectives support at most %d ranks", kMaxPeers);
  const PeerRegionLayout L = peer_region_layout(tp, e->cfg.hidden);
  {
    cudaError_t er = cudaMalloc(&e->peer_region, L.total);
    if (er != cudaSuccess) return fail(LSK_ERR_NOMEM, "cudaMalloc(peer region, %zu) failed: %s", L.total, cudaGetErrorString(er));
  }
  CU(cudaMemset(e->peer_region, 0, L.total));
  CU(cudaDeviceSynchronize());
  cudaIpcMemHandle_t mine;
  CU(cudaIpcGetMemHandle(&mine, e->peer_region));
  const size_t hb = sizeof(cudaIpcMemHandle_t);
  unsigned char* d_h = nullptr;
  CU(cudaMalloc((void**)&d_h, hb * tp));
  CU(cudaMemcpy(d_h + hb * rank, &mine, hb, cudaMemcpyHostToDevice));
  NC(ncclAllGather(d_h + hb * rank, d_h, hb, ncclUint8, e->comm, e->stream));
  CU(cudaStreamSynchronize(e->stream));
  std::vector<cudaIpcMemHandle_t> all(tp);
  CU(cudaMemcpy(all.data(), d_h, hb * tp, cudaMemcpyDeviceToHost));
  cudaFree(d_h);
  int local_ok = 1;
  std::string why;
  for (int r = 0; r < tp; ++r) {
    if (r == rank) { e->peer.base[r] = (unsigned char*)e->peer_region; continue; }
    void* p = nullptr;
    cudaError_t er = cudaIpcOpenMemHandle(&p, all[r], cudaIpcMemLazyEnablePeerAccess);
    if (er != cudaSuccess) {
      local_ok = 0;
      why = cudaGetErrorString(er);
      cudaGetLastError();
      continue;
    }
    e->peer_opened[r] = p;
    e->peer.base[r] = (unsigned char*)p;
  }
  CU(cudaHostAlloc((void**)&e->peer_err_host, sizeof(int), cudaHostAllocMapped));
  *e->peer_err_host = 0;
  CU(cudaHostGetDevicePointer((void**)&e->peer.error, e->peer_err_host, 0));
  e->peer.rank = rank;
  e->peer.size = tp;
  e->peer.hidden = e->cfg.hidden;
  // every rank must take the same path: agree on min(local_ok).  The all-reduce also keeps the
  // ranks together until every mapping exists (nobody pushes into a region before its owner has
  // zeroed it: all did, they produced a handle).
  const float mine_ok = (float)local_ok;
  CU(cudaMemcpyAsync(e->tp_buf, &mine_ok, 4, cudaMemcpyHostToDevice, e->stream));
  NC(ncclAllReduce(e->tp_buf, e->tp_buf, 1, ncclFloat, ncclMin, e->comm, e->stream));
  float all_ok = 0.f;
  CU(cudaMemcpyAsync(&all_ok, e->tp_buf, 4, cudaMemcpyDeviceToHost, e->stream));
  CU(cudaStreamSynchronize(e->stream));
  CU(cudaMemsetAsync(e->tp_buf, 0, 4, e->stream));
  if (all_ok < 0.5f) {
    fprintf(stderr, "[lsk] rank %d: peer mapping unavailable (%s): tensor-parallel collectives fall back to NCCL\n",
            rank, local_ok ? "another rank failed" : why.c_str());
    return LSK_OK;
  }
  e->peer_ok = true;
  return LSK_OK;
}

static int peer_check(lsk_engine* e) {
  if (e->peer_err_host && *(volatile int*)e->peer_err_host)
    return fail(LSK_ERR_NCCL, "one-shot TP collective timed out waiting for another rank");
  return LSK_OK;
}

int lsk_comm_init(lsk_engine* e, const uint8_t id_in[128]) {
  if (!e) return fail(LSK_ERR_INVALID, "null engine");
  if (e->cfg.tp_size == 1) return LSK_OK;
  ncclUniqueId id;
  memcpy(&id, id_in, 128);
  NC(ncclCommInitRank(&e->comm, e->cfg.tp_size, id, e->cfg.tp_rank));
  if (e->want_peer) TRY(peer_setup(e));
  return LSK_OK;
}

static int pack(lsk_engine* e, const __nv_bfloat16* src, int64_t src_ld, int64_t row0, int64_t col0,
                int64_t n_rows, int64_t K, __nv_bfloat16* dst, int64_t dst_row0, int mode, int64_t K_dst = 0) {
  if (K_dst == 0) K_dst = K;
  const int64_t pairs = n_rows * (K / 2);
  int blocks = (int)((pairs + 255) / 256);
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (blocks < 1) blocks = 1;
  pack_rows_kernel<<<blocks, 256, 0, e->stream>>>(src, src_ld, row0, col0, n_rows, K, dst, dst_row0, mode, K_dst, e->cfg.head_dim);
  CU(cudaGetLastError());
  return LSK_OK;
}

static int pack_canon(lsk_engine* e, const __nv_bfloat16* src, int64_t src_ld, int64_t row0, int64_t col0,
                      int64_t n_rows, int64_t K, unsigned char* dst, int64_t dst_row0, int mode, int n_kst) {
  if (!e->pf_tc) return LSK_OK;
  const int64_t total = n_rows * (K / 8);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (blocks < 1) blocks = 1;
  pack_canonical_rows_kernel<<<blocks, 256, 0, e->stream>>>(src, src_ld, row0, col0, n_rows, K, dst, dst_row0, mode,
                                                            n_kst, e->cfg.head_dim);
  CU(cudaGetLastError());
  return LSK_OK;
}

int lsk_load_weights(lsk_engine* e, const lsk_weight_desc* descs, int32_t n) {
  if (!e || !descs) return fail(LSK_ERR_INVALID, "null argument");
  const lsk_config& c = e->cfg;
  const int r = c.tp_rank;
  for (int i = 0; i < n; ++i) {
    const lsk_weight_desc& d = descs[i];
    const __nv_bfloat16* src = static_cast<const __nv_bfloat16*>(d.data);
    auto expect = [&](int64_t rows, int64_t cols) -> int {
      if (d.rows != rows || d.cols != cols)
        return fail(LSK_ERR_INVALID, "weight role %d layer %d: shape [%lld,%lld], expected [%lld,%lld]",
                    d.role, d.layer, (long long)d.rows, (long long)d.cols, (long long)rows, (long long)cols);
      return LSK_OK;
    };
    const bool per_layer = d.role >= LSK_W_LN1;
    if (per_layer && (d.layer < 0 || d.layer >= c.n_layers)) return fail(LSK_ERR_INVALID, "bad layer %d", d.layer);
    LayerWeights* L = per_layer ? &e->layers[d.layer] : nullptr;
    const int64_t h = c.hidden, qd = (int64_t)c.n_heads * c.head_dim, kvd = (int64_t)c.n_kv_heads * c.head_dim;
    switch (d.role) {
      case LSK_W_EMBED:
        TRY(expect(c.vocab, h));
        CU(cudaMemcpyAsync(e->embed, src, (size_t)c.vocab * h * 2, cudaMemcpyDeviceToDevice, e->stream));
        e->globals_loaded |= 1u;
        break;
      case LSK_W_FINAL_NORM:
        TRY(expect(h, 1));
        CU(cudaMemcpyAsync(e->final_norm, src, h * 2, cudaMemcpyDeviceToDevice, e->stream));
        e->globals_loaded |= 2u;
        break;
      case LSK_W_LM_HEAD:
        TRY(expect(c.vocab, h));
        TRY(pack(e, src, h, (int64_t)r * e->vocab_l, 0, e->vocab_l, h, e->lm_head, 0, MAP_PLAIN));
        if (e->lm_tc) {
          pack_canonical_kernel<<<148 * 8, 256, 0, e->stream>>>(src, h, (int64_t)r * e->vocab_l, e->vocab_l, h,
                                                              reinterpret_cast<uint4*>(e->lm_head_tc), e->lm_tc_tiles);
          CU(cudaGetLastError());
        }
        e->globals_loaded |= 4u;
        break;
      case LSK_W_LN1:
        TRY(expect(h, 1));
        CU(cudaMemcpyAsync(L->ln1, src, h * 2, cudaMemcpyDeviceToDevice, e->stream));
        break;
      case LSK_W_LN2:
        TRY(expect(h, 1));
        CU(cudaMemcpyAsync(L->ln2, src, h * 2, cudaMemcpyDeviceToDevice, e->stream));
        break;
      case LSK_W_Q:
        TRY(expect(qd, h));
        TRY(pack(e, src, h, (int64_t)r * e->q_rows, 0, e->q_rows, h, L->wqkv, 0, MAP_ROPE_HEADS));
        TRY(pack_canon(e, src, h, (int64_t)r * e->q_rows, 0, e->q_rows, h, L->wqkv_c, 0, MAP_ROPE_HEADS, e->kst_h));
        break;
      case LSK_W_K:
        TRY(expect(kvd, h));
        TRY(pack(e, src, h, (int64_t)r * e->kv_rows, 0, e->kv_rows, h, L->wqkv, e->q_rows, MAP_ROPE_HEADS));
        TRY(pack_canon(e, src, h, (int64_t)r * e->kv_rows, 0, e->kv_rows, h, L->wqkv_c, e->q_rows, MAP_ROPE_HEADS, e->kst_h));
        break;
      case LSK_W_V:
        TRY(expect(kvd, h));
        TRY(pack(e, src, h, (int64_t)r * e->kv_rows, 0, e->kv_rows, h, L->wqkv, e->q_rows + e->kv_rows, MAP_PLAIN));
        TRY(pack_canon(e, src, h, (int64_t)r * e->kv_rows, 0, e->kv_rows, h, L->wqkv_c, e->q_rows + e->kv_rows, MAP_PLAIN, e->kst_h));
        break;
      case LSK_W_O:   // row-parallel: this rank's input features = its heads
        TRY(expect(h, qd));
        TRY(pack(e, src, qd, 0, (int64_t)r * e->q_rows, h, e->q_rows, L->wo, 0, MAP_PLAIN));
        TRY(pack_canon(e, src, qd, 0, (int64_t)r * e->q_rows, h, e->q_rows, L->wo_c, 0, MAP_PLAIN, e->kst_q));
        break;
      case LSK_W_GATE:
        TRY(expect(c.inter, h));
        TRY(pack(e, src, h, (int64_t)r * e->inter_l, 0, e->inter_l, h, L->wgu, 0, MAP_GATE));
        TRY(pack_canon(e, src, h, (int64_t)r * e->inter_l, 0, e->inter_l, h, L->wgu_c, 0, MAP_GATE, e->kst_h));
        break;
      case LSK_W_UP:
        TRY(expect(c.inter, h));
        TRY(pack(e, src, h, (int64_t)r * e->inter_l, 0, e->inter_l, h, L->wgu, 0, MAP_UP));
        TRY(pack_canon(e, src, h, (int64_t)r * e->inter_l, 0, e->inter_l, h, L->wgu_c, 0, MAP_UP, e->kst_h));
        break;
      case LSK_W_DOWN:
        TRY(expect(h, c.inter));
        TRY(pack(e, src, c.inter, 0, (int64_t)r * e->inter_l, h, e->inter_l, L->wd, 0, MAP_PLAIN, e->inter_l_pad));
        TRY(pack_canon(e, src, c.inter, 0, (int64_t)r * e->inter_l, h, e->inter_l, L->wd_c, 0, MAP_PLAIN, e->kst_i));
        break;
      default:
        return fail(LSK_ERR_INVALID, "unknown weight role %d", d.role);
    }
    if (L) L->loaded |= 1u << d.role;
  }
  CU(cudaStreamSynchronize(e->stream));
  return LSK_OK;
}

int lsk_weights_complete(const lsk_engine* e) {
  if (!e) return 0;
  if (e->globals_loaded != 7u) return 0;
  const unsigned need = (1u << LSK_W_LN1) | (1u << LSK_W_Q) | (1u << LSK_W_K) | (1u << LSK_W_V) |
                        (1u << LSK_W_O) | (1u << LSK_W_LN2) | (1u << LSK_W_GATE) | (1u << LSK_W_UP) |
                        (1u << LSK_W_DOWN);
  for (const auto& L : e->layers)
    if ((L.loaded & need) != need) return 0;
  return 1;
}

int lsk_begin(lsk_engine* e, const lsk_generation* gen) {
  if (!e || !gen) return fail(LSK_ERR_INVALID, "null argument");
  if (!lsk_weights_complete(e)) return fail(LSK_ERR_STATE, "weights not fully loaded");
  if (gen->n_eos < 0 || gen->n_eos > LSK_MAX_EOS) return fail(LSK_ERR_INVALID, "n_eos out of range");
  if (gen->exit_layer > e->cfg.n_layers) return fail(LSK_ERR_INVALID, "exit_layer > n_layers");
  if (gen->no_repeat_ngram_size < 0 || gen->no_repeat_ngram_size > 16)
    return fail(LSK_ERR_INVALID, "no_repeat_ngram_size must be in [0, 16]");
  if (gen->no_repeat_ngram_size > 0 && !e->logits) {
    cudaError_t er = cudaMalloc((void**)&e->logits, (size_t)kMaxRows * e->vocab_l_pad * 4);
    if (er != cudaSuccess) return fail(LSK_ERR_NOMEM, "cudaMalloc failed: %s", cudaGetErrorString(er));
  }
  if (gen->sample) {
    if (!(gen->temperature > 0.f)) return fail(LSK_ERR_INVALID, "temperature must be > 0");
    auto alloc0 = [&](float** p, size_t n) -> int {
      if (*p) return LSK_OK;
      cudaError_t er = cudaMalloc((void**)p, n * 4);
      if (er != cudaSuccess) return fail(LSK_ERR_NOMEM, "cudaMalloc failed: %s", cudaGetErrorString(er));
      return LSK_OK;
    };
    TRY(alloc0(&e->logits, (size_t)kMaxRows * e->vocab_l_pad));
    TRY(alloc0(&e->probs_d, (size_t)kMaxRows * e->cfg.vocab));
    TRY(alloc0(&e->probs_v, (size_t)kMaxRows * e->cfg.vocab));
    TRY(alloc0(&e->samp_scratch, (size_t)e->cfg.vocab));
    if (e->cfg.tp_size > 1) {
      TRY(alloc0(&e->logits_gath, (size_t)e->cfg.tp_size * kMaxRows * e->vocab_l_pad));
      TRY(alloc0(&e->logits_full, (size_t)kMaxRows * e->cfg.vocab));
    }
  }
  e->gen = *gen;
  GenParams gp{};
  gp.n_eos = gen->n_eos;
  for (int i = 0; i < gen->n_eos; ++i) gp.eos[i] = gen->eos_ids[i];
  gp.sample = gen->sample; gp.temperature = gen->temperature; gp.top_k = gen->top_k; gp.top_p = gen->top_p;
  gp.seed = gen->seed;
  CU(cudaMemcpyAsync(e->gen_dev, &gp, sizeof(gp), cudaMemcpyHostToDevice, e->stream));
  CU(cudaMemsetAsync(e->state, 0, sizeof(DevState), e->stream));
  CU(cudaStreamSynchronize(e->stream));
  e->began = true;
  e->prefilled = false;
  e->host_len = 0;
  return LSK_OK;
}

int lsk_prefill(lsk_engine* e, const int32_t* ids, int32_t n) {
  if (!e || !ids) return fail(LSK_ERR_INVALID, "null argument");
  if (!e->began) return fail(LSK_ERR_STATE, "lsk_begin must precede lsk_prefill");
  if (n < 1) return fail(LSK_ERR_INVALID, "empty prompt");
  if (n + 1 > e->cfg.max_ctx) return fail(LSK_ERR_CTX, "prompt of %d tokens exceeds max_ctx %d", n, e->cfg.max_ctx);
  for (int i = 0; i < n; ++i)
    if (ids[i] < 0 || ids[i] >= e->cfg.vocab) return fail(LSK_ERR_INVALID, "token id %d out of range", ids[i]);
  const lsk_config& c = e->cfg;
  CU(cudaEventRecord(e->ev0, e->stream));
  CU(cudaMemcpyAsync(e->d_prompt, ids, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  // ids[0 .. n-2] through every layer; no LM head: the reference discards those logits too
  // (self_speculation_generator.py:177).  Prompts longer than one decode block go through the
  // tcgen05 GEMMs 128 tokens per weight pass (prefill_tc.cuh), short ones through the decode
  // kernels in blocks of <= 16 rows.
  if (e->pf_tc && n - 1 > e->max_rows) {
    for (int c0 = 0; c0 < n - 1; c0 += kPfTokens) {
      const int m = (n - 1 - c0) < kPfTokens ? (n - 1 - c0) : kPfTokens;
      TRY(enqueue_prefill_chunk(e, c0, m));
    }
  } else {
    for (int c0 = 0; c0 < n - 1; c0 += e->max_rows) {
      const int m = (n - 1 - c0) < e->max_rows ? (n - 1 - c0) : e->max_rows;
      CU(launch(e, embed_tokens_kernel, dim3(m), dim3(256), 0, (const __nv_bfloat16*)e->embed, c.hidden,
                (const int*)(e->d_prompt + c0), e->hidden, c.hidden));
      for (int l = 0; l < c.n_layers; ++l)
        TRY(enqueue_layer(e, l, 0, m, e->d_zero, c0, e->layers[(l + 1) % c.n_layers].wqkv,
                          (size_t)(e->q_rows + 2 * e->kv_rows) * c.hidden * 2));
    }
  }
  set_state_kernel<<<1, 1, 0, e->stream>>>(e->state, n - 1, ids[n - 1], 0, n);
  CU(cudaGetLastError());
  CU(cudaEventRecord(e->ev1, e->stream));
  CU(cudaEventSynchronize(e->ev1));
  CU(cudaEventElapsedTime(&e->last_ms, e->ev0, e->ev1));
  TRY(peer_check(e));
  e->host_len = n - 1;
  e->prefilled = true;
  return LSK_OK;
}

static void copy_result(const lsk_engine* e, lsk_round_out* out) {
  const RoundResult& r = *e->res_host;
  out->n_drafted = r.n_drafted;
  out->n_matches = r.n_matches;
  out->n_emitted = r.n_emitted;
  out->kv_len = r.kv_len;
  for (int i = 0; i < kMaxRows; ++i) {
    out->draft_ids[i] = r.draft_ids[i];
    out->emitted_ids[i] = r.emitted_ids[i];
    out->verified_ids[i] = r.verified_ids[i];
  }
}

int lsk_round(lsk_engine* e, int32_t d_req, lsk_round_out* out) {
  if (!e || !out) return fail(LSK_ERR_INVALID, "null argument");
  if (!e->prefilled) return fail(LSK_ERR_STATE, "lsk_prefill must precede lsk_round");
  if (d_req < 0 || d_req + 1 > e->max_rows) return fail(LSK_ERR_INVALID, "d_req %d out of [0,%d]", d_req, e->max_rows - 1);
  const int E = e->gen.exit_layer;
  if (E < 1 || E > e->cfg.n_layers) return fail(LSK_ERR_INVALID, "self-speculation needs 1 <= exit_layer <= n_layers (got %d)", E);
  if (e->host_len + d_req + 2 > e->max_pos) return fail(LSK_ERR_CTX, "context %d + %d exceeds max_ctx", e->host_len, d_req + 1);
  const int seq = ++e->seq;
  const long long key = ((long long)E << 20) | ((long long)d_req << 8) | (e->gen.sample ? 4 : 0) | 1 |
                        ((long long)e->gen.no_repeat_ngram_size << 32);
  TRY(run_cached(e, key, [&]() { return enqueue_round(e, E, d_req, 0); }));
  (void)seq;
  TRY(peer_check(e));
  copy_result(e, out);
  e->host_len = out->kv_len;
  return LSK_OK;
}

int lsk_ar_step(lsk_engine* e, int32_t* token_out) {
  if (!e || !token_out) return fail(LSK_ERR_INVALID, "null argument");
  if (!e->prefilled) return fail(LSK_ERR_STATE, "lsk_prefill must precede lsk_ar_step");
  if (e->host_len + 2 > e->max_pos) return fail(LSK_ERR_CTX, "context exceeds max_ctx");
  const int nl = (e->gen.exit_layer > 0 && e->gen.exit_layer <= e->cfg.n_layers) ? e->gen.exit_layer : e->cfg.n_layers;
  const long long key = ((long long)nl << 20) | (e->gen.sample ? 4 : 0) | 2 | ((long long)e->gen.no_repeat_ngram_size << 32);
  TRY(run_cached(e, key, [&]() { return enqueue_ar(e, nl, 0); }));
  TRY(peer_check(e));
  *token_out = e->res_host->emitted_ids[0];
  e->host_len = e->res_host->kv_len;
  return LSK_OK;
}

int lsk_profile_round(lsk_engine* e, int32_t d_req, lsk_round_out* out, float* class_ms,
                      int64_t* class_launches, float* total_ms) {
  if (!e || !out || !class_ms || !class_launches) return fail(LSK_ERR_INVALID, "null argument");
  if (!e->prefilled) return fail(LSK_ERR_STATE, "lsk_prefill must precede lsk_profile_round");
  if (d_req < 0 || d_req > LSK_MAX_SPEC) return fail(LSK_ERR_INVALID, "d_req out of range");
  const int E = e->gen.exit_layer;
  if (E < 1 || E > e->cfg.n_layers) return fail(LSK_ERR_INVALID, "bad exit_layer");
  if (e->host_len + d_req + 2 > e->max_pos) return fail(LSK_ERR_CTX, "context exceeds max_ctx");
  e->profiling = true;
  e->prof_events.clear();
  CU(cudaEventRecord(e->ev0, e->stream));
  int st = enqueue_round(e, E, d_req, 0);
  e->profiling = false;
  if (st != LSK_OK) return st;
  CU(cudaEventRecord(e->ev1, e->stream));
  CU(cudaEventSynchronize(e->ev1));
  CU(cudaEventElapsedTime(&e->last_ms, e->ev0, e->ev1));
  if (total_ms) *total_ms = e->last_ms;
  for (int i = 0; i < CLS_COUNT; ++i) { class_ms[i] = 0.f; class_launches[i] = 0; }
  for (auto& pe : e->prof_events) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, pe.second.first, pe.second.second);
    class_ms[pe.first] += ms;
    class_launches[pe.first] += 1;
    cudaEventDestroy(pe.second.first);
    cudaEventDestroy(pe.second.second);
  }
  e->prof_events.clear();
  copy_result(e, out);
  e->host_len = out->kv_len;
  return LSK_OK;
}

// Teacher-forced block (parity tests): the m given token ids as rows 0..m-1 at positions
// len .. len+m-1 through ALL layers and the LM head (logits kept: needs LSK_FLAG_KEEP_LOGITS).
// Nothing is committed: the rows' K/V entries land beyond the committed length and are
// overwritten by the next real step.  This is forward() of llama_model_utils.py:155-209 on a
// block of m tokens on top of the committed context.
int lsk_debug_forward_rows(lsk_engine* e, const int32_t* ids, int32_t m) {
  if (!e || !ids) return fail(LSK_ERR_INVALID, "null argument");
  if (!e->prefilled) return fail(LSK_ERR_STATE, "lsk_prefill must precede lsk_debug_forward_rows");
  if (!e->keep_logits) return fail(LSK_ERR_STATE, "engine created without LSK_FLAG_KEEP_LOGITS");
  if (m < 1 || m > e->max_rows) return fail(LSK_ERR_INVALID, "m %d out of [1,%d]", m, e->max_rows);
  if (e->host_len + m + 1 > e->max_pos) return fail(LSK_ERR_CTX, "context exceeds max_ctx");
  const lsk_config& c = e->cfg;
  for (int i = 0; i < m; ++i)
    if (ids[i] < 0 || ids[i] >= c.vocab) return fail(LSK_ERR_INVALID, "token id %d out of range", ids[i]);
  // staged in a buffer of their own: d_prompt is the token history the n-gram ban reads
  CU(cudaMemcpyAsync(e->d_dbg_ids, ids, (size_t)m * 4, cudaMemcpyHostToDevice, e->stream));
  e->cur_class = CLS_MISC;
  CU(launch(e, embed_tokens_kernel, dim3(m), dim3(256), 0, (const __nv_bfloat16*)e->embed, c.hidden,
            (const int*)e->d_dbg_ids, e->hidden, c.hidden));
  for (int l = 0; l < c.n_layers; ++l) TRY(enqueue_layer(e, l, 0, m, &e->state->len, 0));
  const int keep_sample = e->gen.sample;
  e->gen.sample = 0;
  const int keep_ban = e->gen.no_repeat_ngram_size;
  e->gen.no_repeat_ngram_size = 0;
  const int st = enqueue_lm_head(e, 0, m, 0);
  e->gen.no_repeat_ngram_size = keep_ban;
  e->gen.sample = keep_sample;
  if (st != LSK_OK) return st;
  CU(cudaStreamSynchronize(e->stream));
  TRY(peer_check(e));
  return LSK_OK;
}

int lsk_kv_len(const lsk_engine* e, int32_t* len_out) {
  if (!e || !len_out) return fail(LSK_ERR_INVALID, "null argument");
  *len_out = e->host_len;
  return LSK_OK;
}

int lsk_debug_set_page_table(lsk_engine* e, const int32_t* pages, int32_t n) {
  if (!e || !pages || n != e->n_pages) return fail(LSK_ERR_INVALID, "page table must have %d entries", e ? e->n_pages : 0);
  std::vector<char> seen(n, 0);
  for (int i = 0; i < n; ++i) {
    if (pages[i] < 0 || pages[i] >= n || seen[pages[i]]) return fail(LSK_ERR_INVALID, "page table is not a permutation");
    seen[pages[i]] = 1;
  }
  CU(cudaMemcpyAsync(e->page_table, pages, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  CU(cudaStreamSynchronize(e->stream));
  return LSK_OK;
}

int lsk_debug_read(lsk_engine* e, int32_t what, int32_t layer, int64_t index, float* dst, int64_t n) {
  if (!e || !dst) return fail(LSK_ERR_INVALID, "null argument");
  CU(cudaStreamSynchronize(e->stream));
  if (what == LSK_DBG_HIDDEN) {
    if (n > (int64_t)kMaxRows * e->cfg.hidden) return fail(LSK_ERR_INVALID, "too many floats");
    CU(cudaMemcpy(dst, e->hidden, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return LSK_OK;
  }
  if (what == LSK_DBG_PROBS_DRAFT || what == LSK_DBG_PROBS_VERIFY) {
    const float* src = what == LSK_DBG_PROBS_DRAFT ? e->probs_d : e->probs_v;
    if (!src) return fail(LSK_ERR_STATE, "no sampling generation has run");
    if (n > (int64_t)kMaxRows * e->cfg.vocab) return fail(LSK_ERR_INVALID, "too many floats");
    CU(cudaMemcpy(dst, src, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return LSK_OK;
  }
  if (what == LSK_DBG_RESIDUAL) {
    if (!e->samp_scratch) return fail(LSK_ERR_STATE, "no sampling generation has run");
    if (n > (int64_t)e->cfg.vocab) return fail(LSK_ERR_INVALID, "too many floats");
    CU(cudaMemcpy(dst, e->samp_scratch, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return LSK_OK;
  }
  if (what == LSK_DBG_LOGITS) {
    if (!e->logits) return fail(LSK_ERR_STATE, "engine created without LSK_FLAG_KEEP_LOGITS");
    if (n > (int64_t)kMaxRows * e->vocab_l_pad) return fail(LSK_ERR_INVALID, "too many floats");
    CU(cudaMemcpy(dst, e->logits, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return LSK_OK;
  }
  if (what == LSK_DBG_KROW || what == LSK_DBG_VROW) {
    const int hd = e->cfg.head_dim;
    if (layer < 0 || layer >= e->cfg.n_layers || n != hd) return fail(LSK_ERR_INVALID, "bad layer / n (one row = head_dim floats)");
    const int64_t head = index / e->cfg.max_ctx, pos = index % e->cfg.max_ctx;
    if (head >= e->kv_heads_l) return fail(LSK_ERR_INVALID, "bad kv head");
    std::vector<int> pt(e->n_pages);
    CU(cudaMemcpy(pt.data(), e->page_table, pt.size() * 4, cudaMemcpyDeviceToHost));
    const __nv_bfloat16* pool = (what == LSK_DBG_KROW ? e->kpool : e->vpool) + (size_t)layer * e->pool_layer_elems;
    // one token row is contiguous; its 16-byte chunks are swizzled (common.cuh: kv_elem_offset)
    const __nv_bfloat16* src = pool + kv_elem_offset(hd, pt[pos >> 6], e->kv_heads_l, (int)head, (int)(pos & 63), 0) -
                               (size_t)(kv_chunk_swizzle(hd, (int)(pos & 63)) * 8);
    std::vector<__nv_bfloat16> tmp(hd);
    CU(cudaMemcpy(tmp.data(), src, (size_t)hd * 2, cudaMemcpyDeviceToHost));
    for (int i = 0; i < hd; ++i)
      dst[i] = __bfloat162float(tmp[(((i >> 3) ^ kv_chunk_swizzle(hd, (int)(pos & 63))) << 3) + (i & 7)]);
    return LSK_OK;
  }
  return fail(LSK_ERR_INVALID, "unknown debug selector %d", what);
}

// algorithmic bytes (SURVEY.md §8(d)), per GPU: packed weights streamed once per layer call,
// LM head once per head call, KV entries of the visible context once per layer call.
static double layer_weight_bytes(const lsk_engine* e) {
  const double h = e->cfg.hidden;
  return 2.0 * ((double)(e->q_rows + 2 * e->kv_rows) * h + h * e->q_rows + 3.0 * e->inter_l * h);
}
int lsk_round_bytes(const lsk_engine* e, int32_t d, int32_t ctx, double* out) {
  if (!e || !out) return fail(LSK_ERR_INVALID, "null argument");
  const int E = e->gen.exit_layer, L = e->cfg.n_layers;
  const double wl = layer_weight_bytes(e), wh = 2.0 * e->vocab_l * e->cfg.hidden;
  const double kv_tok = 2.0 * 2.0 * e->kv_rows;
  const double layer_calls = (double)(d + 1) * E + (L - E);
  *out = layer_calls * wl + (d + 1) * wh + layer_calls * ctx * kv_tok;
  return LSK_OK;
}
int lsk_ar_bytes(const lsk_engine* e, int32_t ctx, double* out) {
  if (!e || !out) return fail(LSK_ERR_INVALID, "null argument");
  const int nl = (e->gen.exit_layer > 0) ? e->gen.exit_layer : e->cfg.n_layers;
  *out = nl * (layer_weight_bytes(e) + ctx * 2.0 * 2.0 * e->kv_rows) + 2.0 * e->vocab_l * e->cfg.hidden;
  return LSK_OK;
}
int lsk_launch_count(const lsk_engine* e, int64_t* out) {
  if (!e || !out) return fail(LSK_ERR_INVALID, "null argument");
  *out = e->launches;
  return LSK_OK;
}
int lsk_last_device_ms(const lsk_engine* e, float* out) {
  if (!e || !out) return fail(LSK_ERR_INVALID, "null argument");
  *out = e->last_ms;
  return LSK_OK;
}

// Host-side schedule of one skinny GEMM (no GPU needed): what the launcher would do for
// y[m, n_rows] = x[m, K] . W^T with the given prologue / epilogue kinds on `sm_count` SMs.
int lsk_plan_gemm(int64_t n_rows, int64_t K, int32_t m, int32_t pro, int32_t epi, int32_t sm_count,
                  lsk_gemm_plan* out) {
  if (!out || n_rows % 16 || K % 32 || m < 1 || m > kMaxRows || sm_count < 1)
    return fail(LSK_ERR_INVALID, "bad plan query");
  const GemmPlan p = make_plan((int)n_rows, (int)K, sm_count);
  const int NT = m <= 8 ? 1 : 2;
  const GemmSched sc = plan_sched(NT, m, pro, epi, p, sm_count);
  out->ok = sc.ok ? 1 : 0;
  out->nt = NT;
  out->tiles_per_pass = sc.tpp;
  out->n_chunks = sc.n_chunks;
  out->chunk_cols = sc.kc_sbs * 32;
  out->ring_stages = sc.n_stages;
  out->stage_bytes = kStageBytes;
  out->grid = sc.grid;
  out->block = kGemmThreads;
  out->smem_bytes = (int64_t)sc.smem;
  out->smem_limit = kSmemMax;
  out->n_tiles = p.n_tiles;
  return LSK_OK;
}

// Host-side launch plan of the attention kernel for `m` query rows (no GPU needed).
int lsk_plan_attention(int32_t head_dim, int32_t n_heads, int32_t n_kv_heads_local, int32_t m, int32_t sm_count,
                       lsk_attn_plan* out) {
  if (!out || (head_dim != 32 && head_dim != 64 && head_dim != 128) || n_heads < 1 || n_kv_heads_local < 1 ||
      n_heads % n_kv_heads_local || m < 1 || sm_count < 1)
    return fail(LSK_ERR_INVALID, "bad attention plan query");
  const int group = n_heads / n_kv_heads_local;
  const int splits = attn_default_splits(sm_count, n_kv_heads_local);
  const AttnLaunchPlan p = plan_attention_launch(head_dim, group, m, n_kv_heads_local, splits, kAttnMaxStages, sm_count);
  out->ok = p.ok ? 1 : 0;
  out->n_splits = splits;
  out->ring_stages = p.stages;
  out->grid = n_kv_heads_local * splits;
  out->block = kAttnThreads;
  out->row_blocks = (group * m + 15) / 16;
  out->kv_refetched_per_row_block = p.sp.reload_per_rb;
  out->smem_bytes = (int64_t)p.smem;
  out->smem_limit = kSmemMax;
  return LSK_OK;
}

// ---- stand-alone kernel entry points (unit tests / micro-benchmarks) ---------------------
int lsk_test_pack(const void* w, int64_t n, int64_t k, void* packed) {
  if (!w || !packed || n % 16 || k % 32) return fail(LSK_ERR_INVALID, "need n %% 16 == 0 and k %% 32 == 0");
  const int64_t pairs = n * (k / 2);
  int blocks = (int)((pairs + 255) / 256);
  if (blocks > 148 * 32) blocks = 148 * 32;
  pack_rows_kernel<<<blocks, 256>>>((const __nv_bfloat16*)w, k, 0, 0, n, k, (__nv_bfloat16*)packed, 0, MAP_PLAIN, k, 128);
  CU(cudaGetLastError());
  CU(cudaDeviceSynchronize());
  return LSK_OK;
}

int lsk_test_gemm(const void* packed, int64_t n, int64_t k, const void* x, int32_t m, float* y,
                  int32_t iters, float* avg_ms) {
  if (!packed || !x || !y || n % 16 || k % 32 || m < 1 || m > kMaxRows) return fail(LSK_ERR_INVALID, "bad gemm test shape");
  lsk_engine tmp;   // only the launch plumbing is used
  int dev = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&tmp.sm_count, cudaDevAttrMultiProcessorCount, dev));
  CU(cudaStreamCreateWithFlags(&tmp.stream, cudaStreamNonBlocking));
  tmp.use_pdl = true;
  GemmPlan p = make_plan((int)n, (int)k, tmp.sm_count);
  GemmArgs a{};
  a.W = (const uint4*)packed;
  a.M = m;
  a.x_bf16 = (const __nv_bfloat16*)x; a.xb_ld = (int)k;
  a.out_f32 = y; a.out_ld = (int)n;
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  int st = launch_gemm<PRO_BF16, EPI_STORE>(&tmp, p, a);   // warm-up + result
  if (st != LSK_OK) return st;
  CU(cudaStreamSynchronize(tmp.stream));
  if (iters > 0) {
    CU(cudaEventRecord(e0, tmp.stream));
    for (int i = 0; i < iters; ++i) {
      st = launch_gemm<PRO_BF16, EPI_STORE>(&tmp, p, a);
      if (st != LSK_OK) return st;
    }
    CU(cudaEventRecord(e1, tmp.stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (avg_ms) *avg_ms = ms / iters;
  }
  CU(cudaEventDestroy(e0));
  CU(cudaEventDestroy(e1));
  CU(cudaStreamDestroy(tmp.stream));
  tmp.stream = nullptr;
  return LSK_OK;
}

// natural K/V [kv_head][ctx][hd] -> the engine's paged pool layout (one layer)
__global__ void paginate_kv_kernel(const __nv_bfloat16* __restrict__ src, int n_kv, int ctx, int kHeadDim,
                                   const int* __restrict__ page_table, __nv_bfloat16* __restrict__ pool) {
  const int64_t total = (int64_t)n_kv * ctx * (kHeadDim / 8);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ch = (int)(i % (kHeadDim / 8));
    const int pos = (int)((i / (kHeadDim / 8)) % ctx);
    const int h = (int)(i / ((int64_t)(kHeadDim / 8) * ctx));
    const uint4 v = *reinterpret_cast<const uint4*>(src + ((size_t)h * ctx + pos) * kHeadDim + ch * 8);
    const int page = page_table[pos >> 6];
    *reinterpret_cast<uint4*>(pool + kv_elem_offset(kHeadDim, page, n_kv, h, pos & 63, ch * 8)) = v;
  }
}

// Stand-alone attention (unit test / micro-benchmark): m query rows at positions ctx-m .. ctx-1
// attend causally to keys 0 .. ctx-1.  q / out: [m][n_heads * 128] bf16; k / v: natural
// [n_kv_heads][ctx][128] bf16 (k already rotated); page_perm (host, may be null) permutes the
// logical -> physical page map.  Same launch path as the engine (cluster kernel).
int lsk_test_attn(const void* q, const void* k, const void* v, int32_t n_heads, int32_t n_kv_heads,
                  int32_t head_dim, int32_t ctx, int32_t m, int32_t n_splits, const int32_t* page_perm, void* out,
                  int32_t iters, float* avg_ms) {
  const int kHeadDim = head_dim;
  if (head_dim != 32 && head_dim != 64 && head_dim != 128) return fail(LSK_ERR_INVALID, "head_dim %d unsupported", head_dim);
  if (!q || !k || !v || !out || n_heads < 1 || n_kv_heads < 1 || n_heads % n_kv_heads || ctx < m || m < 1 ||
      m > kMaxRows || n_splits < 1 || n_splits > 8)
    return fail(LSK_ERR_INVALID, "bad attention test shape");
  lsk_engine tmp;
  {
    int dev = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&tmp.sm_count, cudaDevAttrMultiProcessorCount, dev));
  }
  CU(cudaStreamCreateWithFlags(&tmp.stream, cudaStreamNonBlocking));
  tmp.use_pdl = true;
  const int n_pages = (ctx + kPageTokens - 1) / kPageTokens;
  const size_t pool_elems = (size_t)n_pages * n_kv_heads * kPageTokens * kHeadDim;
  __nv_bfloat16 *kp = nullptr, *vp = nullptr;
  int *pt = nullptr, *len = nullptr;
  CU(cudaMalloc((void**)&kp, pool_elems * 2));
  CU(cudaMalloc((void**)&vp, pool_elems * 2));
  CU(cudaMalloc((void**)&pt, (size_t)n_pages * 4));
  CU(cudaMalloc((void**)&len, 4));
  CU(cudaMemsetAsync(kp, 0, pool_elems * 2, tmp.stream));
  CU(cudaMemsetAsync(vp, 0, pool_elems * 2, tmp.stream));
  std::vector<int> pth(n_pages);
  for (int i = 0; i < n_pages; ++i) pth[i] = page_perm ? page_perm[i] : i;
  for (int i = 0; i < n_pages; ++i)
    if (pth[i] < 0 || pth[i] >= n_pages) return fail(LSK_ERR_INVALID, "bad page permutation");
  const int base = ctx - m;
  CU(cudaMemcpyAsync(pt, pth.data(), (size_t)n_pages * 4, cudaMemcpyHostToDevice, tmp.stream));
  CU(cudaMemcpyAsync(len, &base, 4, cudaMemcpyHostToDevice, tmp.stream));
  paginate_kv_kernel<<<148 * 4, 256, 0, tmp.stream>>>((const __nv_bfloat16*)k, n_kv_heads, ctx, head_dim, pt, kp);
  paginate_kv_kernel<<<148 * 4, 256, 0, tmp.stream>>>((const __nv_bfloat16*)v, n_kv_heads, ctx, head_dim, pt, vp);
  CU(cudaGetLastError());
  AttnArgs a{};
  a.q = (const __nv_bfloat16*)q; a.q_ld = n_heads * kHeadDim;
  a.out = (__nv_bfloat16*)out; a.out_ld = n_heads * kHeadDim;
  a.kpool = kp; a.vpool = vp; a.page_table = pt; a.base_len = len; a.pos_off = 0; a.M = m;
  a.group = n_heads / n_kv_heads; a.n_kv_heads = n_kv_heads; a.n_splits = n_splits;
  a.scale = 1.0f / sqrtf((float)kHeadDim);
  int st = launch_attention(&tmp, a, head_dim);
  if (st != LSK_OK) return st;
  CU(cudaStreamSynchronize(tmp.stream));
  if (iters > 0) {
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, tmp.stream));
    for (int i = 0; i < iters; ++i) {
      st = launch_attention(&tmp, a, head_dim);
      if (st != LSK_OK) return st;
    }
    CU(cudaEventRecord(e1, tmp.stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (avg_ms) *avg_ms = ms / iters;
    CU(cudaEventDestroy(e0));
    CU(cudaEventDestroy(e1));
  }
  cudaFree(kp); cudaFree(vp); cudaFree(pt); cudaFree(len);
  CU(cudaStreamDestroy(tmp.stream));
  tmp.stream = nullptr;
  return LSK_OK;
}

// tcgen05 LM head on caller-provided device buffers (unit test / micro-benchmark of lmhead_tc.cuh)
int lsk_test_lmhead_tc(const void* w, int64_t n, int64_t k, const float* x, const void* norm_w, float eps,
                       int32_t m, float* logits, float* best_val, int32_t* best_idx, int32_t iters,
                       float* avg_ms) {
  if (!w || !x || !norm_w || !best_val || !best_idx || n < 1 || k % kTcStageK || m < 1 || m > kMaxRows)
    return fail(LSK_ERR_INVALID, "bad tcgen05 LM-head test shape");
  int stages = kTcMaxStages;
  while (stages >= 3 && lmhead_tc_smem_bytes((int)k, stages) > (size_t)kSmemMax) --stages;
  if (stages < 3) return fail(LSK_ERR_INVALID, "hidden %lld does not fit the tcgen05 LM head", (long long)k);
  int dev = 0, sms = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int n_tiles = (int)((n + kTcTileRows - 1) / kTcTileRows);
  const int waves = (n_tiles + sms - 1) / sms;
  const int grid = (n_tiles + waves - 1) / waves;
  unsigned char* canon = nullptr;
  float* cval = nullptr;
  int* cidx = nullptr;
  CU(cudaMalloc((void**)&canon, (size_t)n_tiles * kTcTileRows * k * 2));
  CU(cudaMalloc((void**)&cval, (size_t)grid * kMaxRows * 4));
  CU(cudaMalloc((void**)&cidx, (size_t)grid * kMaxRows * 4));
  pack_canonical_kernel<<<148 * 8, 256>>>((const __nv_bfloat16*)w, k, 0, n, k, reinterpret_cast<uint4*>(canon), n_tiles);
  CU(cudaGetLastError());
  CU(cudaFuncSetAttribute(lmhead_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
  LmHeadTcArgs t{};
  t.W = canon; t.n_tiles = n_tiles; t.K = (int)k; t.M = m; t.n_stages = stages;
  t.x_f32 = x; t.x_ld = (int)k; t.norm_w = (const __nv_bfloat16*)norm_w; t.eps = eps;
  t.logits = logits; t.logits_ld = (int)n; t.n_valid_rows = (int)n; t.vocab_off = 0;
  t.part_val = cval; t.part_idx = cidx;
  const size_t smem = lmhead_tc_smem_bytes((int)k, stages);
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  lmhead_tc_kernel<<<grid, kTcThreads, smem>>>(t);
  CU(cudaGetLastError());
  rank_best_kernel<<<1, 256>>>(cval, cidx, grid, m, best_val, best_idx);
  CU(cudaGetLastError());
  CU(cudaDeviceSynchronize());
  if (iters > 0) {
    CU(cudaEventRecord(e0));
    for (int i = 0; i < iters; ++i) lmhead_tc_kernel<<<grid, kTcThreads, smem>>>(t);
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (avg_ms) *avg_ms = ms / iters;
  }
  CU(cudaEventDestroy(e0));
  CU(cudaEventDestroy(e1));
  cudaFree(canon); cudaFree(cval); cudaFree(cidx);
  return LSK_OK;
}

}  // extern "C"
