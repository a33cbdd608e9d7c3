// Library-level entry points and the index-generation driver (C ABI).
//
// lcrec_indexer_* restates the main body of the reference script index/generate_indices.py:85-128
// on the device: PASS 0 = encoder + fused argmin residual quantisation for all items (chunked so
// that 10 M x 4096 fp32 inputs can be streamed), then up to `max_rounds` collision rounds, each =
// sort/unique on packed codes -> per-group Sinkhorn on the last level -> overwrite the last code.
// The reference re-runs the encoder on every group every round; the latents are the same numbers
// (up to GEMM batch-shape rounding, SURVEY.md F5), so PASS 0 keeps the residual entering the last
// level (128 B/item) and the rounds never touch the 16 KB/item embeddings again.
#include <stdarg.h>
#include <string.h>

#include <utility>
#include <vector>

#include <nvtx3/nvToolsExt.h>     // header-only in CUDA 12: ranges cost a few ns unless a tool (nsys / ncu --nvtx) is attached

#include "common.cuh"

namespace lcrec {

// NVTX range per stage (SURVEY section 5, tracing row): every ProfScope of the library is also an NVTX range named after its tag
static const char* stage_name(int tag) {
  static const char* mlp[] = {"lcrec/mlp_layer1", "lcrec/mlp_layer2", "lcrec/mlp_layer3", "lcrec/mlp_layer4", "lcrec/mlp_layer5",
                              "lcrec/mlp_layer6", "lcrec/mlp_layer7", "lcrec/mlp_layer8+"};
  if (tag == 0) return "lcrec/input_operand_split";
  if (tag >= 1 && tag <= 16) return mlp[tag - 1 < 7 ? tag - 1 : 7];
  switch (tag) {
    case 17: return "lcrec/tail_operand_splits";
    case 20: return "lcrec/rq_quantize";
    case 21: return "lcrec/collision_check";
    case 22: return "lcrec/sinkhorn_groups_round1";
    case 23: return "lcrec/sinkhorn_groups_later_rounds";
    case 24: return "lcrec/sinkhorn_warp_classes";
    case 26: return "lcrec/sinkhorn_literal_rerun";
    default: return "lcrec/stage";
  }
}

static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int num_sms() {
  static int sms = -1;
  if (sms < 0) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0)
      sms = v;
    else
      return 148;
  }
  return sms;
}

// ---- per-stage profiling
static bool g_prof_on = false;
static bool g_prof_suspended = false;      // stream capture in progress: timing events must not become graph nodes
struct ProfPair { cudaEvent_t a, b; int tag; };
static std::vector<ProfPair> g_prof_pairs;
static std::vector<cudaEvent_t> g_prof_pool;
static cudaEvent_t g_prof_open[kProfTags];

static cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
void prof_begin(int tag, cudaStream_t st) {
  nvtxRangePushA(stage_name(tag));
  if (!g_prof_on || g_prof_suspended || tag < 0 || tag >= kProfTags) return;
  cudaEvent_t e = prof_event();
  cudaEventRecord(e, st);
  g_prof_open[tag] = e;
}
void prof_end(int tag, cudaStream_t st) {
  nvtxRangePop();
  if (!g_prof_on || g_prof_suspended || tag < 0 || tag >= kProfTags || !g_prof_open[tag]) return;
  cudaEvent_t e = prof_event();
  cudaEventRecord(e, st);
  g_prof_pairs.push_back({g_prof_open[tag], e, tag});
  g_prof_open[tag] = nullptr;
}

}  // namespace lcrec

using namespace lcrec;

extern "C" int lcrec_profile_enable(int on) {
  g_prof_on = on != 0;
  return LCREC_OK;
}
// Synchronises, then adds the elapsed ms of every recorded pair to ms[tag] and the pair count to
// calls[tag] (both arrays of 32 entries, host memory); clears the record.
extern "C" int lcrec_profile_collect(double* ms, int64_t* calls) {
  LC_ARG(ms && calls);
  LC_CUDA(cudaDeviceSynchronize());
  for (auto& p : g_prof_pairs) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, p.a, p.b) == cudaSuccess) { ms[p.tag] += t; calls[p.tag] += 1; }
    g_prof_pool.push_back(p.a); g_prof_pool.push_back(p.b);
  }
  g_prof_pairs.clear();
  (void)cudaGetLastError();
  return LCREC_OK;
}

extern "C" int lcrec_version(void) { return 100; }

extern "C" const char* lcrec_strerror(int code) {
  switch (code) {
    case LCREC_OK: return "ok";
    case LCREC_ERR_ARG: return "invalid argument";
    case LCREC_ERR_CUDA: return "CUDA error";
    case LCREC_ERR_UNSUPPORTED: return "unsupported shape or device";
    case LCREC_ERR_NOMEM: return "workspace too small or out of memory";
    case LCREC_ERR_NUMERIC: return "numeric guard failed";
    default: return "unknown error";
  }
}

extern "C" const char* lcrec_last_error(void) { return g_err; }

extern "C" int64_t lcrec_launch_count(void) { return g_launches.load(); }

extern "C" int lcrec_device_check(void) {
  static int cached = -1;
  if (cached == LCREC_OK) return LCREC_OK;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { set_error("no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e)); cudaGetLastError(); return LCREC_ERR_CUDA; }
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) { set_error("cudaDeviceGetAttribute: %s", cudaGetErrorString(e)); cudaGetLastError(); return LCREC_ERR_CUDA; }
  if (major != 10) { set_error("device compute capability %d.x is not sm_100 (B200); kernels are built for sm_100a only", major); return LCREC_ERR_UNSUPPORTED; }
  cached = LCREC_OK;
  return LCREC_OK;
}

// ====================================================================== indexer
struct lcrec_indexer {
  lcrec_mlp_t* enc = nullptr;
  int in_dim = 0, D = 0, L = 0;
  std::vector<const float*> cb;
  std::vector<int32_t> K;
  double eps = 0.003; int iters = 50;
  int64_t max_items = 0, chunk_rows = 0;
  int64_t* codes = nullptr; float* resid = nullptr; float* z = nullptr;
  void* mlp_ws = nullptr; int64_t mlp_ws_bytes = 0;
  int64_t* offsets = nullptr; int64_t* members = nullptr; int64_t* counts = nullptr; int32_t* flags = nullptr;
  void* col_ws = nullptr; int64_t col_ws_bytes = 0;
  void* sk_ws = nullptr; int64_t sk_ws_bytes = 0;
  int64_t* seg_offsets = nullptr; int64_t* seg_members = nullptr; int64_t* seg_counts = nullptr;   // prefix segments
  void* seg_ws = nullptr; int64_t seg_ws_bytes = 0;
  int32_t* seg_active[2] = {nullptr, nullptr}; int32_t* seg_active_count = nullptr;   // ping-pong lists + 2 counters
  float* stage[2] = {nullptr, nullptr};
  int64_t* counts_host = nullptr;   // pinned: 4 counts + flags
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  // late collision rounds as CUDA-graph replays (one graph per parity of the active-segment ping-pong)
  cudaStream_t round_stream = nullptr; cudaEvent_t round_ev = nullptr;
  cudaGraphExec_t round_exec[2] = {nullptr, nullptr};
  int64_t round_launches[2] = {0, 0};
  const int64_t* rg_codes = nullptr; const float* rg_resid = nullptr; int64_t rg_n = -1; int rg_key = -1;
  bool rg_failed = false;
};

extern "C" int lcrec_mlp_in_dim(const lcrec_mlp_t* m);
extern "C" int lcrec_mlp_out_dim(const lcrec_mlp_t* m);

#define IX_ALLOC(ptr, bytes)                                                                     \
  do {                                                                                           \
    if (cudaMalloc((void**)&(ptr), (size_t)(bytes)) != cudaSuccess) {                            \
      set_error("indexer: cudaMalloc(%lld) failed: %s", (long long)(bytes), cudaGetErrorString(cudaGetLastError())); \
      lcrec_indexer_destroy(ix);                                                                 \
      return LCREC_ERR_NOMEM;                                                                    \
    }                                                                                            \
  } while (0)

extern "C" int lcrec_indexer_create(lcrec_mlp_t* encoder, int e_dim, int n_levels, const float* const* codebooks,
                                    const int32_t* n_codes, double last_epsilon, int sk_iters, int64_t max_items,
                                    int64_t chunk_rows, lcrec_indexer_t** out) {
  LC_ARG(encoder && e_dim > 0 && n_levels >= 1 && n_levels <= LCREC_MAX_LEVELS && codebooks && n_codes && out);
  LC_ARG(max_items > 0 && chunk_rows > 0 && last_epsilon > 0.0 && sk_iters >= 0);
  LC_ARG(lcrec_mlp_out_dim(encoder) == e_dim);
  LC_TRY(lcrec_device_check());
  lcrec_indexer* ix = new lcrec_indexer();
  ix->enc = encoder; ix->in_dim = lcrec_mlp_in_dim(encoder); ix->D = e_dim; ix->L = n_levels;
  ix->cb.assign(codebooks, codebooks + n_levels); ix->K.assign(n_codes, n_codes + n_levels);
  ix->eps = last_epsilon; ix->iters = sk_iters; ix->max_items = max_items;
  ix->chunk_rows = std::min(chunk_rows, max_items);
  IX_ALLOC(ix->codes, sizeof(int64_t) * max_items * n_levels);
  IX_ALLOC(ix->resid, sizeof(float) * max_items * e_dim);
  IX_ALLOC(ix->z, sizeof(float) * max_items * e_dim);      // latents of all rows of one pass0 call: ONE fused RQ launch
  ix->mlp_ws_bytes = lcrec_mlp_workspace_bytes(encoder, ix->chunk_rows);
  IX_ALLOC(ix->mlp_ws, ix->mlp_ws_bytes);
  IX_ALLOC(ix->offsets, sizeof(int64_t) * (max_items + 1));
  IX_ALLOC(ix->members, sizeof(int64_t) * max_items);
  IX_ALLOC(ix->counts, sizeof(int64_t) * 8);
  ix->flags = reinterpret_cast<int32_t*>(ix->counts + 4);
  ix->col_ws_bytes = lcrec_collisions_workspace_bytes(max_items);
  IX_ALLOC(ix->col_ws, ix->col_ws_bytes);
  ix->sk_ws_bytes = lcrec_sinkhorn_groups_workspace_bytes(max_items, n_codes[n_levels - 1]);
  IX_ALLOC(ix->sk_ws, ix->sk_ws_bytes);
  IX_ALLOC(ix->seg_offsets, sizeof(int64_t) * (max_items + 1));
  IX_ALLOC(ix->seg_members, sizeof(int64_t) * max_items);
  IX_ALLOC(ix->seg_counts, sizeof(int64_t) * 8);
  ix->seg_ws_bytes = lcrec_segment_collisions_workspace_bytes(max_items / 2 + 1);
  IX_ALLOC(ix->seg_ws, ix->seg_ws_bytes);
  IX_ALLOC(ix->seg_active[0], sizeof(int32_t) * (max_items / 2 + 2));
  IX_ALLOC(ix->seg_active[1], sizeof(int32_t) * (max_items / 2 + 2));
  IX_ALLOC(ix->seg_active_count, sizeof(int32_t) * 2);
  if (cudaMallocHost((void**)&ix->counts_host, sizeof(int64_t) * 8) != cudaSuccess) {
    set_error("indexer: cudaMallocHost failed"); lcrec_indexer_destroy(ix); return LCREC_ERR_NOMEM;
  }
  *out = ix;
  return LCREC_OK;
}

extern "C" int lcrec_indexer_destroy(lcrec_indexer_t* ix) {
  if (!ix) return LCREC_OK;
  cudaFree(ix->codes); cudaFree(ix->resid); cudaFree(ix->z); cudaFree(ix->mlp_ws); cudaFree(ix->offsets);
  cudaFree(ix->members); cudaFree(ix->counts); cudaFree(ix->col_ws); cudaFree(ix->sk_ws);
  cudaFree(ix->seg_offsets); cudaFree(ix->seg_members); cudaFree(ix->seg_counts); cudaFree(ix->seg_ws);
  cudaFree(ix->seg_active[0]); cudaFree(ix->seg_active[1]); cudaFree(ix->seg_active_count);
  cudaFree(ix->stage[0]); cudaFree(ix->stage[1]);
  if (ix->counts_host) cudaFreeHost(ix->counts_host);
  for (int i = 0; i < 2; ++i) { if (ix->ev_copied[i]) cudaEventDestroy(ix->ev_copied[i]); if (ix->ev_consumed[i]) cudaEventDestroy(ix->ev_consumed[i]); }
  if (ix->copy_stream) cudaStreamDestroy(ix->copy_stream);
  for (int i = 0; i < 2; ++i) if (ix->round_exec[i]) cudaGraphExecDestroy(ix->round_exec[i]);
  if (ix->round_ev) cudaEventDestroy(ix->round_ev);
  if (ix->round_stream) cudaStreamDestroy(ix->round_stream);
  delete ix;
  return LCREC_OK;
}

extern "C" int64_t* lcrec_indexer_codes(lcrec_indexer_t* ix) { return ix ? ix->codes : nullptr; }
extern "C" float* lcrec_indexer_resid(lcrec_indexer_t* ix) { return ix ? ix->resid : nullptr; }

namespace lcrec {
int rq_quantize_select(const float* z, int64_t n, int64_t n_select, int e_dim, int n_levels, const float* const* codebooks,
                       const int32_t* n_codes, int n_levels_run, int resid_level, int64_t* codes, float* xq, float* resid_last,
                       double* sq_err, void* stream);      // rq_fused.cu
}

// PASS 0 of n device rows into table rows [row_offset, row_offset + n), the RQ kernel path chosen as for n_select rows
static int pass0_rows(lcrec_indexer_t* ix, const void* x, int dtype, int64_t n, int64_t row_offset, int64_t n_select,
                      void* stream) {
  const int64_t row_bytes = dtype_bytes(dtype) * ix->in_dim;
  for (int64_t s = 0; s < n; s += ix->chunk_rows) {
    const int64_t m = std::min(ix->chunk_rows, n - s);
    LC_TRY(lcrec_mlp_forward_ex(ix->enc, static_cast<const char*>(x) + s * row_bytes, dtype, m, ix->z + s * ix->D, nullptr,
                                ix->mlp_ws, ix->mlp_ws_bytes, stream));
  }
  ProfScope prof(20, (cudaStream_t)stream);
  return rq_quantize_select(ix->z, n, n_select, ix->D, ix->L, ix->cb.data(), ix->K.data(), ix->L, ix->L - 1,
                            ix->codes + row_offset * ix->L, nullptr, ix->resid + row_offset * ix->D, nullptr, stream);
}

// PASS 0 for rows [row_offset, row_offset + n) (generate_indices.py:85-95); x of element type dtype
extern "C" int lcrec_indexer_pass0_ex(lcrec_indexer_t* ix, const void* x, int dtype, int64_t n, int64_t row_offset, void* stream) {
  LC_ARG(dtype_ok(dtype));
  LC_ARG(ix && n >= 0 && row_offset >= 0 && row_offset + n <= ix->max_items);
  if (n == 0) return LCREC_OK;
  LC_ARG(x != nullptr);
  return pass0_rows(ix, x, dtype, n, row_offset, n, stream);
}

// The pieces in which host input of n_total rows is streamed: chunks of chunk_rows rows, the last chunk cut into up to four
// pieces (>= 8192 rows each).  The copies are the bottleneck (55 GB/s of pinned H2D against ~14 M items/s of compute), so
// what is left after the LAST copy lands - that chunk's encoder pass - is pure tail: cutting it leaves only a quarter of it
// to encode when the link goes idle.  Every piece keeps >= 8192 rows, so it gets the same kernel choices as a full chunk
// (tensor-core RQ path from 4096 rows on).  A pure function of (n_total, chunk_rows): a block of a larger job is cut along
// the same pieces (lcrec_indexer_pass0_host_ex).
static void host_pieces(int64_t n_total, int64_t chunk_rows, std::vector<std::pair<int64_t, int64_t>>& pieces) {
  pieces.clear();
  for (int64_t s0 = 0; s0 < n_total; s0 += chunk_rows) {
    const int64_t m0 = std::min(chunk_rows, n_total - s0);
    if (s0 + m0 < n_total) { pieces.emplace_back(s0, m0); continue; }
    const int64_t k = std::max<int64_t>(1, std::min<int64_t>(4, m0 / 8192));
    const int64_t q = ceil_div(m0, k);
    for (int64_t t = 0; t < m0; t += q) pieces.emplace_back(s0 + t, std::min(q, m0 - t));
  }
}

// PASS 0 of global rows [row_begin, row_begin + n) of an n_total-row job from host memory into table rows [0, n):
// double-buffered H2D on the indexer's copy stream, compute on `stream` (the fp32-sized staging buffers also hold a piece of
// half rows).  The block is cut along the pieces of host_pieces(n_total, chunk_rows) and every part is quantised with the
// RQ path of its whole piece, so codes and residuals are bit-identical to those rows of the single-call PASS 0 over all
// n_total rows.  Returns once every row has been copied; the compute stays ordered on `stream`.
extern "C" int lcrec_indexer_pass0_host_ex(lcrec_indexer_t* ix, const void* x_host, int dtype, int64_t n_total, int64_t row_begin,
                                           int64_t n, void* stream) {
  LC_ARG(dtype_ok(dtype));
  LC_ARG(ix && n >= 0 && row_begin >= 0 && n_total >= 0 && row_begin <= n_total && n <= n_total - row_begin && n <= ix->max_items);
  if (n == 0) return LCREC_OK;
  LC_ARG(x_host != nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  if (!ix->copy_stream) {
    LC_CUDA(cudaStreamCreateWithFlags(&ix->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      LC_CUDA(cudaEventCreateWithFlags(&ix->ev_copied[i], cudaEventDisableTiming));
      LC_CUDA(cudaEventCreateWithFlags(&ix->ev_consumed[i], cudaEventDisableTiming));
      LC_CUDA(cudaMalloc((void**)&ix->stage[i], sizeof(float) * ix->chunk_rows * ix->in_dim));
    }
  }
  std::vector<std::pair<int64_t, int64_t>> pieces;
  host_pieces(n_total, ix->chunk_rows, pieces);
  const int64_t row_bytes = dtype_bytes(dtype) * ix->in_dim;
  const int64_t end = row_begin + n;
  int64_t c = 0;      // parts streamed so far
  for (const auto& pc : pieces) {
    const int64_t s = std::max(pc.first, row_begin), e = std::min(pc.first + pc.second, end);
    if (s >= e) continue;
    const int b = (int)(c & 1);
    // also for the first two parts: the previous call's last passes over stage[b] may still be queued on `stream` (this
    // entry returns once the copies land, not the compute); an event never recorded counts as complete
    LC_CUDA(cudaStreamWaitEvent(ix->copy_stream, ix->ev_consumed[b], 0));
    LC_CUDA(cudaMemcpyAsync(ix->stage[b], static_cast<const char*>(x_host) + (s - row_begin) * row_bytes, (e - s) * row_bytes,
                            cudaMemcpyHostToDevice, ix->copy_stream));
    LC_CUDA(cudaEventRecord(ix->ev_copied[b], ix->copy_stream));
    LC_CUDA(cudaStreamWaitEvent(st, ix->ev_copied[b], 0));
    LC_TRY(pass0_rows(ix, ix->stage[b], dtype, e - s, s - row_begin, pc.second, stream));
    LC_CUDA(cudaEventRecord(ix->ev_consumed[b], st));
    ++c;
  }
  LC_CUDA(cudaStreamSynchronize(ix->copy_stream));      // the caller's host rows may be released on return
  return LCREC_OK;
}

extern "C" int lcrec_indexer_pass0(lcrec_indexer_t* ix, const float* x, int64_t n, int64_t row_offset, void* stream) {
  return lcrec_indexer_pass0_ex(ix, x, kDtypeF32, n, row_offset, stream);
}

static int g_use_segments = 1;
// 1 (default): after the first round the collision check runs inside the prefix segments (no global re-sort);
// 0: every round re-sorts all items (the original path; used to cross-check).
extern "C" int lcrec_indexer_set_segments(int on) { g_use_segments = on ? 1 : 0; return LCREC_OK; }

// One collision check of codes (n x L) into ix->offsets / members / counts, counts copied to the pinned host block
// (8 int64: n_unique, n_groups, rows, max_mult, flag words, segment fallback).  Synchronises the stream.
// seg_round: -1 = global sort; k >= 0 = k-th check inside the prefix segments (0 examines all segments, later ones
// only those that collided in the previous check)
static int collide_and_fetch(lcrec_indexer_t* ix, const int64_t* codes, int64_t n, int seg_round, cudaStream_t st) {
  {
    ProfScope prof(21, st);
    if (seg_round >= 0) {
      const int in = (seg_round + 1) & 1, out = seg_round & 1;
      LC_CUDA(cudaMemsetAsync(ix->seg_active_count + out, 0, sizeof(int32_t), st));
      LC_TRY(lcrec_collisions_in_segments_active(codes, n, ix->L, ix->L - 1, ix->seg_offsets, ix->seg_members, ix->seg_counts + 1,
                                                 n / 2 + 1, seg_round > 0 ? ix->seg_active[in] : nullptr,
                                                 seg_round > 0 ? ix->seg_active_count + in : nullptr, ix->seg_active[out],
                                                 ix->seg_active_count + out, ix->offsets, ix->members, ix->counts, ix->seg_ws,
                                                 ix->seg_ws_bytes, st));
    } else
      LC_TRY(lcrec_collisions(codes, n, ix->L, ix->K.data(), ix->offsets, ix->members, ix->counts, ix->col_ws,
                              ix->col_ws_bytes, st));
  }
  LC_CUDA(cudaMemcpyAsync(ix->counts_host, ix->counts, sizeof(int64_t) * 8, cudaMemcpyDeviceToHost, st));
  LC_CUDA(cudaStreamSynchronize(st));
  return LCREC_OK;
}

// Later collision rounds without a host round trip per round (lcrec_indexer_set_speculative).  Once the first check inside the
// prefix segments has passed (no segment too large for the on-chip sort - the segments never change afterwards, only last-level
// codes do) a round can be enqueued BLIND: check -> account -> Sinkhorn with worst-case launch bounds; the kernels read the group
// count on the device and a round without collisions is a chain of empty launches.
//   0: one host read of the counts per round (the synchronous loop);
//   1: every remaining round enqueued blind on the caller's stream, one host read at the end.  Measured NOT faster on one B200
//      (profiles/r2_speculative_rounds.txt): ~20 launches per round, the host's launch rate becomes the bound;
//   2 (default): as soon as a round has at most kLateGroups groups the blind round is captured ONCE into a CUDA graph (two graphs:
//      the active-segment lists ping-pong) and the remaining rounds are graph replays in batches of kRoundBatch with one host
//      read per batch (stop when a check finds no group).  Late rounds are bound by launch gaps and the latency of one group, not
//      by work: a replay runs the ~16 nodes back to back.
// Results and stats are identical in all three modes (tests/test_gpu_loop_ledger.py).
static int g_speculative = 2;
extern "C" int lcrec_indexer_set_speculative(int on) { g_speculative = on < 0 ? 0 : (on > 2 ? 2 : on); return LCREC_OK; }
constexpr int64_t kLateGroups = 888;      // = kColLateGroups of sinkhorn.cu: from here on every group runs on the column kernels
constexpr int kRoundBatch = 6;
__global__ void round_account_kernel(int64_t* counts) {      // counts[6] += rounds that resolved, counts[7] += their rows
  if (counts[1] > 0) { counts[6] += 1; counts[7] += counts[2]; }
}

// One blind round on `st`: check number seg_round (>= 1) inside the segments, account, Sinkhorn.  hint: -1 = any group count,
// -2 = few groups expected (column kernels for every size class)
static int enqueue_blind_round(lcrec_indexer_t* ix, int64_t* codes, const float* resid, int64_t n, int seg_round, int64_t hint,
                               cudaStream_t st) {
  const int in = (seg_round + 1) & 1, out = seg_round & 1;
  LC_CUDA(cudaMemsetAsync(ix->seg_active_count + out, 0, sizeof(int32_t), st));
  LC_TRY(lcrec_collisions_in_segments_active(codes, n, ix->L, ix->L - 1, ix->seg_offsets, ix->seg_members, ix->seg_counts + 1,
                                             n / 2 + 1, ix->seg_active[in], ix->seg_active_count + in, ix->seg_active[out],
                                             ix->seg_active_count + out, ix->offsets, ix->members, ix->counts, ix->seg_ws,
                                             ix->seg_ws_bytes, st));
  round_account_kernel<<<1, 1, 0, st>>>(ix->counts);
  LC_LAUNCH_CHECK("round_account_kernel");
  return lcrec_sinkhorn_groups_ex(resid, ix->D, ix->cb[ix->L - 1], ix->K[ix->L - 1], ix->offsets, ix->members, ix->counts + 1,
                                  n / 2, n, hint, ix->eps, ix->iters, codes, ix->L, ix->L - 1, 1, 0, ix->flags, ix->sk_ws,
                                  ix->sk_ws_bytes, st);
}

namespace lcrec { int sinkhorn_config_key(); }      // sinkhorn.cu: the kernel-selection switches a captured round depends on

// The two round graphs for (codes, resid, n) and the current kernel-selection switches; captured on the indexer's own stream
// (the caller's may be the legacy default stream, which cannot be captured).  Nothing executes during capture.
static int ensure_round_graphs(lcrec_indexer_t* ix, int64_t* codes, const float* resid, int64_t n) {
  if (ix->rg_failed) return LCREC_ERR_CUDA;
  if (!ix->round_stream) {
    if (cudaStreamCreateWithFlags(&ix->round_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ix->round_ev, cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); ix->rg_failed = true; return LCREC_ERR_CUDA; }
  }
  const int key = sinkhorn_config_key();
  if (ix->round_exec[0] && ix->round_exec[1] && ix->rg_codes == codes && ix->rg_resid == resid && ix->rg_n == n && ix->rg_key == key) return LCREC_OK;
  for (int i = 0; i < 2; ++i) if (ix->round_exec[i]) { cudaGraphExecDestroy(ix->round_exec[i]); ix->round_exec[i] = nullptr; }
  for (int parity = 0; parity < 2; ++parity) {
    const int64_t l0 = g_launches.load();
    g_prof_suspended = true;
    cudaGraph_t graph = nullptr;
    int rc = LCREC_OK;
    if (cudaStreamBeginCapture(ix->round_stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) rc = LCREC_ERR_CUDA;
    if (rc == LCREC_OK) {
      rc = enqueue_blind_round(ix, codes, resid, n, 2 + parity, -2, ix->round_stream);
      if (cudaStreamEndCapture(ix->round_stream, &graph) != cudaSuccess || graph == nullptr) rc = rc == LCREC_OK ? LCREC_ERR_CUDA : rc;
    }
    g_prof_suspended = false;
    ix->round_launches[parity] = g_launches.load() - l0;
    g_launches.fetch_sub(ix->round_launches[parity]);      // capture launched nothing
    if (rc == LCREC_OK && cudaGraphInstantiate(&ix->round_exec[parity], graph, 0) != cudaSuccess) rc = LCREC_ERR_CUDA;
    if (graph) cudaGraphDestroy(graph);
    if (rc != LCREC_OK) {
      (void)cudaGetLastError();
      for (int i = 0; i < 2; ++i) if (ix->round_exec[i]) { cudaGraphExecDestroy(ix->round_exec[i]); ix->round_exec[i] = nullptr; }
      ix->rg_failed = true;      // this indexer stays on the synchronous loop
      return rc;
    }
  }
  ix->rg_codes = codes; ix->rg_resid = resid; ix->rg_n = n; ix->rg_key = key;
  return LCREC_OK;
}

static int check_flags(int32_t f) {
  if (f & 2) { set_error("indexer: workspace for oversized collision groups exhausted"); return LCREC_ERR_NOMEM; }
  if (f & 4) { set_error("indexer: amplitude > 0 failed (vq.py:59)"); return LCREC_ERR_NUMERIC; }
  return LCREC_OK;
}

// generate_indices.py:108-128 on codes (n x L, device, updated in place) with the residuals entering the last level.
static int rounds_impl(lcrec_indexer_t* ix, int64_t* codes, const float* resid, int64_t n, int max_rounds, int64_t* stats,
                       cudaStream_t st) {
  int64_t rounds = 0, g1 = 0, r1 = 0, tot_rows = 0;
  bool use_seg = g_use_segments && ix->L >= 2, have_seg = false;
  int seg_round = 0;
  LC_CUDA(cudaMemsetAsync(ix->counts, 0, sizeof(int64_t) * 8, st));     // incl. the flag words (accumulated by atomicOr)
  const int64_t* c = ix->counts_host;
  while (true) {
    const bool resolve = rounds < max_rounds;
    LC_TRY(collide_and_fetch(ix, codes, n, have_seg ? seg_round++ : -1, st));
    if (have_seg && c[5] != 0) {            // a segment too large for the on-chip sort: back to the global sort for good
      have_seg = use_seg = false;
      LC_CUDA(cudaMemsetAsync(ix->counts + 5, 0, sizeof(int64_t), st));
      LC_TRY(collide_and_fetch(ix, codes, n, -1, st));
    }
    LC_TRY(check_flags((int32_t)(c[4] & 0xffffffff)));
    const int64_t groups = c[1], rows = c[2];
    if (c[0] == n || !resolve || groups == 0) break;
    if (rounds == 0) { g1 = groups; r1 = rows; }
    if (use_seg && !have_seg) {
      ProfScope prof(21, st);
      LC_TRY(lcrec_prefix_segments(codes, n, ix->L, ix->K.data(), ix->seg_offsets, ix->seg_members, ix->seg_counts, ix->col_ws,
                                   ix->col_ws_bytes, st));
      have_seg = true;
    }
    {
      ProfScope prof(rounds == 0 ? 22 : 23, st);      // 22 = first round, 23 = later rounds
      LC_TRY(lcrec_sinkhorn_groups_ex(resid, ix->D, ix->cb[ix->L - 1], ix->K[ix->L - 1], ix->offsets, ix->members,
                                      ix->counts + 1, groups, rows, c[3], ix->eps, ix->iters, codes, ix->L, ix->L - 1, 1, 0,
                                      ix->flags, ix->sk_ws, ix->sk_ws_bytes, st));
    }
    tot_rows += rows;
    ++rounds;
    const bool blind_ok = have_seg && seg_round >= 1 && ix->K[ix->L - 1] <= 256 && rounds < max_rounds;
    if (g_speculative == 2 && blind_ok && groups <= kLateGroups && ensure_round_graphs(ix, codes, resid, n) == LCREC_OK) {
      // the rest of the loop as graph replays: the indexer's stream takes over from the caller's and hands back by a host wait
      LC_CUDA(cudaEventRecord(ix->round_ev, st));
      LC_CUDA(cudaStreamWaitEvent(ix->round_stream, ix->round_ev, 0));
      int64_t enq = rounds;
      while (enq < max_rounds) {
        const int64_t b = std::min<int64_t>(kRoundBatch, max_rounds - enq);
        {
          ProfScope prof(23, ix->round_stream);      // (covers the checks of these rounds as well)
          for (int64_t i = 0; i < b; ++i) {
            const int parity = seg_round & 1;
            LC_CUDA(cudaGraphLaunch(ix->round_exec[parity], ix->round_stream));
            count_launch((int)ix->round_launches[parity]);
            ++seg_round;
          }
        }
        enq += b;
        LC_CUDA(cudaMemcpyAsync(ix->counts_host, ix->counts, sizeof(int64_t) * 8, cudaMemcpyDeviceToHost, ix->round_stream));
        LC_CUDA(cudaStreamSynchronize(ix->round_stream));
        if (c[1] == 0) break;      // the last check found no group (and its Sinkhorn was a chain of empty launches)
      }
      if (c[1] != 0) LC_TRY(collide_and_fetch(ix, codes, n, seg_round++, st));      // max_rounds reached: the check after the last round
      LC_TRY(check_flags((int32_t)(c[4] & 0xffffffff)));
      rounds += c[6];
      tot_rows += c[7];
      break;
    }
    if (g_speculative == 1 && blind_ok) {
      for (int64_t r = rounds; r < max_rounds; ++r) {
        ProfScope prof(23, st);
        LC_TRY(enqueue_blind_round(ix, codes, resid, n, seg_round++, -1, st));
      }
      LC_TRY(collide_and_fetch(ix, codes, n, seg_round++, st));      // the check after the last round (statistics, flags)
      LC_TRY(check_flags((int32_t)(c[4] & 0xffffffff)));
      rounds += c[6];
      tot_rows += c[7];
      break;
    }
  }
  int32_t f[2];
  LC_CUDA(cudaMemcpyAsync(f, ix->flags, sizeof(f), cudaMemcpyDeviceToHost, st));
  LC_CUDA(cudaStreamSynchronize(st));
  LC_TRY(check_flags(f[0]));
  if (stats) {
    stats[0] = rounds; stats[1] = c[0]; stats[2] = g1; stats[3] = r1; stats[4] = tot_rows; stats[5] = c[3];
    stats[6] = f[0] & 1; stats[7] = 0;
  }
  return LCREC_OK;
}

static int indexer_rounds(lcrec_indexer_t* ix, int64_t n, int max_rounds, int64_t* stats, cudaStream_t st) {
  return rounds_impl(ix, ix->codes, ix->resid, n, max_rounds, stats, st);
}

// The collision rounds alone on caller-owned device arrays (codes n x L updated in place; resid n x e_dim = residual
// entering the last level).  stats_host as in lcrec_indexer_run_host.
extern "C" int lcrec_indexer_resolve(lcrec_indexer_t* ix, int64_t* codes, const float* resid, int64_t n, int max_rounds,
                                     int64_t* stats_host, void* stream) {
  LC_ARG(ix && n >= 0 && n <= ix->max_items && max_rounds >= 0);
  if (n == 0) { if (stats_host) memset(stats_host, 0, 8 * sizeof(int64_t)); return LCREC_OK; }
  LC_ARG(codes && resid);
  return rounds_impl(ix, codes, resid, n, max_rounds, stats_host, (cudaStream_t)stream);
}

// One round on the indexer's own table (teacher-forced parity tests): check + resolve; counts_host (4 int64).
extern "C" int lcrec_indexer_round(lcrec_indexer_t* ix, int64_t n, int64_t* counts_host, void* stream) {
  LC_ARG(ix && n >= 0 && n <= ix->max_items);
  cudaStream_t st = (cudaStream_t)stream;
  LC_CUDA(cudaMemsetAsync(ix->counts, 0, sizeof(int64_t) * 8, st));
  LC_TRY(collide_and_fetch(ix, ix->codes, n, -1, st));
  const int64_t groups = ix->counts_host[1], rows = ix->counts_host[2];
  if (groups > 0) {
    ProfScope prof(22, st);
    LC_TRY(lcrec_sinkhorn_groups(ix->resid, ix->D, ix->cb[ix->L - 1], ix->K[ix->L - 1], ix->offsets, ix->members,
                                 ix->counts + 1, groups, rows, ix->eps, ix->iters, ix->codes, ix->L, ix->L - 1,
                                 ix->flags, ix->sk_ws, ix->sk_ws_bytes, st));
  }
  if (counts_host) memcpy(counts_host, ix->counts_host, sizeof(int64_t) * 4);
  return LCREC_OK;
}

extern "C" int lcrec_indexer_run_device(lcrec_indexer_t* ix, const float* x, int64_t n, int max_rounds, int64_t* codes,
                                        int64_t* stats_host, void* stream) {
  return lcrec_indexer_run_device_ex(ix, x, kDtypeF32, n, max_rounds, codes, stats_host, stream);
}

extern "C" int lcrec_indexer_run_device_ex(lcrec_indexer_t* ix, const void* x, int dtype, int64_t n, int max_rounds, int64_t* codes,
                                           int64_t* stats_host, void* stream) {
  LC_ARG(dtype_ok(dtype));
  LC_ARG(ix && n >= 0 && n <= ix->max_items && max_rounds >= 0);
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) { if (stats_host) memset(stats_host, 0, 8 * sizeof(int64_t)); return LCREC_OK; }
  LC_TRY(lcrec_indexer_pass0_ex(ix, x, dtype, n, 0, stream));
  LC_TRY(indexer_rounds(ix, n, max_rounds, stats_host, st));
  if (codes && codes != ix->codes)
    LC_CUDA(cudaMemcpyAsync(codes, ix->codes, sizeof(int64_t) * n * ix->L, cudaMemcpyDeviceToDevice, st));
  return LCREC_OK;
}

extern "C" int lcrec_indexer_run_host(lcrec_indexer_t* ix, const float* x_host, int64_t n, int max_rounds,
                                      int64_t* codes_host, int64_t* stats_host, void* stream) {
  return lcrec_indexer_run_host_ex(ix, x_host, kDtypeF32, n, max_rounds, codes_host, stats_host, stream);
}

extern "C" int lcrec_indexer_run_host_ex(lcrec_indexer_t* ix, const void* x_host, int dtype, int64_t n, int max_rounds,
                                         int64_t* codes_host, int64_t* stats_host, void* stream) {
  LC_ARG(dtype_ok(dtype));
  LC_ARG(ix && n >= 0 && n <= ix->max_items && max_rounds >= 0);
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) { if (stats_host) memset(stats_host, 0, 8 * sizeof(int64_t)); return LCREC_OK; }
  LC_ARG(x_host && codes_host);
  LC_TRY(lcrec_indexer_pass0_host_ex(ix, x_host, dtype, n, 0, n, stream));
  LC_TRY(indexer_rounds(ix, n, max_rounds, stats_host, st));
  LC_CUDA(cudaMemcpyAsync(codes_host, ix->codes, sizeof(int64_t) * n * ix->L, cudaMemcpyDeviceToHost, st));
  LC_CUDA(cudaStreamSynchronize(st));
  return LCREC_OK;
}
