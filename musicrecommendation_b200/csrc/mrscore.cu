// mrscore.cu — the C-ABI of include/mrscore.h: handle, data residency in HBM, and the batch pipeline K1 -> K2 -> K3.
//
// HBM layout (DESIGN.md §2):
//   train CSR  (user -> songs)   tr_ptr i64[T+1], tr_col i32[nnz]        MusicRecommender.scala:55  trainUsersToSongsMap
//   train CSC  (song -> users)   csc_ptr i64[S+1], csc_idx i32[nnz]      MusicRecommender.scala:60  songsToUsersMap (train part)
//   qv u32[T], qd u32[S]         rint(2^24 / sqrt(deg)), rint(2^26 / sqrt(deg))   cosine denominators MR:147 / MR:237 in fixed point
//   rsa f64[U], rsd f64[S]       2^-24 / sqrt(deg), 2^-26 / sqrt(deg)              the other half of each denominator
//   A_tr  u8[T][pitchS], A_trT u8[S][pitchT]   dense 0/1 operands of the tensor-core count GEMM (tensor engine only)
//   user space, per batch of 128 test users: Ct u16[T][128], Sint_u / Sint_i i64[128][spitch], G i32[rows][ldg], select bits
//   item space: head rows G16 / Gq32 (once per train set), Sint_u / Sint_i i64[batch][spitch] with batch = as many test users as fit
//   (plan_item_batches), balanced work groups of the head pass, per-slice tail scatter -> mask -> top-k -> streamed copy of the result
#include "../../include/mrscore.h"
#include "mr_common.cuh"
#include "mr_kernels.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <numeric>
#include <string>
#include <queue>
#include <mutex>
#include <thread>
#include <vector>

using namespace mr;

namespace {

constexpr int kSplitLen = 4096;   // listeners per K2 work item
// largest degrees whose fixed-point cosine factor stays within 1e-5 relative: 0.5 * sqrt(deg) / 2^k <= 1e-5  <=>  deg <= (2e-5 * 2^k)^2
constexpr int kMaxDegUbm = 112589;      // (2e-5 * 2^24)^2 = 112 589.99
constexpr int kPreStreams = 4;          // streams of the in-place head-row build (start_head_rows): 113.8 / 82.9 / 75.8 / 73.4 ms with 1 / 2 / 3 / 4
constexpr int kPreExtraStreams = 3;     // at most 1 + 3 (MRSCORE_PRE_STREAMS)
constexpr int kMaxDegIbm = 1801439;     // (2e-5 * 2^26)^2 = 1 801 439.85
constexpr size_t kCallerReserve = 6ULL << 30;   // HBM the item-space batch plan leaves for the caller's context and small workspaces

struct TopkOut { int32_t* song; double* score; int32_t* len; };   // one top-k result: song [U][k], score [U][k], len [U]

}  // namespace

struct mr_handle {
  int device = 0; int num_sms = 148; unsigned flags = 0; int engine = MR_ENGINE_AUTO;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr; cudaEvent_t ev_slice = nullptr;   // mr_topk streams finished slices of the result to the host beside the compute
  // Batch pipeline of the item-space top-k (run_batches): the head pass of batch b + 1 is issued on `stream` while the tail scatter, mask
  // and select of batch b run on slice_stream (higher priority); the two batches use the two Sint panels (a pure model needs only one).
  // ev_head[p] / ev_done[p]: head pass / slices of the batch in panel p.
  cudaStream_t slice_stream = nullptr; cudaEvent_t ev_head[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
  cudaStream_t slice_stream2 = nullptr; cudaEvent_t ev_join = nullptr;   // single-batch calls alternate their slices between the two slice streams
  std::string err;
  long long launches = 0; size_t dev_bytes = 0;
  std::vector<void*> allocs;          // allocated once per handle (mr_load, the sqrt tables of similar songs / users, peer buffers), freed in mr_destroy
  // train
  int T = 0, S = 0; long long nnz_tr = 0; bool loaded = false;
  long long *d_tr_ptr = nullptr, *d_csc_ptr = nullptr; int *d_tr_col = nullptr, *d_csc_idx = nullptr;
  // Song window (MR_OPT_SONG_WINDOW_LO / _HI, the song partition of distributed.scala:459-461): only the songs [win_lo, win_hi) are scored.
  // Internally song ids are ROTATED by win_lo (id' = id - win_lo mod S), so that the scored columns are [0, n_cols) of every array and
  // kernel while histories still refer to all S songs; CSR rows stay ascending (their in-window entries become a prefix that ends at
  // d_tr_end[v] / d_te_end[u]); only the ranked ids handed back are shifted by win_lo again.  Without a window n_cols = S, *_end = *_ptr + 1.
  int win_lo = 0, win_hi = 0, n_cols = 0; bool windowed = false;
  const long long *d_tr_end = nullptr, *d_te_end = nullptr;
  // asynchronous head-row build (mr_prepare_async): the kernels run on pre_stream, ev_pre marks their end; head_pending until the
  // exception list has been read back and uploaded (finish_head_rows, by the first call that needs the rows)
  cudaStream_t pre_stream = nullptr; cudaEvent_t ev_pre = nullptr; bool head_pending = false; unsigned int* h_n_ex = nullptr;
  cudaStream_t pre_extra[kPreExtraStreams] = {}; cudaEvent_t ev_pre_extra[kPreExtraStreams] = {};   // extra streams of the in-place row build (chunks rotate over them)
  HeadExceptions pend_ex{};
  unsigned int* d_topk_stats = nullptr;   // [4] counters since mr_load: [0, 3) of the top-k select (BlendParams::stats), [3] audience columns through the radix select
  uint32_t *d_qv = nullptr, *d_qd = nullptr; double* d_rsd = nullptr; float* d_rsd_up = nullptr;
  std::vector<int32_t> deg_song, deg_song_train;
  struct SongInfo { int head; uint32_t v; };   // head row or -1; v = q_26(d_s) of a head song, train listeners of a tail song
  int2* d_song_info = nullptr;                 // the same records on the device (k7_testlists.cu)
  std::vector<SongInfo> song_info;             // per song, 8 bytes: the one random access per test entry in mr_set_test_users
  uint32_t max_qv = 0;                         // largest UBM weight q_24(|I_v|) of a train user (number of byte planes of the tensor precompute)
  unsigned long long max_qsum = 0;             // max over songs of song_qsum
  std::vector<unsigned long long> song_qsum;   // per song: sum of qv over its train listeners = upper bound of any Gq entry of its row
  bool ubm_int_ok = false;                     // every UBM numerator of the current shard is provably < 2^52 (top-k may rank the integers)
  int *d_item_song = nullptr, *d_item_len = nullptr; long long* d_item_begin = nullptr; uint8_t* d_item_split = nullptr; int n_items = 0;
  long long pitchS = 0, pitchT = 0, spitch = 0, ldg = 0; size_t dense_bytes = 0;
  uint8_t *d_Atr = nullptr, *d_AtrT = nullptr;
  // item-space engine: head songs and their precomputed rows
  int space_flag = MR_SPACE_AUTO; int space = MR_SPACE_USER; int n_head = 0; bool head_ready = false;
  int item_batch_cap = 0;              // MRSCORE_ITEM_BATCH: upper bound on test users per item-space batch (0 = as many as fit in HBM)
  int batch_rows = kUserBatch;         // test users per batch of the current shard = rows of the Sint panels
  int head_words_u = 4, head_words_i = 4, head_threads = 128, n_groups = 0;   // head_rowsum: 32-bit words per row load (UBM / IBM pass), groups per batch
  int4 *d_seg = nullptr, *d_grp_hdr = nullptr; int *d_ge_row = nullptr, *d_split_rows = nullptr; uint32_t* d_ge_q = nullptr; int seg_cap = 1, ent_cap = 1;
  std::vector<int> h_split_ptr;   // balanced work groups per batch
  std::vector<int> head_index;         // song -> head row or -1
  int* d_head_song = nullptr; long long* d_head_lst_ptr = nullptr;
  uint16_t* d_g16 = nullptr; uint32_t* d_gq32 = nullptr;   // packed head rows, slots SL_HEAD_G16 / SL_HEAD_GQ32 (kept across mr_invalidate_prepared)
  int n_head_staged = 0;               // rows [0, n_head_staged) are built in a 64-bit staging area and packed; the rest directly in place
  bool head_packed = false; int head_planes = 0;   // last head-row build: packed 64-bit accumulator; byte planes of the tensor engine (0 = scatter)
  long long opt_head_min_deg = 0;      // mr_set_option(MR_OPT_HEAD_MIN_DEG): 0 = default rule
  long long* d_ex_ptr = nullptr; int* d_ex_song = nullptr; uint32_t* d_ex_g = nullptr; unsigned long long* d_ex_gq = nullptr; long long n_ex = 0;
  long long *d_hu_ptr = nullptr; int *d_hu_row = nullptr, *d_hu_song = nullptr; uint32_t* d_hu_q = nullptr;
  int *d_tu_user = nullptr, *d_tu_song = nullptr; long long* d_tu_lptr = nullptr; std::vector<long long> h_tu_ptr, h_tu_lptr; long long n_head_entries = 0, n_tail_entries = 0;
  // test shard (freed / reallocated by mr_set_test_users)
  int U = 0; long long nnz_te = 0; bool have_test = false;
  // grow-only device buffers of the test shard, its results and the workspaces: steady-state mr_set_test_users / mr_topk calls do no cudaMalloc
  enum { SL_TE_PTR, SL_TE_COL, SL_TE_GROW, SL_RSA, SL_PAIR_BASE, SL_ROWS, SL_HU_PTR, SL_HU_ROW, SL_HU_SONG, SL_HU_Q, SL_TU_USER,
         SL_TU_SONG, SL_TU_LPTR, SL_TU_PTR, SL_EX_PTR, SL_EX_SONG, SL_EX_G, SL_EX_GQ, SL_L_FLAG, SL_L_HEADPOS, SL_L_DEG, SL_L_LSUM, SL_L_TMP, SL_COPY_DESC, SL_SEG, SL_GRP_HDR, SL_GE_ROW, SL_GE_Q, SL_SPLIT_ROWS, SL_SINT_U, SL_SINT_I, SL_SEL, SL_GRAM_IDS, SL_DENSE, SL_OUT_PACK, SL_TE_END, SL_PRE_G, SL_PRE_GQ, SL_PRE_EXC, SL_EVAL_MM, SL_EVAL_COLMAP, SL_EVAL_CNT, SL_LAB_PTR, SL_LAB_COL, SL_AGG_SPLIT, SL_MULTI_OUT, SL_SIM_IDS, SL_SIM_EV, SL_SIM_Q, SL_SIM_OUT, SL_SIM_LIDS, SL_SIM_LOUT, SL_SIM_SQU, SL_GRAM_G, SL_GRAM_A, SL_HEAD_G16, SL_HEAD_GQ32, SL_AUD_OUT, SL_AUD_Q, SL_FLT_BITS, SL_FLT_COLS, SL_FLT_EX_PTR, SL_FLT_EX_COL, SL_N };
  void* slot_p[SL_N] = {}; size_t slot_cap[SL_N] = {};
  long long *d_te_ptr = nullptr, *d_pair_base = nullptr; int *d_te_col = nullptr, *d_te_grow = nullptr; double* d_rsa = nullptr;
  std::vector<long long> h_te_ptr; std::vector<int> h_te_col;
  std::vector<long long> batch_row_off; int* d_rows = nullptr; int max_batch_rows = 0;
  long long pair_index_base = 0, n_pairs_total = 0;
  // workspaces
  uint8_t *d_Ate = nullptr, *d_Aj = nullptr; uint16_t* d_ct = nullptr; long long *d_sint_u = nullptr, *d_sint_i = nullptr;
  uint32_t* d_wi = nullptr;             // IBM user-space weighted counts u32[T][128] (sparse engine)
  unsigned int* d_carry_count = nullptr; uint2* d_carry_events = nullptr; unsigned int carry_cap = 1u << 20;   // MRSCORE_CARRY_CAP
  unsigned int* h_carry_seen = nullptr; int carry_seen_cap = 0;   // pinned, one event count per user batch of the current call
  long long carry_events = 0;           // carry events of the last scoring call (sparse user-space IBM; 0 for any other call)
  uint64_t* d_sel = nullptr; long long sel_pitch = 0; int32_t* d_g = nullptr;   // d_g / d_Aj: the Gram workspace, slots SL_GRAM_G / SL_GRAM_A
  double* d_dense = nullptr;
  // results
  TopkOut out{}; int out_k = 0; bool have_topk = false; size_t out_pack_bytes = 0;   // the single-model result, a TopkBlock in SL_OUT_PACK
  // results of the last mr_topk_multi_device: entry i is the i-th TopkBlock of the SL_MULTI_OUT slot
  int multi_n = 0, multi_k = 0;
  long long passes = 0;   // scoring passes since mr_load: batches whose score panels were built
  // streamed evaluation (mr_eval_range* / mr_eval_counts*).  gen counts the calls that may rewrite the score panels; after a range pass
  // over a single-batch item-space shard the panels still hold the masked numerators of the model set (eval_n entries of eval_models,
  // eval_params, eval_seeds), and a count pass of the same set at the same gen reuses them instead of scoring again.
  unsigned long long gen = 0, eval_gen = ~0ULL; int eval_n = 0; int eval_models[16] = {}; double eval_params[16] = {}; uint64_t eval_seeds[16] = {};
  unsigned long long* d_eval_mm = nullptr;   // [2] min / max bit patterns of the range pass
  EvalCounts ec{};                           // device state of the count pass
  // similar songs (mr_similar_songs): sqrt(deg_song_all) per song, built on the first call; rows answered by each path since mr_load
  double* d_sim_sqd = nullptr; long long sim_short_rows = 0, sim_long_rows = 0;
  // similar users (mr_similar_users): sqrt(deg_train) per train user, built on the first call; sqrt(deg_test) per test user of the shard
  // (slot SL_SIM_SQU), rebuilt on the first call after each mr_set_test_users; rows answered by each path since mr_load
  std::vector<int32_t> deg_train, deg_test;
  double *d_simu_sqt = nullptr, *d_simu_squ = nullptr; bool simu_squ_ok = false; long long simu_short_rows = 0, simu_long_rows = 0;
  long long explain_rows = 0;   // mr_explain: count rows built since mr_load
  long long audience_rows = 0;  // mr_song_audience: query rows answered since mr_load
  // filtered top-k (mr_set_topk_filter, DESIGN.md §4.11): the in-window part of the current shard's filter, dropped by mr_set_test_users.
  // flt_n_allow: allowed columns of the window (d_flt_cols, ascending; bitmap d_flt_bits), -1 = every column; flt_n_ex: in-window exclusion
  // entries (rows d_flt_ex_ptr [U + 1] over columns d_flt_ex_col).  Rows answered by each path since mr_load.
  bool flt_on = false; int flt_n_allow = -1; long long flt_n_ex = 0;
  uint32_t* d_flt_bits = nullptr; int* d_flt_cols = nullptr; long long* d_flt_ex_ptr = nullptr; int* d_flt_ex_col = nullptr;
  long long flt_full_rows = 0, flt_cand_rows = 0;
  // profiling
  cudaEvent_t ev[2] = {nullptr, nullptr}; double t_ms[MR_T_N] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
};

namespace {

int fail(mr_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  if (h) h->err = buf;
  return code;
}

#define MR_CUDA(h, expr)                                                                                       \
  do {                                                                                                         \
    cudaError_t e__ = (expr);                                                                                  \
    if (e__ != cudaSuccess)                                                                                    \
      return fail(h, e__ == cudaErrorMemoryAllocation ? MR_ERR_OOM : MR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                                                \
  } while (0)

#define MR_LAUNCH(h, expr)                                                                     \
  do {                                                                                         \
    int rc__ = (expr);                                                                         \
    (h)->launches++;                                                                           \
    if (rc__ != 0) {                                                                           \
      cudaError_t e__ = cudaGetLastError();                                                    \
      return fail(h, MR_ERR_CUDA, "%s failed: rc=%d (%s)", #expr, rc__, cudaGetErrorString(e__)); \
    }                                                                                          \
  } while (0)

template <class Tp>
int dev_alloc(mr_handle* h, Tp** out, size_t count, std::vector<void*>& owner) {
  void* p = nullptr;
  size_t bytes = std::max<size_t>(count, 1) * sizeof(Tp);
  MR_CUDA(h, cudaMalloc(&p, bytes));
  owner.push_back(p);
  h->dev_bytes += bytes;
  *out = static_cast<Tp*>(p);
  return MR_OK;
}

template <class Tp>
int slot_alloc(mr_handle* h, int slot, Tp** out, size_t count, bool exact = false) {
  const size_t bytes = std::max<size_t>(count, 1) * sizeof(Tp);
  if (h->slot_cap[slot] < bytes) {
    if (h->slot_p[slot]) { cudaFree(h->slot_p[slot]); h->dev_bytes -= h->slot_cap[slot]; h->slot_p[slot] = nullptr; h->slot_cap[slot] = 0; }
    const size_t cap = exact ? bytes : bytes + bytes / 4 + 256;
    void* p = nullptr;
    MR_CUDA(h, cudaMalloc(&p, cap));
    h->slot_p[slot] = p; h->slot_cap[slot] = cap; h->dev_bytes += cap;
  }
  *out = static_cast<Tp*>(h->slot_p[slot]);
  return MR_OK;
}

template <class Tp>
int slot_upload(mr_handle* h, int slot, Tp** out, const Tp* src, size_t count) {
  int rc = slot_alloc(h, slot, out, count);
  if (rc) return rc;
  if (count) MR_CUDA(h, cudaMemcpyAsync(*out, src, count * sizeof(Tp), cudaMemcpyHostToDevice, h->stream));
  return MR_OK;
}

template <class Tp>
int dev_upload(mr_handle* h, Tp** out, const Tp* src, size_t count, std::vector<void*>& owner) {
  int rc = dev_alloc(h, out, count, owner);
  if (rc) return rc;
  if (count) MR_CUDA(h, cudaMemcpyAsync(*out, src, count * sizeof(Tp), cudaMemcpyHostToDevice, h->stream));
  return MR_OK;
}

// The temporaries of one call, counted in dev_bytes while they live.  They are freed when the owner goes out of scope, on every return
// path, once the stream they are used on has drained.
struct Scratch {
  mr_handle* h; cudaStream_t st;
  std::vector<void*> bufs; size_t bytes = 0;
  Scratch(mr_handle* hh, cudaStream_t s) : h(hh), st(s) {}
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
  ~Scratch() {
    if (bufs.empty()) return;
    cudaStreamSynchronize(st);
    for (void* p : bufs) cudaFree(p);
    h->dev_bytes -= bytes;
  }
  template <class Tp>
  int alloc(Tp** out, size_t count) {
    const int rc = dev_alloc(h, out, count, bufs);
    if (!rc) bytes += std::max<size_t>(count, 1) * sizeof(Tp);
    return rc;
  }
  template <class Tp>
  int upload(Tp** out, const Tp* src, size_t count) {
    const int rc = alloc(out, count);
    if (rc) return rc;
    if (count) MR_CUDA(h, cudaMemcpyAsync(*out, src, count * sizeof(Tp), cudaMemcpyHostToDevice, st));
    return MR_OK;
  }
};

inline uint32_t q_of(int32_t deg, double scale) { return deg <= 0 ? 0u : static_cast<uint32_t>(llrint(scale / std::sqrt(static_cast<double>(deg)))); }
inline double rs_of(int32_t deg, double inv) { return deg <= 0 ? 0.0 : inv / std::sqrt(static_cast<double>(deg)); }
inline long long round_up(long long x, long long m) { return (x + m - 1) / m * m; }

// f(lo, hi) over disjoint row ranges on a few host threads.  The per-shard host work of mr_set_test_users (CSR validation, id rotation,
// cosine factors: O(test entries)) sits on the calling thread inside every end-to-end step; a rank of an 8-GPU job shares the host with
// seven others, hence at most hardware threads / 8 (and at most 8) workers.
template <class F>
void parallel_rows(int n, F&& f) {
  const int hw = static_cast<int>(std::thread::hardware_concurrency());
  const int t = std::max(1, std::min(8, hw / 8));
  if (n < 16384 || t == 1) { f(0, n); return; }
  const int chunk = (n + t - 1) / t;
  std::vector<std::thread> workers;
  for (int i = 1; i < t; ++i) workers.emplace_back([&f, i, chunk, n] { f(std::min(n, i * chunk), std::min(n, (i + 1) * chunk)); });
  f(0, std::min(n, chunk));
  for (auto& w : workers) w.join();
}

int check_csr(mr_handle* h, const char* what, int n_rows, int n_cols, const int64_t* ptr, const int32_t* col) {
  if (!ptr || (!col && ptr[n_rows] > 0)) return fail(h, MR_ERR_BAD_ARG, "%s: null CSR arrays", what);
  if (ptr[0] != 0) return fail(h, MR_ERR_BAD_ARG, "%s: rowptr[0] != 0", what);
  for (int r = 0; r < n_rows; ++r)
    if (ptr[r + 1] < ptr[r]) return fail(h, MR_ERR_BAD_ARG, "%s: rowptr not monotone at row %d", what, r);
  // the first offending row (smallest index) is reported, whichever thread finds it
  struct Bad { int row = -1; int kind = 0; int col = 0; };
  Bad best; std::mutex mu;
  parallel_rows(n_rows, [&](int lo, int hi) {
    Bad b;
    for (int r = lo; r < hi && b.row < 0; ++r) {
      for (int64_t i = ptr[r]; i < ptr[r + 1]; ++i) {
        if (col[i] < 0 || col[i] >= n_cols) { b.row = r; b.kind = 1; b.col = col[i]; break; }
        if (i > ptr[r] && col[i] <= col[i - 1]) { b.row = r; b.kind = 2; break; }
      }
    }
    if (b.row >= 0) {
      std::lock_guard<std::mutex> g(mu);
      if (best.row < 0 || b.row < best.row) best = b;
    }
  });
  const Bad& b = best;
  if (b.row >= 0 && b.kind == 1) return fail(h, MR_ERR_BAD_ARG, "%s: column id %d out of range at row %d", what, b.col, b.row);
  if (b.row >= 0) return fail(h, MR_ERR_BAD_ARG, "%s row %d not ascending/unique", what, b.row);
  return MR_OK;
}

struct PhaseTimer {   // CUDA events on the library stream (or the given one) around one phase (only with MR_PROFILE)
  mr_handle* h; int phase; bool on; cudaStream_t st;
  PhaseTimer(mr_handle* hh, int ph, cudaStream_t s = nullptr) : h(hh), phase(ph), on((hh->flags & MR_PROFILE) != 0), st(s ? s : hh->stream) {
    if (on) cudaEventRecord(h->ev[0], st);
  }
  ~PhaseTimer() {
    if (!on) return;
    cudaEventRecord(h->ev[1], st);
    cudaEventSynchronize(h->ev[1]);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]) == cudaSuccess) h->t_ms[phase] += ms;
  }
};

// In place over n_rows count rows ld apart: c -> float(c) * (rs(sq_row[rows[r]]) * rs(sq_col[j])) with rs(x) = float(1.0 / x), 0 where x = 0
// (degree 0).  The sqrt tables are correctly rounded (launch_sqrt_deg) and the build uses --fmad=false, so each value has the bits of
// the same formula on the host.  An element's int32 and its float share the 4 bytes, read and written by one thread.
__global__ void count_to_cos_kernel(int32_t* __restrict__ g, long long ld, const int* __restrict__ rows, int n_rows, int n_cols,
                                    const double* __restrict__ sq_row, const double* __restrict__ sq_col) {
  auto rs = [](double x) { return x > 0 ? static_cast<float>(1.0 / x) : 0.0f; };
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < static_cast<long long>(n_rows) * n_cols;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / n_cols), j = static_cast<int>(i % n_cols);
    int32_t& e = g[r * ld + j];
    e = __float_as_int(static_cast<float>(e) * (rs(sq_row[rows[r]]) * rs(sq_col[j])));
  }
}
__global__ void iota_kernel(int* p, int start, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = start + i;
}

// ---- K1 for one batch of test users -> Ct u16[T][128]
int count_ubm_batch(mr_handle* h, int b0, int nb) {
  if (h->engine == MR_ENGINE_TENSOR) {
    {
      PhaseTimer t(h, MR_T_EXPAND);
      MR_LAUNCH(h, launch_expand_rows(h->d_te_ptr, h->d_te_col, nullptr, b0, nb, kUserBatch, h->pitchS, h->d_Ate, h->stream));
    }
    PhaseTimer t(h, MR_T_COUNT);
    MR_LAUNCH(h, launch_count_gemm(h->d_Ate, kUserBatch, h->d_Atr, h->T, h->pitchS, kUserBatch, h->T, EPI_U16_T, h->d_ct, kUserBatch,
                                   h->num_sms, h->stream));
  } else {
    PhaseTimer t(h, MR_T_COUNT);
    MR_LAUNCH(h, launch_sparse_count_u16t(h->d_te_ptr, h->d_te_col, b0, nb, h->d_csc_ptr, h->d_csc_idx, h->d_ct, h->T, h->stream));
  }
  return MR_OK;
}

// Exact intersection-count rows of one query kind: G[r][c] = |items(rows[r]) ∩ items(c)| for the n_cols candidates c, rows ld apart, in
// the Gram workspace.  Tensor engine: the query rows expanded to 0/1 rows of `pitch` bytes, times the candidates' dense operand B (n_cols
// rows).  Sparse engine: the walk query -> items (q_ptr / q_idx) -> candidates (c_ptr / c_idx), one atomic per event.
//   Gram rows (song x song):        q = inverted index, c = train rows, B = A_tr^T, pitch = pitchT, n_cols = S, ld = ldg
//   user rows (test x train user):  q = test rows, c = inverted index, B = A_tr, pitch = pitchS, n_cols = T, ld = T padded to 32
struct CountRows {
  const long long* q_ptr; const int* q_idx; const long long* c_ptr; const int* c_idx;
  const uint8_t* B; long long pitch; int n_cols; long long ld;
};
CountRows song_count_rows(const mr_handle* h) { return {h->d_csc_ptr, h->d_csc_idx, h->d_tr_ptr, h->d_tr_col, h->d_AtrT, h->pitchT, h->S, h->ldg}; }
CountRows user_count_rows(const mr_handle* h) { return {h->d_te_ptr, h->d_te_col, h->d_csc_ptr, h->d_csc_idx, h->d_Atr, h->pitchS, h->T, round_up(h->T, 32)}; }

int count_rows(mr_handle* h, const CountRows& cr, const int* d_rows, int n_rows) {
  if (h->engine == MR_ENGINE_TENSOR) {
    const int rows_pad = static_cast<int>(round_up(n_rows, 128));
    {
      PhaseTimer t(h, MR_T_EXPAND);
      MR_LAUNCH(h, launch_expand_rows(cr.q_ptr, cr.q_idx, d_rows, 0, n_rows, rows_pad, cr.pitch, h->d_Aj, h->stream));
    }
    PhaseTimer t(h, MR_T_COUNT);
    MR_LAUNCH(h, launch_count_gemm(h->d_Aj, rows_pad, cr.B, cr.n_cols, cr.pitch, n_rows, cr.n_cols, EPI_I32, h->d_g, cr.ld, h->num_sms,
                                   h->stream));
  } else {
    PhaseTimer t(h, MR_T_COUNT);
    for (int r0 = 0; r0 < n_rows; r0 += 32768) {
      const int n = std::min(32768, n_rows - r0);
      MR_LAUNCH(h, launch_sparse_gram_rows(d_rows + r0, n, cr.q_ptr, cr.q_idx, cr.c_ptr, cr.c_idx, h->d_g + static_cast<long long>(r0) * cr.ld,
                                           cr.ld, h->stream));
    }
  }
  return MR_OK;
}

// ---- K1 for a list of Gram rows (device array of song ids) -> G i32[n_rows][ldg]
int gram_rows(mr_handle* h, const int* d_rows, int n_rows) { return count_rows(h, song_count_rows(h), d_rows, n_rows); }

// the Gram workspace for n_rows count rows of a kind (default: Gram rows): ld ints per row, and on the tensor engine the expanded query rows
int ensure_gram_ws(mr_handle* h, int n_rows, long long ld = 0, long long a_pitch = 0) {
  const size_t rows = static_cast<size_t>(round_up(std::max(n_rows, 1), 128));
  const int rc = slot_alloc(h, mr_handle::SL_GRAM_G, &h->d_g, rows * (ld ? ld : h->ldg), true);
  if (rc || h->engine != MR_ENGINE_TENSOR) return rc;
  return slot_alloc(h, mr_handle::SL_GRAM_A, &h->d_Aj, rows * (a_pitch ? a_pitch : h->pitchT), true);
}

// Item-space: compute the rows G[h][:], Gq[h][:] of the head songs once per train set (lazily, on first use, or mr_prepare).
// Head rows are ordered by train degree, descending.  Two construction paths, both from the inverted index:
//   staged rows [0, n_head_staged): the most popular songs, whose entries can exceed 16 / 32 bits — one packed 64-bit accumulator per
//     entry in an L2-resident staging chunk, then pack_head_rows_kernel writes the 6-byte form + the exact exception list;
//   direct rows [n_head_staged, n_head): every song whose weighted listener sum is < 2^32 and whose train degree is < 2^16 — no entry
//     of such a row can overflow, so the events are added straight into the final u16 / u32 arrays (32-bit L2 atomics), an L2-sized
//     chunk of rows at a time: zero the chunk (it stays dirty in L2), scatter into it, let it drain to HBM once.  This path moves
//     6 bytes per entry instead of 8 (zero) + 8 (read) + 6 (write) and has no pack pass: it is what made the sparse 85 % of the head
//     rows cheap (they carry few events but paid the full dense staging traffic).
// On the tensor engine (dense-friendly shapes) every row is staged and computed by K1: one 0/1 count GEMM + byte-plane GEMMs of the weights.
int finish_head_rows(mr_handle* h);

// Launch the whole build on stream st (the library stream, or pre_stream for mr_prepare_async) and leave the handle in the
// head_pending state; nothing here waits for the device except the tensor engine's temporary operands.
int start_head_rows(mr_handle* h, cudaStream_t st) {
  if (h->head_ready || h->head_pending) return MR_OK;
  int rc;
  if (st != h->stream) {   // the build overwrites rows that earlier work on the library stream may still be reading
    MR_CUDA(h, cudaEventRecord(h->ev_pre, h->stream));
    MR_CUDA(h, cudaStreamWaitEvent(st, h->ev_pre, 0));
  }
  const bool dbg = getenv("MRSCORE_DEBUG_TIMING") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms_since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(now() - t).count(); };
  auto t_start = now();
  const size_t n = static_cast<size_t>(std::max(h->n_head, 1)) * h->spitch;   // allocated once per handle; a failed or invalidated precompute reuses it
  if ((rc = slot_alloc(h, mr_handle::SL_HEAD_G16, &h->d_g16, n, true)) || (rc = slot_alloc(h, mr_handle::SL_HEAD_GQ32, &h->d_gq32, n, true))) return rc;
  const bool tensor = h->engine == MR_ENGINE_TENSOR && h->n_head > 0 && h->T < (1 << 23);
  const int n_staged = tensor ? h->n_head : h->n_head_staged;
  // number of byte planes the weights q_24(|I_v|) need (3 when every train user has >= 2 songs: q < 2^24)
  int n_planes = 1;
  while (n_planes < 4 && (static_cast<unsigned long long>(h->max_qv) >> (8 * n_planes)) != 0) ++n_planes;
  // staging chunk.  Tensor engine: <= 8 GiB of (u32 + u64) rows, a multiple of the 128-row GEMM tile.  Scatter path: small enough
  // (<= 64 MiB) that the rows being built stay L2-resident, so the integer atomics are resolved in L2 instead of as DRAM read-modify-writes.
  long long chunk = 1; bool packed = false;
  if (tensor) {
    chunk = (8LL << 30) / (h->spitch * 12) / 128 * 128;
    chunk = std::max<long long>(128, std::min<long long>(chunk, 4096));
  } else if (n_staged > 0) {
    // one packed 64-bit accumulator per entry when no weighted sum can reach 2^44 and no count 2^20 (any realistic data set)
    packed = h->max_qsum < (1ULL << 44) && *std::max_element(h->deg_song_train.begin(), h->deg_song_train.end()) < (1 << 20) &&
             !getenv("MRSCORE_PRECOMPUTE_UNPACKED");
    chunk = std::max<long long>(4, std::min<long long>((64LL << 20) / (h->spitch * (packed ? 8 : 12)), 4096));
    if (const char* e = getenv("MRSCORE_PRECOMPUTE_CHUNK")) chunk = std::max(1LL, atoll(e));
  }
  h->head_packed = packed; h->head_planes = tensor ? n_planes : 0;
  // The staging rows and the exception list live in grow-only slots of the handle: a rebuild (mr_invalidate_prepared + mr_prepare, i.e.
  // every step of a job that counts the model build) does no cudaMalloc / cudaFree — next to 100+ GB of live allocations those cost
  // tens to hundreds of milliseconds, more than the kernels of a song partition's precompute.  Only the tensor engine's dense operands
  // (small shapes) are temporary.
  Scratch tmp(h, st);
  uint32_t* g_stage = nullptr; unsigned long long* gq_stage = nullptr;
  HeadExceptions ex{};
  ex.capacity = n_staged > 0 ? (1u << 24) : 1u;
  const size_t stage_entries = n_staged > 0 ? static_cast<size_t>(chunk) * h->spitch : 1;
  {
    char* xb = nullptr;                 // [count (16 B)] [gq_extra u64] [row i32] [song i32] [g_extra u32]
    const size_t cap = ex.capacity;
    if ((rc = slot_alloc(h, mr_handle::SL_PRE_G, &g_stage, packed ? 1 : stage_entries, true)) ||
        (rc = slot_alloc(h, mr_handle::SL_PRE_GQ, &gq_stage, stage_entries, true)) || (rc = slot_alloc(h, mr_handle::SL_PRE_EXC, &xb, 16 + cap * 20, true))) return rc;
    ex.count = reinterpret_cast<unsigned int*>(xb);
    ex.gq_extra = reinterpret_cast<unsigned long long*>(xb + 16);
    ex.row = reinterpret_cast<int*>(xb + 16 + cap * 8);
    ex.song = reinterpret_cast<int*>(xb + 16 + cap * 12);
    ex.g_extra = reinterpret_cast<uint32_t*>(xb + 16 + cap * 16);
  }
  cudaError_t e = cudaMemsetAsync(ex.count, 0, sizeof(unsigned int), st);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "memset: %s", cudaGetErrorString(e));
  uint8_t *a_rows = nullptr, *b_plane = nullptr;
  if (tensor) {
    if ((rc = tmp.alloc(&a_rows, static_cast<size_t>(chunk) * h->pitchT)) ||
        (rc = tmp.alloc(&b_plane, static_cast<size_t>(h->S) * h->pitchT * n_planes))) return rc;
    // the GEMM epilogues write only the columns < S: the pad columns of the staging rows must not hold garbage (pack reads the full pitch)
    e = cudaMemsetAsync(g_stage, 0, stage_entries * sizeof(uint32_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(gq_stage, 0, stage_entries * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "memset: %s", cudaGetErrorString(e));
    // the byte planes of q_24(|I_v|) as weighted B operands (built once, reused by every chunk)
    PhaseTimer t(h, MR_T_EXPAND, st);
    for (int plane = 0; plane < n_planes; ++plane) {
      int lrc = launch_expand_rows_weighted(h->d_csc_ptr, h->d_csc_idx, h->d_qv, plane, h->S, h->pitchT,
                                            b_plane + static_cast<size_t>(plane) * h->S * h->pitchT, st);
      h->launches++;
      if (lrc) return fail(h, MR_ERR_CUDA, "launch_expand_rows_weighted failed");
    }
  }
  if (dbg) { cudaStreamSynchronize(st); fprintf(stderr, "[mrscore] precompute: allocations %.1f ms (staged rows %d in chunks of %lld, direct rows %d)\n", ms_since(t_start), n_staged, chunk, h->n_head - n_staged); }
  auto t_loop = now();
  for (int r0 = 0; r0 < n_staged; r0 += static_cast<int>(chunk)) {
    const int nr = std::min<int>(static_cast<int>(chunk), n_staged - r0);
    if (tensor) {
      // G = A_head · A_trT^T as one 0/1 count GEMM; Gq as byte-plane GEMMs (255 * T < 2^31 keeps each plane exact in int32)
      const int n_pad = static_cast<int>(round_up(nr, 128));
      {
        PhaseTimer t(h, MR_T_EXPAND, st);
        int lrc = launch_expand_rows(h->d_csc_ptr, h->d_csc_idx, h->d_head_song + r0, 0, nr, n_pad, h->pitchT, a_rows, st);
        h->launches++;
        if (lrc) return fail(h, MR_ERR_CUDA, "launch_expand_rows failed");
      }
      PhaseTimer t(h, MR_T_COUNT, st);
      int lrc = launch_count_gemm(a_rows, n_pad, h->d_AtrT, h->S, h->pitchT, nr, h->S, EPI_I32, g_stage, h->spitch, h->num_sms, st);
      h->launches++;
      for (int plane = 0; plane < n_planes && !lrc; ++plane) {
        lrc = launch_count_gemm(a_rows, n_pad, b_plane + static_cast<size_t>(plane) * h->S * h->pitchT, h->S, h->pitchT, nr, h->S, EPI_ACC_U64,
                                gq_stage, h->spitch, h->num_sms, st, 8 * plane, plane > 0);
        h->launches++;
      }
      if (lrc) return fail(h, MR_ERR_CUDA, "launch_count_gemm failed: rc=%d (%s)", lrc, cudaGetErrorString(cudaGetLastError()));
    } else {
      PhaseTimer t(h, MR_T_PRECOMPUTE, st);
      int lrc = launch_gram_head_scatter(h->d_head_song, h->d_head_lst_ptr, r0, r0 + nr, h->d_csc_ptr, h->d_csc_idx, h->d_tr_ptr, h->d_tr_end,
                                         h->d_tr_col, h->d_qv, g_stage, gq_stage, h->spitch, packed ? 1 : 0, h->num_sms, st);
      h->launches++;
      if (lrc) return fail(h, MR_ERR_CUDA, "launch_gram_head_scatter failed");
    }
    PhaseTimer t(h, MR_T_PRECOMPUTE, st);
    int lrc = launch_pack_head_rows(g_stage, gq_stage, packed ? 1 : 0, r0, nr, h->spitch, h->n_cols, h->d_g16, h->d_gq32, ex, h->num_sms, st);
    h->launches++;
    if (lrc) return fail(h, MR_ERR_CUDA, "launch_pack_head_rows failed");
  }
  if (dbg) { cudaStreamSynchronize(st); fprintf(stderr, "[mrscore] precompute: staged rows %.1f ms\n", ms_since(t_loop)); }
  if (n_staged < h->n_head) {
    // direct rows: an L2-sized chunk of final rows at a time
    long long mb = 48;
    if (const char* ev = getenv("MRSCORE_DIRECT_CHUNK_MB")) mb = std::max(1LL, atoll(ev));
    const long long dchunk = std::max<long long>(1, (mb << 20) / (h->spitch * 6));
    PhaseTimer t(h, MR_T_PRECOMPUTE, st);
    // Several streams (kPreStreams): the chunks are independent (disjoint rows) and each one is three short enqueues (two memsets + a
    // kernel of ~1.3 waves), so consecutive chunks rotate over `st` and the extra build streams and the next chunk's CTAs start while
    // the previous grid drains: 113.8 -> 73.4 ms for the 32 k rows of the MSD-shaped set with four streams (profiles/r02_summary.md §10).
    // Not under MR_PROFILE (the phase timer brackets `st` only).
    int n_streams = kPreStreams;
    if (const char* ev = getenv("MRSCORE_PRE_STREAMS")) n_streams = std::max(1, std::min(atoi(ev), 1 + kPreExtraStreams));
    if (h->flags & MR_PROFILE) n_streams = 1;
    auto sync_extra = [&] { for (int i = 0; i < kPreExtraStreams; ++i) cudaStreamSynchronize(h->pre_extra[i]); };
    for (int i = 0; i + 1 < n_streams; ++i) {
      if ((e = cudaEventRecord(h->ev_pre_extra[i], st)) != cudaSuccess || (e = cudaStreamWaitEvent(h->pre_extra[i], h->ev_pre_extra[i], 0)) != cudaSuccess)
        return fail(h, MR_ERR_CUDA, "head-row precompute: %s", cudaGetErrorString(e));
    }
    int ci = 0;
    for (int r0 = n_staged; r0 < h->n_head; r0 += static_cast<int>(dchunk), ++ci) {
      const int nr = std::min<int>(static_cast<int>(dchunk), h->n_head - r0);
      const int si = ci % n_streams;
      int lrc = launch_gram_head_direct(h->d_head_song, h->d_head_lst_ptr, r0, r0 + nr, h->d_csc_ptr, h->d_csc_idx, h->d_tr_ptr, h->d_tr_end,
                                        h->d_tr_col, h->d_qv, h->d_g16, h->d_gq32, h->spitch, h->num_sms, si ? h->pre_extra[si - 1] : st);
      h->launches++;
      if (lrc) { sync_extra(); return fail(h, MR_ERR_CUDA, "launch_gram_head_direct failed"); }
    }
    for (int i = 0; i + 1 < n_streams; ++i) {   // `st` joins the extra streams
      if ((e = cudaEventRecord(h->ev_pre_extra[i], h->pre_extra[i])) != cudaSuccess || (e = cudaStreamWaitEvent(st, h->ev_pre_extra[i], 0)) != cudaSuccess) {
        sync_extra();
        return fail(h, MR_ERR_CUDA, "head-row precompute: %s", cudaGetErrorString(e));
      }
    }
  }
  // the exception count travels to pinned host memory behind the kernels; finish_head_rows picks it up
  e = cudaMemcpyAsync(h->h_n_ex, ex.count, sizeof(unsigned int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaEventRecord(h->ev_pre, st);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "head-row precompute: %s", cudaGetErrorString(e));
  if (dbg) fprintf(stderr, "[mrscore] precompute: launched after %.1f ms\n", ms_since(t_start));
  h->pend_ex = ex;
  h->head_pending = true;
  return MR_OK;
}

// Complete a started build: wait for its kernels, turn the exception list into a CSR by head row (host sort; it is a few thousand
// entries on MSD-shaped data) and order the library stream behind the build.
int finish_head_rows(mr_handle* h) {
  if (h->head_ready) return MR_OK;
  if (!h->head_pending) return fail(h, MR_ERR_STATE, "no head-row build in flight");
  int rc;
  h->head_pending = false;
  const HeadExceptions ex = h->pend_ex;
  cudaError_t e = cudaEventSynchronize(h->ev_pre);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "head-row precompute: %s", cudaGetErrorString(e));
  const unsigned int n_ex = *h->h_n_ex;
  if (n_ex > ex.capacity) return fail(h, MR_ERR_OOM, "head-row exception list overflowed (%u entries)", n_ex);
  std::vector<int> xr(n_ex), xs(n_ex); std::vector<uint32_t> xg(n_ex); std::vector<unsigned long long> xq(n_ex);
  if (n_ex) {
    e = cudaMemcpy(xr.data(), ex.row, n_ex * sizeof(int), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(xs.data(), ex.song, n_ex * sizeof(int), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(xg.data(), ex.g_extra, n_ex * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(xq.data(), ex.gq_extra, n_ex * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "head-row exception list: %s", cudaGetErrorString(e));
  }
  std::vector<unsigned int> order(n_ex);
  for (unsigned int i = 0; i < n_ex; ++i) order[i] = i;
  std::sort(order.begin(), order.end(), [&](unsigned int a, unsigned int b) { return xr[a] != xr[b] ? xr[a] < xr[b] : xs[a] < xs[b]; });
  std::vector<long long> ex_ptr(static_cast<size_t>(h->n_head) + 1, 0);
  std::vector<int> es(n_ex); std::vector<uint32_t> eg(n_ex); std::vector<unsigned long long> eq(n_ex);
  for (unsigned int i = 0; i < n_ex; ++i) { const unsigned int o = order[i]; ex_ptr[xr[o] + 1]++; es[i] = xs[o]; eg[i] = xg[o]; eq[i] = xq[o]; }
  for (int r = 0; r < h->n_head; ++r) ex_ptr[r + 1] += ex_ptr[r];
  if ((rc = slot_upload(h, mr_handle::SL_EX_PTR, &h->d_ex_ptr, ex_ptr.data(), ex_ptr.size()))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_EX_SONG, &h->d_ex_song, es.data(), es.size()))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_EX_G, &h->d_ex_g, eg.data(), eg.size()))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_EX_GQ, &h->d_ex_gq, eq.data(), eq.size()))) return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  h->n_ex = n_ex;
  h->head_ready = true;
  return MR_OK;
}

int ensure_head_rows(mr_handle* h) {
  if (h->head_ready) return MR_OK;
  int rc = start_head_rows(h, h->stream);
  if (rc) return rc;
  return finish_head_rows(h);
}

// Batch plan of the current test shard.  User space: 128-user batches (UMMA M).  Item space: as many test users per batch as the Sint
// panels (two models, 8 bytes per (user, song)) fit in HBM next to the head rows — a large batch shares the row tiles of popular
// songs among more users (head_rowsum_kernel) — split evenly, plus per batch the balanced work groups of head_rowsum_kernel:
// segments (Sint row, head-entry range) packed longest-first into n_groups bins of equal total length.
constexpr int kPlanTooLarge = -100;   // a work group exceeds the shared-memory staging area: the caller retries with smaller batches

int plan_item_batches_once(mr_handle* h, const std::vector<long long>& hu_ptr, int rows_cap) {
  int rc;
  const int U = h->U;
  h->batch_rows = kUserBatch;
  const size_t panel_rows_have = std::min(h->slot_cap[mr_handle::SL_SINT_U], h->slot_cap[mr_handle::SL_SINT_I]) / (static_cast<size_t>(h->spitch) * 8);
  if (h->space == MR_SPACE_ITEM && static_cast<size_t>(U) <= panel_rows_have && (h->item_batch_cap <= 0 || U <= h->item_batch_cap) &&
      (rows_cap <= 0 || U <= rows_cap) && h->slot_cap[mr_handle::SL_SEL] >= static_cast<size_t>(U) * h->sel_pitch * 8) {
    h->batch_rows = std::max(kUserBatch, U);   // the panels of an earlier shard already hold this one as a single batch: no memory query
  } else if (h->space == MR_SPACE_ITEM) {
    size_t free_b = 0, total_b = 0;
    MR_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    const size_t per_row = static_cast<size_t>(h->spitch) * 16 + static_cast<size_t>(h->sel_pitch) * 8;
    size_t avail = free_b + h->slot_cap[mr_handle::SL_SINT_U] + h->slot_cap[mr_handle::SL_SINT_I] + h->slot_cap[mr_handle::SL_SEL];
    size_t reserve = kCallerReserve;   // left for the caller's context (torch, NCCL buffers, gathered top-k blocks) and small workspaces
    if (!h->head_ready && h->slot_cap[mr_handle::SL_HEAD_G16] == 0) reserve += static_cast<size_t>(std::max(h->n_head, 1)) * h->spitch * 6 + (1ULL << 30);   // head rows + staging come later
    long long max_rows = avail > reserve ? static_cast<long long>((avail - reserve) / per_row) : 0;
    max_rows = std::max<long long>(max_rows, kUserBatch);
    if (h->item_batch_cap > 0) max_rows = std::min<long long>(max_rows, h->item_batch_cap);
    if (rows_cap > 0) max_rows = std::min<long long>(max_rows, std::max(rows_cap, kUserBatch));
    const int n_batches = static_cast<int>((U + max_rows - 1) / max_rows);
    h->batch_rows = std::max(kUserBatch, (U + n_batches - 1) / n_batches);
  }
  const size_t rows = static_cast<size_t>(h->batch_rows);
  if ((rc = slot_alloc(h, mr_handle::SL_SINT_U, &h->d_sint_u, rows * h->spitch, true))) return rc;
  if ((rc = slot_alloc(h, mr_handle::SL_SINT_I, &h->d_sint_i, rows * h->spitch, true))) return rc;
  if ((rc = slot_alloc(h, mr_handle::SL_SEL, &h->d_sel, rows * h->sel_pitch, true))) return rc;
  if (h->space != MR_SPACE_ITEM) return MR_OK;

  const int G = h->n_groups, B = h->batch_rows;
  const int n_batches = (U + B - 1) / B;
  std::vector<int4> seg, grp_hdr, copy_desc; std::vector<int> split_rows;
  long long ge_size = 0;   // entries of the group-ordered copies (segments padded to multiples of 4)
  h->h_split_ptr.assign(1, 0);
  h->seg_cap = 1; h->ent_cap = 1;
  struct Item { int row, e0, e1, acc; };
  std::vector<Item> items; std::vector<std::vector<int>> bins(G);
  for (int bi = 0; bi < n_batches; ++bi) {
    const int b0 = bi * B, nb = std::min(B, U - b0);
    const long long entries = hu_ptr[b0 + nb] - hu_ptr[b0];
    // a segment costs its entries plus ~3 entry-equivalents for the Sint row it writes (8 B/song against 4 or 2 B/song per entry)
    constexpr int kRowCost = 3;
    const long long share = (entries + static_cast<long long>(kRowCost) * nb + G - 1) / G;
    const int cap = static_cast<int>(std::max<long long>(32, share));
    items.clear();
    for (int b = 0; b < nb; ++b) {
      const int e0 = static_cast<int>(hu_ptr[b0 + b]), e1 = static_cast<int>(hu_ptr[b0 + b + 1]), n = e1 - e0;
      if (n <= cap) { items.push_back({b, e0, e1, 0}); continue; }
      const int parts = (n + cap - 1) / cap;
      for (int p = 0; p < parts; ++p) items.push_back({b, e0 + static_cast<int>(static_cast<long long>(n) * p / parts), e0 + static_cast<int>(static_cast<long long>(n) * (p + 1) / parts), 1});
      split_rows.push_back(b);
    }
    h->h_split_ptr.push_back(static_cast<int>(split_rows.size()));
    // Longest-processing-time packing into G bins of equal cost: every item goes to the currently lightest bin.  Costs are small
    // integers and the minimum load never decreases, so the priority queue is a bucket queue (bins listed by load, a cursor that only
    // moves up): O(items + largest load) instead of a heap operation per user, which at 110 000 users per shard was half of
    // mr_set_test_users.  (A plain sequential fill balances the cost model just as well but measured 30 % slower in head_rowsum: LPT
    // mixes long and short segments in every bin, which averages out what the model gets wrong.)
    {   // counting sort by length, descending, stable
      int max_n = 0;
      for (const Item& it : items) max_n = std::max(max_n, it.e1 - it.e0);
      std::vector<int> start(static_cast<size_t>(max_n) + 2, 0);
      for (const Item& it : items) start[max_n - (it.e1 - it.e0) + 1]++;
      for (int i = 0; i <= max_n; ++i) start[i + 1] += start[i];
      std::vector<Item> sorted(items.size());
      for (const Item& it : items) sorted[start[max_n - (it.e1 - it.e0)]++] = it;
      items.swap(sorted);
    }
    for (auto& v : bins) v.clear();
    {
      std::vector<std::vector<int>> by_load(static_cast<size_t>(2 * (share + cap) + 64));
      by_load[0].resize(G);
      for (int g = 0; g < G; ++g) by_load[0][g] = G - 1 - g;      // pop_back hands out bin 0 first
      size_t cur = 0;
      for (size_t i = 0; i < items.size(); ++i) {
        while (by_load[cur].empty()) ++cur;
        const int g = by_load[cur].back(); by_load[cur].pop_back();
        bins[g].push_back(static_cast<int>(i));
        const size_t nl = cur + static_cast<size_t>(items[i].e1 - items[i].e0 + kRowCost);
        if (nl >= by_load.size()) by_load.resize(nl + nl / 2 + 1);
        by_load[nl].push_back(g);
      }
    }
    for (int g = 0; g < G; ++g) {   // the group's segments and entries, contiguous: the CTA stages them in shared memory
      const int seg0 = static_cast<int>(seg.size());
      const long long ent0 = ge_size;
      for (int i : bins[g]) {
        const int local = static_cast<int>(ge_size - ent0), n = items[i].e1 - items[i].e0;
        seg.push_back(make_int4(items[i].row, local, local + n, items[i].acc));
        if (n > 0) copy_desc.push_back(make_int4(items[i].e0, static_cast<int>(ge_size), n, 0));   // gathered on the device
        ge_size += n;
      }
      const int n_seg = static_cast<int>(seg.size()) - seg0, n_ent = static_cast<int>(ge_size - ent0);
      grp_hdr.push_back(make_int4(seg0, n_seg, static_cast<int>(ent0), n_ent));
      h->seg_cap = std::max(h->seg_cap, n_seg); h->ent_cap = std::max(h->ent_cap, n_ent);
    }
  }
  if (ge_size >= (1LL << 31)) return fail(h, MR_ERR_BAD_ARG, "too many head entries in one shard");
  if (static_cast<size_t>(h->seg_cap) * 16 + static_cast<size_t>(h->ent_cap) * 8 > 48 * 1024) {
    if (h->batch_rows > kUserBatch) return kPlanTooLarge;
    return fail(h, MR_ERR_BAD_ARG, "head_rowsum work group too large for shared-memory staging (%d segments, %d entries)", h->seg_cap, h->ent_cap);
  }
  if ((rc = slot_upload(h, mr_handle::SL_SEG, &h->d_seg, seg.data(), seg.size()))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_GRP_HDR, &h->d_grp_hdr, grp_hdr.data(), grp_hdr.size()))) return rc;
  int4* d_desc = nullptr;
  if ((rc = slot_upload(h, mr_handle::SL_COPY_DESC, &d_desc, copy_desc.data(), copy_desc.size()))) return rc;
  if ((rc = slot_alloc(h, mr_handle::SL_GE_ROW, &h->d_ge_row, static_cast<size_t>(ge_size)))) return rc;
  if ((rc = slot_alloc(h, mr_handle::SL_GE_Q, &h->d_ge_q, static_cast<size_t>(ge_size)))) return rc;
  MR_LAUNCH(h, launch_gather_group_entries(d_desc, static_cast<int>(copy_desc.size()), h->d_hu_row, h->d_hu_q, h->d_ge_row, h->d_ge_q, h->stream));
  if ((rc = slot_upload(h, mr_handle::SL_SPLIT_ROWS, &h->d_split_rows, split_rows.data(), split_rows.size()))) return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));   // the staging vectors above are pageable and go out of scope
  return MR_OK;
}

// A shard with very many head entries per work group (small S with many users per batch, or few groups) is split into more batches
// until a group's segments and entries fit the 48 KB staging area of head_rowsum_kernel.
int plan_item_batches(mr_handle* h, const std::vector<long long>& hu_ptr) {
  int rows_cap = 0;
  for (;;) {
    const int rc = plan_item_batches_once(h, hu_ptr, rows_cap);
    if (rc != kPlanTooLarge) return rc;
    rows_cap = std::max(kUserBatch, h->batch_rows / 2);
  }
}

// The layout of one top-k result block: song i32[U][k] | score f64[U][k] | len i32[U], the song and len parts rounded up to 16 bytes, so
// that a caller can ship a whole result with a single transfer (mr_topk_packed).
struct TopkBlock {
  size_t score_off, len_off, bytes;
  TopkBlock(int U, int k)
      : score_off(static_cast<size_t>(round_up(static_cast<long long>(U) * k * 4, 16))), len_off(score_off + static_cast<size_t>(U) * k * 8),
        bytes(len_off + static_cast<size_t>(round_up(static_cast<long long>(U) * 4, 16))) {}
  TopkOut at(char* base) const {
    return {reinterpret_cast<int32_t*>(base), reinterpret_cast<double*>(base + score_off), reinterpret_cast<int32_t*>(base + len_off)};
  }
};

// Enqueue on st the copy of users [u0, u0 + n) of the device result src into the caller's host buffers dst (both indexed by user).
int copy_topk(mr_handle* h, const TopkOut& dst, const TopkOut& src, int k, int u0, int n, cudaStream_t st) {
  const size_t o = static_cast<size_t>(u0) * k, m = static_cast<size_t>(n) * k;
  MR_CUDA(h, cudaMemcpyAsync(dst.song + o, src.song + o, m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  MR_CUDA(h, cudaMemcpyAsync(dst.score + o, src.score + o, m * sizeof(double), cudaMemcpyDeviceToHost, st));
  MR_CUDA(h, cudaMemcpyAsync(dst.len + u0, src.len + u0, static_cast<size_t>(n) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  return MR_OK;
}

// DENSE: where the fp64 rows go.  ALL: out[u][s] for every test user (mr_score_dense).  USERS: out[i][s] for the listed users
// (DIST getRanks1 granularity).  SONGS: d_out[i][u] for the listed songs, gathered on the device (DIST getRanks2 granularity).
struct DenseOut { enum Kind { ALL, USERS, SONGS } kind; double* out; const int32_t* ids; int n_ids; const int* d_ids; double* d_out; };

// A model set (DESIGN.md §4.6): the entries one scoring of the shard serves.  The single-model calls run a set of one.
constexpr int kMaxSet = 16;
struct ModelSet {
  int n = 0;
  BlendParams bp[kMaxSet];
  TopkOut out[kMaxSet] = {};   // TOPK: each entry's device result
  // eval consumers: the entries grouped for the fused kernels; grp_stoch[g] = the STOCH entry whose select plane group g reads, or -1
  int n_groups = 0; EvalGroup grp[kMaxSet]; int grp_stoch[kMaxSet] = {};
  int n_stoch = 0;
  bool needs(int panel_model) const {   // UBM panel: some entry is not IBM; IBM panel: some entry is not UBM
    for (int i = 0; i < n; ++i) if (bp[i].model != (panel_model == MODEL_UBM ? MODEL_IBM : MODEL_UBM)) return true;
    return false;
  }
  ModelSet() = default;
  explicit ModelSet(int model) : n(1) { memset(&bp[0], 0, sizeof bp[0]); bp[0].model = model; }   // one model without blend parameters
};

// What a scoring run hands the masked panels to: the top-k select, the fp64 rows, the streamed evaluateModel passes (DESIGN.md §4.5), or
// the column select of song audiences (DESIGN.md §4.10).
enum class Consumer { TOPK, DENSE, EVAL_RANGE, EVAL_COUNT, AUDIENCE };
struct Run {
  ModelSet set;
  Consumer what = Consumer::TOPK;
  int k = 0;                            // TOPK: list length
  const DenseOut* dense = nullptr;      // DENSE: where the rows go
  const TopkOut* topk_host = nullptr;   // TOPK in item space: the caller's buffers, filled slice by slice from entry 0 on copy_stream
  bool reuse = false;                   // EVAL_COUNT: the panels hold this set's masked numerators (resident reuse): no scoring at all
  const int2* aud_q = nullptr;          // AUDIENCE: [aud_n] device (column, list row), ascending column; the running lists are set.out[0]
  int aud_n = 0;
  // TOPK under a filter (DESIGN.md §4.11): the exclusion rows masked after the listened pairs (ex_ptr [U + 1], or null), and the candidate
  // path over the allowed columns cand_cols [n_cand] instead of the full-row select (whose bitmap, if any, is in each entry's BlendParams)
  const long long* ex_ptr = nullptr; const int* ex_col = nullptr;
  bool candidate = false; const int* cand_cols = nullptr; int n_cand = 0;
  bool eval() const { return what == Consumer::EVAL_RANGE || what == Consumer::EVAL_COUNT; }
};

// The consumers of one masked slice: per entry the select (after its blend's select plane), or per group the fused eval kernels (after
// the group's STOCH plane, unless the plane of the set's only STOCH entry is still in place from the range pass).
int consume_slice(mr_handle* h, const Run& run, long long* su, long long* si, uint64_t* sel, int u0, int n, cudaStream_t st) {
  const ModelSet& set = run.set;
  if (run.what == Consumer::AUDIENCE) {   // the column select runs once per batch (audience_columns); a slice only builds its select plane
    const BlendParams& bp = set.bp[0];
    if (bp.model == MODEL_AGG || bp.model == MODEL_STOCH)
      MR_LAUNCH(h, launch_select_bits(bp, h->d_te_ptr, h->d_te_col, u0, n, h->n_cols, sel, h->sel_pitch, st));
    return MR_OK;
  }
  if (run.what == Consumer::TOPK) {
    for (int e = 0; e < set.n; ++e) {
      const BlendParams& bp = set.bp[e];
      const bool blend_sel = bp.model == MODEL_AGG || bp.model == MODEL_STOCH;
      if (blend_sel) MR_LAUNCH(h, launch_select_bits(bp, h->d_te_ptr, h->d_te_col, u0, n, h->n_cols, sel, h->sel_pitch, st));
      if (run.candidate) {
        MR_LAUNCH(h, launch_candidate_topk(bp, bp.model != MODEL_IBM ? su : nullptr, bp.model != MODEL_UBM ? si : nullptr, h->spitch,
                                           blend_sel ? sel : nullptr, h->sel_pitch, u0, n, run.cand_cols, run.n_cand, h->d_rsa, h->d_rsd, run.k,
                                           set.out[e].song, set.out[e].score, set.out[e].len, st));
        continue;
      }
      MR_LAUNCH(h, launch_topk(bp, h->d_te_ptr, bp.model != MODEL_IBM ? su : nullptr, bp.model != MODEL_UBM ? si : nullptr, h->spitch,
                               blend_sel ? sel : nullptr, h->sel_pitch, u0, n, h->n_cols, h->d_rsa, h->d_rsd, run.k, set.out[e].song,
                               set.out[e].score, set.out[e].len, st));
    }
    return MR_OK;
  }
  const bool plane_resident = run.reuse && set.n_stoch == 1;
  for (int g = 0; g < set.n_groups; ++g) {
    const int se = set.grp_stoch[g];
    if (se >= 0 && !plane_resident)
      MR_LAUNCH(h, launch_select_bits(set.bp[se], h->d_te_ptr, h->d_te_col, u0, n, h->n_cols, sel, h->sel_pitch, st));
    if (run.what == Consumer::EVAL_RANGE) {
      MR_LAUNCH(h, launch_eval_range(set.grp[g], su, si, h->spitch, sel, h->sel_pitch, u0, n, h->n_cols, h->d_rsa, h->d_rsd, h->d_eval_mm, st));
    } else {
      EvalCounts ec = h->ec;
      if (g > 0) ec.nlab = nullptr;   // label counts do not depend on the model: the first group takes them
      MR_LAUNCH(h, launch_eval_count(set.grp[g], su, si, h->spitch, sel, h->sel_pitch, u0, n, h->n_cols, h->d_rsa, h->d_rsd, ec, st));
    }
  }
  return MR_OK;
}

// AUDIENCE: the column select of the whole masked batch [b0, b0 + nb) (panels and select plane from row 0 of the batch) on st, after every
// slice of the batch, into the running lists.
int audience_columns(mr_handle* h, const Run& run, const long long* su, const long long* si, int b0, int nb, cudaStream_t st) {
  const BlendParams& bp = run.set.bp[0];
  const TopkOut& l = run.set.out[0];
  const AudienceArgs a{bp.model, bp.alpha, bp.one_minus_alpha, su, si, h->spitch, h->d_sel, h->sel_pitch, h->d_rsa, h->d_rsd, run.aud_q,
                       l.song, l.score, l.len, h->d_topk_stats + 3};
  PhaseTimer t(h, MR_T_TOPK, st);
  MR_LAUNCH(h, launch_audience(a, run.aud_n, b0, nb, run.k, st));
  return MR_OK;
}

// Item space, the head pass of batch bi (users [b0, b0 + nb)) on the library stream into pu (models bit 0, UBM) / pi (bit 1, IBM), after
// the event release of the slices that last read these panels (or null): zero the split rows, head_rowsum, exception fixup.
int head_pass(mr_handle* h, int bi, int b0, int nb, int models, long long* pu, long long* pi, cudaEvent_t release) {
  PhaseTimer t(h, MR_T_HEAD_ROWSUM);
  if (release) MR_CUDA(h, cudaStreamWaitEvent(h->stream, release, 0));
  const int4* grp = h->d_grp_hdr + static_cast<long long>(bi) * h->n_groups;
  const int sp0 = h->h_split_ptr[bi], n_split = h->h_split_ptr[bi + 1] - sp0;
  for (int m = 1; m <= 2; ++m) {
    if (!(models & m)) continue;
    long long* const panel = m == 1 ? pu : pi;
    if (n_split) MR_LAUNCH(h, launch_zero_rows(h->d_split_rows + sp0, n_split, panel, h->spitch, h->stream));
    MR_LAUNCH(h, launch_head_rowsum(m, m == 1 ? h->head_words_u : h->head_words_i, h->head_threads, grp, h->n_groups, h->d_seg, h->d_ge_row,
                                    h->d_ge_q, h->seg_cap, h->ent_cap, h->d_g16, h->d_gq32, h->spitch, h->n_cols, panel, h->spitch, h->stream));
  }
  if (h->n_ex > 0)
    MR_LAUNCH(h, launch_head_fixup(models, h->d_hu_ptr, h->d_hu_row, h->d_hu_song, h->d_hu_q, b0, nb, h->d_ex_ptr, h->d_ex_song, h->d_ex_g,
                                   h->d_ex_gq, pu, pi, h->spitch, h->stream));
  return MR_OK;
}

// How a call cuts the item-space batches into slices: panels (as head_pass), users per slice, tail-scatter lanes, whether the consumers
// read the select plane (the blends' bits for the top-k, STOCH's for the eval kernels; AGG's pick there is its split column), and the two
// streams consecutive slices alternate between.  Per slice the atomics of one tail-scatter launch stay within a few GB of the Sint panels
// (measured optimum 300-600 users; kTailSubBatch users of whole rows = ~1.8 GB of a panel; a song partition's rows are shorter).
struct Slicing { int models, users, lanes; bool sel; cudaStream_t st[2]; };

// Item space, the slices of batch b0: tail scatter, then (DENSE takes the whole batch) mask, consumers and the streamed host copy.
int item_slices(mr_handle* h, const Run& run, const Slicing& sl, int b0, int nb, long long* pu, long long* pi) {
  for (int s0 = 0; s0 < nb; s0 += sl.users) {
    const int sn = std::min(sl.users, nb - s0), u0 = b0 + s0;
    cudaStream_t const ts = sl.st[(s0 / sl.users) & 1];
    if (!run.reuse) {
      PhaseTimer t(h, MR_T_TAIL_SCATTER);
      const long long e0 = h->h_tu_ptr[u0], e1 = h->h_tu_ptr[u0 + sn];
      MR_LAUNCH(h, launch_tail_scatter(sl.models, h->d_tu_user, h->d_tu_song, h->d_tu_lptr, e0, e1, h->d_csc_ptr, h->d_csc_idx, h->d_tr_ptr,
                                       h->d_tr_end, h->d_tr_col, h->d_qv, h->d_qd, b0, pu, pi, h->spitch, h->h_tu_lptr[e1] - h->h_tu_lptr[e0],
                                       sl.lanes, ts));
    }
    if (run.what == Consumer::DENSE) continue;
    PhaseTimer t(h, run.eval() ? MR_T_OTHER : MR_T_TOPK);
    long long* su = (sl.models & 1) ? pu + static_cast<long long>(s0) * h->spitch : nullptr;
    long long* si = (sl.models & 2) ? pi + static_cast<long long>(s0) * h->spitch : nullptr;
    uint64_t* sel = sl.sel ? h->d_sel + static_cast<long long>(s0) * h->sel_pitch : nullptr;
    if (!run.reuse) MR_LAUNCH(h, launch_mask_listened(h->d_te_ptr, h->d_te_end, h->d_te_col, u0, sn, su, si, h->spitch, ts));
    if (run.ex_ptr) MR_LAUNCH(h, launch_mask_listened(run.ex_ptr, run.ex_ptr + 1, run.ex_col, u0, sn, su, si, h->spitch, ts));
    if (const int rc = consume_slice(h, run, su, si, sel, u0, sn, ts)) return rc;
    if (run.topk_host) {
      MR_CUDA(h, cudaEventRecord(h->ev_slice, ts));
      MR_CUDA(h, cudaStreamWaitEvent(h->copy_stream, h->ev_slice, 0));
      if (const int rc = copy_topk(h, *run.topk_host, run.set.out[0], run.k, u0, sn, h->copy_stream)) return rc;
    }
  }
  return MR_OK;
}

// User space, K1 + K2 of the 128-user batch b0 into d_sint_u (UBM) and d_sint_i (IBM: sparse weighted counts, or the batch's Gram rows).
int user_panels(mr_handle* h, int b0, int nb, bool need_ubm, bool need_ibm) {
  const AggItems items{h->d_item_song, h->d_item_begin, h->d_item_len, h->d_item_split, h->n_items};
  if (need_ubm) {
    if (const int rc = count_ubm_batch(h, b0, nb)) return rc;
    PhaseTimer t(h, MR_T_AGG_UBM);
    MR_CUDA(h, cudaMemsetAsync(h->d_sint_u, 0, static_cast<size_t>(kUserBatch) * h->spitch * sizeof(long long), h->stream));
    MR_LAUNCH(h, launch_aggregate_ubm(items, h->d_csc_idx, h->d_qv, h->d_ct, h->T, h->d_sint_u, h->spitch, h->num_sms, h->stream));
  }
  if (!need_ibm) return MR_OK;
  if (h->engine == MR_ENGINE_SPARSE) {
    // user-space formulation: weighted intersection counts, then the same inverted-index gather as UBM
    CarryList carry{h->d_carry_count, h->d_carry_events, h->carry_cap};
    {
      PhaseTimer t(h, MR_T_COUNT);
      MR_LAUNCH(h, launch_sparse_wcount_u32(h->d_te_ptr, h->d_te_col, b0, nb, h->d_csc_ptr, h->d_csc_idx, h->d_qd, h->d_wi, h->T, carry, h->stream));
    }
    PhaseTimer t(h, MR_T_AGG_IBM);
    MR_CUDA(h, cudaMemsetAsync(h->d_sint_i, 0, static_cast<size_t>(kUserBatch) * h->spitch * sizeof(long long), h->stream));
    MR_LAUNCH(h, launch_aggregate_w32(items, h->d_csc_idx, h->d_wi, h->T, h->d_sint_i, h->spitch, h->num_sms, h->stream));
    MR_LAUNCH(h, launch_carry_fixup(carry, h->d_tr_ptr, h->d_tr_col, h->d_sint_i, h->spitch, h->stream));
    MR_CUDA(h, cudaMemcpyAsync(h->h_carry_seen + b0 / kUserBatch, h->d_carry_count, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->stream));
    return MR_OK;
  }
  const int bi = b0 / kUserBatch;
  const long long r_off = h->batch_row_off[bi];
  const int n_rows = static_cast<int>(h->batch_row_off[bi + 1] - r_off);
  int rc;
  if (n_rows > 0 && (rc = gram_rows(h, h->d_rows + r_off, n_rows))) return rc;
  PhaseTimer t(h, MR_T_AGG_IBM);
  MR_LAUNCH(h, launch_aggregate_ibm(h->d_te_ptr, h->d_te_col, h->d_te_grow, h->d_qd, b0, nb, h->d_g, h->ldg, h->S, h->d_sint_i, h->spitch, h->stream));
  return MR_OK;
}

// DENSE: the masked panel rows of batch b0 as fp64 scores of model, kDenseChunk users at a time, to where d says.
int dense_out(mr_handle* h, int model, const long long* panel, const DenseOut& d, int b0, int nb) {
  for (int c0 = 0; c0 < nb; c0 += kDenseChunk) {
    const int cn = std::min(kDenseChunk, nb - c0), r0 = b0 + c0;
    MR_LAUNCH(h, launch_dense_scores(model, panel + static_cast<long long>(c0) * h->spitch, h->spitch, r0, cn, h->n_cols, h->d_rsa, h->d_rsd,
                                     h->d_dense, h->stream));
    if (d.kind == DenseOut::ALL) {
      MR_CUDA(h, cudaMemcpyAsync(d.out + static_cast<long long>(r0) * h->n_cols, h->d_dense, static_cast<size_t>(cn) * h->n_cols * sizeof(double),
                                 cudaMemcpyDeviceToHost, h->stream));
    } else if (d.kind == DenseOut::USERS) {
      for (int i = 0; i < d.n_ids; ++i) {
        const int r = d.ids[i] - r0;
        if (r < 0 || r >= cn) continue;
        MR_CUDA(h, cudaMemcpyAsync(d.out + static_cast<long long>(i) * h->n_cols, h->d_dense + static_cast<long long>(r) * h->n_cols,
                                   static_cast<size_t>(h->n_cols) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
      }
    } else {
      MR_LAUNCH(h, launch_gather_columns(h->d_dense, cn, h->n_cols, d.d_ids, d.n_ids, d.d_out, h->U, r0, h->stream));
    }
    MR_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  return MR_OK;
}

// One scoring of the shard (DESIGN.md §4.2): per batch, build the score panels the set needs, mask them, and hand them to run.what.
int run_batches(mr_handle* h, const Run& run) {
  const bool need_ubm = run.set.needs(MODEL_UBM), need_ibm = run.set.needs(MODEL_IBM);
  const int pure = need_ubm && need_ibm ? -1 : (need_ubm ? MODEL_UBM : MODEL_IBM);   // the one panel the set needs, if only one
  const bool item_space = h->space == MR_SPACE_ITEM;
  int rc;
  // the Gram workspace of the user-space IBM panel (allocated in item space too, which does not read it: it counts in device_bytes)
  if (need_ibm && h->engine != MR_ENGINE_SPARSE && (rc = ensure_gram_ws(h, h->max_batch_rows))) return rc;
  if (!run.reuse) ++h->gen;
  if (item_space && (rc = ensure_head_rows(h))) return rc;
  const int batch = item_space ? h->batch_rows : kUserBatch;
  // the sparse user-space IBM panel: each batch's carry-event count lands in its own zeroed slot of this call (user_panels), so the
  // check below sees exactly the batches of this call.  The sync first: a call that failed mid-shard may have left copies in flight.
  const bool carries = need_ibm && !item_space && h->engine == MR_ENGINE_SPARSE;
  const int n_user_batches = (h->U + kUserBatch - 1) / kUserBatch;
  h->carry_events = 0;
  if (carries) {
    MR_CUDA(h, cudaStreamSynchronize(h->stream));
    if (h->carry_seen_cap < n_user_batches) {
      if (h->h_carry_seen) cudaFreeHost(h->h_carry_seen);
      h->h_carry_seen = nullptr; h->carry_seen_cap = 0;
      MR_CUDA(h, cudaMallocHost(reinterpret_cast<void**>(&h->h_carry_seen), static_cast<size_t>(n_user_batches) * sizeof(unsigned int)));
      h->carry_seen_cap = n_user_batches;
    }
    memset(h->h_carry_seen, 0, static_cast<size_t>(n_user_batches) * sizeof(unsigned int));
  }
  // Batch pipeline (item-space top-k of a pure model over >= 2 batches; not under MR_PROFILE, whose phase timers serialise the
  // stream): the head pass of batch b + 1 is issued on the library stream while the tail scatter, mask and select of batch b run on
  // slice_stream.  A pure model leaves the other model's Sint panel idle, so consecutive batches alternate between the two panels: no
  // extra memory.  Head passes stay in order on h->stream, slices in order on slice_stream; ev_head[p] releases the slices of the batch
  // in panel p, ev_done[p] releases panel p for the head pass two batches later; the last batch joins slice_stream back into h->stream.
  // What it buys is the kernel boundaries (the next kernel's CTAs start while the previous grid drains): 727 -> 701 ms for the two
  // models of the one-GPU job.  Making the kernels truly share the SMs was measured and is WORSE (profiles/r02_summary.md §8): the head
  // pass lives on every resident CTA working on the same song tile out of L2, and a select streaming 48 GB through L2 beside it breaks that.
  // A set that needs both panels (a blend, or UBM and IBM entries) cannot alternate them across batches: it takes the alternating slices.
  const bool pipelined = item_space && run.what != Consumer::DENSE && pure >= 0 && !(h->flags & MR_PROFILE) &&
                         h->U > batch && !getenv("MRSCORE_NO_PIPELINE");
  // Every other item-space top-k (one batch, e.g. a GPU's share of a song-partitioned job, or a blend) puts consecutive slices on two
  // alternating streams instead: same idea, the boundaries between the slices' kernels (107.6 -> 105.1 ms for both models of a 1/8 song
  // partition; next to the batch pipeline it adds nothing).  The two streams' kernels have different shared-memory carve-outs and never
  // share an SM; asking for matched carve-outs makes them do so and is slower (profiles/r02_summary.md §8).
  const bool alternating = item_space && run.what != Consumer::DENSE && !pipelined && !(h->flags & MR_PROFILE) && !getenv("MRSCORE_NO_PIPELINE");
  const bool streamed = pipelined || alternating;   // the slices run off the library stream and are joined back into it
  // On an error return from the streamed region the library stream is still ordered behind both slice streams, so that nothing the
  // failed call left on them races the next call on the library stream.
  struct JoinOnError {
    mr_handle* h; bool armed;
    ~JoinOnError() {
      for (cudaStream_t s : {h->slice_stream, h->slice_stream2})
        if (armed && s && cudaEventRecord(h->ev_join, s) == cudaSuccess) cudaStreamWaitEvent(h->stream, h->ev_join, 0);
    }
  } join{h, streamed};
  Slicing sl{(need_ubm ? 1 : 0) | (need_ibm ? 2 : 0), 0, 0, false, {h->stream, h->stream}};
  const long long sub_fit = static_cast<long long>(kTailSubBatch) * round_up(h->S, 32) / h->spitch / (2 * h->num_sms) * (2 * h->num_sms);
  sl.users = static_cast<int>(std::max<long long>(kTailSubBatch, std::min<long long>(sub_fit, 1 << 20)));
  sl.lanes = 2LL * h->n_cols >= h->S ? 32 : (4LL * h->n_cols >= h->S ? 16 : 8);
  for (int e = 0; e < run.set.n; ++e) sl.sel = sl.sel || run.set.bp[e].model == MODEL_STOCH || (!run.eval() && run.set.bp[e].model == MODEL_AGG);
  if (streamed) { sl.st[0] = h->slice_stream; sl.st[1] = alternating ? h->slice_stream2 : h->slice_stream; }
  for (int b0 = 0; b0 < h->U; b0 += batch) {
    const int bi = b0 / batch, nb = std::min(batch, h->U - b0);
    if (!run.reuse) ++h->passes;
    if (item_space) {
      const int par = pipelined ? (bi & 1) ^ (pure == MODEL_IBM ? 1 : 0) : 0;   // panel of this batch: 0 = d_sint_u, 1 = d_sint_i
      // the panels of this batch by role (pipelined: the pure model's panel alternates between the two allocations)
      long long* const panel = par ? h->d_sint_i : h->d_sint_u;
      long long* const pu = pipelined ? (pure == MODEL_UBM ? panel : nullptr) : h->d_sint_u;
      long long* const pi = pipelined ? (pure == MODEL_IBM ? panel : nullptr) : h->d_sint_i;
      // the slices that last used this panel (two batches ago in the batch pipeline, else the previous batch) must have left it
      cudaEvent_t const release = streamed && bi >= (pipelined ? 2 : 1) ? h->ev_done[par] : nullptr;
      if (!run.reuse && (rc = head_pass(h, bi, b0, nb, sl.models, pu, pi, release))) return rc;
      if (streamed) {
        MR_CUDA(h, cudaEventRecord(h->ev_head[par], h->stream));
        MR_CUDA(h, cudaStreamWaitEvent(sl.st[0], h->ev_head[par], 0));
        if (alternating) MR_CUDA(h, cudaStreamWaitEvent(sl.st[1], h->ev_head[par], 0));
      }
      if ((rc = item_slices(h, run, sl, b0, nb, pu, pi))) return rc;
      if (alternating) {   // the batch's slices end on st[0]
        MR_CUDA(h, cudaEventRecord(h->ev_join, sl.st[1]));
        MR_CUDA(h, cudaStreamWaitEvent(sl.st[0], h->ev_join, 0));
      }
      if (run.what == Consumer::AUDIENCE && (rc = audience_columns(h, run, pu, pi, b0, nb, sl.st[0]))) return rc;
      if (streamed) {
        MR_CUDA(h, cudaEventRecord(h->ev_done[par], sl.st[0]));
        if (b0 + batch >= h->U) {   // last batch: the library stream joins the slices (of the last two batches in the batch pipeline)
          MR_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_done[par], 0));
          if (pipelined) MR_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_done[par ^ 1], 0));
        }
      }
      if (run.what != Consumer::DENSE) continue;   // the slices have consumed the batch
    } else if ((rc = user_panels(h, b0, nb, need_ubm, need_ibm))) {
      return rc;
    }
    // the whole batch on the library stream (user space; the dense rows in item space): mask, then the dense rows or the consumers
    long long* const su = need_ubm ? h->d_sint_u : nullptr;
    long long* const si = need_ibm ? h->d_sint_i : nullptr;
    {
      PhaseTimer t(h, run.eval() ? MR_T_OTHER : MR_T_TOPK);   // closed before audience_columns opens its own timer on the same events
      MR_LAUNCH(h, launch_mask_listened(h->d_te_ptr, h->d_te_end, h->d_te_col, b0, nb, su, si, h->spitch, h->stream));
      if (run.ex_ptr) MR_LAUNCH(h, launch_mask_listened(run.ex_ptr, run.ex_ptr + 1, run.ex_col, b0, nb, su, si, h->spitch, h->stream));
      rc = run.what == Consumer::DENSE ? dense_out(h, run.set.bp[0].model, su ? su : si, *run.dense, b0, nb)
                                       : consume_slice(h, run, su, si, h->d_sel, b0, nb, h->stream);
      if (rc) return rc;
    }
    if (run.what == Consumer::AUDIENCE && (rc = audience_columns(h, run, su, si, b0, nb, h->stream))) return rc;
  }
  join.armed = false;
  if (carries) {
    // the carry list of the u32 weighted-count panel must not have overflowed in any batch (it never does on real data: an event
    // needs more than ~64 songs shared between one test user and one train user)
    MR_CUDA(h, cudaStreamSynchronize(h->stream));
    unsigned int worst = 0;
    for (int i = 0; i < n_user_batches; ++i) { h->carry_events += h->h_carry_seen[i]; worst = std::max(worst, h->h_carry_seen[i]); }
    if (worst > h->carry_cap)
      return fail(h, MR_ERR_OOM, "IBM weighted-count carry list overflowed (%u events > capacity %u)", worst, h->carry_cap);
  }
  return MR_OK;
}

int make_blend_params(mr_handle* h, int model, double param, uint64_t seed, long long n_total, BlendParams* bp) {
  memset(bp, 0, sizeof *bp);
  bp->model = model;
  bp->ubm_int_ok = h->ubm_int_ok ? 1 : 0;
  bp->rsd_up = h->d_rsd_up;
  bp->te_end = h->d_te_end; bp->song_off = h->win_lo; bp->stats = h->d_topk_stats;
  if (model < MR_UBM || model > MR_STOCH) return fail(h, MR_ERR_BAD_ARG, "unknown model selector %d", model);
  if (model == MR_LC) { bp->alpha = param; bp->one_minus_alpha = 1 - param; }   // rank1 * alpha + rank2 * (1 - alpha), MR:328
  if (model == MR_AGG) {
    if (!(param >= 0 && param <= 1)) return fail(h, MR_ERR_PARAM_RANGE, "Percentage must be between 0 and 1");   // MR:366-369 (NaN fails too)
    bp->agg_threshold = static_cast<long long>(param * static_cast<double>(n_total));                        // MR:372 .toInt
  }
  if (model == MR_STOCH) {
    if (!(param >= 0 && param <= 1)) return fail(h, MR_ERR_PARAM_RANGE, "Probability must be between 0 and 1");   // MR:434-437
    bp->prob = param; bp->seed = seed;
  }
  return MR_OK;
}

}  // namespace

// =====================================================================================================================
#pragma GCC visibility push(default)
extern "C" {

int mr_create(mr_handle** out, const int* device_ids, int n_devices, unsigned flags) {
  if (!out) return MR_ERR_BAD_ARG;
  *out = nullptr;
  mr_handle* h = new mr_handle();
  *out = h;   // returned even on failure so that mr_last_error works; caller still calls mr_destroy
  if (n_devices != 1 || !device_ids) return fail(h, MR_ERR_BAD_ARG, "n_devices must be 1 (one process per GPU), got %d", n_devices);
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(h, MR_ERR_CUDA, "no CUDA device: %s — libmrscore has no CPU fallback", cudaGetErrorString(e));
  h->device = device_ids[0];
  if (h->device < 0 || h->device >= count) return fail(h, MR_ERR_BAD_ARG, "device id %d out of range (%d devices)", h->device, count);
  MR_CUDA(h, cudaSetDevice(h->device));
  cudaDeviceProp prop;
  MR_CUDA(h, cudaGetDeviceProperties(&prop, h->device));
  if (prop.major != 10) return fail(h, MR_ERR_CUDA, "device %d is sm_%d%d; libmrscore is built for sm_100a only", h->device, prop.major, prop.minor);
  h->num_sms = prop.multiProcessorCount;
  h->flags = flags;
  h->engine = flags & MR_ENGINE_MASK;
  h->space_flag = flags & MR_SPACE_MASK;
  MR_CUDA(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  MR_CUDA(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  MR_CUDA(h, cudaEventCreateWithFlags(&h->ev_slice, cudaEventDisableTiming));
  MR_CUDA(h, cudaStreamCreateWithFlags(&h->pre_stream, cudaStreamNonBlocking));
  MR_CUDA(h, cudaEventCreateWithFlags(&h->ev_pre, cudaEventDisableTiming));
  for (int i = 0; i < kPreExtraStreams; ++i) {
    MR_CUDA(h, cudaStreamCreateWithFlags(&h->pre_extra[i], cudaStreamNonBlocking));
    MR_CUDA(h, cudaEventCreateWithFlags(&h->ev_pre_extra[i], cudaEventDisableTiming));
  }
  {
    int prio_lo = 0, prio_hi = 0;
    MR_CUDA(h, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));   // numerically lower = higher priority; `stream` has the default (lowest)
    MR_CUDA(h, cudaStreamCreateWithPriority(&h->slice_stream, cudaStreamNonBlocking, prio_hi));
    MR_CUDA(h, cudaStreamCreateWithPriority(&h->slice_stream2, cudaStreamNonBlocking, prio_hi));
    MR_CUDA(h, cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) {
      MR_CUDA(h, cudaEventCreateWithFlags(&h->ev_head[i], cudaEventDisableTiming));
      MR_CUDA(h, cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
    }
  }
  MR_CUDA(h, cudaMallocHost(reinterpret_cast<void**>(&h->h_n_ex), sizeof(unsigned int)));
  *h->h_n_ex = 0;
  MR_CUDA(h, cudaEventCreate(&h->ev[0]));
  MR_CUDA(h, cudaEventCreate(&h->ev[1]));
  return MR_OK;
}

void mr_destroy(mr_handle* h) {
  if (!h) return;
  if (h->stream) { cudaSetDevice(h->device); cudaStreamSynchronize(h->stream); }
  if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
  if (h->ev_slice) cudaEventDestroy(h->ev_slice);
  if (h->pre_stream) { cudaStreamSynchronize(h->pre_stream); cudaStreamDestroy(h->pre_stream); }
  if (h->ev_pre) cudaEventDestroy(h->ev_pre);
  for (int i = 0; i < kPreExtraStreams; ++i) {
    if (h->pre_extra[i]) { cudaStreamSynchronize(h->pre_extra[i]); cudaStreamDestroy(h->pre_extra[i]); }
    if (h->ev_pre_extra[i]) cudaEventDestroy(h->ev_pre_extra[i]);
  }
  if (h->slice_stream) { cudaStreamSynchronize(h->slice_stream); cudaStreamDestroy(h->slice_stream); }
  if (h->slice_stream2) { cudaStreamSynchronize(h->slice_stream2); cudaStreamDestroy(h->slice_stream2); }
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  for (int i = 0; i < 2; ++i) { if (h->ev_head[i]) cudaEventDestroy(h->ev_head[i]); if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]); }
  if (h->h_n_ex) cudaFreeHost(h->h_n_ex);
  for (int i = 0; i < mr_handle::SL_N; ++i) if (h->slot_p[i]) cudaFree(h->slot_p[i]);
  for (void* p : h->allocs) cudaFree(p);
  if (h->h_carry_seen) cudaFreeHost(h->h_carry_seen);
  if (h->ev[0]) cudaEventDestroy(h->ev[0]);
  if (h->ev[1]) cudaEventDestroy(h->ev[1]);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

const char* mr_last_error(const mr_handle* h) { return h ? h->err.c_str() : "null handle"; }

int mr_load(mr_handle* h, int n_train, int n_test, int n_songs, const int64_t* tr_rowptr, const int32_t* tr_col,
            const int64_t* te_rowptr, const int32_t* te_col, const int32_t* deg_train, const int32_t* deg_test,
            const int32_t* deg_song_all) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (h->loaded) return fail(h, MR_ERR_STATE, "mr_load called twice on one handle");
  ++h->gen;
  if (n_train <= 0 || n_songs <= 0 || n_test < 0 || !deg_train || !deg_song_all) return fail(h, MR_ERR_BAD_ARG, "bad sizes / null degree arrays");
  int rc = check_csr(h, "train", n_train, n_songs, tr_rowptr, tr_col);
  if (rc) return rc;
  // The fixed-point cosine factors q_k(deg) = rint(2^k / sqrt(deg)) carry a relative rounding error of up to 0.5 * sqrt(deg) / 2^k
  // (DESIGN.md §3); beyond these degrees it would exceed the 1e-5 the scores are specified to (north_star): refuse instead of degrading.
  for (int v = 0; v < n_train; ++v)
    if (deg_train[v] > kMaxDegUbm) return fail(h, MR_ERR_BAD_ARG, "train user %d has %d songs: above %d the 2^24 fixed-point UBM weight leaves the 1e-5 score tolerance", v, deg_train[v], kMaxDegUbm);
  for (int s = 0; s < n_songs; ++s)
    if (deg_song_all[s] > kMaxDegIbm) return fail(h, MR_ERR_BAD_ARG, "song %d has %d listeners: above %d the 2^26 fixed-point IBM weight leaves the 1e-5 score tolerance", s, deg_song_all[s], kMaxDegIbm);
  MR_CUDA(h, cudaSetDevice(h->device));
  const int T = n_train, S = n_songs;
  const long long nnz = tr_rowptr[T];
  h->T = T; h->S = S; h->nnz_tr = nnz;
  // song window: rotate the song ids so that the window becomes the columns [0, n_cols) (see mr_handle)
  if (h->win_hi > S || h->win_lo >= (h->win_hi ? h->win_hi : S)) return fail(h, MR_ERR_BAD_ARG, "song window [%d,%d) outside [0,%d)", h->win_lo, h->win_hi, S);
  if (h->win_hi == 0) h->win_hi = S;
  h->windowed = h->win_lo > 0 || h->win_hi < S;
  h->n_cols = h->win_hi - h->win_lo;
  std::vector<int32_t> rot_col, rot_deg; std::vector<long long> tr_wend;
  if (h->windowed) {
    // the windowed path exists in the item-space formulation with inverted-index counts only
    if (h->engine == MR_ENGINE_TENSOR || h->space_flag == MR_SPACE_USER)
      return fail(h, MR_ERR_BAD_ARG, "a song window needs MR_ENGINE_SPARSE / MR_SPACE_ITEM (or AUTO)");
    h->engine = MR_ENGINE_SPARSE; h->space_flag = MR_SPACE_ITEM;
    const int lo = h->win_lo, up = S - lo;
    rot_col.resize(static_cast<size_t>(std::max<long long>(nnz, 1))); tr_wend.resize(T);
    for (int v = 0; v < T; ++v) {
      const int32_t* b = tr_col + tr_rowptr[v]; const int32_t* e = tr_col + tr_rowptr[v + 1];
      const int32_t* m = std::lower_bound(b, e, lo);             // [b, m) < lo <= [m, e)
      int32_t* o = rot_col.data() + tr_rowptr[v];
      for (const int32_t* p = m; p < e; ++p) *o++ = *p - lo;
      for (const int32_t* p = b; p < m; ++p) *o++ = *p + up;
      tr_wend[v] = tr_rowptr[v] + (std::lower_bound(m, e, h->win_hi) - m);
    }
    rot_deg.resize(S);
    for (int s = 0; s < S; ++s) rot_deg[s < lo ? s + up : s - lo] = deg_song_all[s];
    tr_col = rot_col.data(); deg_song_all = rot_deg.data();
  }
  h->pitchS = round_up(S, 128); h->pitchT = round_up(T, 128);
  h->spitch = round_up(h->n_cols, 32); h->ldg = round_up(S, 32);
  h->deg_song.assign(deg_song_all, deg_song_all + S);
  h->deg_train.assign(deg_train, deg_train + T);
  h->deg_song_train.assign(S, 0);
  for (long long i = 0; i < nnz; ++i) h->deg_song_train[tr_col[i]]++;

  // inverted index (counting sort; listeners of a song ascending because rows are visited in order)
  std::vector<long long> csc_ptr(static_cast<size_t>(S) + 1, 0);
  for (long long i = 0; i < nnz; ++i) csc_ptr[tr_col[i] + 1]++;
  for (int s = 0; s < S; ++s) csc_ptr[s + 1] += csc_ptr[s];
  std::vector<int> csc_idx(static_cast<size_t>(std::max<long long>(nnz, 1)));
  {
    std::vector<long long> fill(csc_ptr.begin(), csc_ptr.end() - 1);
    for (int v = 0; v < T; ++v)
      for (long long i = tr_rowptr[v]; i < tr_rowptr[v + 1]; ++i) csc_idx[fill[tr_col[i]]++] = v;
  }
  // fixed-point cosine factors
  std::vector<uint32_t> qv(T), qd(S);
  std::vector<double> rsd(S);
  for (int v = 0; v < T; ++v) { qv[v] = q_of(deg_train[v], kQScaleUbm); h->max_qv = std::max(h->max_qv, qv[v]); }
  for (int s = 0; s < S; ++s) { qd[s] = q_of(deg_song_all[s], kQScaleIbm); rsd[s] = rs_of(deg_song_all[s], kQInvIbm); }
  h->song_qsum.assign(S, 0);
  for (int s = 0; s < S; ++s)
    for (long long i = csc_ptr[s]; i < csc_ptr[s + 1]; ++i) h->song_qsum[s] += qv[csc_idx[i]];
  // K2 work items: <= kSplitLen listeners each, longest first
  struct Item { int song; long long begin; int len; uint8_t split; };
  std::vector<Item> items;
  for (int s = 0; s < S; ++s) {
    const long long len = csc_ptr[s + 1] - csc_ptr[s];
    for (long long o = 0; o < len; o += kSplitLen)
      items.push_back({s, csc_ptr[s] + o, static_cast<int>(std::min<long long>(kSplitLen, len - o)), static_cast<uint8_t>(len > kSplitLen)});
  }
  std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.len > b.len; });
  h->n_items = static_cast<int>(items.size());
  std::vector<int> it_song(items.size()), it_len(items.size());
  std::vector<long long> it_begin(items.size());
  std::vector<uint8_t> it_split(items.size());
  for (size_t i = 0; i < items.size(); ++i) { it_song[i] = items[i].song; it_begin[i] = items[i].begin; it_len[i] = items[i].len; it_split[i] = items[i].split; }

  std::vector<long long> trp(tr_rowptr, tr_rowptr + T + 1);
  if ((rc = dev_upload(h, &h->d_tr_ptr, trp.data(), trp.size(), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_tr_col, tr_col, static_cast<size_t>(nnz), h->allocs))) return rc;
  if ((rc = dev_alloc(h, &h->d_topk_stats, 4, h->allocs))) return rc;
  MR_CUDA(h, cudaMemsetAsync(h->d_topk_stats, 0, 4 * sizeof(unsigned int), h->stream));
  h->d_tr_end = h->d_tr_ptr + 1;
  if (h->windowed) {
    long long* d_end = nullptr;
    if ((rc = dev_upload(h, &d_end, tr_wend.data(), tr_wend.size(), h->allocs))) return rc;
    h->d_tr_end = d_end;
  }
  if ((rc = dev_upload(h, &h->d_csc_ptr, csc_ptr.data(), csc_ptr.size(), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_csc_idx, csc_idx.data(), static_cast<size_t>(nnz), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_qv, qv.data(), qv.size(), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_qd, qd.data(), qd.size(), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_rsd, rsd.data(), rsd.size(), h->allocs))) return rc;
  {  // rsd rounded UP to fp32: the top-k select bounds IBM scores from above with it
    std::vector<float> up(S);
    for (int s = 0; s < S; ++s) { float f = static_cast<float>(rsd[s]); if (static_cast<double>(f) < rsd[s]) f = std::nextafterf(f, INFINITY); up[s] = f; }
    if ((rc = dev_upload(h, &h->d_rsd_up, up.data(), up.size(), h->allocs))) return rc;
    MR_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  if ((rc = dev_upload(h, &h->d_item_song, it_song.data(), it_song.size(), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_item_begin, it_begin.data(), it_begin.size(), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_item_len, it_len.data(), it_len.size(), h->allocs))) return rc;
  if ((rc = dev_upload(h, &h->d_item_split, it_split.data(), it_split.size(), h->allocs))) return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));   // host staging vectors go out of scope below

  // engine choice: dense operands A_tr (T x pitchS) and A_tr^T (S x pitchT) must fit comfortably
  h->dense_bytes = static_cast<size_t>(T) * h->pitchS + static_cast<size_t>(S) * h->pitchT;
  if (h->engine == MR_ENGINE_AUTO) {
    size_t free_b = 0, total_b = 0;
    MR_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    h->engine = (h->dense_bytes < free_b / 3) ? MR_ENGINE_TENSOR : MR_ENGINE_SPARSE;
  }
  if (h->engine == MR_ENGINE_TENSOR) {
    if ((rc = dev_alloc(h, &h->d_Atr, static_cast<size_t>(T) * h->pitchS, h->allocs))) return rc;
    if ((rc = dev_alloc(h, &h->d_AtrT, static_cast<size_t>(S) * h->pitchT, h->allocs))) return rc;
    if ((rc = dev_alloc(h, &h->d_Ate, static_cast<size_t>(kUserBatch) * h->pitchS, h->allocs))) return rc;
    PhaseTimer t(h, MR_T_EXPAND);
    MR_LAUNCH(h, launch_expand_rows(h->d_tr_ptr, h->d_tr_col, nullptr, 0, T, T, h->pitchS, h->d_Atr, h->stream));
    MR_LAUNCH(h, launch_expand_rows(h->d_csc_ptr, h->d_csc_idx, nullptr, 0, S, S, h->pitchT, h->d_AtrT, h->stream));
  } else {
    h->dense_bytes = 0;
  }
  // per-batch workspaces
  if ((rc = dev_alloc(h, &h->d_ct, static_cast<size_t>(T) * kUserBatch, h->allocs))) return rc;
  if (h->engine == MR_ENGINE_SPARSE) {
    if ((rc = dev_alloc(h, &h->d_wi, static_cast<size_t>(T) * kUserBatch, h->allocs))) return rc;
    // test aid: a small carry list lets a test reach its overflow error, which real data cannot (it needs ~10^6 wrapping pairs)
    if (const char* e = getenv("MRSCORE_CARRY_CAP")) h->carry_cap = static_cast<unsigned int>(std::max(1LL, std::min<long long>(atoll(e), 1LL << 20)));
    if ((rc = dev_alloc(h, &h->d_carry_count, 1, h->allocs))) return rc;
    if ((rc = dev_alloc(h, &h->d_carry_events, h->carry_cap, h->allocs))) return rc;
  }
  if (const char* e = getenv("MRSCORE_ITEM_BATCH")) h->item_batch_cap = std::max(128, atoi(e));   // developer override of MR_OPT_ITEM_BATCH
  if (const char* e = getenv("MRSCORE_HEAD_WORDS_U")) { const int w = atoi(e); if (w == 1 || w == 2 || w == 4) h->head_words_u = w; }
  if (const char* e = getenv("MRSCORE_HEAD_WORDS_I")) { const int w = atoi(e); if (w == 1 || w == 2 || w == 4) h->head_words_i = w; }
  if (const char* e = getenv("MRSCORE_HEAD_THREADS")) { const int t = atoi(e); if (t == 32 || t == 64 || t == 128 || t == 256) h->head_threads = t; }
  h->n_groups = h->num_sms * std::min(32, kHeadCtasPerSm * 256 / h->head_threads);   // one wave of resident CTAs = one song tile for the whole batch
  if (const char* e = getenv("MRSCORE_HEAD_GROUPS")) h->n_groups = std::max(1, atoi(e));   // test aid: few groups -> several users per group on small shards
  h->sel_pitch = (h->n_cols + 63) / 64;
  // item-space head: songs with enough train listeners that a dense precomputed row beats expanding them per test user
  {
    long long min_deg = std::max<long long>(2, S / 6000);   // below ~64 listeners expanding a song on the fly is cheaper than streaming its row
    if (h->opt_head_min_deg > 0) min_deg = h->opt_head_min_deg;
    if (const char* e = getenv("MRSCORE_HEAD_MIN_DEG")) min_deg = std::max(1LL, atoll(e));
    size_t free_b = 0, total_b = 0;
    MR_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    const long long max_rows = static_cast<long long>((free_b / 100 * 47) / (static_cast<size_t>(h->spitch) * 6));   // packed rows: 6 B per entry; the rest holds the Sint panels
    std::vector<int> order(S);
    for (int s = 0; s < S; ++s) order[s] = s;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return csc_ptr[a + 1] - csc_ptr[a] > csc_ptr[b + 1] - csc_ptr[b]; });
    h->head_index.assign(S, -1);
    std::vector<int> head_song; std::vector<long long> lst_ptr(1, 0);
    for (int r = 0; r < S && r < max_rows; ++r) {
      const int s = order[r]; const long long d = csc_ptr[s + 1] - csc_ptr[s];
      if (d < min_deg) break;
      h->head_index[s] = static_cast<int>(head_song.size());
      head_song.push_back(s); lst_ptr.push_back(lst_ptr.back() + d);
    }
    h->n_head = static_cast<int>(head_song.size());
    // rows from n_head_staged on can be built in place: no entry of theirs can overflow 16 / 32 bits (ensure_head_rows)
    h->n_head_staged = h->n_head;
    while (h->n_head_staged > 0) {
      const int s = head_song[h->n_head_staged - 1];
      if (h->song_qsum[s] >= (1ULL << 32) || csc_ptr[s + 1] - csc_ptr[s] >= 65536) break;
      --h->n_head_staged;
    }
    if (getenv("MRSCORE_PRECOMPUTE_STAGE_ALL")) h->n_head_staged = h->n_head;
    h->song_info.resize(S);
    for (int s = 0; s < S; ++s) h->song_info[s] = {h->head_index[s], h->head_index[s] >= 0 ? qd[s] : static_cast<uint32_t>(h->deg_song_train[s])};
    h->max_qsum = *std::max_element(h->song_qsum.begin(), h->song_qsum.end());
    static_assert(sizeof(mr_handle::SongInfo) == sizeof(int2), "SongInfo is uploaded as int2");
    if ((rc = dev_upload(h, &h->d_song_info, reinterpret_cast<const int2*>(h->song_info.data()), h->song_info.size(), h->allocs))) return rc;
    if ((rc = dev_upload(h, &h->d_head_song, head_song.data(), head_song.size(), h->allocs))) return rc;
    if ((rc = dev_upload(h, &h->d_head_lst_ptr, lst_ptr.data(), lst_ptr.size(), h->allocs))) return rc;
  }
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  h->loaded = true; h->passes = 0;
  if (n_test > 0) return mr_set_test_users(h, n_test, te_rowptr, te_col, deg_test, 0, 0);
  return MR_OK;
}

int mr_set_test_users(mr_handle* h, int n_test, const int64_t* te_rowptr, const int32_t* te_col, const int32_t* deg_test,
                      int64_t pair_index_base, int64_t n_pairs_total) {
  if (!h || !h->loaded) return fail(h, MR_ERR_STATE, "mr_load has not succeeded on this handle");
  if (n_test <= 0 || !deg_test) return fail(h, MR_ERR_BAD_ARG, "n_test must be > 0 and deg_test non-null");
  int rc = check_csr(h, "test", n_test, h->S, te_rowptr, te_col);
  if (rc) return rc;
  for (int u = 0; u < n_test; ++u)
    if (te_rowptr[u + 1] - te_rowptr[u] > 65535) return fail(h, MR_ERR_BAD_ARG, "test user %d has more than 65535 visible songs (u16 count panel)", u);
  const bool dbg = getenv("MRSCORE_DEBUG_TIMING") != nullptr;
  auto t_dbg = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!dbg) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[mrscore] set_test_users: %s %.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_dbg).count());
    t_dbg = now;
  };
  MR_CUDA(h, cudaSetDevice(h->device));
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  lap("check_csr + sync");
  h->have_test = false; h->have_topk = false; h->out_k = 0; h->multi_n = 0; h->flt_on = false; ++h->gen;
  const int U = n_test; const long long nnz = te_rowptr[U];
  h->U = U; h->nnz_te = nnz;
  h->deg_test.assign(deg_test, deg_test + U); h->simu_squ_ok = false;
  h->h_te_ptr.assign(te_rowptr, te_rowptr + U + 1);
  if (h->windowed) h->h_te_col.resize(static_cast<size_t>(nnz)); else h->h_te_col.assign(te_col, te_col + nnz);   // a window rewrites every row below
  std::vector<double> rsa(U);
  std::vector<long long> pair_base(static_cast<size_t>(U) + 1);
  pair_base[0] = pair_index_base;
  parallel_rows(U, [&](int lo, int hi) { for (int u = lo; u < hi; ++u) rsa[u] = rs_of(deg_test[u], kQInvUbm); });
  for (int u = 0; u < U; ++u) pair_base[u + 1] = pair_base[u] + (h->S - (te_rowptr[u + 1] - te_rowptr[u]));   // unlistened songs of u (MR:109)
  h->pair_index_base = pair_index_base;
  h->n_pairs_total = n_pairs_total > 0 ? n_pairs_total : pair_base[U] - pair_index_base;
  std::vector<long long> te_wend;
  if (h->windowed) {
    // rotate the rows like the train rows (mr_load); the pair index of column c of user u in MAIN:57-59 order is
    // pair_base[u] + (c + win_lo) - (listened songs below win_lo) - (listened songs of the window below c): fold the constants into pair_base
    const int lo = h->win_lo, up = h->S - lo;
    te_wend.resize(U);
    int32_t* const rot = h->h_te_col.data();
    const int win_hi = h->win_hi;
    parallel_rows(U, [&](int u_lo, int u_hi) {
      for (int u = u_lo; u < u_hi; ++u) {
        const int32_t* b = te_col + te_rowptr[u]; const int32_t* e = te_col + te_rowptr[u + 1];
        const int32_t* m = std::lower_bound(b, e, lo);
        int32_t* o = rot + te_rowptr[u];
        for (const int32_t* p = m; p < e; ++p) *o++ = *p - lo;
        for (const int32_t* p = b; p < m; ++p) *o++ = *p + up;
        te_wend[u] = te_rowptr[u] + (std::lower_bound(m, e, win_hi) - m);
        pair_base[u] += lo - (m - b);
      }
    });
    te_col = h->h_te_col.data();
  }
  // per batch: sorted union of the visible songs (the Gram rows the batch needs) and each entry's row index in it — only the
  // tensor engine's user-space IBM path consumes them
  const int n_batches = (U + kUserBatch - 1) / kUserBatch;
  std::vector<int> rows_all; std::vector<int> grow(h->engine == MR_ENGINE_TENSOR ? static_cast<size_t>(std::max<long long>(nnz, 1)) : 1);
  h->batch_row_off.assign(static_cast<size_t>(n_batches) + 1, 0);
  h->max_batch_rows = 0;
  if (h->engine == MR_ENGINE_TENSOR) {
    for (int b = 0; b < n_batches; ++b) {
      const long long e0 = te_rowptr[b * kUserBatch], e1 = te_rowptr[std::min(U, (b + 1) * kUserBatch)];
      std::vector<int> uni(te_col + e0, te_col + e1);
      std::sort(uni.begin(), uni.end());
      uni.erase(std::unique(uni.begin(), uni.end()), uni.end());
      for (long long e = e0; e < e1; ++e) grow[e] = static_cast<int>(std::lower_bound(uni.begin(), uni.end(), te_col[e]) - uni.begin());
      rows_all.insert(rows_all.end(), uni.begin(), uni.end());
      h->batch_row_off[b + 1] = static_cast<long long>(rows_all.size());
      h->max_batch_rows = std::max<int>(h->max_batch_rows, static_cast<int>(uni.size()));
    }
  }
  lap("host arrays");
  if ((rc = slot_upload(h, mr_handle::SL_TE_PTR, &h->d_te_ptr, h->h_te_ptr.data(), h->h_te_ptr.size()))) return rc;
  h->d_te_end = h->d_te_ptr + 1;
  if (h->windowed) {
    long long* d_end = nullptr;
    if ((rc = slot_upload(h, mr_handle::SL_TE_END, &d_end, te_wend.data(), te_wend.size()))) return rc;
    h->d_te_end = d_end;
  }
  if ((rc = slot_upload(h, mr_handle::SL_TE_COL, &h->d_te_col, h->h_te_col.data(), static_cast<size_t>(nnz)))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_TE_GROW, &h->d_te_grow, grow.data(), grow.size()))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_RSA, &h->d_rsa, rsa.data(), rsa.size()))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_PAIR_BASE, &h->d_pair_base, pair_base.data(), pair_base.size()))) return rc;
  if ((rc = slot_upload(h, mr_handle::SL_ROWS, &h->d_rows, rows_all.data(), rows_all.size()))) return rc;
  lap("uploads 1");
  {  // item-space work lists (k7_testlists.cu): per user the precomputed head rows it sums, and its tail songs expanded on the fly
    std::vector<long long> hu_ptr(static_cast<size_t>(U) + 1, 0);
    h->h_tu_ptr.assign(static_cast<size_t>(U) + 1, 0);
    const size_t n1 = static_cast<size_t>(nnz) + 1;
    int *d_flag = nullptr, *d_head_pos = nullptr; long long *d_deg = nullptr, *d_lsum = nullptr, *d_tu_ptr = nullptr; char* d_tmp = nullptr;
    const size_t tmp_bytes = test_lists_temp_bytes(nnz);
    if ((rc = slot_alloc(h, mr_handle::SL_L_FLAG, &d_flag, n1)) || (rc = slot_alloc(h, mr_handle::SL_L_HEADPOS, &d_head_pos, n1)) ||
        (rc = slot_alloc(h, mr_handle::SL_L_DEG, &d_deg, n1)) || (rc = slot_alloc(h, mr_handle::SL_L_LSUM, &d_lsum, n1)) ||
        (rc = slot_alloc(h, mr_handle::SL_L_TMP, &d_tmp, tmp_bytes)) || (rc = slot_alloc(h, mr_handle::SL_TU_PTR, &d_tu_ptr, hu_ptr.size())) ||
        (rc = slot_alloc(h, mr_handle::SL_HU_PTR, &h->d_hu_ptr, hu_ptr.size())) || (rc = slot_alloc(h, mr_handle::SL_HU_ROW, &h->d_hu_row, n1)) ||
        (rc = slot_alloc(h, mr_handle::SL_HU_SONG, &h->d_hu_song, n1)) || (rc = slot_alloc(h, mr_handle::SL_HU_Q, &h->d_hu_q, n1)) ||
        (rc = slot_alloc(h, mr_handle::SL_TU_USER, &h->d_tu_user, n1)) || (rc = slot_alloc(h, mr_handle::SL_TU_SONG, &h->d_tu_song, n1)) ||
        (rc = slot_alloc(h, mr_handle::SL_TU_LPTR, &h->d_tu_lptr, n1)))
      return rc;
    MR_LAUNCH(h, launch_build_test_lists(h->d_te_ptr, h->d_te_col, U, nnz, h->d_song_info, d_flag, d_head_pos, d_deg, d_lsum, d_tmp, tmp_bytes, h->d_hu_row,
                                         h->d_hu_song, h->d_hu_q, h->d_hu_ptr, h->d_tu_user, h->d_tu_song, h->d_tu_lptr, d_tu_ptr, h->stream));
    MR_CUDA(h, cudaMemcpyAsync(hu_ptr.data(), h->d_hu_ptr, hu_ptr.size() * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    MR_CUDA(h, cudaMemcpyAsync(h->h_tu_ptr.data(), d_tu_ptr, h->h_tu_ptr.size() * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    long long longest = 0;   // overlaps the device work
    for (int u = 0; u < U; ++u) longest = std::max<long long>(longest, te_rowptr[u + 1] - te_rowptr[u]);
    // Sint_u[u][s] = sum_{j in I_u} Gq[j][s] <= sum_{j in I_u} qsum[j]: below 2^52 the top-k select may rank the UBM integers.  The cheap
    // bound (longest row x largest qsum) decides almost always; otherwise the exact per-user sums do.
    h->ubm_int_ok = static_cast<long double>(h->max_qsum) * static_cast<long double>(longest) < 4503599627370496.0L;
    if (!h->ubm_int_ok) {
      unsigned long long worst = 0;
      for (int u = 0; u < U; ++u) {
        unsigned long long bound = 0;
        for (long long e = te_rowptr[u]; e < te_rowptr[u + 1]; ++e) bound += h->song_qsum[te_col[e]];
        worst = std::max(worst, bound);
      }
      h->ubm_int_ok = worst < (1ULL << 52);
    }
    // test aid: the fp64 UBM select, which data reaches only past ~2^28 train listens, on any shard (it must give the same lists)
    if (getenv("MRSCORE_UBM_FP64_SELECT")) h->ubm_int_ok = false;
    MR_CUDA(h, cudaStreamSynchronize(h->stream));
    h->n_head_entries = hu_ptr[U]; h->n_tail_entries = h->h_tu_ptr[U];
    h->h_tu_lptr.resize(static_cast<size_t>(h->n_tail_entries) + 1);
    MR_CUDA(h, cudaMemcpyAsync(h->h_tu_lptr.data(), h->d_tu_lptr, h->h_tu_lptr.size() * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    lap("device work lists");
    h->space = h->space_flag == MR_SPACE_AUTO ? (U >= 1024 ? MR_SPACE_ITEM : MR_SPACE_USER) : h->space_flag;
    if ((rc = plan_item_batches(h, hu_ptr))) return rc;
    lap("plan_item_batches");
  }
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  h->have_test = true;
  return MR_OK;
}

static int require_loaded(mr_handle* h) {
  if (!h || !h->loaded) return fail(h, MR_ERR_STATE, "mr_load has not succeeded on this handle");
  cudaError_t e = cudaSetDevice(h->device);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  return MR_OK;
}

static int require_test(mr_handle* h) {
  if (!h) return MR_ERR_STATE;
  if (!h->loaded || !h->have_test) return fail(h, MR_ERR_STATE, "no data loaded (mr_load / mr_set_test_users)");
  return require_loaded(h);
}

int mr_gram_rows_device(mr_handle* h, int s0, int s1, int32_t** dev_out, int64_t* ld) {
  int rc = require_loaded(h);
  if (rc) return rc;
  if (!dev_out || !ld) return fail(h, MR_ERR_BAD_ARG, "null output");
  if (h->windowed) return fail(h, MR_ERR_STATE, "Gram rows are not available on a handle with a song window (its song ids are rotated)");
  if (s0 < 0 || s1 > h->S || s0 >= s1) return fail(h, MR_ERR_BAD_ARG, "song range [%d,%d) outside [0,%d)", s0, s1, h->S);
  const int n = s1 - s0;
  if ((rc = ensure_gram_ws(h, n))) return rc;
  int* d_ids = nullptr;
  if ((rc = slot_alloc(h, mr_handle::SL_GRAM_IDS, &d_ids, static_cast<size_t>(n)))) return rc;
  iota_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(d_ids, s0, n);
  h->launches++;
  if ((rc = gram_rows(h, d_ids, n))) return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  *dev_out = h->d_g; *ld = h->ldg;
  return MR_OK;
}

int mr_peer_alloc(mr_handle* h, uint64_t bytes, void** dev_ptr, unsigned char* handle_out_64) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (!dev_ptr || !handle_out_64 || bytes == 0) return fail(h, MR_ERR_BAD_ARG, "null output / zero size");
  MR_CUDA(h, cudaSetDevice(h->device));
  void* p = nullptr;
  MR_CUDA(h, cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t hd;
  cudaError_t e = cudaIpcGetMemHandle(&hd, p);
  if (e != cudaSuccess) { cudaFree(p); return fail(h, MR_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  memcpy(handle_out_64, &hd, 64);
  MR_CUDA(h, cudaMemsetAsync(p, 0, bytes, h->stream));
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  h->allocs.push_back(p);
  h->dev_bytes += bytes;
  *dev_ptr = p;
  return MR_OK;
}

int mr_peer_open(mr_handle* h, const unsigned char* handle_64, void** dev_ptr) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (!dev_ptr || !handle_64) return fail(h, MR_ERR_BAD_ARG, "null argument");
  MR_CUDA(h, cudaSetDevice(h->device));
  cudaIpcMemHandle_t hd;
  memcpy(&hd, handle_64, 64);
  MR_CUDA(h, cudaIpcOpenMemHandle(dev_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
  return MR_OK;
}

int mr_peer_close(mr_handle* h, void* dev_ptr) {
  if (!h || !h->stream) return MR_ERR_STATE;
  MR_CUDA(h, cudaSetDevice(h->device));
  MR_CUDA(h, cudaIpcCloseMemHandle(dev_ptr));
  return MR_OK;
}

static int gram_rows_scatter_impl(mr_handle* h, int s0, int s1, void* const* slot_ptrs, int n_owners, int rows_per_owner, int64_t ld, bool sync);
int mr_gram_rows_scatter(mr_handle* h, int s0, int s1, void* const* slot_ptrs, int n_owners, int rows_per_owner, int64_t ld) {
  return gram_rows_scatter_impl(h, s0, s1, slot_ptrs, n_owners, rows_per_owner, ld, true);
}
int mr_gram_rows_scatter_async(mr_handle* h, int s0, int s1, void* const* slot_ptrs, int n_owners, int rows_per_owner, int64_t ld) {
  return gram_rows_scatter_impl(h, s0, s1, slot_ptrs, n_owners, rows_per_owner, ld, false);
}

int mr_peer_signal(mr_handle* h, void* const* flag_ptrs, int n, uint64_t value) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (!flag_ptrs || n < 1 || n > 8) return fail(h, MR_ERR_BAD_ARG, "1..8 flag pointers expected");
  MR_CUDA(h, cudaSetDevice(h->device));
  PeerFlags f{};
  for (int i = 0; i < n; ++i) f.p[i] = static_cast<unsigned long long*>(flag_ptrs[i]);
  MR_LAUNCH(h, launch_peer_signal(f, n, value, h->stream));
  return MR_OK;
}

int mr_peer_wait(mr_handle* h, const void* flags, int n, uint64_t value) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (!flags || n < 1 || n > 8) return fail(h, MR_ERR_BAD_ARG, "1..8 flags expected");
  MR_CUDA(h, cudaSetDevice(h->device));
  MR_LAUNCH(h, launch_peer_wait(static_cast<const unsigned long long*>(flags), n, value, h->stream));
  return MR_OK;
}

int mr_sync(mr_handle* h) {
  if (!h || !h->stream) return MR_ERR_STATE;
  MR_CUDA(h, cudaSetDevice(h->device));
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  return MR_OK;
}

static int gram_rows_scatter_impl(mr_handle* h, int s0, int s1, void* const* slot_ptrs, int n_owners, int rows_per_owner, int64_t ld, bool sync) {
  int rc = require_loaded(h);
  if (rc) return rc;
  if (h->engine != MR_ENGINE_TENSOR) return fail(h, MR_ERR_STATE, "mr_gram_rows_scatter needs the tensor engine (the scatter is the GEMM epilogue)");
  if (h->windowed) return fail(h, MR_ERR_STATE, "Gram rows are not available on a handle with a song window (its song ids are rotated)");
  if (s0 < 0 || s1 > h->S || s0 >= s1) return fail(h, MR_ERR_BAD_ARG, "song range [%d,%d) outside [0,%d)", s0, s1, h->S);
  const int n = s1 - s0;
  if (!slot_ptrs || n_owners < 1 || n_owners > 8 || rows_per_owner < 1 || static_cast<long long>(n_owners) * rows_per_owner < n || ld < h->S)
    return fail(h, MR_ERR_BAD_ARG, "bad slot table (owners %d, rows per owner %d, ld %lld)", n_owners, rows_per_owner, static_cast<long long>(ld));
  const int rows_pad = static_cast<int>(round_up(n, 128));
  if ((rc = slot_alloc(h, mr_handle::SL_GRAM_A, &h->d_Aj, static_cast<size_t>(rows_pad) * h->pitchT, true))) return rc;   // no G: the GEMM scatters
  int* d_ids = nullptr;
  if ((rc = slot_alloc(h, mr_handle::SL_GRAM_IDS, &d_ids, static_cast<size_t>(n)))) return rc;
  iota_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(d_ids, s0, n);
  h->launches++;
  {
    PhaseTimer t(h, MR_T_EXPAND);
    MR_LAUNCH(h, launch_expand_rows(h->d_csc_ptr, h->d_csc_idx, d_ids, 0, n, rows_pad, h->pitchT, h->d_Aj, h->stream));
  }
  int32_t* slots[8];
  for (int i = 0; i < n_owners; ++i) slots[i] = static_cast<int32_t*>(slot_ptrs[i]);
  PhaseTimer t(h, MR_T_COUNT);
  MR_LAUNCH(h, launch_count_gemm(h->d_Aj, rows_pad, h->d_AtrT, h->S, h->pitchT, n, h->S, EPI_I32_SCATTER, nullptr, ld, h->num_sms, h->stream, 0, 0,
                                 slots, n_owners, rows_per_owner));
  if (sync) MR_CUDA(h, cudaStreamSynchronize(h->stream));
  return MR_OK;
}

// ---- similar songs and similar users (DESIGN.md §4.7, §4.8, k8_similar.cu).  Both use only the train replica (and the test shard's rows)
// and their own slots: the score panels, the select plane, the head rows, the top-k blocks and gen stay as they are; the count rows of the
// long path go to the Gram workspace (ensure_gram_ws).
static constexpr int kSimClassCap[] = {256, 1024, 4096, kSimShortMax};   // short-path launches by E_q: 12 * cap bytes of shared memory per CTA
static constexpr size_t kSimWindowBytes = 256ULL << 20;   // short-path results: the query list in windows of rows whose block fits this
static constexpr size_t kSimMargin = 512ULL << 20;        // device memory the long path's chunk sizing leaves free

// One query kind of the similar-items driver: the two-level lists and sqrt tables of the kernels, the count rows of the long path and
// the counters of mr_get_info.
struct SimKind {
  const char* name;   // "similar songs" / "similar users", for messages
  SimLists lists;
  CountRows counts;
  long long *short_rows, *long_rows;
};

// the sqrt of n degrees, correctly rounded on the device, into out (the degrees pass through the SL_SIM_IDS slot)
static int sqrt_table(mr_handle* h, const int32_t* deg, int n, double* out) {
  int* d_deg = nullptr;
  const int rc = slot_upload(h, mr_handle::SL_SIM_IDS, &d_deg, deg, static_cast<size_t>(n));
  if (rc) return rc;
  MR_LAUNCH(h, launch_sqrt_deg(d_deg, n, out, h->stream));
  return MR_OK;
}

// Rows per chunk of count rows of kind cr for n_rows rows (the long rows of similar_lists, the keys of mr_explain), each row needing
// row_bytes of its own besides: up to 1024 rows, as many as the Gram workspace holds already or as fit in the free device memory less
// kSimMargin, in multiples of 128; MRSCORE_SIM_CHUNK caps it (test aid: force a multi-chunk run).  Sizes the workspace for the chunk.
static int count_chunk(mr_handle* h, const CountRows& cr, size_t row_bytes, int n_rows, const char* name, int* out) {
  const bool tensor = h->engine == MR_ENGINE_TENSOR;
  const size_t ws_row = static_cast<size_t>(cr.ld) * sizeof(int32_t) + (tensor ? static_cast<size_t>(cr.pitch) : 0);
  long long have = static_cast<long long>(h->slot_cap[mr_handle::SL_GRAM_G] / (static_cast<size_t>(cr.ld) * sizeof(int32_t)));   // rows the workspace holds already
  if (tensor) have = std::min<long long>(have, static_cast<long long>(h->slot_cap[mr_handle::SL_GRAM_A] / cr.pitch));
  size_t free_b = 0, total_b = 0;
  MR_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
  const long long grow = static_cast<long long>((free_b > kSimMargin ? free_b - kSimMargin : 0) / (ws_row + row_bytes)) / 128 * 128;
  long long chunk = std::min<long long>(1024, std::max(have, grow));
  if (const char* e = getenv("MRSCORE_SIM_CHUNK")) chunk = std::min(chunk, std::max(1LL, atoll(e)));
  chunk = std::min<long long>(chunk, n_rows);
  if (chunk < 1)
    return fail(h, MR_ERR_OOM, "%s: one chunk of 128 count rows needs %zu bytes of device memory beyond a %zu-byte margin, %zu are free",
                name, 128 * (ws_row + row_bytes), kSimMargin, free_b);
  *out = static_cast<int>(chunk);
  return ensure_gram_ws(h, *out, cr.ld, cr.pitch);
}

// sqrt(d_s) of every song (similar songs, IBM explanations), once per handle
static int ensure_sqrt_songs(mr_handle* h) {
  if (h->d_sim_sqd) return MR_OK;
  double* sq = nullptr;
  int rc;
  if ((rc = dev_alloc(h, &sq, static_cast<size_t>(h->S), h->allocs)) || (rc = sqrt_table(h, h->deg_song.data(), h->S, sq))) return rc;
  h->d_sim_sqd = sq;
  return MR_OK;
}

// sqrt(|I_v|) of the train users, once per handle, and sqrt(|I_u|) of the test users, once per shard (similar users, UBM explanations)
static int ensure_sqrt_users(mr_handle* h) {
  int rc;
  if (!h->d_simu_sqt) {
    double* sq = nullptr;
    if ((rc = dev_alloc(h, &sq, static_cast<size_t>(h->T), h->allocs)) || (rc = sqrt_table(h, h->deg_train.data(), h->T, sq))) return rc;
    h->d_simu_sqt = sq;
  }
  if (!h->simu_squ_ok) {
    if ((rc = slot_alloc(h, mr_handle::SL_SIM_SQU, &h->d_simu_squ, static_cast<size_t>(h->U))) ||
        (rc = sqrt_table(h, h->deg_test.data(), h->U, h->d_simu_squ))) return rc;
    h->simu_squ_ok = true;
  }
  return MR_OK;
}

// The query ids are checked by the caller.  E_q of every query is read back to split the queries into short and long rows.
static int similar_lists(mr_handle* h, const SimKind& kind, const int32_t* ids, int n, int k, int32_t* out_song, double* out_score, int32_t* out_len) {
  cudaStream_t st = h->stream;
  int rc;
  int* d_ids = nullptr;
  long long* d_ev = nullptr;
  if ((rc = slot_upload(h, mr_handle::SL_SIM_IDS, &d_ids, ids, static_cast<size_t>(n))) ||
      (rc = slot_alloc(h, mr_handle::SL_SIM_EV, &d_ev, static_cast<size_t>(n)))) return rc;
  std::vector<long long> ev(static_cast<size_t>(n));
  {
    PhaseTimer t(h, MR_T_OTHER);
    MR_LAUNCH(h, launch_sim_events(d_ids, n, kind.lists, d_ev, st));
  }
  MR_CUDA(h, cudaMemcpyAsync(ev.data(), d_ev, static_cast<size_t>(n) * sizeof(long long), cudaMemcpyDeviceToHost, st));
  MR_CUDA(h, cudaStreamSynchronize(st));
  long long short_max = kSimShortMax;   // MRSCORE_SIM_SHORT_MAX can lower the limit (0: every row long), never raise it
  if (const char* e = getenv("MRSCORE_SIM_SHORT_MAX")) short_max = std::max(0LL, std::min<long long>(kSimShortMax, atoll(e)));

  // short rows: the query list in windows of W rows; one launch per size class; the window's block goes to out rows [r0, r1) in one copy.
  // The block's rows of long queries hold nothing meaningful; the long path below overwrites them on the host.
  constexpr int kClasses = static_cast<int>(sizeof kSimClassCap / sizeof kSimClassCap[0]);
  const size_t row_bytes = static_cast<size_t>(k) * 12 + 4;
  size_t w_rows = std::min<size_t>(static_cast<size_t>(n), kSimWindowBytes / row_bytes);
  if (const char* e = getenv("MRSCORE_SIM_WINDOW")) w_rows = std::min<size_t>(w_rows, static_cast<size_t>(std::max(1LL, atoll(e))));   // test aid: many windows
  const int W = static_cast<int>(std::max<size_t>(1, w_rows));
  std::vector<int> long_rows;
  {
    const TopkBlock blk(W, k);
    char* base = nullptr; int* d_q = nullptr;
    if ((rc = slot_alloc(h, mr_handle::SL_SIM_OUT, &base, blk.bytes)) || (rc = slot_alloc(h, mr_handle::SL_SIM_Q, &d_q, 2 * static_cast<size_t>(W)))) return rc;
    const TopkOut dev = blk.at(base);
    std::vector<int> q(2 * static_cast<size_t>(W));   // query ids [0, W), window rows [W, 2W), grouped by class
    for (int r0 = 0; r0 < n; r0 += W) {
      const int r1 = std::min(n, r0 + W);
      int cnt[kClasses] = {}, off[kClasses + 1] = {};
      auto cls = [&](long long e) { int c = 0; while (c < kClasses - 1 && kSimClassCap[c] < e) ++c; return c; };
      for (int r = r0; r < r1; ++r)
        if (ev[r] <= short_max) ++cnt[cls(ev[r])]; else long_rows.push_back(r);
      for (int c = 0; c < kClasses; ++c) off[c + 1] = off[c] + cnt[c];
      const int n_short = off[kClasses];
      if (n_short == 0) continue;
      int fill[kClasses];
      std::copy(off, off + kClasses, fill);
      for (int r = r0; r < r1; ++r)
        if (ev[r] <= short_max) { const int p = fill[cls(ev[r])]++; q[p] = ids[r]; q[W + p] = r - r0; }
      MR_CUDA(h, cudaMemcpyAsync(d_q, q.data(), static_cast<size_t>(n_short) * sizeof(int), cudaMemcpyHostToDevice, st));
      MR_CUDA(h, cudaMemcpyAsync(d_q + W, q.data() + W, static_cast<size_t>(n_short) * sizeof(int), cudaMemcpyHostToDevice, st));
      {
        PhaseTimer t(h, MR_T_OTHER);
        for (int c = 0; c < kClasses; ++c)
          if (cnt[c]) MR_LAUNCH(h, launch_similar_short(d_q + off[c], d_q + W + off[c], cnt[c], kSimClassCap[c], kind.lists, k, dev.song, dev.score,
                                                        dev.len, st));
      }
      const size_t o = static_cast<size_t>(r0) * k;
      if ((rc = copy_topk(h, TopkOut{out_song + o, out_score + o, out_len + r0}, dev, k, 0, r1 - r0, st))) return rc;
      *kind.short_rows += n_short;
    }
  }
  // long rows: exact count rows in chunks (count GEMM or inverted-index counts), the select over each chunk, then the rows to the caller
  if (!long_rows.empty()) {
    const int n_long = static_cast<int>(long_rows.size());
    const CountRows& cr = kind.counts;
    int C = 0;
    if ((rc = count_chunk(h, cr, row_bytes, n_long, kind.name, &C))) return rc;
    const TopkBlock blk(C, k);
    char* base = nullptr; int* d_rows = nullptr;
    if ((rc = slot_alloc(h, mr_handle::SL_SIM_LOUT, &base, blk.bytes)) || (rc = slot_alloc(h, mr_handle::SL_SIM_LIDS, &d_rows, static_cast<size_t>(C)))) return rc;
    const TopkOut dev = blk.at(base);
    std::vector<int> rows(static_cast<size_t>(C));
    std::vector<int32_t> hs(static_cast<size_t>(C) * k), hl(static_cast<size_t>(C));
    std::vector<double> hv(static_cast<size_t>(C) * k);
    for (int c0 = 0; c0 < n_long; c0 += C) {
      const int nc = std::min(C, n_long - c0);
      for (int j = 0; j < nc; ++j) rows[j] = ids[long_rows[c0 + j]];
      MR_CUDA(h, cudaMemcpyAsync(d_rows, rows.data(), static_cast<size_t>(nc) * sizeof(int), cudaMemcpyHostToDevice, st));
      if ((rc = count_rows(h, cr, d_rows, nc))) return rc;
      {
        PhaseTimer t(h, MR_T_TOPK);
        MR_LAUNCH(h, launch_similar_rows(d_rows, nc, h->d_g, cr.ld, cr.n_cols, kind.lists, k, dev.song, dev.score, dev.len, st));
      }
      if ((rc = copy_topk(h, TopkOut{hs.data(), hv.data(), hl.data()}, dev, k, 0, nc, st))) return rc;
      MR_CUDA(h, cudaStreamSynchronize(st));
      for (int j = 0; j < nc; ++j) {
        const size_t r = static_cast<size_t>(long_rows[c0 + j]);
        memcpy(out_song + r * k, hs.data() + static_cast<size_t>(j) * k, static_cast<size_t>(k) * sizeof(int32_t));
        memcpy(out_score + r * k, hv.data() + static_cast<size_t>(j) * k, static_cast<size_t>(k) * sizeof(double));
        out_len[r] = hl[j];
      }
    }
    *kind.long_rows += n_long;
  }
  MR_CUDA(h, cudaStreamSynchronize(st));
  return MR_OK;
}

int mr_similar_songs(mr_handle* h, const int32_t* song_ids, int n, int k, int32_t* out_song, double* out_score, int32_t* out_len) {
  int rc = require_loaded(h);
  if (rc) return rc;
  if (h->windowed) return fail(h, MR_ERR_STATE, "similar songs are not available on a handle with a song window (its song ids are rotated)");
  if (k < 1 || k > 1024) return fail(h, MR_ERR_BAD_ARG, "k = %d outside [1, 1024]", k);
  if (n < 0) return fail(h, MR_ERR_BAD_ARG, "n = %d < 0", n);
  if (n == 0) return MR_OK;
  if (!song_ids || !out_song || !out_score || !out_len) return fail(h, MR_ERR_BAD_ARG, "null query or output array");
  for (int r = 0; r < n; ++r)
    if (song_ids[r] < 0 || song_ids[r] >= h->S) return fail(h, MR_ERR_BAD_ARG, "query %d: song id %d outside [0,%d)", r, song_ids[r], h->S);
  if ((rc = ensure_sqrt_songs(h))) return rc;
  const SimKind kind{"similar songs", SimLists{h->d_csc_ptr, h->d_csc_idx, h->d_tr_ptr, h->d_tr_col, h->d_sim_sqd, h->d_sim_sqd, true},
                     song_count_rows(h), &h->sim_short_rows, &h->sim_long_rows};
  return similar_lists(h, kind, song_ids, n, k, out_song, out_score, out_len);
}

int mr_similar_users(mr_handle* h, const int32_t* user_idx, int n, int k, int32_t* out_user, double* out_score, int32_t* out_len) {
  int rc = require_test(h);
  if (rc) return rc;
  if (k < 1 || k > 1024) return fail(h, MR_ERR_BAD_ARG, "k = %d outside [1, 1024]", k);
  if (n < 0) return fail(h, MR_ERR_BAD_ARG, "n = %d < 0", n);
  if (n == 0) return MR_OK;
  if (!user_idx || !out_user || !out_score || !out_len) return fail(h, MR_ERR_BAD_ARG, "null query or output array");
  for (int r = 0; r < n; ++r)
    if (user_idx[r] < 0 || user_idx[r] >= h->U) return fail(h, MR_ERR_BAD_ARG, "query %d: test user index %d outside [0,%d)", r, user_idx[r], h->U);
  if ((rc = ensure_sqrt_users(h))) return rc;
  const SimKind kind{"similar users", SimLists{h->d_te_ptr, h->d_te_col, h->d_csc_ptr, h->d_csc_idx, h->d_simu_squ, h->d_simu_sqt, false},
                     user_count_rows(h), &h->simu_short_rows, &h->simu_long_rows};
  return similar_lists(h, kind, user_idx, n, k, out_user, out_score, out_len);
}

// ---- parity probes (mr_counts_*, mr_similarity_*): rows [r0, r1) of count rows cr to the caller's [r1 - r0][n_cols], as int32 (out_i32)
// or as cosines (out_f32, count_to_cos_kernel over the sqrt tables sq_row / sq_col), in chunks sized as the long rows of similar_lists.
// Like the similar calls they keep to the Gram workspace and SL_GRAM_IDS: the score panels, the select plane and gen stay as they are.
static int count_probe(mr_handle* h, const CountRows& cr, int r0, int r1, int32_t* out_i32, float* out_f32, const double* sq_row,
                       const double* sq_col) {
  if (r0 == r1) return MR_OK;
  int C = 0, rc;
  int* d_ids = nullptr;
  if ((rc = count_chunk(h, cr, 0, r1 - r0, "parity probe", &C)) || (rc = slot_alloc(h, mr_handle::SL_GRAM_IDS, &d_ids, static_cast<size_t>(C))))
    return rc;
  char* out = out_i32 ? reinterpret_cast<char*>(out_i32) : reinterpret_cast<char*>(out_f32);   // both are 4-byte elements
  const size_t row = static_cast<size_t>(cr.n_cols) * 4;
  for (int c0 = r0; c0 < r1; c0 += C) {
    const int nc = std::min(C, r1 - c0);
    iota_kernel<<<(nc + 255) / 256, 256, 0, h->stream>>>(d_ids, c0, nc);
    h->launches++;
    if ((rc = count_rows(h, cr, d_ids, nc))) return rc;
    if (out_f32) {
      PhaseTimer t(h, MR_T_OTHER);
      count_to_cos_kernel<<<h->num_sms * 4, 256, 0, h->stream>>>(h->d_g, cr.ld, d_ids, nc, cr.n_cols, sq_row, sq_col);
      h->launches++;
    }
    MR_CUDA(h, cudaMemcpy2DAsync(out + static_cast<size_t>(c0 - r0) * row, row, h->d_g, static_cast<size_t>(cr.ld) * 4, row, nc,
                                 cudaMemcpyDeviceToHost, h->stream));
    MR_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  return MR_OK;
}

int mr_counts_ubm(mr_handle* h, int32_t* out_UxT) {
  int rc = require_test(h);
  if (rc) return rc;
  if (!out_UxT) return fail(h, MR_ERR_BAD_ARG, "null output");
  return count_probe(h, user_count_rows(h), 0, h->U, out_UxT, nullptr, nullptr, nullptr);
}

int mr_similarity_ubm(mr_handle* h, float* out_UxT) {
  int rc = require_test(h);
  if (rc) return rc;
  if (!out_UxT) return fail(h, MR_ERR_BAD_ARG, "null output");
  if ((rc = ensure_sqrt_users(h))) return rc;
  return count_probe(h, user_count_rows(h), 0, h->U, nullptr, out_UxT, h->d_simu_squ, h->d_simu_sqt);
}

static int check_gram_range(mr_handle* h, int s0, int s1) {
  int rc = require_loaded(h);   // Gram rows need only the train replica
  if (rc) return rc;
  if (h->windowed) return fail(h, MR_ERR_STATE, "Gram rows are not available on a handle with a song window (its song ids are rotated)");
  if (s0 < 0 || s1 > h->S || s0 > s1) return fail(h, MR_ERR_BAD_ARG, "song range [%d,%d) outside [0,%d)", s0, s1, h->S);
  return MR_OK;
}

int mr_counts_ibm(mr_handle* h, int s0, int s1, int32_t* out_rows) {
  if (!out_rows) return fail(h, MR_ERR_BAD_ARG, "null output");
  const int rc = check_gram_range(h, s0, s1);
  return rc ? rc : count_probe(h, song_count_rows(h), s0, s1, out_rows, nullptr, nullptr, nullptr);
}

int mr_similarity_ibm(mr_handle* h, int s0, int s1, float* out_rows) {
  if (!out_rows) return fail(h, MR_ERR_BAD_ARG, "null output");
  int rc = check_gram_range(h, s0, s1);
  if (rc || (rc = ensure_sqrt_songs(h))) return rc;
  return count_probe(h, song_count_rows(h), s0, s1, nullptr, out_rows, h->d_sim_sqd, h->d_sim_sqd);
}

// ---- explanations (DESIGN.md §4.9, k8_similar.cu explain_pairs_kernel): the contributors of (test user, song) scores of UBM or IBM.  The
// pairs are grouped by the key whose count row serves them (UBM: the test user, row c(u, .); IBM: the song, Gram row g(s, .)); the
// distinct keys go through count_rows in chunks sized as the long rows of similar_lists, and the pairs of each chunk through
// explain_pairs_kernel in windows whose results fit kSimWindowBytes.  Slots: the keys, pair descriptors and results use the similar
// calls' SL_SIM_LIDS, SL_SIM_Q and SL_SIM_LOUT (no call keeps anything in them), the count rows the Gram workspace.
int mr_explain(mr_handle* h, int model, const int32_t* user_idx, const int32_t* song_ids, int n, int m, int32_t* out_id, double* out_term,
               int64_t* out_num, int32_t* out_len, int32_t* out_count, int64_t* out_total, double* out_score) {
  int rc = require_test(h);
  if (rc) return rc;
  if (h->windowed) return fail(h, MR_ERR_STATE, "explanations are not available on a handle with a song window (its song ids are rotated)");
  if (model != MR_UBM && model != MR_IBM) return fail(h, MR_ERR_BAD_ARG, "model %d: explanations exist for MR_UBM and MR_IBM only", model);
  if (m < 1 || m > 1024) return fail(h, MR_ERR_BAD_ARG, "m = %d outside [1, 1024]", m);
  if (n < 0) return fail(h, MR_ERR_BAD_ARG, "n = %d < 0", n);
  if (n == 0) return MR_OK;
  if (!user_idx || !song_ids || !out_id || !out_term || !out_num || !out_len || !out_count || !out_total || !out_score)
    return fail(h, MR_ERR_BAD_ARG, "null pair or output array");
  for (int r = 0; r < n; ++r) {
    if (user_idx[r] < 0 || user_idx[r] >= h->U) return fail(h, MR_ERR_BAD_ARG, "pair %d: test user index %d outside [0,%d)", r, user_idx[r], h->U);
    if (song_ids[r] < 0 || song_ids[r] >= h->S) return fail(h, MR_ERR_BAD_ARG, "pair %d: song id %d outside [0,%d)", r, song_ids[r], h->S);
  }
  const bool ubm = model == MR_UBM;
  if ((rc = ubm ? ensure_sqrt_users(h) : ensure_sqrt_songs(h))) return rc;
  cudaStream_t st = h->stream;
  const int32_t* key_of = ubm ? user_idx : song_ids;
  const int32_t* other_of = ubm ? song_ids : user_idx;
  // the pairs sorted by key; keys[i] is the i-th distinct key, its pairs are order[kbeg[i] .. kbeg[i + 1])
  std::vector<int> order(static_cast<size_t>(n));
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key_of[a] < key_of[b]; });
  std::vector<int> keys, kbeg;
  for (int p = 0; p < n; ++p)
    if (p == 0 || key_of[order[p]] != keys.back()) { keys.push_back(key_of[order[p]]); kbeg.push_back(p); }
  kbeg.push_back(n);
  const int n_keys = static_cast<int>(keys.size());

  // results of a window of W pairs: term f64 [W][m] | num i64 [W][m] | total i64 [W] | score f64 [W] | id i32 [W][m] | len i32 [W] | count i32 [W]
  const size_t pair_bytes = static_cast<size_t>(m) * 20 + 24;
  const int W = static_cast<int>(std::max<size_t>(1, std::min<size_t>(static_cast<size_t>(n), kSimWindowBytes / pair_bytes)));
  const size_t Wm = static_cast<size_t>(W) * m;
  auto at = [&](char* b) {
    ExplainOut o;
    o.term = reinterpret_cast<double*>(b);
    o.num = reinterpret_cast<long long*>(o.term + Wm);
    o.total = o.num + Wm;
    o.score = reinterpret_cast<double*>(o.total + W);
    o.id = reinterpret_cast<int*>(o.score + W);
    o.len = o.id + Wm;
    o.count = o.len + W;
    return o;
  };
  char* base = nullptr; int2* d_pairs = nullptr; int* d_keys = nullptr;
  if ((rc = slot_alloc(h, mr_handle::SL_SIM_LOUT, &base, W * pair_bytes)) || (rc = slot_alloc(h, mr_handle::SL_SIM_Q, &d_pairs, static_cast<size_t>(W))))
    return rc;
  const CountRows cr = ubm ? user_count_rows(h) : song_count_rows(h);
  int C = 0;
  if ((rc = count_chunk(h, cr, sizeof(int), n_keys, "explanations", &C))) return rc;
  if ((rc = slot_alloc(h, mr_handle::SL_SIM_LIDS, &d_keys, static_cast<size_t>(C)))) return rc;
  const ExplainArgs a{d_keys, d_pairs, h->d_g, cr.ld, ubm ? h->d_csc_ptr : h->d_te_ptr, ubm ? h->d_csc_idx : h->d_te_col, h->d_te_ptr,
                      h->d_te_col, ubm ? h->d_simu_squ : h->d_sim_sqd, ubm ? h->d_simu_sqt : h->d_sim_sqd, ubm ? h->d_qv : h->d_qd,
                      ubm ? h->d_rsa : h->d_rsd};
  const ExplainOut dev = at(base);
  std::vector<char> hb(W * pair_bytes);
  const ExplainOut hst = at(hb.data());
  std::vector<int2> desc(static_cast<size_t>(W));
  for (int k0 = 0; k0 < n_keys; k0 += C) {
    const int nc = std::min(C, n_keys - k0);
    MR_CUDA(h, cudaMemcpyAsync(d_keys, keys.data() + k0, static_cast<size_t>(nc) * sizeof(int), cudaMemcpyHostToDevice, st));
    if ((rc = count_rows(h, cr, d_keys, nc))) return rc;
    h->explain_rows += nc;
    int ki = k0;
    for (int w0 = kbeg[k0]; w0 < kbeg[k0 + nc]; w0 += W) {
      const int nw = std::min(W, kbeg[k0 + nc] - w0);
      for (int j = 0; j < nw; ++j) {
        while (kbeg[ki + 1] <= w0 + j) ++ki;
        desc[j] = make_int2(ki - k0, other_of[order[w0 + j]]);
      }
      MR_CUDA(h, cudaMemcpyAsync(d_pairs, desc.data(), static_cast<size_t>(nw) * sizeof(int2), cudaMemcpyHostToDevice, st));
      {
        PhaseTimer t(h, MR_T_TOPK);
        MR_LAUNCH(h, launch_explain_pairs(model, a, nw, m, dev, st));
      }
      const size_t nwm = static_cast<size_t>(nw) * m;
      MR_CUDA(h, cudaMemcpyAsync(hst.term, dev.term, nwm * sizeof(double), cudaMemcpyDeviceToHost, st));
      MR_CUDA(h, cudaMemcpyAsync(hst.num, dev.num, nwm * sizeof(long long), cudaMemcpyDeviceToHost, st));
      MR_CUDA(h, cudaMemcpyAsync(hst.id, dev.id, nwm * sizeof(int), cudaMemcpyDeviceToHost, st));
      MR_CUDA(h, cudaMemcpyAsync(hst.total, dev.total, static_cast<size_t>(nw) * sizeof(long long), cudaMemcpyDeviceToHost, st));
      MR_CUDA(h, cudaMemcpyAsync(hst.score, dev.score, static_cast<size_t>(nw) * sizeof(double), cudaMemcpyDeviceToHost, st));
      MR_CUDA(h, cudaMemcpyAsync(hst.len, dev.len, static_cast<size_t>(nw) * sizeof(int), cudaMemcpyDeviceToHost, st));
      MR_CUDA(h, cudaMemcpyAsync(hst.count, dev.count, static_cast<size_t>(nw) * sizeof(int), cudaMemcpyDeviceToHost, st));
      MR_CUDA(h, cudaStreamSynchronize(st));
      for (int j = 0; j < nw; ++j) {   // into the caller's rows
        const size_t r = static_cast<size_t>(order[w0 + j]), o = static_cast<size_t>(j) * m;
        memcpy(out_id + r * m, hst.id + o, static_cast<size_t>(m) * sizeof(int32_t));
        memcpy(out_term + r * m, hst.term + o, static_cast<size_t>(m) * sizeof(double));
        memcpy(out_num + r * m, hst.num + o, static_cast<size_t>(m) * sizeof(int64_t));
        out_len[r] = hst.len[j]; out_count[r] = hst.count[j]; out_total[r] = hst.total[j]; out_score[r] = hst.score[j];
      }
    }
  }
  MR_CUDA(h, cudaStreamSynchronize(st));
  return MR_OK;
}

int mr_score_dense(mr_handle* h, int model, double* out_UxS) {
  int rc = require_test(h);
  if (rc) return rc;
  if (model != MR_UBM && model != MR_IBM) return fail(h, MR_ERR_BAD_ARG, "mr_score_dense: model must be MR_UBM or MR_IBM");
  if (!out_UxS) return fail(h, MR_ERR_BAD_ARG, "null output");
  if ((rc = slot_alloc(h, mr_handle::SL_DENSE, &h->d_dense, static_cast<size_t>(std::min(h->batch_rows, kDenseChunk)) * h->n_cols))) return rc;
  const DenseOut dout{DenseOut::ALL, out_UxS, nullptr, 0, nullptr, nullptr};
  Run run{ModelSet(model), Consumer::DENSE, 0, &dout};
  return run_batches(h, run);
}

static int score_subset(mr_handle* h, int model, const int32_t* ids, int n, double* out, bool songs) {
  int rc = require_test(h);
  if (rc) return rc;
  if (model != MR_UBM && model != MR_IBM) return fail(h, MR_ERR_BAD_ARG, "model must be MR_UBM or MR_IBM");
  if (n < 0 || (n > 0 && (!ids || !out))) return fail(h, MR_ERR_BAD_ARG, "null id list / output");
  const int first = songs ? h->win_lo : 0, limit = songs ? h->win_lo + h->n_cols : h->U;   // songs: the scored columns (the window, if one is set)
  for (int i = 0; i < n; ++i)
    if (ids[i] < first || ids[i] >= limit) return fail(h, MR_ERR_BAD_ARG, "%s id %d out of range [%d,%d)", songs ? "song" : "test user", ids[i], first, limit);
  if (n == 0) return MR_OK;
  if ((rc = slot_alloc(h, mr_handle::SL_DENSE, &h->d_dense, static_cast<size_t>(std::min(h->batch_rows, kDenseChunk)) * h->n_cols))) return rc;
  Scratch tmp(h, h->stream);
  DenseOut dout{songs ? DenseOut::SONGS : DenseOut::USERS, out, ids, n, nullptr, nullptr};
  if (songs) {
    int* d_ids = nullptr;
    std::vector<int> cols(ids, ids + n);
    for (int& c : cols) c -= h->win_lo;
    if ((rc = tmp.upload(&d_ids, cols.data(), static_cast<size_t>(n))) || (rc = tmp.alloc(&dout.d_out, static_cast<size_t>(n) * h->U))) return rc;
    dout.d_ids = d_ids;
  }
  Run run{ModelSet(model), Consumer::DENSE, 0, &dout};
  if ((rc = run_batches(h, run))) return rc;
  if (songs) {
    cudaError_t e = cudaMemcpyAsync(out, dout.d_out, static_cast<size_t>(n) * h->U * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "mr_score_songs copy-out: %s", cudaGetErrorString(e));
  }
  return MR_OK;
}

int mr_score_users(mr_handle* h, int model, const int32_t* user_idx, int n, double* out_nxS) { return score_subset(h, model, user_idx, n, out_nxS, false); }
int mr_score_songs(mr_handle* h, int model, const int32_t* song_ids, int n, double* out_nxU) { return score_subset(h, model, song_ids, n, out_nxU, true); }

int mr_map_at_k(mr_handle* h, int k, const int32_t* top_song, const int32_t* top_len, int n_users, const int64_t* lab_rowptr, const int32_t* lab_col,
                double* out_map, double* out_ap) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (k < 1 || n_users <= 0 || !lab_rowptr || !out_map) return fail(h, MR_ERR_BAD_ARG, "null / empty arguments");
  if ((top_song == nullptr) != (top_len == nullptr)) return fail(h, MR_ERR_BAD_ARG, "top_song and top_len must both be given or both be null");
  int rc = check_csr(h, "label", n_users, INT_MAX, lab_rowptr, lab_col);   // song ids are only compared: any id >= 0 is in range
  if (rc) return rc;
  const long long n_lab = lab_rowptr[n_users];
  MR_CUDA(h, cudaSetDevice(h->device));
  const int* d_song = nullptr; const int* d_len = nullptr;
  Scratch tmp(h, h->stream);
  if (!top_song) {   // rank the device-resident result of the last mr_topk_device / mr_topk
    if (!h->have_topk || h->out_k != k || n_users != h->U) return fail(h, MR_ERR_STATE, "no top-%d result of %d users on the device", k, n_users);
    d_song = h->out.song; d_len = h->out.len;
  } else {
    int *ds = nullptr, *dl = nullptr;
    if ((rc = tmp.upload(&ds, top_song, static_cast<size_t>(n_users) * k)) || (rc = tmp.upload(&dl, top_len, static_cast<size_t>(n_users)))) return rc;
    d_song = ds; d_len = dl;
  }
  std::vector<long long> lp(lab_rowptr, lab_rowptr + n_users + 1);
  long long* d_lp = nullptr; int* d_lc = nullptr; double* d_ap = nullptr;
  if ((rc = tmp.upload(&d_lp, lp.data(), lp.size())) || (rc = tmp.upload(&d_lc, lab_col, static_cast<size_t>(n_lab))) ||
      (rc = tmp.alloc(&d_ap, static_cast<size_t>(n_users)))) return rc;
  int lrc;
  {
    PhaseTimer t(h, MR_T_OTHER);
    lrc = launch_map_at_k(d_song, d_len, n_users, k, d_lp, d_lc, d_ap, h->stream);
    h->launches++;
  }
  std::vector<double> ap(n_users);
  cudaError_t e = lrc ? cudaErrorLaunchFailure : cudaMemcpyAsync(ap.data(), d_ap, static_cast<size_t>(n_users) * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "mr_map_at_k: %s", cudaGetErrorString(e));
  double total = 0.0; long long n_eval = 0;
  for (int u = 0; u < n_users; ++u) {
    if (lab_rowptr[u + 1] > lab_rowptr[u]) { total += ap[u]; ++n_eval; }   // left fold in ascending user order, users without labels skipped
    if (out_ap) out_ap[u] = ap[u];
  }
  *out_map = n_eval > 0 ? total / static_cast<double>(n_eval) : 0.0;
  return MR_OK;
}

int mr_set_option(mr_handle* h, int option, int64_t value) {
  if (!h) return MR_ERR_STATE;
  ++h->gen;
  switch (option) {
    case MR_OPT_HEAD_MIN_DEG:
      if (h->loaded) return fail(h, MR_ERR_STATE, "MR_OPT_HEAD_MIN_DEG must be set before mr_load (it selects the head songs)");
      if (value < 0) return fail(h, MR_ERR_BAD_ARG, "MR_OPT_HEAD_MIN_DEG must be >= 0");
      h->opt_head_min_deg = value;
      return MR_OK;
    case MR_OPT_SONG_WINDOW_LO:
    case MR_OPT_SONG_WINDOW_HI:
      if (h->loaded) return fail(h, MR_ERR_STATE, "the song window must be set before mr_load (ids are rotated and the head rows sized by it)");
      if (value < 0 || value > 0x7fffffff) return fail(h, MR_ERR_BAD_ARG, "song window bound out of range");
      (option == MR_OPT_SONG_WINDOW_LO ? h->win_lo : h->win_hi) = static_cast<int>(value);
      return MR_OK;
    case MR_OPT_ITEM_BATCH:
      if (value < 0) return fail(h, MR_ERR_BAD_ARG, "MR_OPT_ITEM_BATCH must be >= 0");
      h->item_batch_cap = value > 0 ? static_cast<int>(std::max<int64_t>(128, std::min<int64_t>(value, 1 << 30))) : 0;
      return MR_OK;
    default:
      return fail(h, MR_ERR_BAD_ARG, "unknown option %d", option);
  }
}

int mr_invalidate_prepared(mr_handle* h) {
  const int rc = require_loaded(h);
  if (rc) return rc;
  const cudaError_t e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "mr_invalidate_prepared: %s", cudaGetErrorString(e));
  if (h->head_pending) { cudaEventSynchronize(h->ev_pre); h->head_pending = false; }   // a build in flight is abandoned once it has drained
  h->head_ready = false; h->n_ex = 0; ++h->gen;
  return MR_OK;
}

int mr_blend_dense(mr_handle* h, int kind, double param, uint64_t seed, const double* ubm, const double* ibm, double* out,
                   int64_t n_pairs, int64_t first_index, int64_t n_total) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (kind != MR_LC && kind != MR_AGG && kind != MR_STOCH) return fail(h, MR_ERR_BAD_ARG, "mr_blend_dense: kind must be MR_LC, MR_AGG or MR_STOCH");
  if (n_pairs < 0 || (n_pairs > 0 && (!ubm || !ibm || !out))) return fail(h, MR_ERR_BAD_ARG, "null arrays");
  BlendParams bp;
  int rc = make_blend_params(h, kind, param, seed, n_total > 0 ? n_total : n_pairs, &bp);
  if (rc) return rc;
  if (n_pairs == 0) return MR_OK;
  MR_CUDA(h, cudaSetDevice(h->device));
  Scratch tmp(h, h->stream);
  double *du = nullptr, *di = nullptr, *dout = nullptr;
  if ((rc = tmp.alloc(&du, n_pairs)) || (rc = tmp.alloc(&di, n_pairs)) || (rc = tmp.alloc(&dout, n_pairs))) return rc;
  cudaError_t e = cudaMemcpyAsync(du, ubm, n_pairs * sizeof(double), cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(di, ibm, n_pairs * sizeof(double), cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) {
    PhaseTimer t(h, MR_T_OTHER);
    int lrc = launch_blend_arrays(bp, du, di, dout, n_pairs, first_index, h->stream);
    h->launches++;
    if (lrc) e = cudaErrorLaunchFailure;
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, n_pairs * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "mr_blend_dense: %s", cudaGetErrorString(e));
  return MR_OK;
}

int mr_evaluate_dense(mr_handle* h, const double* scores_UxS, int n_users, int n_songs, const int64_t* lab_rowptr, const int32_t* lab_col,
                      int n_thresholds, double* out_map) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (!scores_UxS || !lab_rowptr || !out_map || n_users <= 0 || n_songs <= 0) return fail(h, MR_ERR_BAD_ARG, "null / empty arguments");
  if (n_thresholds != 10 && n_thresholds != 11) return fail(h, MR_ERR_BAD_ARG, "n_thresholds must be 10 (MR:590) or 11 (DIST:395)");
  const long long n_lab = lab_rowptr[n_users];
  if (n_lab <= 0 || !lab_col) return fail(h, MR_ERR_BAD_ARG, "empty label set");
  int rc = check_csr(h, "label", n_users, INT_MAX, lab_rowptr, lab_col);   // eval_ap_kernel scores only ids < n_songs
  if (rc) return rc;
  MR_CUDA(h, cudaSetDevice(h->device));
  std::vector<int> new_songs(lab_col, lab_col + n_lab);                       // newSongs = distinct label songs (MR:72, 79)
  std::sort(new_songs.begin(), new_songs.end());
  new_songs.erase(std::unique(new_songs.begin(), new_songs.end()), new_songs.end());
  const int n_new = static_cast<int>(new_songs.size());
  std::vector<long long> lp(lab_rowptr, lab_rowptr + n_users + 1);
  Scratch tmp(h, h->stream);
  double *d_scores = nullptr, *d_ap = nullptr; long long* d_lp = nullptr; int *d_lc = nullptr, *d_new = nullptr; unsigned long long* d_mm = nullptr;
  if ((rc = tmp.upload(&d_scores, scores_UxS, static_cast<size_t>(n_users) * n_songs)) || (rc = tmp.upload(&d_lp, lp.data(), lp.size())) ||
      (rc = tmp.upload(&d_lc, lab_col, static_cast<size_t>(n_lab))) || (rc = tmp.upload(&d_new, new_songs.data(), new_songs.size())) ||
      (rc = tmp.alloc(&d_ap, static_cast<size_t>(n_new))) || (rc = tmp.alloc(&d_mm, 2))) return rc;
  int lrc;
  {
    PhaseTimer t(h, MR_T_OTHER);
    lrc = launch_evaluate(d_scores, n_users, n_songs, d_lp, d_lc, d_new, n_new, n_thresholds, d_mm, d_ap, h->num_sms, h->stream);
    h->launches += 2;
  }
  std::vector<double> ap(n_new);
  cudaError_t e = lrc ? cudaErrorLaunchFailure : cudaMemcpyAsync(ap.data(), d_ap, n_new * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "mr_evaluate_dense: %s", cudaGetErrorString(e));
  double total = 0.0;
  for (int c = 0; c < n_new; ++c) total += ap[c];                              // foldLeft(0.0)(_+_), MR:626
  *out_map = total / n_new;
  return MR_OK;
}

// ---- streamed evaluateModel (MR:521-639; DESIGN.md §4.5)
namespace {
const double kEvalTh[11] = {0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0};   // the TH literals of eval_ap_kernel

// doubles -> unsigned integers in the same order (negative values included), and back
inline unsigned long long ord_key(double x) { unsigned long long b; memcpy(&b, &x, 8); return (b >> 63) ? ~b : b | (1ULL << 63); }
inline double from_key(unsigned long long k) { const unsigned long long b = (k >> 63) ? k & ~(1ULL << 63) : ~k; double x; memcpy(&x, &b, 8); return x; }

// c_t = the least double x in [mn, mx] with RN(RN(x - mn) / RN(mx - mn)) > TH[t], +inf when there is none.  The normalisation is
// monotone non-decreasing in x (RN subtraction, RN division by a positive number), so a bisection over the ordered bit patterns finds it.
void eval_cutoffs(double mn, double mx, int n_thresholds, double* out) {
  const double range = mx - mn;
  auto f = [&](double x) { return (x - mn) / range; };
  for (int t = 0; t < n_thresholds; ++t) {
    out[t] = std::numeric_limits<double>::infinity();
    if (!(range > 0) || !(f(mx) > kEvalTh[t])) continue;
    unsigned long long lo = ord_key(mn), hi = ord_key(mx);
    while (lo < hi) {
      const unsigned long long mid = lo + (hi - lo) / 2;
      if (f(from_key(mid)) > kEvalTh[t]) hi = mid; else lo = mid + 1;
    }
    out[t] = from_key(hi);
  }
}

// A model set from the caller's parallel arrays, every entry checked before any GPU work (what: the caller's name in the messages;
// name_entries: the message names the first bad entry, as the set calls do).  The LC alpha must be in [0, 1]: the select and the
// evaluator rank IEEE bit patterns of non-negative scores.  The reference's linear combination accepts any alpha (MR:317-330 has no
// range check) and mr_blend_dense follows it, but outside [0,1] a blended score can be negative, which has no place in a ranking of
// cosine sums (documented deviation, DESIGN.md §3).
int make_set(mr_handle* h, int n, const int* models, const double* params, const uint64_t* seeds, const char* what, bool name_entries,
             ModelSet* set) {
  if (n < 1 || n > kMaxSet) return fail(h, MR_ERR_BAD_ARG, "%s: n_models = %d outside 1..%d", what, n, kMaxSet);
  if (!models || !params || !seeds) return fail(h, MR_ERR_BAD_ARG, "%s: null model arrays", what);
  set->n = n; set->n_stoch = 0;
  for (int i = 0; i < n; ++i) {
    int rc;
    if (models[i] == MR_LC && !(params[i] >= 0 && params[i] <= 1))
      rc = fail(h, MR_ERR_PARAM_RANGE, "%s: alpha of the linear combination must be between 0 and 1", what);
    else
      rc = make_blend_params(h, models[i], params[i], seeds[i], h->n_pairs_total, &set->bp[i]);
    if (rc) {
      if (name_entries) h->err = "entry " + std::to_string(i) + ": " + h->err;
      return rc;
    }
    set->bp[i].pair_base = h->d_pair_base;
    if (models[i] == MR_STOCH) ++set->n_stoch;
  }
  return MR_OK;
}

// The evaluation form of a set: checks, the AGG split columns (one [U] array per AGG entry, on the library stream)
// and the consumer groups.  Each STOCH entry heads a group of its own (the group reads the one select plane); the other entries fill
// the groups in entry order, kEvalGroupMax to a launch.
int eval_set(mr_handle* h, int n, const int* models, const double* params, const uint64_t* seeds, bool name_entries, ModelSet* set) {
  int rc = require_test(h);
  if (rc) return rc;
  if ((rc = make_set(h, n, models, params, seeds, "evaluation", name_entries, set))) return rc;
  int n_agg = 0;
  for (int e = 0; e < n; ++e) { set->bp[e].stats = nullptr; n_agg += set->bp[e].model == MODEL_AGG; }
  int* d_split = nullptr;
  if (n_agg && (rc = slot_alloc(h, mr_handle::SL_AGG_SPLIT, &d_split, static_cast<size_t>(n_agg) * h->U))) return rc;
  set->n_groups = 0;
  auto add = [&](int g, int e) {
    EvalGroup& G = set->grp[g];
    const int m = G.n++;
    G.model[m] = set->bp[e].model; G.alpha[m] = set->bp[e].alpha; G.oma[m] = set->bp[e].one_minus_alpha; G.out[m] = e; G.split[m] = nullptr;
    for (unsigned long long& c : G.cut[m]) c = ~0ULL;
  };
  auto open_group = [&](int stoch) { const int g = set->n_groups++; memset(&set->grp[g], 0, sizeof(EvalGroup)); set->grp_stoch[g] = stoch; return g; };
  for (int e = 0; e < n; ++e)
    if (set->bp[e].model == MODEL_STOCH) add(open_group(e), e);
  for (int e = 0, j = 0; e < n; ++e) {
    if (set->bp[e].model == MODEL_STOCH) continue;
    int g = 0;
    while (g < set->n_groups && set->grp[g].n == kEvalGroupMax) ++g;
    if (g == set->n_groups) open_group(-1);
    add(g, e);
    if (set->bp[e].model == MODEL_AGG) {
      int* split = d_split + static_cast<size_t>(j++) * h->U;
      set->grp[g].split[set->grp[g].n - 1] = split;
      MR_LAUNCH(h, launch_agg_split(set->bp[e], h->d_te_ptr, h->d_te_col, h->U, h->n_cols, split, h->stream));
    }
  }
  return MR_OK;
}

void remember_eval_set(mr_handle* h, int n, const int* models, const double* params, const uint64_t* seeds) {
  h->eval_gen = h->gen; h->eval_n = n;
  for (int i = 0; i < n; ++i) { h->eval_models[i] = models[i]; h->eval_params[i] = params[i]; h->eval_seeds[i] = seeds[i]; }
}
bool same_eval_set(const mr_handle* h, int n, const int* models, const double* params, const uint64_t* seeds) {
  if (h->eval_gen != h->gen || h->eval_n != n) return false;
  for (int i = 0; i < n; ++i)
    if (h->eval_models[i] != models[i] || memcmp(&h->eval_params[i], &params[i], sizeof(double)) != 0 || h->eval_seeds[i] != seeds[i]) return false;
  return true;
}

int eval_range_impl(mr_handle* h, int n, const int* models, const double* params, const uint64_t* seeds, bool name_entries, double* out_min,
                    double* out_max) {
  if (!h) return MR_ERR_STATE;
  if (!out_min || !out_max) return fail(h, MR_ERR_BAD_ARG, "null output");
  Run run{ModelSet{}, Consumer::EVAL_RANGE};
  int rc = eval_set(h, n, models, params, seeds, name_entries, &run.set);
  if (rc) return rc;
  if ((rc = slot_alloc(h, mr_handle::SL_EVAL_MM, &h->d_eval_mm, 2 * static_cast<size_t>(n)))) return rc;
  std::vector<unsigned long long> mm(2 * static_cast<size_t>(n));
  for (int e = 0; e < n; ++e) { mm[2 * e] = ~0ULL; mm[2 * e + 1] = 0ULL; }
  MR_CUDA(h, cudaMemcpyAsync(h->d_eval_mm, mm.data(), mm.size() * 8, cudaMemcpyHostToDevice, h->stream));
  if ((rc = run_batches(h, run))) return rc;
  MR_CUDA(h, cudaMemcpyAsync(mm.data(), h->d_eval_mm, mm.size() * 8, cudaMemcpyDeviceToHost, h->stream));
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  remember_eval_set(h, n, models, params, seeds);
  for (int e = 0; e < n; ++e) {
    if (mm[2 * e] == ~0ULL) {   // no emitted pair
      out_min[e] = std::numeric_limits<double>::infinity(); out_max[e] = -std::numeric_limits<double>::infinity();
    } else {
      memcpy(&out_min[e], &mm[2 * e], 8); memcpy(&out_max[e], &mm[2 * e + 1], 8);
    }
  }
  return MR_OK;
}

// MRSCORE_DEBUG_TIMING: the host stages of a count call on stderr
struct HostStages {
  bool on = getenv("MRSCORE_DEBUG_TIMING") != nullptr;
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  std::string line;
  void mark(const char* stage) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    char buf[64];
    snprintf(buf, sizeof buf, " %s=%.2f", stage, std::chrono::duration<double, std::milli>(now - t).count());
    line += buf; t = now;
  }
  void print(int n) const { if (on) fprintf(stderr, "[mrscore] eval_counts host stages (ms), %d model(s):%s\n", n, line.c_str()); }
};

int eval_counts_impl(mr_handle* h, int n, const int* models, const double* params, const uint64_t* seeds, bool name_entries, const double* mn,
                     const double* mx, int n_thresholds, const int64_t* lab_rowptr, const int32_t* lab_col, const int32_t* new_songs, int n_new,
                     int64_t* out_pred, int64_t* out_tp, int64_t* out_nlab) {
  if (!h) return MR_ERR_STATE;
  HostStages hs;
  if (n_thresholds != 10 && n_thresholds != 11) return fail(h, MR_ERR_BAD_ARG, "n_thresholds must be 10 (MR:590) or 11 (DIST:395)");
  if (!lab_rowptr || !new_songs || n_new <= 0 || !out_pred || !out_tp || !out_nlab || !mn || !mx) return fail(h, MR_ERR_BAD_ARG, "null / empty arguments");
  Run run{ModelSet{}, Consumer::EVAL_COUNT};
  int rc = eval_set(h, n, models, params, seeds, name_entries, &run.set);
  if (rc) return rc;
  hs.mark("set");
  const int U = h->U;
  if ((rc = check_csr(h, "label", U, INT_MAX, lab_rowptr, lab_col))) return rc;   // ids beyond the songs are checked against new_songs below
  const long long n_lab = lab_rowptr[U];
  if (new_songs[0] < 0) return fail(h, MR_ERR_BAD_ARG, "new_songs: negative song id");
  for (int i = 1; i < n_new; ++i)
    if (new_songs[i] <= new_songs[i - 1]) return fail(h, MR_ERR_BAD_ARG, "new_songs not strictly ascending at %d", i);
  {   // every label song is in new_songs: a membership table over [0, largest new song] (a binary search per label was 270 ms at MSD scale)
    std::vector<uint8_t> in_new(static_cast<size_t>(new_songs[n_new - 1]) + 1, 0);
    for (int i = 0; i < n_new; ++i) in_new[new_songs[i]] = 1;
    for (long long i = 0; i < n_lab; ++i)
      if (static_cast<size_t>(lab_col[i]) >= in_new.size() || !in_new[lab_col[i]])
        return fail(h, MR_ERR_BAD_ARG, "new_songs lacks label song %d", lab_col[i]);
  }
  for (int e = 0; e < n; ++e)
    if (mx[e] - mn[e] > 0 && !(mn[e] >= 0)) {
      rc = fail(h, MR_ERR_BAD_ARG, "mn must be >= 0 (scores are non-negative)");
      if (name_entries) h->err = "entry " + std::to_string(e) + ": " + h->err;
      return rc;
    }
  hs.mark("label_checks");
  for (int g = 0; g < run.set.n_groups; ++g) {
    EvalGroup& G = run.set.grp[g];
    for (int m = 0; m < G.n; ++m) {
      double cut[11];
      eval_cutoffs(mn[G.out[m]], mx[G.out[m]], n_thresholds, cut);
      for (int t = 0; t < n_thresholds; ++t) memcpy(&G.cut[m][t], &cut[t], 8);
    }
  }
  EvalCounts& ec = h->ec;
  ec = EvalCounts{};
  ec.n_thresholds = n_thresholds; ec.col_lo = h->win_lo;
  std::vector<int> colmap(h->n_cols, -1);   // scored column -> label-song index
  for (int i = 0; i < n_new; ++i)
    if (new_songs[i] >= h->win_lo && new_songs[i] < h->win_lo + h->n_cols) colmap[new_songs[i] - h->win_lo] = i;
  const size_t per = static_cast<size_t>(n_new) * n_thresholds, n_cnt = 2 * per * n + n_new;
  int* d_colmap = nullptr; long long* d_lp = nullptr; int* d_lc = nullptr; unsigned long long* d_cnt = nullptr;
  if ((rc = slot_upload(h, mr_handle::SL_EVAL_COLMAP, &d_colmap, colmap.data(), colmap.size())) ||
      (rc = slot_upload(h, mr_handle::SL_LAB_PTR, &d_lp, reinterpret_cast<const long long*>(lab_rowptr), static_cast<size_t>(U) + 1)) ||
      (rc = slot_upload(h, mr_handle::SL_LAB_COL, &d_lc, lab_col, static_cast<size_t>(n_lab))) ||
      (rc = slot_alloc(h, mr_handle::SL_EVAL_CNT, &d_cnt, n_cnt)))
    return rc;
  MR_CUDA(h, cudaMemsetAsync(d_cnt, 0, n_cnt * sizeof(unsigned long long), h->stream));
  ec.colmap = d_colmap; ec.lab_ptr = d_lp; ec.lab_col = d_lc; ec.pred_b = d_cnt; ec.tp_b = d_cnt + per;
  ec.model_stride = static_cast<long long>(2 * per); ec.nlab = d_cnt + 2 * per * n;
  hs.mark("uploads");
  // resident reuse: a single-batch item-space shard whose panels the range pass of the same set has just filled
  run.reuse = h->space == MR_SPACE_ITEM && h->U <= h->batch_rows && same_eval_set(h, n, models, params, seeds);
  if ((rc = run_batches(h, run))) return rc;
  hs.mark("enqueue");
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  hs.mark("gpu_wait");
  std::vector<unsigned long long> cnt(n_cnt);
  MR_CUDA(h, cudaMemcpyAsync(cnt.data(), d_cnt, n_cnt * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  hs.mark("copy_back");
  for (int e = 0; e < n; ++e) {
    const unsigned long long* pb = cnt.data() + 2 * per * e;
    int64_t* op = out_pred + per * e; int64_t* ot = out_tp + per * e;
    for (int c = 0; c < n_new; ++c) {   // bucket counts -> counts per threshold: predicted at t <=> bucket > t
      long long p = 0, q = 0;
      for (int t = n_thresholds - 1; t >= 0; --t) {
        const size_t i = static_cast<size_t>(c) * n_thresholds + t;
        p += static_cast<long long>(pb[i]); q += static_cast<long long>(pb[per + i]);
        op[i] = p; ot[i] = q;
      }
    }
  }
  for (int c = 0; c < n_new; ++c) out_nlab[c] = static_cast<long long>(cnt[2 * per * n + c]);
  hs.mark("suffix_sums");
  hs.print(n);
  return MR_OK;
}
}  // namespace

int mr_eval_cutoffs(double mn, double mx, int n_thresholds, double* out) {
  if (!out || (n_thresholds != 10 && n_thresholds != 11)) return MR_ERR_BAD_ARG;
  eval_cutoffs(mn, mx, n_thresholds, out);
  return MR_OK;
}

int mr_eval_range(mr_handle* h, int model, double param, uint64_t seed, double* out_min, double* out_max) {
  return eval_range_impl(h, 1, &model, &param, &seed, false, out_min, out_max);
}

int mr_eval_counts(mr_handle* h, int model, double param, uint64_t seed, double mn, double mx, int n_thresholds, const int64_t* lab_rowptr,
                   const int32_t* lab_col, const int32_t* new_songs, int n_new, int64_t* out_pred, int64_t* out_tp, int64_t* out_nlab) {
  return eval_counts_impl(h, 1, &model, &param, &seed, false, &mn, &mx, n_thresholds, lab_rowptr, lab_col, new_songs, n_new, out_pred, out_tp,
                          out_nlab);
}

int mr_eval_range_multi(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, double* out_min,
                        double* out_max) {
  return eval_range_impl(h, n_models, models, params, seeds, true, out_min, out_max);
}

int mr_eval_counts_multi(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, const double* mn,
                         const double* mx, int n_thresholds, const int64_t* lab_rowptr, const int32_t* lab_col, const int32_t* new_songs,
                         int n_new, int64_t* out_pred, int64_t* out_tp, int64_t* out_nlab) {
  return eval_counts_impl(h, n_models, models, params, seeds, true, mn, mx, n_thresholds, lab_rowptr, lab_col, new_songs, n_new, out_pred,
                          out_tp, out_nlab);
}

// fp64 in exactly the operation order of eval_ap_kernel and mr_evaluate_dense; no contraction into FMAs
__attribute__((optimize("fp-contract=off")))
int mr_eval_finish(const int64_t* pred, const int64_t* tp, const int64_t* nlab, int n_new, int n_thresholds, double* out_ap, double* out_map) {
  if (!pred || !tp || !nlab || !out_map || n_new <= 0 || (n_thresholds != 10 && n_thresholds != 11)) return MR_ERR_BAD_ARG;
  double total = 0.0;
  for (int c = 0; c < n_new; ++c) {
    double prec[11], rec[11];
    const long long l = nlab[c];
    for (int t = 0; t < n_thresholds; ++t) {
      const long long p = pred[static_cast<size_t>(c) * n_thresholds + t], x = tp[static_cast<size_t>(c) * n_thresholds + t];
      if (x < 0 || x > p || x > l) return MR_ERR_BAD_ARG;                                     // not counts of one partitioning
      prec[t] = p > 0 ? static_cast<double>(x) / static_cast<double>(p) : 0.0;               // tp / (tp + fp), MR:561-566
      rec[t] = l > 0 ? static_cast<double>(x) / static_cast<double>(l) : 0.0;                // tp / (tp + fn), MR:574-579
    }
    double ap = 0.0;
    for (int t = 0; t < n_thresholds; ++t) {
      double term;
      if (t == n_thresholds - 1) term = 0.0;
      else if (t == n_thresholds - 2) term = (rec[t] - 0.0) * prec[t];
      else term = (rec[t] - rec[t + 1]) * prec[t];
      ap = ap + term;
    }
    if (out_ap) out_ap[c] = ap;
    total += ap;                                                                              // foldLeft(0.0)(_+_), MR:626
  }
  *out_map = total / n_new;
  return MR_OK;
}

// The single-model top-k: a set of one whose result keeps its own slot (SL_OUT_PACK), so that it survives a set call.
static int topk_impl(mr_handle* h, int model, double param, uint64_t seed, int k, const TopkOut* ho) {
  int rc = require_test(h);
  if (rc) return rc;
  if (k < 1 || k > 1024) return fail(h, MR_ERR_BAD_ARG, "k must be in [1,1024], got %d", k);
  Run run{ModelSet(), Consumer::TOPK, k};
  if ((rc = make_set(h, 1, &model, &param, &seed, "getTopK", false, &run.set))) return rc;
  const TopkBlock blk(h->U, k);
  char* base = nullptr;
  if ((rc = slot_alloc(h, mr_handle::SL_OUT_PACK, &base, blk.bytes))) return rc;
  h->out = run.set.out[0] = blk.at(base);
  h->out_pack_bytes = blk.bytes;
  h->out_k = k;
  h->have_topk = false;
  const bool streamed = ho && h->space == MR_SPACE_ITEM;          // the item-space pipeline copies slice by slice
  if (streamed) run.topk_host = ho;
  rc = run_batches(h, run);
  if (streamed) { cudaError_t e = cudaStreamSynchronize(h->copy_stream); if (!rc && e != cudaSuccess) rc = fail(h, MR_ERR_CUDA, "result copy: %s", cudaGetErrorString(e)); }
  if (rc) return rc;
  h->have_topk = true;
  if (ho && !streamed) return mr_topk_fetch(h, k, ho->song, ho->score, ho->len);
  if (ho) MR_CUDA(h, cudaStreamSynchronize(h->stream));
  return MR_OK;
}

int mr_topk_device(mr_handle* h, int model, double param, uint64_t seed, int k) { return topk_impl(h, model, param, seed, k, nullptr); }

int mr_topk_fetch(mr_handle* h, int k, int32_t* out_song, double* out_score, int32_t* out_len) {
  int rc = require_test(h);
  if (rc) return rc;
  if (!h->have_topk || h->out_k != k) return fail(h, MR_ERR_STATE, "no top-%d result on the device (call mr_topk_device first)", k);
  if (!out_song || !out_score || !out_len) return fail(h, MR_ERR_BAD_ARG, "null output");
  if ((rc = copy_topk(h, TopkOut{out_song, out_score, out_len}, h->out, k, 0, h->U, h->stream))) return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  return MR_OK;
}

int mr_topk_device_ptrs(mr_handle* h, int k, void** song, void** score, void** len) {
  int rc = require_test(h);
  if (rc) return rc;
  if (!h->have_topk || h->out_k != k) return fail(h, MR_ERR_STATE, "no top-%d result on the device (call mr_topk_device first)", k);
  if (song) *song = h->out.song;
  if (score) *score = h->out.score;
  if (len) *len = h->out.len;
  return MR_OK;
}

int mr_topk_packed(mr_handle* h, int k, void** base, uint64_t* bytes, uint64_t* score_offset, uint64_t* len_offset) {
  int rc = require_test(h);
  if (rc) return rc;
  if (!h->have_topk || h->out_k != k) return fail(h, MR_ERR_STATE, "no top-%d result on the device (call mr_topk_device first)", k);
  if (base) *base = h->out.song;
  if (bytes) *bytes = h->out_pack_bytes;
  if (score_offset) *score_offset = static_cast<uint64_t>(reinterpret_cast<char*>(h->out.score) - reinterpret_cast<char*>(h->out.song));
  if (len_offset) *len_offset = static_cast<uint64_t>(reinterpret_cast<char*>(h->out.len) - reinterpret_cast<char*>(h->out.song));
  return MR_OK;
}

int mr_topk_merge(mr_handle* h, int k, int n_parts, int n_users, const int32_t* const* part_song, const double* const* part_score,
                  const int32_t* const* part_len, int32_t* out_song, double* out_score, int32_t* out_len) {
  if (!h || !h->stream) return MR_ERR_STATE;
  if (k < 1 || k > 1024 || n_users < 0 || !part_song || !part_score || !part_len || !out_song || !out_score || !out_len)
    return fail(h, MR_ERR_BAD_ARG, "mr_topk_merge: null argument or k outside [1,1024]");
  if (n_parts < 1 || n_parts > kMergeMaxParts) return fail(h, MR_ERR_BAD_ARG, "mr_topk_merge: %d partitions (1..%d)", n_parts, kMergeMaxParts);
  MergeParts p; memset(&p, 0, sizeof p);
  p.n = n_parts;
  for (int i = 0; i < n_parts; ++i) {
    if (!part_song[i] || !part_score[i] || !part_len[i]) return fail(h, MR_ERR_BAD_ARG, "mr_topk_merge: partition %d has a null array", i);
    p.song[i] = part_song[i]; p.score[i] = part_score[i]; p.len[i] = part_len[i];
  }
  MR_CUDA(h, cudaSetDevice(h->device));
  PhaseTimer t(h, MR_T_TOPK);
  MR_LAUNCH(h, launch_merge_topk(p, k, n_users, out_song, out_score, out_len, h->stream));
  return MR_OK;
}

int mr_topk(mr_handle* h, int model, double param, uint64_t seed, int k, int32_t* out_song, double* out_score, int32_t* out_len) {
  if (!out_song || !out_score || !out_len) return fail(h, MR_ERR_BAD_ARG, "null output");
  const TopkOut ho{out_song, out_score, out_len};
  return topk_impl(h, model, param, seed, k, &ho);
}

}  // extern "C"

namespace {

// Fraction of the window's columns below which a filtered top-k ranks the allowed columns (candidate path) instead of streaming the rows
// with the allowed-column bitmap (full-row path): on the MSD shape the candidate path wins at 1 % and loses from 5 % on, for UBM, IBM and
// AGG (DESIGN.md §4.11).  MRSCORE_FILTER_PATH=full|candidate forces a path (developer aid for timing both at one size).
constexpr double kCandidateFrac = 0.03;

// A model set's top-k lists into the SL_MULTI_OUT blocks (mr_topk_multi_device), optionally under the handle's filter.
int topk_set(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k, bool filtered) {
  int rc = require_test(h);
  if (rc) return rc;
  if (k < 1 || k > 1024) return fail(h, MR_ERR_BAD_ARG, "k must be in [1,1024], got %d", k);
  Run run{ModelSet(), Consumer::TOPK, k};
  if ((rc = make_set(h, n_models, models, params, seeds, "getTopK", true, &run.set))) return rc;
  if (filtered) {
    if (!h->flt_on) return fail(h, MR_ERR_STATE, "no top-k filter is set on this shard (mr_set_topk_filter)");
    if (h->flt_n_ex > 0) { run.ex_ptr = h->d_flt_ex_ptr; run.ex_col = h->d_flt_ex_col; }
    const char* force = getenv("MRSCORE_FILTER_PATH");
    run.candidate = h->flt_n_allow >= 0 && h->flt_n_allow < kCandidateFrac * h->n_cols;
    if (force && h->flt_n_allow >= 0) run.candidate = strcmp(force, "candidate") == 0 || (run.candidate && strcmp(force, "full") != 0);
    run.cand_cols = h->d_flt_cols; run.n_cand = std::max(h->flt_n_allow, 0);
    if (!run.candidate && h->flt_n_allow >= 0)
      for (int e = 0; e < run.set.n; ++e) run.set.bp[e].allow = h->d_flt_bits;
  }
  // one block per entry in a grow-only slot of its own: the single-model result (mr_topk_fetch, mr_map_at_k) stays
  const TopkBlock blk(h->U, k);
  const size_t need = blk.bytes * static_cast<size_t>(n_models);
  h->multi_n = 0;
  // it must fit inside the caller's reserve that the batch plan leaves free, and be free now; the plan is not changed for it
  size_t avail = kCallerReserve;
  if (h->slot_cap[mr_handle::SL_MULTI_OUT] < need) {
    size_t free_b = 0, total_b = 0;
    MR_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    avail = std::min(avail, free_b + h->slot_cap[mr_handle::SL_MULTI_OUT]);
  }
  if (need > avail)
    return fail(h, MR_ERR_OOM, "mr_topk_multi: %d top-%d results of %d users need %zu bytes, more than the %zu bytes of the caller's reserve "
                "that are free", n_models, k, h->U, need, avail);
  char* base = nullptr;
  if ((rc = slot_alloc(h, mr_handle::SL_MULTI_OUT, &base, need, true))) return rc;
  for (int e = 0; e < n_models; ++e) run.set.out[e] = blk.at(base + blk.bytes * e);
  if ((rc = run_batches(h, run))) return rc;
  h->multi_n = n_models; h->multi_k = k;
  if (filtered) (run.candidate ? h->flt_cand_rows : h->flt_full_rows) += static_cast<long long>(h->U) * n_models;
  return MR_OK;
}

// The set's lists copied to the caller's host arrays (mr_topk_multi, mr_topk_filtered).
int topk_set_host(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k, int32_t* const* out_song,
                  double* const* out_score, int32_t* const* out_len, bool filtered) {
  if (!h) return MR_ERR_STATE;
  if (n_models < 1 || n_models > kMaxSet) return fail(h, MR_ERR_BAD_ARG, "getTopK: n_models = %d outside 1..%d", n_models, kMaxSet);
  if (!out_song || !out_score || !out_len) return fail(h, MR_ERR_BAD_ARG, "null output");
  for (int e = 0; e < n_models; ++e)
    if (!out_song[e] || !out_score[e] || !out_len[e]) return fail(h, MR_ERR_BAD_ARG, "entry %d: null output", e);
  int rc = topk_set(h, n_models, models, params, seeds, k, filtered);
  if (rc) return rc;
  const TopkBlock blk(h->U, k);
  char* const base = static_cast<char*>(h->slot_p[mr_handle::SL_MULTI_OUT]);
  for (int e = 0; e < n_models; ++e)
    if ((rc = copy_topk(h, TopkOut{out_song[e], out_score[e], out_len[e]}, blk.at(base + blk.bytes * e), k, 0, h->U, h->stream))) return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  return MR_OK;
}

}  // namespace

extern "C" {

int mr_topk_multi_device(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k) {
  return topk_set(h, n_models, models, params, seeds, k, false);
}

int mr_topk_multi_ptrs(mr_handle* h, int i, int k, void** song, void** score, void** len) {
  int rc = require_test(h);
  if (rc) return rc;
  if (h->multi_n == 0 || h->multi_k != k) return fail(h, MR_ERR_STATE, "no top-%d set result on the device (call mr_topk_multi_device first)", k);
  if (i < 0 || i >= h->multi_n) return fail(h, MR_ERR_BAD_ARG, "entry %d outside the set of %d", i, h->multi_n);
  const TopkBlock blk(h->U, k);
  const TopkOut o = blk.at(static_cast<char*>(h->slot_p[mr_handle::SL_MULTI_OUT]) + blk.bytes * i);
  if (song) *song = o.song;
  if (score) *score = o.score;
  if (len) *len = o.len;
  return MR_OK;
}

int mr_topk_multi(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k, int32_t* const* out_song,
                  double* const* out_score, int32_t* const* out_len) {
  return topk_set_host(h, n_models, models, params, seeds, k, out_song, out_score, out_len, false);
}

int mr_set_topk_filter(mr_handle* h, const int32_t* allow_songs, int n_allow, const int64_t* ex_rowptr, const int32_t* ex_col) {
  int rc = require_test(h);
  if (rc) return rc;
  h->flt_on = false;
  if (!allow_songs && n_allow == -1 && !ex_rowptr) return MR_OK;   // cleared
  if (n_allow < -1 || (n_allow > 0 && !allow_songs)) return fail(h, MR_ERR_BAD_ARG, "allowed songs: n_allow = %d with %s list", n_allow, allow_songs ? "a" : "a null");
  for (int i = 0; i < n_allow; ++i)
    if (allow_songs[i] < 0 || allow_songs[i] >= h->S) return fail(h, MR_ERR_BAD_ARG, "allowed song %d (entry %d) out of range [0,%d)", allow_songs[i], i, h->S);
  if (ex_rowptr && (rc = check_csr(h, "exclusions", h->U, h->S, ex_rowptr, ex_col))) return rc;
  // the in-window part, in columns: ids in [win_lo, win_hi) become id - win_lo (window order = id order); the others are dropped
  const int lo = h->win_lo, hi = h->win_lo + h->n_cols, n_words = (h->n_cols + 31) / 32;
  std::vector<uint32_t> bits;
  std::vector<int> cols;
  if (n_allow >= 0) {
    bits.assign(static_cast<size_t>(n_words), 0u);
    for (int i = 0; i < n_allow; ++i)
      if (allow_songs[i] >= lo && allow_songs[i] < hi) bits[(allow_songs[i] - lo) >> 5] |= 1u << ((allow_songs[i] - lo) & 31);
    for (int c = 0; c < h->n_cols; ++c)
      if ((bits[c >> 5] >> (c & 31)) & 1u) cols.push_back(c);
  }
  std::vector<long long> ex_ptr;
  std::vector<int> ex_c;
  long long n_ex = 0;
  if (ex_rowptr) {
    const int U = h->U;
    std::vector<long long> b(U), e(U);   // the in-window entries of a row are one ascending run
    parallel_rows(U, [&](int u_lo, int u_hi) {
      for (int u = u_lo; u < u_hi; ++u) {
        const int32_t *rb = ex_col + ex_rowptr[u], *re = ex_col + ex_rowptr[u + 1];
        b[u] = std::lower_bound(rb, re, lo) - ex_col; e[u] = std::lower_bound(rb, re, hi) - ex_col;
      }
    });
    ex_ptr.assign(static_cast<size_t>(U) + 1, 0);
    for (int u = 0; u < U; ++u) ex_ptr[u + 1] = ex_ptr[u] + (e[u] - b[u]);
    n_ex = ex_ptr[U];
    ex_c.resize(static_cast<size_t>(n_ex));
    parallel_rows(U, [&](int u_lo, int u_hi) {
      for (int u = u_lo; u < u_hi; ++u)
        for (long long i = b[u], o = ex_ptr[u]; i < e[u]; ++i, ++o) ex_c[o] = ex_col[i] - lo;
    });
  }
  // the device copies must fit inside the caller's reserve that the batch plan leaves free, and be free now; the plan is not changed for it
  const int slots[4] = {mr_handle::SL_FLT_BITS, mr_handle::SL_FLT_COLS, mr_handle::SL_FLT_EX_PTR, mr_handle::SL_FLT_EX_COL};
  const size_t bytes[4] = {bits.size() * 4, cols.size() * 4, n_ex > 0 ? ex_ptr.size() * 8 : 0, ex_c.size() * 4};
  size_t need = 0, held = 0; bool grows = false;
  for (int i = 0; i < 4; ++i) { need += bytes[i]; held += h->slot_cap[slots[i]]; grows = grows || h->slot_cap[slots[i]] < bytes[i]; }
  size_t avail = kCallerReserve;
  if (grows) {
    size_t free_b = 0, total_b = 0;
    MR_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    avail = std::min(avail, free_b + held);
  }
  if (need > avail)
    return fail(h, MR_ERR_OOM, "mr_set_topk_filter: the filter needs %zu bytes of device memory, more than the %zu bytes of the caller's reserve "
                "that are free", need, avail);
  if ((rc = slot_upload(h, mr_handle::SL_FLT_BITS, &h->d_flt_bits, bits.data(), bits.size())) ||
      (rc = slot_upload(h, mr_handle::SL_FLT_COLS, &h->d_flt_cols, cols.data(), cols.size())))
    return rc;
  if (n_ex > 0 && ((rc = slot_upload(h, mr_handle::SL_FLT_EX_PTR, &h->d_flt_ex_ptr, ex_ptr.data(), ex_ptr.size())) ||
                   (rc = slot_upload(h, mr_handle::SL_FLT_EX_COL, &h->d_flt_ex_col, ex_c.data(), ex_c.size()))))
    return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));   // the pageable host arrays must outlive their uploads
  h->flt_n_allow = n_allow >= 0 ? static_cast<int>(cols.size()) : -1;
  h->flt_n_ex = n_ex;
  h->flt_on = true;
  return MR_OK;
}

int mr_topk_filtered_device(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k) {
  return topk_set(h, n_models, models, params, seeds, k, true);
}

int mr_topk_filtered(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k, int32_t* const* out_song,
                     double* const* out_score, int32_t* const* out_len) {
  return topk_set_host(h, n_models, models, params, seeds, k, out_song, out_score, out_len, true);
}

int mr_song_audience(mr_handle* h, int model, double param, uint64_t seed, const int32_t* song_ids, int n, int k, int32_t* out_user,
                     double* out_score, int32_t* out_len) {
  int rc = require_test(h);
  if (rc) return rc;
  if (k < 1 || k > 1024) return fail(h, MR_ERR_BAD_ARG, "k must be in [1,1024], got %d", k);
  Run run{ModelSet(), Consumer::AUDIENCE, k};
  if ((rc = make_set(h, 1, &model, &param, &seed, "getSongAudience", false, &run.set))) return rc;
  if (n < 0 || (n > 0 && (!song_ids || !out_user || !out_score || !out_len))) return fail(h, MR_ERR_BAD_ARG, "null song list / output");
  const int lo = h->win_lo, hi = h->win_lo + h->n_cols;
  for (int i = 0; i < n; ++i)
    if (song_ids[i] < lo || song_ids[i] >= hi) return fail(h, MR_ERR_BAD_ARG, "song id %d out of range [%d,%d)", song_ids[i], lo, hi);
  if (n == 0) return MR_OK;
  // the running lists, one TopkBlock of n rows in a grow-only slot of their own (the top-k results stay); it must fit inside the caller's
  // reserve that the batch plan leaves free, and be free now; the plan is not changed for it
  const TopkBlock blk(n, k);
  size_t avail = kCallerReserve;
  if (h->slot_cap[mr_handle::SL_AUD_OUT] < blk.bytes) {
    size_t free_b = 0, total_b = 0;
    MR_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    avail = std::min(avail, free_b + h->slot_cap[mr_handle::SL_AUD_OUT]);
  }
  if (blk.bytes > avail)
    return fail(h, MR_ERR_OOM, "mr_song_audience: %d top-%d lists need %zu bytes, more than the %zu bytes of the caller's reserve that are free",
                n, k, blk.bytes, avail);
  char* base = nullptr;
  int2* d_q = nullptr;
  if ((rc = slot_alloc(h, mr_handle::SL_AUD_OUT, &base, blk.bytes, true))) return rc;
  // the queries by column (rotated into the window), so that CTAs of adjacent columns run together; each keeps its caller's row
  std::vector<int2> q(static_cast<size_t>(n));
  for (int i = 0; i < n; ++i) q[i] = make_int2(song_ids[i] - lo, i);
  std::sort(q.begin(), q.end(), [](const int2& a, const int2& b) { return a.x != b.x ? a.x < b.x : a.y < b.y; });
  if ((rc = slot_upload(h, mr_handle::SL_AUD_Q, &d_q, q.data(), q.size()))) return rc;
  run.set.out[0] = blk.at(base);
  run.aud_q = d_q; run.aud_n = n;
  const TopkOut& l = run.set.out[0];
  MR_CUDA(h, cudaMemsetAsync(l.song, 0xff, static_cast<size_t>(n) * k * sizeof(int32_t), h->stream));   // empty lists: user -1, score 0.0, len 0
  MR_CUDA(h, cudaMemsetAsync(l.score, 0, static_cast<size_t>(n) * k * sizeof(double), h->stream));
  MR_CUDA(h, cudaMemsetAsync(l.len, 0, static_cast<size_t>(n) * sizeof(int32_t), h->stream));
  rc = run_batches(h, run);
  if (!rc) rc = copy_topk(h, TopkOut{out_user, out_score, out_len}, l, k, 0, n, h->stream);
  const cudaError_t e = cudaStreamSynchronize(h->stream);   // also keeps the pageable query list alive until its upload has run
  if (rc) return rc;
  if (e != cudaSuccess) return fail(h, MR_ERR_CUDA, "mr_song_audience: %s", cudaGetErrorString(e));
  h->audience_rows += n;
  return MR_OK;
}

int mr_get_timing(mr_handle* h, double* ms_out, int n) {
  if (!h || !ms_out) return MR_ERR_BAD_ARG;
  for (int i = 0; i < n && i < MR_T_N; ++i) ms_out[i] = h->t_ms[i];
  return MR_OK;
}
int mr_reset_timing(mr_handle* h) {
  if (!h) return MR_ERR_BAD_ARG;
  for (double& t : h->t_ms) t = 0;
  return MR_OK;
}
int mr_get_info(mr_handle* h, int64_t* out, int n) {
  if (!h || !out) return MR_ERR_BAD_ARG;
  unsigned int st[4] = {0, 0, 0, 0};
  if (n > 16 && h->d_topk_stats && cudaMemcpy(st, h->d_topk_stats, sizeof st, cudaMemcpyDeviceToHost) != cudaSuccess) return fail(h, MR_ERR_CUDA, "mr_get_info: reading the select counters failed");
  const int64_t v[34] = {h->engine, h->launches, static_cast<int64_t>(h->dense_bytes), h->n_items, h->num_sms, static_cast<int64_t>(h->dev_bytes), h->space, h->n_head,
                         h->n_head_entries, h->n_tail_entries, h->n_ex, h->batch_rows, h->n_groups,
                         h->h_split_ptr.empty() ? 0 : h->h_split_ptr.back(), h->n_cols, h->win_lo, st[0], st[1], st[2], h->passes,
                         h->sim_short_rows, h->sim_long_rows, h->simu_short_rows, h->simu_long_rows, h->explain_rows,
                         h->audience_rows, st[3], h->flt_full_rows, h->flt_cand_rows,
                         h->carry_events, h->n_head_staged, h->head_packed ? 1 : 0, h->head_planes, h->ubm_int_ok ? 1 : 0};
  for (int i = 0; i < n && i < 34; ++i) out[i] = v[i];
  return MR_OK;
}
int mr_prepare_async(mr_handle* h) {
  const int rc = require_loaded(h);
  if (rc) return rc;
  return start_head_rows(h, h->pre_stream);
}

int mr_prepare(mr_handle* h) {
  int rc = require_loaded(h);
  if (rc) return rc;
  if ((rc = ensure_head_rows(h))) return rc;
  MR_CUDA(h, cudaStreamSynchronize(h->stream));
  return MR_OK;
}
int mr_set_profile(mr_handle* h, int on) {
  if (!h) return MR_ERR_BAD_ARG;
  if (on) h->flags |= MR_PROFILE; else h->flags &= ~static_cast<unsigned>(MR_PROFILE);
  return MR_OK;
}
void* mr_stream(mr_handle* h) { return h ? static_cast<void*>(h->stream) : nullptr; }

}  // extern "C"
#pragma GCC visibility pop
