// k8_similar.cu — the exact top-k of the reference's two cosines for a list of queries (DESIGN.md §4.7, §4.8):
//   similar songs (mr_similar_songs):  sim(i, s) = g(i, s) / (sqrt((double) d_i) * sqrt((double) d_s))   g = |U_i^train ∩ U_s^train| (MR:232),
//                                      d = deg_song_all (MR:237); candidates s != i
//   similar users (mr_similar_users):  w(u, v) = c(u, v) / (sqrt((double) |I_u|) * sqrt((double) |I_v|))   c = |I_u^test ∩ I_v^train| (MR:142-145),
//                                      the degrees as handed to mr_load / mr_set_test_users (MR:147); candidates are train users v
// in the operation order of the CPU formula (the reference's cosineSimilarity, MR:147-148 and MR:237-238), every step correctly rounded
// (__dsqrt_rn, __dmul_rn, __ddiv_rn; the library is built with --fmad=false), so every score has the bits of the CPU formula.  Candidates
// have a count > 0; order: score descending, then candidate id ascending — the composite key (score bits : 64, ~id : 32) of k3_topk.cu.
//
// Both query kinds are one two-level walk (SimLists): query q -> its items q_idx[q_ptr[q] .. q_ptr[q + 1]) -> the candidates of each item
// c_idx[c_ptr[j] .. c_ptr[j + 1]).  Songs: song -> train listeners (inverted index) -> their train histories.  Users: test user -> visible
// songs -> train listeners.  The work of query q is E_q = the number of (item, candidate) events.  Two row paths:
//   short rows (E_q <= kSimShortMax): one CTA per query gathers the candidate ids into shared memory, sorts them, run-lengths them into
//     (id, count), scores each distinct id and sorts the candidates by key; the row never touches HBM and no global atomics are used;
//   long rows: exact int32 count rows from the count engines (mrscore.cu count_rows), then similar_row_topk_kernel, one CTA per row:
//     maximum, linear histogram, then the exact select topk_kernel runs too (mr_common.cuh: bin of the k-th key, MSD radix select inside
//     a crowded bin, collect, bitonic sort, write-out).
// kSelf: similar songs exclude the query song from its own list; a train user is never the test user asking, so similar users exclude none.
//
// Explanations (mr_explain, DESIGN.md §4.9) rank the same two cosines restricted to the contributors of one (test user, song) score:
// explain_pairs_kernel runs the select of the long rows (row_select) over a scan of the pair's contributor list instead of a count row.
#include <climits>

#include "mr_common.cuh"
#include "mr_kernels.h"

namespace mr {

__device__ __forceinline__ double sim_score(int g, double sq_i, double sq_s) {
  const double den = __dmul_rn(sq_i, sq_s);
  return den != 0.0 ? __ddiv_rn(static_cast<double>(g), den) : 0.0;   // naive_*_cos: denominator != 0 ? numerator / denominator : 0
}

// ascending bitonic sort of n_pad (a power of two) ints; every thread of the CTA calls it
__device__ void bitonic_ints(int* a, int n_pad) {
  __syncthreads();
  for (int size = 2; size <= n_pad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < n_pad / 2; i += blockDim.x) {
        const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
        const int x = a[lo], y = a[hi];
        if ((x > y) == ((lo & size) == 0)) { a[lo] = y; a[hi] = x; }
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------- per-call helpers
__global__ void sqrt_deg_kernel(const int* __restrict__ deg, int n, double* __restrict__ out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n) out[s] = __dsqrt_rn(static_cast<double>(deg[s]));
}

int launch_sqrt_deg(const int* deg, int n, double* out, cudaStream_t st) {
  if (n <= 0) return 0;
  sqrt_deg_kernel<<<(n + 255) / 256, 256, 0, st>>>(deg, n, out);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// E_q of every query, one warp per query
__global__ void sim_events_kernel(const int* __restrict__ ids, int n, const long long* __restrict__ q_ptr, const int* __restrict__ q_idx,
                                  const long long* __restrict__ c_ptr, long long* __restrict__ events) {
  const int q = static_cast<int>((blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (q >= n) return;
  const int i = ids[q];
  long long e = 0;
  for (long long l = q_ptr[i] + lane; l < q_ptr[i + 1]; l += 32) { const int j = q_idx[l]; e += c_ptr[j + 1] - c_ptr[j]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
  if (lane == 0) events[q] = e;
}

int launch_sim_events(const int* ids, int n, const SimLists& l, long long* events, cudaStream_t st) {
  if (n <= 0) return 0;
  sim_events_kernel<<<(n + 7) / 8, 256, 0, st>>>(ids, n, l.q_ptr, l.q_idx, l.c_ptr, events);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- short rows: one CTA per query, everything in shared memory
// Dynamic shared memory: key u64[cap] | ids i32[cap], cap a power of two >= E_q of every query of the launch (12 * cap bytes).
// Positions per thread (cap / blockDim.x) must be <= 32: the candidate flags of a thread live in one register mask.
template <bool kSelf>
__global__ void similar_short_kernel(const int* __restrict__ q_ids, const int* __restrict__ q_row, int cap, const long long* __restrict__ q_ptr,
                                     const int* __restrict__ q_idx, const long long* __restrict__ c_ptr, const int* __restrict__ c_idx,
                                     const double* __restrict__ sq_q, const double* __restrict__ sq_c, int k, int* __restrict__ out_song,
                                     double* __restrict__ out_score, int* __restrict__ out_len) {
  extern __shared__ unsigned long long s_dyn[];
  unsigned long long* s_key = s_dyn;
  int* s_ids = reinterpret_cast<int*>(s_dyn + cap);
  __shared__ int s_n, s_cand;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = blockDim.x >> 5;
  const int i = q_ids[blockIdx.x], row = q_row[blockIdx.x];
  if (tid == 0) { s_n = 0; s_cand = 0; }
  __syncthreads();
  // gather the candidate lists of i's items, one warp per item (songs: the train histories of i's train listeners)
  for (long long l = q_ptr[i] + warp; l < q_ptr[i + 1]; l += n_warps) {
    const int j = q_idx[l];
    const long long b = c_ptr[j];
    const int len = static_cast<int>(c_ptr[j + 1] - b);
    int base = 0;
    if (lane == 0) base = atomicAdd(&s_n, len);
    base = __shfl_sync(0xffffffffu, base, 0);
    for (int m = lane; m < len; m += 32) s_ids[base + m] = __ldg(c_idx + b + m);
  }
  __syncthreads();
  const int n = s_n;
  int n_pad = 1;
  while (n_pad < n) n_pad <<= 1;
  for (int p = n + tid; p < n_pad; p += blockDim.x) s_ids[p] = INT_MAX;
  bitonic_ints(s_ids, n_pad);
  // run-length: the first position of each run of equal ids is a candidate (s, g = run length), unless kSelf and s == i
  const double sq_i = sq_q[i];
  uint32_t cand = 0;
  int n_mine = 0;
  for (int p = tid, j = 0; p < n; p += blockDim.x, ++j) {
    const int s = s_ids[p];
    if ((kSelf && s == i) || (p > 0 && s_ids[p - 1] == s)) continue;
    int lo = p + 1, hi = n;                       // end of the run: first position with a larger id
    while (lo < hi) { const int m = (lo + hi) >> 1; if (s_ids[m] <= s) lo = m + 1; else hi = m; }
    s_key[p] = key_bits(sim_score(lo - p, sq_i, __ldg(sq_c + s)));
    cand |= 1u << j;
    ++n_mine;
  }
  if (n_mine) atomicAdd(&s_cand, n_mine);
  __syncthreads();
  // non-candidates sort last: key 0 and song INT_MAX (a candidate's score may be 0.0 only with a zero degree, its song id is < INT_MAX)
  for (int p = tid, j = 0; p < n_pad; p += blockDim.x, ++j)
    if (p >= n || !((cand >> j) & 1u)) { s_key[p] = 0; s_ids[p] = INT_MAX; }
  bitonic_keys(s_key, s_ids, n_pad);
  const int need = min(k, s_cand);
  int* o_song = out_song + static_cast<long long>(row) * k;
  double* o_score = out_score + static_cast<long long>(row) * k;
  for (int j = tid; j < k; j += blockDim.x) {
    if (j < need) { o_song[j] = s_ids[j]; o_score[j] = __longlong_as_double(static_cast<long long>(s_key[j])); }
    else { o_song[j] = -1; o_score[j] = 0.0; }
  }
  if (tid == 0) out_len[row] = need;
}

int launch_similar_short(const int* q_ids, const int* q_row, int n_q, int cap, const SimLists& l, int k, int* out_song, double* out_score,
                         int* out_len, cudaStream_t st) {
  if (n_q <= 0) return 0;
  if (cap < 64 || cap > kSimShortMax || (cap & (cap - 1))) return -2;
  const int threads = cap <= 1024 ? 128 : 256;
  if (cap / threads > 32) return -2;
  const size_t smem = static_cast<size_t>(cap) * 12;
  // the attribute is per device (handles may live on several GPUs of one process); setting it is cheap, so no caching.  Always set: the
  // 48 KB default counts the static shared memory too, which the 4 k class (48 KB dynamic) already exceeds
  auto kern = l.self ? similar_short_kernel<true> : similar_short_kernel<false>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSimShortMax * 12) != cudaSuccess) return -3;
  kern<<<n_q, threads, smem, st>>>(q_ids, q_row, cap, l.q_ptr, l.q_idx, l.c_ptr, l.c_idx, l.sq_q, l.sq_c, k, out_song, out_score, out_len);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- long rows: select over exact int32 count rows, one CTA per row
// f(song, key bits, candidate) for 4 songs per thread per step, the same number of times by every thread (f may use warp collectives)
template <bool kSelf, class F>
__device__ __forceinline__ void scan_counts(const int32_t* __restrict__ g, int n_songs, int self, double sq_i, const double* __restrict__ sq_c, F&& f) {
  for (int base0 = 0; base0 < n_songs; base0 += 4 * kTopkThreads) {
    const int s = base0 + 4 * static_cast<int>(threadIdx.x);
    int4 v = make_int4(0, 0, 0, 0);
    if (s < n_songs) v = __ldg(reinterpret_cast<const int4*>(g + s));   // rows are padded to 32 songs
    const int c[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const bool ok = s + t < n_songs && c[t] > 0 && (!kSelf || s + t != self);
      const unsigned long long kb = ok ? key_bits(sim_score(c[t], sq_i, __ldg(sq_c + s + t))) : 0ULL;
      f(s + t, kb, ok);
    }
  }
}

template <bool kSelf>
__global__ void __launch_bounds__(kTopkThreads, 2)
similar_row_topk_kernel(const int* __restrict__ rows, int n_rows, const int32_t* __restrict__ g, long long ldg, int n_songs,
                        const double* __restrict__ sq_q, const double* __restrict__ sq_c, int k, int* __restrict__ out_song,
                        double* __restrict__ out_score, int* __restrict__ out_len) {
  __shared__ RowSelect sm;
  const int r = blockIdx.x;
  if (r >= n_rows) return;
  const int self = rows[r];
  const double sq_i = sq_q[self];
  const int32_t* row = g + static_cast<long long>(r) * ldg;
  auto scan = [&](auto&& f) { scan_counts<kSelf>(row, n_songs, self, sq_i, sq_c, f); };
  row_select(scan, scan, k, sm, out_song + static_cast<long long>(r) * k, out_score + static_cast<long long>(r) * k, out_len + r);
}

int launch_similar_rows(const int* rows, int n_rows, const int32_t* g, long long ldg, int n_cols, const SimLists& l, int k, int* out_song,
                        double* out_score, int* out_len, cudaStream_t st) {
  if (n_rows <= 0) return 0;
  if (k <= 0 || k > kTopkCap / 2) return -2;
  auto kern = l.self ? similar_row_topk_kernel<true> : similar_row_topk_kernel<false>;
  kern<<<n_rows, kTopkThreads, 0, st>>>(rows, n_rows, g, ldg, n_cols, l.sq_q, l.sq_c, k, out_song, out_score, out_len);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- explanations: the contributors of one (test user, song) score
// One CTA per pair p = (count row a.pairs[p].x of the chunk, other id a.pairs[p].y).  The pair's contributor list is scanned straight
// from the index and each entry's count read from the count row:
//   UBM (key = test user u, other = song s): the train listeners v of s (inverted index), c(u, v) from the row c(u, .);
//   IBM (key = song s, other = test user u): u's visible songs j, g(s, j) from the Gram row g(s, .).
// Since s is not in I_u for an explained pair, j != s holds for every j of I_u.  The first pass also sums num = count * q over all
// contributors: the exact numerator Sint[u, s] of DESIGN.md §3.
template <int kModel>
__global__ void __launch_bounds__(kTopkThreads, 2)
explain_pairs_kernel(const ExplainArgs a, int n, int m, const ExplainOut o) {
  __shared__ RowSelect sm;
  __shared__ unsigned long long s_total;
  const int p = blockIdx.x;
  if (p >= n) return;
  const int tid = threadIdx.x, lane = tid & 31;
  const int2 pr = a.pairs[p];
  const int key = a.keys[pr.x];
  const int u = kModel == MODEL_UBM ? key : pr.y, s = kModel == MODEL_UBM ? pr.y : key;
  const int32_t* row = a.g + static_cast<long long>(pr.x) * a.ld;
  int* o_id = o.id + static_cast<long long>(p) * m;
  double* o_term = o.term + static_cast<long long>(p) * m;
  long long* o_num = o.num + static_cast<long long>(p) * m;
  // a listened pair (s in u's ascending test row) is no pair of the model (MR:109)
  const long long tb = a.te_ptr[u];
  int lo = 0, hi = static_cast<int>(a.te_ptr[u + 1] - tb);
  const int n_u = hi;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(a.te_col + tb + mid) < s) lo = mid + 1; else hi = mid; }
  if (lo < n_u && __ldg(a.te_col + tb + lo) == s) {
    for (int i = tid; i < m; i += kTopkThreads) { o_id[i] = -1; o_term[i] = 0.0; o_num[i] = 0; }
    if (tid == 0) { o.len[p] = 0; o.count[p] = 0; o.total[p] = 0; o.score[p] = __longlong_as_double(0x7ff8000000000000LL); }
    return;
  }
  const int li = kModel == MODEL_UBM ? s : u;
  const long long lb = a.list_ptr[li];
  const int len = static_cast<int>(a.list_ptr[li + 1] - lb);
  const int* list = a.list_idx + lb;
  const double sq_k = a.sq_key[key];
  if (tid == 0) s_total = 0;   // row_select synchronises before anyone adds to it
  long long tot = 0;
  // f(id, key bits, contributor) for one list entry per thread per step; on(id, count) for each contributor
  auto walk = [&](auto&& f, auto&& on) {
    for (int b = 0; b < len; b += kTopkThreads) {
      const int i = b + tid;
      int id = 0, c = 0;
      if (i < len) { id = __ldg(list + i); c = __ldg(row + id); }
      unsigned long long kb = 0;
      if (c > 0) { kb = key_bits(sim_score(c, sq_k, __ldg(a.sq_other + id))); on(id, c); }
      f(id, kb, c > 0);
    }
  };
  auto first = [&](auto&& f) { walk(f, [&](int id, int c) { tot += static_cast<long long>(c) * __ldg(a.q + id); }); };
  auto scan = [&](auto&& f) { walk(f, [](int, int) {}); };
  const int need = row_select(first, scan, m, sm, o_id, o_term, o.len + p);
  for (int i = tid; i < m; i += kTopkThreads) {
    long long v = 0;
    if (i < need) { const int id = sm.id[i]; v = static_cast<long long>(__ldg(row + id)) * __ldg(a.q + id); }
    o_num[i] = v;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, off);
  if (lane == 0 && tot) atomicAdd(&s_total, static_cast<unsigned long long>(tot));
  __syncthreads();
  if (tid == 0) {
    const long long total = static_cast<long long>(s_total);
    o.count[p] = sm.valid;
    o.total[p] = total;
    o.score[p] = __dmul_rn(__ll2double_rn(total), a.rs[kModel == MODEL_UBM ? u : s]);
  }
}

int launch_explain_pairs(int model, const ExplainArgs& a, int n, int m, const ExplainOut& o, cudaStream_t st) {
  if (n <= 0) return 0;
  if (m <= 0 || m > kTopkCap / 2 || (model != MODEL_UBM && model != MODEL_IBM)) return -2;
  auto kern = model == MODEL_UBM ? explain_pairs_kernel<MODEL_UBM> : explain_pairs_kernel<MODEL_IBM>;
  kern<<<n, kTopkThreads, 0, st>>>(a, n, m, o);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mr
