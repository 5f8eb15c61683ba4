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
//   long rows: exact int32 count rows from the count engines (mrscore.cu count_rows), then similar_row_topk_kernel, one CTA per row: the
//     exact path of topk_kernel (maximum, linear histogram, bin of the k-th key, MSD radix select inside a crowded bin, collect, bitonic sort).
// kSelf: similar songs exclude the query song from its own list; a train user is never the test user asking, so similar users exclude none.
#include <climits>

#include "mr_common.cuh"
#include "mr_kernels.h"

namespace mr {

__device__ __forceinline__ double sim_score(int g, double sq_i, double sq_s) {
  const double den = __dmul_rn(sq_i, sq_s);
  return den != 0.0 ? __ddiv_rn(static_cast<double>(g), den) : 0.0;   // naive_*_cos: denominator != 0 ? numerator / denominator : 0
}

__device__ __forceinline__ unsigned long long key_bits(double x) { return static_cast<unsigned long long>(__double_as_longlong(x)); }

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

// bitonic sort of n_pad (key, song) pairs, "better first": key descending, then song ascending
__device__ void bitonic_keys(unsigned long long* key, int* song, int n_pad) {
  __syncthreads();
  for (int size = 2; size <= n_pad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < n_pad / 2; i += blockDim.x) {
        const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
        const unsigned long long ka = key[lo], kb = key[hi];
        const int sa = song[lo], sb = song[hi];
        const bool a_better = ka > kb || (ka == kb && sa < sb);
        if (a_better != ((lo & size) == 0)) { key[lo] = kb; key[hi] = ka; song[lo] = sb; song[hi] = sa; }
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
constexpr int kSimThreads = 512;
constexpr int kSimCap = 2048;     // candidate buffer, bitonic-sorted in shared memory
constexpr int kSimBins = 2048;

// f(song, key bits, candidate) for 4 songs per thread per step, the same number of times by every thread (f may use warp collectives)
template <bool kSelf, class F>
__device__ __forceinline__ void scan_counts(const int32_t* __restrict__ g, int n_songs, int self, double sq_i, const double* __restrict__ sq_c, F&& f) {
  for (int base0 = 0; base0 < n_songs; base0 += 4 * kSimThreads) {
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
__global__ void __launch_bounds__(kSimThreads, 2)
similar_row_topk_kernel(const int* __restrict__ rows, int n_rows, const int32_t* __restrict__ g, long long ldg, int n_songs,
                        const double* __restrict__ sq_q, const double* __restrict__ sq_c, int k, int* __restrict__ out_song,
                        double* __restrict__ out_score, int* __restrict__ out_len) {
  __shared__ unsigned long long s_key[kSimCap];
  __shared__ int s_song[kSimCap];
  __shared__ int s_hist[kSimBins];
  __shared__ unsigned long long s_max[kSimThreads / 32];
  __shared__ int s_count, s_valid;
  __shared__ int s_ctl[3];     // 0: chosen bin / digit, 1: keys strictly above it, 2: keys in it
  const int r = blockIdx.x;
  if (r >= n_rows) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int self = rows[r];
  const double sq_i = sq_q[self];
  const int32_t* row = g + static_cast<long long>(r) * ldg;
  int* o_song = out_song + static_cast<long long>(r) * k;
  double* o_score = out_score + static_cast<long long>(r) * k;
  // ---- maximum key and number of candidates
  if (tid == 0) { s_valid = 0; s_count = 0; }
  __syncthreads();
  unsigned long long mx = 0; int nv = 0;
  scan_counts<kSelf>(row, n_songs, self, sq_i, sq_c, [&](int, unsigned long long kb, bool ok) { if (ok) { ++nv; mx = kb > mx ? kb : mx; } });
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xffffffffu, mx, o); mx = other > mx ? other : mx; nv += __shfl_xor_sync(0xffffffffu, nv, o); }
  if (lane == 0) { s_max[warp] = mx; atomicAdd(&s_valid, nv); }
  for (int i = tid; i < kSimBins; i += kSimThreads) s_hist[i] = 0;
  __syncthreads();
  mx = 0;
  for (int i = 0; i < kSimThreads / 32; ++i) mx = s_max[i] > mx ? s_max[i] : mx;
  const int need = min(k, s_valid);
  if (need == 0) {
    for (int i = tid; i < k; i += kSimThreads) { o_song[i] = -1; o_score[i] = 0.0; }
    if (tid == 0) out_len[r] = 0;
    return;
  }
  const double max_score = __longlong_as_double(static_cast<long long>(mx));
  const double scale = max_score > 0.0 ? __ddiv_rn(static_cast<double>(kSimBins - 1), max_score) : 0.0;
  auto bin_of = [&](unsigned long long kb) -> uint32_t {   // monotone in the key
    const int d = __double2int_rz(__dmul_rn(__longlong_as_double(static_cast<long long>(kb)), scale));
    return static_cast<uint32_t>(d > kSimBins - 1 ? kSimBins - 1 : d);
  };
  // ---- linear histogram of the candidates, then the bin holding the need-th best key (warp 0, suffix search)
  scan_counts<kSelf>(row, n_songs, self, sq_i, sq_c, [&](int, unsigned long long kb, bool ok) { hist_add(s_hist, ok ? bin_of(kb) : 0u, ok, lane); });
  __syncthreads();
  if (warp == 0) {
    int part = 0;
    for (int i = 0; i < kSimBins / 32; ++i) part += s_hist[lane * (kSimBins / 32) + i];
    int above_lane = 0;
    for (int l = 0; l < 32; ++l) { const int pp = __shfl_sync(0xffffffffu, part, l); if (l > lane) above_lane += pp; }
    if (above_lane < need && above_lane + part >= need) {
      int cum = above_lane, chosen = lane * (kSimBins / 32);
      for (int i = kSimBins / 32 - 1; i >= 0; --i) {
        const int bin = lane * (kSimBins / 32) + i;
        if (cum + s_hist[bin] >= need) { chosen = bin; break; }
        cum += s_hist[bin];
      }
      s_ctl[0] = chosen; s_ctl[1] = cum; s_ctl[2] = s_hist[chosen];
    }
  }
  __syncthreads();
  const uint32_t cbin = static_cast<uint32_t>(s_ctl[0]);
  int above = s_ctl[1];
  unsigned long long phi = 0; uint32_t plo = 0; int nd = 0;
  if (above + s_ctl[2] > kSimCap) {
    // crowded bin (thousands of exact ties, e.g. g = 1 against songs of one degree): MSD radix select of the (need - above) best keys in it
    for (;;) {
      __syncthreads();
      for (int i = tid; i < 256; i += kSimThreads) s_hist[i] = 0;
      __syncthreads();
      scan_counts<kSelf>(row, n_songs, self, sq_i, sq_c, [&](int s, unsigned long long kb, bool ok) {
        const uint32_t inv = ~static_cast<uint32_t>(s);
        ok = ok && bin_of(kb) == cbin && prefix_cmp(kb, inv, phi, plo, nd) == 0;
        hist_add(s_hist, ok ? key_digit(kb, inv, nd) : 0u, ok, lane);
      });
      __syncthreads();
      if (tid == 0) {
        const int want = need - above;
        int cum = 0, chosen = 0;
        for (int d = 255; d >= 0; --d) {
          if (cum + s_hist[d] >= want) { chosen = d; break; }
          cum += s_hist[d];
        }
        s_ctl[0] = chosen; s_ctl[1] = above + cum; s_ctl[2] = s_hist[chosen];
      }
      __syncthreads();
      const int chosen = s_ctl[0];
      above = s_ctl[1];
      if (nd < 8) phi |= static_cast<unsigned long long>(chosen) << (56 - 8 * nd);
      else plo |= static_cast<uint32_t>(chosen) << (24 - 8 * (nd - 8));
      ++nd;
      if (above + s_ctl[2] <= kSimCap || nd == 12) break;
    }
  }
  // ---- collect every key in a higher bin, plus the keys of bin cbin at or above the radix prefix
  __syncthreads();
  scan_counts<kSelf>(row, n_songs, self, sq_i, sq_c, [&](int s, unsigned long long kb, bool ok) {
    if (ok) {
      const uint32_t bn = bin_of(kb);
      ok = bn > cbin || (bn == cbin && prefix_cmp(kb, ~static_cast<uint32_t>(s), phi, plo, nd) >= 0);
    }
    const uint32_t m = __ballot_sync(0xffffffffu, ok);
    if (m) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&s_count, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (ok) {
        const int pos = base + __popc(m & ((1u << lane) - 1));
        if (pos < kSimCap) { s_key[pos] = kb; s_song[pos] = s; }
      }
    }
  });
  __syncthreads();
  const int n_cand = min(s_count, kSimCap);
  int n_sort = 1;
  while (n_sort < n_cand) n_sort <<= 1;
  for (int i = n_cand + tid; i < n_sort; i += kSimThreads) { s_key[i] = 0; s_song[i] = INT_MAX; }   // sorts last
  bitonic_keys(s_key, s_song, n_sort);
  for (int i = tid; i < k; i += kSimThreads) {
    if (i < need) { o_song[i] = s_song[i]; o_score[i] = __longlong_as_double(static_cast<long long>(s_key[i])); }
    else { o_song[i] = -1; o_score[i] = 0.0; }
  }
  if (tid == 0) out_len[r] = need;
}

int launch_similar_rows(const int* rows, int n_rows, const int32_t* g, long long ldg, int n_cols, const SimLists& l, int k, int* out_song,
                        double* out_score, int* out_len, cudaStream_t st) {
  if (n_rows <= 0) return 0;
  if (k <= 0 || k > kSimCap / 2) return -2;
  auto kern = l.self ? similar_row_topk_kernel<true> : similar_row_topk_kernel<false>;
  kern<<<n_rows, kSimThreads, 0, st>>>(rows, n_rows, g, ldg, n_cols, l.sq_q, l.sq_c, k, out_song, out_score, out_len);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mr
