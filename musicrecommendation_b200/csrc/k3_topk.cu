// k3_topk.cu — kernel K3: fp64 score finalisation, model blends and the per-user top-k select.
//
// Score finalisation (canonical arithmetic, DESIGN.md §3):   ubm = (double)Sint_u * rsa[u],  ibm = (double)Sint_i * rsd[s]
// Blends (MusicRecommender.scala, element i = index of (user, song) in the (user asc, song asc) order of main.scala:57-59):
//   LinearCombination   rank1 * alpha + rank2 * (1 - alpha)                         MR:328   (rank1 = UBM, rank2 = IBM)
//   Aggregation         i < (pct * N).toInt ? ibm : ubm                              MR:372, 381-382
//   Stochastic          java.util.Random(seed): (i+1)-th nextFloat() < prob ? ibm : ubm   MR:439, 447 (sequential version)
// Top-k (new derived output, SURVEY.md §8a A8): per test user, unlistened songs ordered by score descending, then song id
//   ascending; first min(k, S - |I_u|).
// All fp64 products/sums use explicit round-to-nearest intrinsics so that no FMA contraction can change the bits.
#include "mr_common.cuh"
#include "mr_kernels.h"

namespace mr {

// ---------------------------------------------------------------- listened-pair sentinel (getModel's filter, MR:109)
// te_end[u] = end of the row's scored columns: te_ptr[u + 1], or — with a song window — the end of the in-window prefix of the row
__global__ void mask_listened_kernel(const long long* __restrict__ te_ptr, const long long* __restrict__ te_end, const int* __restrict__ te_col,
                                     int u0, int n_users, long long* sint_u, long long* sint_i, long long spitch) {
  const int b = blockIdx.x;
  if (b >= n_users) return;
  const long long beg = te_ptr[u0 + b], end = te_end[u0 + b];
  for (long long i = beg + threadIdx.x; i < end; i += blockDim.x) {
    const int s = te_col[i];
    if (sint_u) sint_u[static_cast<long long>(b) * spitch + s] = kListened;
    if (sint_i) sint_i[static_cast<long long>(b) * spitch + s] = kListened;
  }
}

int launch_mask_listened(const long long* te_ptr, const long long* te_end, const int* te_col, int u0, int n_users, long long* sint_u,
                         long long* sint_i, long long spitch, cudaStream_t st) {
  if (n_users <= 0) return 0;
  mask_listened_kernel<<<n_users, 128, 0, st>>>(te_ptr, te_end, te_col, u0, n_users, sint_u, sint_i, spitch);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- dense fp64 model rows (small configs / parity probes)
__global__ void dense_scores_kernel(int model, const long long* __restrict__ sint, long long spitch, int u0, int n_songs,
                                    const double* __restrict__ rsa, const double* __restrict__ rsd, double* __restrict__ out) {
  const int b = blockIdx.y;
  const double rsu = rsa[u0 + b];
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n_songs; s += gridDim.x * blockDim.x) {
    const long long v = sint[static_cast<long long>(b) * spitch + s];
    double r;
    if (v < 0) r = __longlong_as_double(0x7ff8000000000000LL);   // NaN marks a pair the reference does not emit
    else r = model == MODEL_UBM ? __dmul_rn(__ll2double_rn(v), rsu) : __dmul_rn(__ll2double_rn(v), rsd[s]);
    out[static_cast<long long>(b) * n_songs + s] = r;
  }
}

int launch_dense_scores(int model, const long long* sint, long long spitch, int u0, int n_users, int n_songs, const double* rsa,
                        const double* rsd, double* out, cudaStream_t st) {
  if (n_users <= 0 || n_songs <= 0) return 0;
  int gx = (n_songs + 255) / 256;
  if (gx > 1024) gx = 1024;
  dense_scores_kernel<<<dim3(gx, n_users), 256, 0, st>>>(model, sint, spitch, u0, n_songs, rsa, rsd, out);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// Columns of a chunk of dense model rows, transposed: out[i * out_ld + u_base + r] = dense[r][songs[i]] — the per-song granularity of
// distributed.scala's getRanks2(song) (DIST:214-221, 285-292): one song against every test user.
__global__ void gather_columns_kernel(const double* __restrict__ dense, int n_rows, int n_songs, const int* __restrict__ songs, int n_sel,
                                      double* __restrict__ out, long long out_ld, int u_base) {
  const long long n = static_cast<long long>(n_sel) * n_rows;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < n; t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(t / n_rows), r = static_cast<int>(t % n_rows);
    out[i * out_ld + u_base + r] = dense[static_cast<long long>(r) * n_songs + songs[i]];
  }
}

int launch_gather_columns(const double* dense, int n_rows, int n_songs, const int* songs, int n_sel, double* out, long long out_ld, int u_base,
                          cudaStream_t st) {
  if (n_rows <= 0 || n_sel <= 0) return 0;
  const long long n = static_cast<long long>(n_sel) * n_rows;
  const int grid = static_cast<int>(n + 255 < 256LL * 148 * 8 ? (n + 255) / 256 : 148 * 8);
  gather_columns_kernel<<<grid, 256, 0, st>>>(dense, n_rows, n_songs, songs, n_sel, out, out_ld, u_base);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- java.util.Random (48-bit LCG) with O(log n) jump-ahead
constexpr unsigned long long kLcgA = 0x5DEECE66DULL, kLcgC = 0xBULL, kLcgMask = (1ULL << 48) - 1;

__host__ __device__ inline unsigned long long lcg_jump(unsigned long long state, unsigned long long n) {
  unsigned long long acc_mul = 1, acc_add = 0, cur_mul = kLcgA, cur_add = kLcgC;
  while (n) {
    if (n & 1) { acc_mul = (acc_mul * cur_mul) & kLcgMask; acc_add = (acc_add * cur_mul + cur_add) & kLcgMask; }
    cur_add = ((cur_mul + 1) * cur_add) & kLcgMask;
    cur_mul = (cur_mul * cur_mul) & kLcgMask;
    n >>= 1;
  }
  return (acc_mul * state + acc_add) & kLcgMask;
}

// Selection bit per (user, song): 1 -> take the IBM score, 0 -> UBM.  One thread per 64-song word.
__global__ void select_bits_kernel(BlendParams bp, const long long* __restrict__ te_ptr, const int* __restrict__ te_col, int u0,
                                   int n_songs, uint64_t* __restrict__ sel, long long sel_pitch_words) {
  const int b = blockIdx.y;
  const int u = u0 + b;
  const int n_words = (n_songs + 63) / 64;
  const long long beg = te_ptr[u], end = bp.te_end[u];
  const int* row = te_col + beg;
  const int row_len = static_cast<int>(end - beg);
  for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += gridDim.x * blockDim.x) {
    const int s0 = w * 64;
    int lo = 0, hi = row_len;                       // listened songs with id < s0
    while (lo < hi) { const int m = (lo + hi) >> 1; if (row[m] < s0) lo = m + 1; else hi = m; }
    int p = lo;
    long long idx = bp.pair_base[u] + s0 - p;        // index of the first unlistened song >= s0 in MAIN:57-59 order
    unsigned long long state = 0;
    if (bp.model == MODEL_STOCH) state = lcg_jump((bp.seed ^ kLcgA) & kLcgMask, static_cast<unsigned long long>(idx));
    uint64_t bits = 0;
    const int s_end = min(s0 + 64, n_songs);
    for (int s = s0; s < s_end; ++s) {
      if (p < row_len && row[p] == s) { ++p; continue; }   // listened: not in the model, consumes no index / no draw
      bool pick;
      if (bp.model == MODEL_AGG) {
        pick = idx < bp.agg_threshold;
      } else {
        state = (state * kLcgA + kLcgC) & kLcgMask;
        const float f = static_cast<float>(static_cast<int>(state >> 24)) / static_cast<float>(1 << 24);   // nextFloat()
        pick = static_cast<double>(f) < bp.prob;
      }
      bits |= static_cast<uint64_t>(pick) << (s - s0);
      ++idx;
    }
    sel[static_cast<long long>(b) * sel_pitch_words + w] = bits;
  }
}

int launch_select_bits(const BlendParams& bp, const long long* te_ptr, const int* te_col, int u0, int n_users, int n_songs,
                       uint64_t* sel, long long sel_pitch_words, cudaStream_t st) {
  if (n_users <= 0 || n_songs <= 0) return 0;
  const int n_words = (n_songs + 63) / 64;
  int gx = (n_words + 127) / 128;
  select_bits_kernel<<<dim3(gx, n_users), 128, 0, st>>>(bp, te_ptr, te_col, u0, n_songs, sel, sel_pitch_words);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// AGG's select bits as one column per user.  In select_bits_kernel the index of an unlistened column s is pair_base[u] + f(s) with
// f(s) = s - (listened songs < s), and the bit is idx < agg_threshold, i.e. f(s) < m = agg_threshold - pair_base[u].  f grows by one
// per unlistened column, so the unlistened columns with bit 1 are exactly those below split[u] = m + #{j : row[j] - j < m} (row[j] - j is
// non-decreasing along the ascending row, so that count is a binary search), clamped to [0, n_songs].
__global__ void agg_split_kernel(BlendParams bp, const long long* __restrict__ te_ptr, const int* __restrict__ te_col, int n_users,
                                 int n_songs, int* __restrict__ split) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n_users) return;
  const long long m = bp.agg_threshold - bp.pair_base[u];
  if (m <= 0) { split[u] = 0; return; }
  if (m >= n_songs) { split[u] = n_songs; return; }
  const long long beg = te_ptr[u];
  const int* row = te_col + beg;
  int lo = 0, hi = static_cast<int>(bp.te_end[u] - beg);
  while (lo < hi) { const int j = (lo + hi) >> 1; if (row[j] - j < m) lo = j + 1; else hi = j; }
  split[u] = static_cast<int>(m + lo < n_songs ? m + lo : n_songs);
}

int launch_agg_split(const BlendParams& bp, const long long* te_ptr, const int* te_col, int n_users, int n_songs, int* split, cudaStream_t st) {
  if (n_users <= 0) return 0;
  agg_split_kernel<<<(n_users + 255) / 256, 256, 0, st>>>(bp, te_ptr, te_col, n_users, n_songs, split);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- top-k select
// One CTA per test user.  Keys are the composite (score bits : 64, ~song : 32), so "larger key" == "better" with ties broken by
// the smaller song id; scores are >= 0, so their IEEE bit patterns order like unsigned integers.
// Every bin map below is monotone in the key and only ever a PRE-FILTER; exactness comes from the final sort of the collected keys.
//   long rows (S > 16384), fast path — 1.25 passes over the row:
//     A1  maximum over every 8th chunk of the row (1/8 of it)
//     A2  2048-bin logarithmic histogram (64 bins per binade below the maximum) over the same chunks; the bin above which about
//         1.46 k / 8 sampled keys lie gives the cut
//     B   ONE full pass collects the keys at or above the cut; accepted when min(k, valid) <= collected <= 2048
//     For the pure UBM model the score (double)Sint * rsu is strictly monotone in the integer numerator, so A1/A2/B work on the
//     integers (one 64-bit compare per song in B) and only the collected keys are converted to fp64.  The other models evaluate the
//     fp64 score per song (blends included) and compare its bit pattern.
//     valid = S - |I_u| needs no counting: the listened pairs are exactly the sentinel entries (getModel's filter, MR:109).
//   otherwise / on reject:  exact path — full linear histogram, the bin holding the k-th best key, collect pass
//   degenerate rows (thousands of exact ties such as all-zero rows, or a bin more crowded than the candidate buffer): exact
//                           most-significant-digit radix select (8-bit digits of the 96-bit key) inside the chosen bin
// The collected keys (<= 2048) are bitonic-sorted exactly in shared memory: key descending, song ascending.
// The exact select (bin search, radix select, collect, sort, write-out) is shared with similar_row_topk_kernel (mr_common.cuh).

struct KeyCtx {
  int model; double rsu, alpha, oma;
  const long long* su; const long long* si; const double* rsd; const uint64_t* sel;
};

// L2 prefetches.  The select streams a row in dependent rounds (a thread has one or two 32-byte loads in flight, then computes), so a
// round costs a full DRAM latency.  Short rows (a song partition: a few hundred KB per user) are pulled into L2 whole by a handful of
// bulk prefetches when the CTA starts — the sampled passes and the collect pass then hit L2, and the row crosses HBM once instead of
// 1.25-1.5 times; long rows prefetch the lines the collect pass will need kPrefetchRounds rounds ahead.
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void prefetch_l2_line(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
constexpr int kPrefetchRounds = 4;
constexpr int kShortRow = 65536;      // rows up to this many songs are prefetched whole

__device__ __forceinline__ void prefetch_row(const long long* row, int n_songs) {
  if (!row) return;
  const long long bytes = static_cast<long long>((n_songs + 31) / 32 * 32) * 8;      // rows are padded to 32 songs
  for (long long off = static_cast<long long>(threadIdx.x) * 2048; off < bytes; off += static_cast<long long>(kTopkThreads) * 2048)
    prefetch_l2_bulk(reinterpret_cast<const char*>(row) + off, static_cast<uint32_t>(min(2048LL, bytes - off)));
}

// Stream the row: f(song, key bits, valid) is called for 4 songs per thread per iteration, the same number of times by every
// thread of the CTA (so f may use warp collectives); valid is false for listened pairs and past the end of the row.
// ubm_min: for the pure UBM model the score is monotone in the integer numerator, so the caller may pass the smallest numerator
// worth looking at; rows entries below it are reported as valid with key 0 and cost no fp64 work at all.
template <class F>
__device__ __forceinline__ void scan_row(const KeyCtx& c, int n_songs, F&& f, int chunk_stride = 1, long long ubm_min = 0) {
  for (int base = 0; base < n_songs; base += 4 * kTopkThreads * chunk_stride) {
    const int s = base + 4 * static_cast<int>(threadIdx.x);
    long long a[4] = {-1, -1, -1, -1}, b[4] = {-1, -1, -1, -1};
    double rd[4] = {0, 0, 0, 0};
    uint64_t selw = 0;
    if (s < n_songs) {   // rows are padded to a multiple of 32 songs, so the 4-wide loads stay inside the row
      if (c.model != MODEL_IBM) {
        const longlong2 x = *reinterpret_cast<const longlong2*>(c.su + s), y = *reinterpret_cast<const longlong2*>(c.su + s + 2);
        a[0] = x.x; a[1] = x.y; a[2] = y.x; a[3] = y.y;
      }
      if (c.model != MODEL_UBM) {
        const longlong2 x = *reinterpret_cast<const longlong2*>(c.si + s), y = *reinterpret_cast<const longlong2*>(c.si + s + 2);
        b[0] = x.x; b[1] = x.y; b[2] = y.x; b[3] = y.y;
#pragma unroll
        for (int t = 0; t < 4; ++t) rd[t] = s + t < n_songs ? c.rsd[s + t] : 0.0;
      }
      if (c.model >= MODEL_AGG) selw = c.sel[s >> 6] >> (s & 63);
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      bool ok = s + t < n_songs;
      if (c.model != MODEL_IBM) ok = ok && a[t] >= 0;
      if (c.model != MODEL_UBM) ok = ok && b[t] >= 0;
      unsigned long long kb = 0;
      if (ok && (c.model != MODEL_UBM || a[t] >= ubm_min)) kb = static_cast<unsigned long long>(__double_as_longlong(
                  blend_score(c.model, a[t], b[t], c.rsu, rd[t], c.alpha, c.oma, (selw >> t) & 1ULL)));
      f(s + t, kb, ok);
    }
  }
}

// ---- fast path helpers.  "Proxy" p of a song: the integer numerator (pure UBM) or the fp64 score bits (every other model); the
// logarithmic bin of a proxy keeps its exponent and 6 mantissa bits: lb(p) = bits(float_rz(p)) >> 17 resp. bits(double) >> 46.
__device__ __forceinline__ uint32_t logbits_int(long long a) { return a > 0 ? __float_as_uint(__ll2float_rz(a)) >> 17 : 0u; }
__device__ __forceinline__ uint32_t logbits_key(unsigned long long kb) { return static_cast<uint32_t>(kb >> 46); }

// Visit the row 4 songs per thread per step, two steps in flight: f(song of the first of 4, a[4], b[4], rsd[4], select word) with a = -1 /
// b = -1 where the model does not use that panel; entries past the end of the row are reported as listened (-1).
template <bool kInt, class F>
__device__ __forceinline__ void visit_row(const KeyCtx& c, int n_songs, int chunk_stride, F&& f) {
  constexpr int kSteps = kInt ? 2 : 1;                          // steps in flight (the fp64 models already load three arrays per step)
  const int step = 4 * kTopkThreads * chunk_stride;
  const bool ahead = chunk_stride == 1 && n_songs > kShortRow && (threadIdx.x & 3) == 0;   // one thread per 128-byte line
  for (int base0 = 0; base0 < n_songs; base0 += kSteps * step) {   // the same trip count for every thread: f may use warp collectives
    const int base = base0 + 4 * static_cast<int>(threadIdx.x);
    if (ahead) {
#pragma unroll
      for (int h = 0; h < kSteps; ++h) {
        const int sp = base + (kPrefetchRounds * kSteps + h) * step;
        if (sp < n_songs) {
          if (kInt || c.model != MODEL_IBM) prefetch_l2_line(c.su + sp);
          if (!kInt && c.model != MODEL_UBM) prefetch_l2_line(c.si + sp);
        }
      }
    }
    long long a[kSteps][4], b[kSteps][4]; double rd[kSteps][4]; uint64_t selw[kSteps];
#pragma unroll
    for (int h = 0; h < kSteps; ++h) {
      const int s = base + h * step;
      selw[h] = 0;
#pragma unroll
      for (int t = 0; t < 4; ++t) { a[h][t] = -1; b[h][t] = -1; rd[h][t] = 0.0; }
      if (s < n_songs) {   // rows are padded to a multiple of 32 songs, so the 4-wide loads stay inside the row
        if (kInt || c.model != MODEL_IBM) {
          const longlong2 x = __ldcs(reinterpret_cast<const longlong2*>(c.su + s)), y = __ldcs(reinterpret_cast<const longlong2*>(c.su + s + 2));
          a[h][0] = x.x; a[h][1] = x.y; a[h][2] = y.x; a[h][3] = y.y;
        }
        if (!kInt && c.model != MODEL_UBM) {
          const longlong2 x = __ldcs(reinterpret_cast<const longlong2*>(c.si + s)), y = __ldcs(reinterpret_cast<const longlong2*>(c.si + s + 2));
          b[h][0] = x.x; b[h][1] = x.y; b[h][2] = y.x; b[h][3] = y.y;
          if (s + 4 <= n_songs) {
            const double2 r0 = __ldg(reinterpret_cast<const double2*>(c.rsd + s)), r1 = __ldg(reinterpret_cast<const double2*>(c.rsd + s + 2));
            rd[h][0] = r0.x; rd[h][1] = r0.y; rd[h][2] = r1.x; rd[h][3] = r1.y;
          } else {
#pragma unroll
            for (int t = 0; t < 4; ++t) if (s + t < n_songs) rd[h][t] = __ldg(c.rsd + s + t);
          }
        }
        if (!kInt && c.model >= MODEL_AGG) selw[h] = c.sel[s >> 6] >> (s & 63);
        if (s + 4 > n_songs) {   // only the last quad of a row can reach past its end
#pragma unroll
          for (int t = 0; t < 4; ++t) if (s + t >= n_songs) { a[h][t] = -1; b[h][t] = -1; }
        }
      }
    }
#pragma unroll
    for (int h = 0; h < kSteps; ++h) f(base + h * step, a[h], b[h], rd[h], selw[h]);
  }
}

// proxy of one song (0 = not a candidate: listened, past the end, or a zero score — zero scores are only ever needed when fewer than k
// positive ones exist, which the acceptance test catches)
template <bool kInt>
__device__ __forceinline__ unsigned long long proxy_of(const KeyCtx& c, long long a, long long b, double rd, bool pick) {
  if (kInt) return a > 0 ? static_cast<unsigned long long>(a) : 0ULL;
  bool ok = true;
  if (c.model != MODEL_IBM) ok = ok && a >= 0;
  if (c.model != MODEL_UBM) ok = ok && b >= 0;
  return ok ? static_cast<unsigned long long>(__double_as_longlong(blend_score(c.model, a, b, c.rsu, rd, c.alpha, c.oma, pick))) : 0ULL;
}

// Pass B of the pure IBM model.  The score (double)Sint_i * rsd[s] depends on the song, so there is no integer threshold; instead a
// round-up fp32 product bounds the fp64 score from above — float_ru(Sint) * rsd_up[s] (rsd_up = rsd rounded up to fp32, product
// rounded up) >= the exact product >= its fp64 rounding — and only songs whose bound reaches the threshold (rounded down to fp32)
// are evaluated exactly.  12 bytes per song instead of 16, no fp64 work per song, and two steps of loads in flight per thread.
__device__ __forceinline__ void ibm_collect_pass(const KeyCtx& c, const float* __restrict__ rsd_up, int n_songs, unsigned long long thr,
                                                 unsigned long long* s_key, int* s_song, int* s_count) {
  const float t_f = __double2float_rd(__longlong_as_double(static_cast<long long>(thr)));
  constexpr int kSteps = 2;
  const int step = 4 * kTopkThreads;
  const bool ahead = n_songs > kShortRow && (threadIdx.x & 3) == 0;
  for (int base0 = 0; base0 < n_songs; base0 += kSteps * step) {
    if (ahead) {
#pragma unroll
      for (int h = 0; h < kSteps; ++h) {
        const int sp = base0 + (kPrefetchRounds * kSteps + h) * step + 4 * static_cast<int>(threadIdx.x);
        if (sp < n_songs) prefetch_l2_line(c.si + sp);
      }
    }
    long long b[kSteps][4]; float r[kSteps][4];
#pragma unroll
    for (int h = 0; h < kSteps; ++h) {
      const int s = base0 + h * step + 4 * static_cast<int>(threadIdx.x);
#pragma unroll
      for (int t = 0; t < 4; ++t) { b[h][t] = -1; r[h][t] = 0.f; }
      if (s < n_songs) {
        const longlong2 x = __ldcs(reinterpret_cast<const longlong2*>(c.si + s)), y = __ldcs(reinterpret_cast<const longlong2*>(c.si + s + 2));
        b[h][0] = x.x; b[h][1] = x.y; b[h][2] = y.x; b[h][3] = y.y;
        if (s + 4 <= n_songs) { const float4 f = __ldg(reinterpret_cast<const float4*>(rsd_up + s)); r[h][0] = f.x; r[h][1] = f.y; r[h][2] = f.z; r[h][3] = f.w; }
        else {
#pragma unroll
          for (int t = 0; t < 4; ++t) { if (s + t < n_songs) r[h][t] = __ldg(rsd_up + s + t); else b[h][t] = -1; }
        }
      }
    }
#pragma unroll
    for (int h = 0; h < kSteps; ++h) {
      const int s = base0 + h * step + 4 * static_cast<int>(threadIdx.x);
      // songs whose upper bound reaches the threshold are rare (a few per thousand): exact score, and one shared-memory atomic per
      // surviving song — no ballots or shuffles in the common case
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        if (b[h][t] > 0 && __fmul_ru(__ll2float_ru(b[h][t]), r[h][t]) >= t_f) {
          const unsigned long long kb = static_cast<unsigned long long>(__double_as_longlong(__dmul_rn(__ll2double_rn(b[h][t]), __ldg(c.rsd + s + t))));
          if (kb >= thr) {
            const int pos = atomicAdd(s_count, 1);
            if (pos < kTopkCap) { s_key[pos] = kb; s_song[pos] = s + t; }
          }
        }
      }
    }
  }
}

// Fast path for long rows; returns true when the candidate buffer holds a superset of the top `need` keys (s_count of them).
// *scale_out = the linear-bin scale of the exact path (from the sampled maximum), so a rejected row continues there.
template <bool kInt>
__device__ __forceinline__ bool topk_fast_path(const KeyCtx& c, int n_songs, int stride, int k, int need, unsigned long long* s_key, int* s_song,
                                               int* s_hist, unsigned long long* s_max, int* s_count, int* s_ctl, double* max_score_out, const float* __restrict__ rsd_up) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // ---- A1: sampled maximum of the proxy
  unsigned long long mx = 0;
  visit_row<kInt>(c, n_songs, stride, [&](int, const long long* a, const long long* b, const double* rd, uint64_t selw) {
#pragma unroll
    for (int t = 0; t < 4; ++t) { const unsigned long long p = proxy_of<kInt>(c, a[t], b[t], rd[t], (selw >> t) & 1ULL); mx = p > mx ? p : mx; }
  });
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xffffffffu, mx, o); mx = other > mx ? other : mx; }
  if (lane == 0) s_max[warp] = mx;
  for (int i = tid; i < kTopkBins; i += kTopkThreads) s_hist[i] = 0;
  if (tid == 0) *s_count = 0;
  __syncthreads();
  mx = 0;
  for (int i = 0; i < kTopkThreads / 32; ++i) mx = s_max[i] > mx ? s_max[i] : mx;
  *max_score_out = kInt ? __dmul_rn(__ll2double_rn(static_cast<long long>(mx)), c.rsu) : __longlong_as_double(static_cast<long long>(mx));
  const uint32_t top = kInt ? logbits_int(static_cast<long long>(mx)) : logbits_key(mx);
  auto bin_of = [&](unsigned long long p) -> uint32_t {     // 0 for p == 0; monotone in p; the sampled maximum lands in the top bin
    if (p == 0) return 0u;
    const uint32_t lb = kInt ? logbits_int(static_cast<long long>(p)) : logbits_key(p);
    const int d = static_cast<int>(kTopkBins - 1) - (static_cast<int>(top) - static_cast<int>(lb));
    return static_cast<uint32_t>(d < 1 ? 1 : (d > kTopkBins - 1 ? kTopkBins - 1 : d));
  };
  // ---- A2: histogram over the same chunks
  visit_row<kInt>(c, n_songs, stride, [&](int, const long long* a, const long long* b, const double* rd, uint64_t selw) {
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const unsigned long long p = proxy_of<kInt>(c, a[t], b[t], rd[t], (selw >> t) & 1ULL);
      hist_add(s_hist, bin_of(p), p != 0, lane);
    }
  });
  __syncthreads();
  // ---- the cut: highest bin with at least `want` sampled keys in it or above, bin 0 when the sample holds fewer; bins >= 2 only, so the
  // threshold is a real proxy value.  Keys aimed at above the cut: k plus 3 sigma of the sampling noise (every 8th chunk: sigma of the
  // full-row count ~ sqrt(8 * want) ~ 75 for k = 500) — 730 for k = 500, so that the collected keys land in [~520, ~950]: at least k, and
  // the final sort stays at 1024 slots
  if (warp == 0) find_bin(s_hist, (k + (46 * k) / 100 + stride - 1) / stride, false, s_ctl);
  __syncthreads();
  const int cut = s_ctl[0];
  if (cut < 2) return false;                     // too few positive keys in the sample: let the exact path decide
  // smallest proxy whose bin is >= cut: log bits >= top - (2047 - cut)
  const long long lb_cut = static_cast<long long>(top) - (kTopkBins - 1 - cut);
  if (lb_cut <= 0) return false;
  unsigned long long thr;
  if (kInt) thr = static_cast<unsigned long long>(__float2ll_ru(__uint_as_float(static_cast<uint32_t>(lb_cut) << 17)));
  else thr = static_cast<unsigned long long>(lb_cut) << 46;
  // ---- B: one full pass, collect every song whose proxy is at or above the threshold
  if (!kInt && c.model == MODEL_IBM && rsd_up) {
    ibm_collect_pass(c, rsd_up, n_songs, thr, s_key, s_song, s_count);
    __syncthreads();
    return *s_count >= need && *s_count <= kTopkCap;
  }
  // Candidates are ~2 per thousand songs: a thread that holds some reserves their slots with ONE shared-memory atomic (no ballots or
  // shuffles in the common no-candidate case; the order inside the buffer is irrelevant, it is sorted afterwards).
  // (the integer path keeps the raw numerators in the buffer and converts the few hundred survivors to fp64 after the pass)
  const long long thr_int = static_cast<long long>(thr);            // >= 1: a listened pair (-1) or a zero score never passes
  visit_row<kInt>(c, n_songs, 1, [&](int s, const long long* a, const long long* b, const double* rd, uint64_t selw) {
    unsigned long long p[4];
    int n_ok = 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      if (kInt) { p[t] = static_cast<unsigned long long>(a[t]); n_ok += a[t] >= thr_int ? 1 : 0; }
      else { p[t] = proxy_of<kInt>(c, a[t], b[t], rd[t], (selw >> t) & 1ULL); n_ok += p[t] >= thr ? 1 : 0; }
    }
    if (n_ok) {
      int pos = atomicAdd(s_count, n_ok);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        if (kInt ? a[t] >= thr_int : p[t] >= thr) {
          if (pos < kTopkCap) { s_key[pos] = p[t]; s_song[pos] = s + t; }
          ++pos;
        }
      }
    }
  });
  if (kInt) {
    __syncthreads();
    const int n = min(*s_count, kTopkCap);
    for (int i = threadIdx.x; i < n; i += kTopkThreads)
      s_key[i] = static_cast<unsigned long long>(__double_as_longlong(__dmul_rn(__ll2double_rn(static_cast<long long>(s_key[i])), c.rsu)));
  }
  __syncthreads();
  return *s_count >= need && *s_count <= kTopkCap;
}

// Trim before the final sort: only the best `need` keys have to be ordered.  The candidates (k plus the sampling margin, ~750 for
// k = 500) would take a 1024-slot bitonic network although `need` fits 512 slots: a linear histogram of their scores finds the bin of the
// need-th best, the keys in that bin or above (>= need of them, normally < 512) are compacted to the front, and the network halves (the
// sort was 1/3 of the kernel's instructions on the 48 k-song rows of a song partition, profiles/r02_topk_partition.md).  Returns the new
// candidate count (unchanged when the keys are all tied or the chosen bin is too crowded).  A function of its own so that its registers
// do not weigh on the streaming passes of the kernel.
__device__ __noinline__ int trim_candidates(unsigned long long* s_key, int* s_song, int* s_hist, unsigned long long* s_max, int* s_ctl,
                                            int* s_count, int n_cand, int need) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long kv[2]; int sv[2];
  unsigned long long kmax = 0, kmin = ~0ULL;
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int i = tid + e * kTopkThreads;
    kv[e] = i < n_cand ? s_key[i] : 0ULL; sv[e] = i < n_cand ? s_song[i] : 0;
    if (i < n_cand) { kmax = kv[e] > kmax ? kv[e] : kmax; kmin = kv[e] < kmin ? kv[e] : kmin; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long a = __shfl_xor_sync(0xffffffffu, kmax, o), b = __shfl_xor_sync(0xffffffffu, kmin, o);
    kmax = a > kmax ? a : kmax; kmin = b < kmin ? b : kmin;
  }
  __syncthreads();                                     // every candidate is in registers; the scratch arrays are free
  if (lane == 0) s_max[warp] = kmax;
  for (int i = tid; i < kTopkBins; i += kTopkThreads) s_hist[i] = 0;
  __syncthreads();
  kmax = 0;
  for (int i = 0; i < kTopkThreads / 32; ++i) kmax = s_max[i] > kmax ? s_max[i] : kmax;
  __syncthreads();
  if (lane == 0) s_max[warp] = kmin;                   // the minimum through a second round on the same scratch array
  __syncthreads();
  kmin = ~0ULL;
  for (int i = 0; i < kTopkThreads / 32; ++i) kmin = s_max[i] < kmin ? s_max[i] : kmin;
  const double d_lo = __longlong_as_double(static_cast<long long>(kmin)), d_hi = __longlong_as_double(static_cast<long long>(kmax));
  if (!(d_hi > d_lo)) return n_cand;                   // all candidates tied (uniform across the CTA): nothing to trim by score
  const double tscale = __ddiv_rn(static_cast<double>(kTopkBins - 1), __dsub_rn(d_hi, d_lo));
  int tb[2];
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int d = __double2int_rz(__dmul_rn(__dsub_rn(__longlong_as_double(static_cast<long long>(kv[e])), d_lo), tscale));
    tb[e] = d < 0 ? 0 : (d > kTopkBins - 1 ? kTopkBins - 1 : d);                     // monotone in the key
    if (tid + e * kTopkThreads < n_cand) atomicAdd(&s_hist[tb[e]], 1);
  }
  __syncthreads();
  if (warp == 0) find_bin(s_hist, need, false, s_ctl);   // the highest bin with at least `need` keys in it or above (n_cand >= need)
  __syncthreads();
  const int tbin = s_ctl[0], kept = s_ctl[1] + s_ctl[2];
  if (kept < need || kept > kTopkThreads) return n_cand;   // (uniform) a crowded bin: keep the whole buffer
  __syncthreads();
  if (tid == 0) *s_count = 0;
  __syncthreads();
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    if (tid + e * kTopkThreads < n_cand && tb[e] >= tbin) {
      const int pos = atomicAdd(s_count, 1);
      s_key[pos] = kv[e]; s_song[pos] = sv[e];
    }
  }
  __syncthreads();
  return *s_count;
}

__global__ void __launch_bounds__(kTopkThreads, 2)
topk_kernel(BlendParams bp, const long long* __restrict__ te_ptr, const long long* __restrict__ sint_u, const long long* __restrict__ sint_i, long long spitch,
            const uint64_t* __restrict__ sel, long long sel_pitch_words, int u0, int n_songs, const double* __restrict__ rsa,
            const double* __restrict__ rsd, int k, int* __restrict__ out_song, double* __restrict__ out_score,
            int* __restrict__ out_len) {
  __shared__ unsigned long long s_key[kTopkCap];
  __shared__ int s_song[kTopkCap];
  __shared__ int s_hist[kTopkBins];
  __shared__ unsigned long long s_max[kTopkThreads / 32];
  __shared__ int s_count;
  __shared__ int s_ctl[4];     // 0: chosen bin / digit, 1: keys strictly above it, 2: keys in it, 3: need

  const int b = blockIdx.x;
  const int u = u0 + b;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  KeyCtx c;
  c.model = bp.model; c.rsu = rsa[u]; c.alpha = bp.alpha; c.oma = bp.one_minus_alpha;
  c.su = sint_u ? sint_u + static_cast<long long>(b) * spitch : nullptr;
  c.si = sint_i ? sint_i + static_cast<long long>(b) * spitch : nullptr;
  c.rsd = rsd;
  c.sel = sel ? sel + static_cast<long long>(b) * sel_pitch_words : nullptr;
  int* o_song = out_song + static_cast<long long>(u) * k;
  double* o_score = out_score + static_cast<long long>(u) * k;

  if (n_songs <= kShortRow) { prefetch_row(c.su, n_songs); prefetch_row(c.si, n_songs); }
  const int stride = n_songs > 16384 ? 8 : 1;   // the rows of a song partition (S / 8 = 48 k songs at MSD scale) take the sampled path too
  const int n_valid = n_songs - static_cast<int>(bp.te_end[u] - te_ptr[u]);   // scored pairs of this user (MR:109)
  int need = 0;
  bool collected = false;
  double max_score = 0.0;
  if (stride > 1) {
    need = min(k, n_valid);
    if (c.model == MODEL_UBM && bp.ubm_int_ok && c.rsu > 0.0)
      collected = topk_fast_path<true>(c, n_songs, stride, k, need, s_key, s_song, s_hist, s_max, &s_count, s_ctl, &max_score, nullptr);
    else
      collected = topk_fast_path<false>(c, n_songs, stride, k, need, s_key, s_song, s_hist, s_max, &s_count, s_ctl, &max_score, bp.rsd_up);
    __syncthreads();
  } else {
    // ---- short rows: exact maximum
    unsigned long long mx = 0;
    scan_row(c, n_songs, [&](int, unsigned long long kb, bool ok) { if (ok && kb > mx) mx = kb; });
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xffffffffu, mx, o); mx = other > mx ? other : mx; }
    if (lane == 0) s_max[warp] = mx;
    __syncthreads();
    mx = 0;
    for (int i = 0; i < kTopkThreads / 32; ++i) mx = s_max[i] > mx ? s_max[i] : mx;
    max_score = __longlong_as_double(static_cast<long long>(mx));
  }
  // linear bin map of the exact path; any scale keeps it monotone (scores above a sampled maximum share the top bin)
  const double scale = max_score > 0.0 ? __ddiv_rn(static_cast<double>(kTopkBins - 1), max_score) : 0.0;
  auto bin_of = [&](unsigned long long kb) -> uint32_t {
    const int d = __double2int_rz(__dmul_rn(__longlong_as_double(static_cast<long long>(kb)), scale));
    return static_cast<uint32_t>(d > kTopkBins - 1 ? kTopkBins - 1 : d);
  };
  auto scan = [&](auto&& f) { scan_row(c, n_songs, f); };
  if (!collected) {
    if (tid == 0 && bp.stats) atomicAdd(bp.stats + (stride > 1 ? 0 : 1), 1u);   // rows the fast path handed back / short rows
    // ---- exact histogram over the whole row
    for (int i = tid; i < kTopkBins; i += kTopkThreads) s_hist[i] = 0;
    __syncthreads();
    scan([&](int, unsigned long long kb, bool ok) { hist_add(s_hist, ok ? bin_of(kb) : 0u, ok, lane); });
    __syncthreads();
    // ---- exact path: the bin holding the k-th best key from the full histogram
    if (warp == 0) {
      const int want = find_bin(s_hist, k, true, s_ctl);
      if (lane == 0) s_ctl[3] = want;
    }
    __syncthreads();
    need = s_ctl[3];
    if (need > 0) {
      const uint32_t cbin = static_cast<uint32_t>(s_ctl[0]);
      int above = s_ctl[1];                 // keys strictly better than everything still undecided
      unsigned long long phi = 0; uint32_t plo = 0; int nd = 0;
      if (above + s_ctl[2] > kTopkCap) {
        if (tid == 0 && bp.stats) atomicAdd(bp.stats + 2, 1u);   // degenerate rows
        radix_refine(scan, bin_of, cbin, need, above, phi, plo, nd, s_hist, s_ctl);
      }
      collect_keys(scan, bin_of, cbin, phi, plo, nd, s_key, s_song, &s_count);   // pass C
    }
  }
  if (need == 0) {
    write_list(s_key, s_song, 0, k, 0, o_song, o_score, out_len + u);
    return;
  }
  __syncthreads();
  int n_cand = min(s_count, kTopkCap);
  if (n_cand > kTopkThreads && n_cand <= 2 * kTopkThreads && need <= kTopkThreads)
    n_cand = trim_candidates(s_key, s_song, s_hist, s_max, s_ctl, &s_count, n_cand, need);
  sort_keys(s_key, s_song, n_cand);
  write_list(s_key, s_song, need, k, bp.song_off, o_song, o_score, out_len + u);
}

int launch_topk(const BlendParams& bp, const long long* te_ptr, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                long long sel_pitch_words, int u0, int n_users, int n_songs, const double* rsa, const double* rsd, int k,
                int* out_song, double* out_score, int* out_len, cudaStream_t st) {
  if (n_users <= 0) return 0;
  if (k <= 0 || k > kTopkCap / 2) return -2;
  topk_kernel<<<n_users, kTopkThreads, 0, st>>>(bp, te_ptr, sint_u, sint_i, spitch, sel, sel_pitch_words, u0, n_songs, rsa, rsd, k,
                                                out_song, out_score, out_len);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- join of the ranked lists of several song partitions
// One CTA per test user.  The n lists (each ordered by score descending, song id ascending — disjoint song sets, so the order over their
// union is strict) are staged in shared memory; an element's position in the merged order is its own index plus, for every other list,
// the number of that list's elements that precede it (one binary search each); the first k positions are written.  This is the
// driver-side `.collect` + ranking of the reference's song partitioning (distributed.scala:459-461, 477-479).
__device__ __forceinline__ bool merge_precedes(double sa, int ia, double sb, int ib) { return sa > sb || (sa == sb && ia < ib); }

__global__ void __launch_bounds__(256)
merge_topk_kernel(MergeParts p, int k, int n_users, int* __restrict__ out_song, double* __restrict__ out_score, int* __restrict__ out_len) {
  extern __shared__ double s_merge[];
  double* s_score = s_merge;                                             // [n][k]
  int* s_song = reinterpret_cast<int*>(s_merge + p.n * k);              // [n][k]
  __shared__ int s_len[kMergeMaxParts];
  const int u = blockIdx.x;
  if (u >= n_users) return;
  if (threadIdx.x < p.n) s_len[threadIdx.x] = max(0, min(k, p.len[threadIdx.x][u]));
  __syncthreads();
  for (int a = 0; a < p.n; ++a) {
    const int la = s_len[a];
    for (int i = threadIdx.x; i < la; i += blockDim.x) {
      s_score[a * k + i] = p.score[a][static_cast<long long>(u) * k + i];
      s_song[a * k + i] = p.song[a][static_cast<long long>(u) * k + i];
    }
  }
  int total = 0;
  for (int a = 0; a < p.n; ++a) total += s_len[a];
  const int need = min(k, total);
  __syncthreads();
  int* o_song = out_song + static_cast<long long>(u) * k;
  double* o_score = out_score + static_cast<long long>(u) * k;
  for (int e = threadIdx.x; e < p.n * k; e += blockDim.x) {
    const int a = e / k, i = e - a * k;
    if (i >= s_len[a]) continue;
    const double sc = s_score[e]; const int sg = s_song[e];
    int rank = i;
    for (int b = 0; b < p.n && rank < need; ++b) {
      if (b == a) continue;
      int lo = 0, hi = s_len[b];                                        // elements of list b that precede (sc, sg)
      while (lo < hi) { const int m = (lo + hi) >> 1; if (merge_precedes(s_score[b * k + m], s_song[b * k + m], sc, sg)) lo = m + 1; else hi = m; }
      rank += lo;
    }
    if (rank < need) { o_song[rank] = sg; o_score[rank] = sc; }
  }
  for (int i = need + threadIdx.x; i < k; i += blockDim.x) { o_song[i] = -1; o_score[i] = 0.0; }
  if (threadIdx.x == 0) out_len[u] = need;
}

int launch_merge_topk(const MergeParts& p, int k, int n_users, int* out_song, double* out_score, int* out_len, cudaStream_t st) {
  if (n_users <= 0) return 0;
  if (p.n < 1 || p.n > kMergeMaxParts || k < 1) return -2;
  const size_t smem = static_cast<size_t>(p.n) * k * 12;
  if (smem > 200 * 1024) return -3;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(merge_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess) return -4;
  merge_topk_kernel<<<n_users, 256, smem, st>>>(p, k, n_users, out_song, out_score, out_len);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- blends on materialised model arrays (MR:317-481)
__global__ void blend_arrays_kernel(BlendParams bp, const double* __restrict__ ubm, const double* __restrict__ ibm,
                                    double* __restrict__ out, long long n, long long first_index) {
  // each thread owns a contiguous chunk so the sequential Random stream is replayed with one jump per chunk
  const long long n_threads = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long chunk = (n + n_threads - 1) / n_threads;
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long lo = t * chunk, hi = min(n, lo + chunk);
  if (lo >= hi) return;
  unsigned long long state = 0;
  if (bp.model == MODEL_STOCH) state = lcg_jump((bp.seed ^ kLcgA) & kLcgMask, static_cast<unsigned long long>(first_index + lo));
  for (long long i = lo; i < hi; ++i) {
    double r;
    if (bp.model == MODEL_LC) {
      r = __dadd_rn(__dmul_rn(ubm[i], bp.alpha), __dmul_rn(ibm[i], bp.one_minus_alpha));
    } else if (bp.model == MODEL_AGG) {
      r = (first_index + i < bp.agg_threshold) ? ibm[i] : ubm[i];
    } else {
      state = (state * kLcgA + kLcgC) & kLcgMask;
      const float f = static_cast<float>(static_cast<int>(state >> 24)) / static_cast<float>(1 << 24);
      r = (static_cast<double>(f) < bp.prob) ? ibm[i] : ubm[i];
    }
    out[i] = r;
  }
}

int launch_blend_arrays(const BlendParams& bp, const double* ubm, const double* ibm, double* out, long long n,
                        long long first_index, cudaStream_t st) {
  if (n <= 0) return 0;
  blend_arrays_kernel<<<148 * 4, 256, 0, st>>>(bp, ubm, ibm, out, n, first_index);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mr
