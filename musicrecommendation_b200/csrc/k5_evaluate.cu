// k5_evaluate.cu — the reference's evaluation metric on the GPU (SURVEY.md §8f N2).
//
// MusicRecommender.scala:521-639: scores are min-max normalised over the WHOLE model (MR:524-529); for each threshold t in
// 0.0, 0.1, ... (10 values, MR:590; distributed.scala:395 uses 11) the predictions are { (u, s) : normalised score > t }; for each
// distinct label song c the confusion counts over test users (MR:541-553) give precision / recall (MR:561-579) and
//   AP(c) = sum_{i < n-2} (R_i - R_{i+1}) P_i + R_{n-2} P_{n-2} + 0        (MR:600-610, List.sum = left fold from 0.0)
// mAP = (sum_c AP(c)) / |label songs|  (MR:626, summed on the host in ascending song order = the oracle's canonical order).
// The reference spends 62-75 s per model on this at 2000 / 100 users (README:940-944).  All fp64 operations use explicit
// round-to-nearest intrinsics, so the result is bit-identical to the CPU restatement.
#include "mr_common.cuh"
#include "mr_kernels.h"

namespace mr {

// min / max over the emitted (non-NaN) scores; scores are >= 0 so their bit patterns order like unsigned integers
__global__ void eval_minmax_kernel(const double* __restrict__ scores, long long n, unsigned long long* __restrict__ mn,
                                   unsigned long long* __restrict__ mx) {
  unsigned long long lo = ~0ULL, hi = 0ULL;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const double x = scores[i];
    if (x == x) {
      const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(x));
      lo = b < lo ? b : lo; hi = b > hi ? b : hi;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long a = __shfl_xor_sync(0xffffffffu, lo, o), c = __shfl_xor_sync(0xffffffffu, hi, o);
    lo = a < lo ? a : lo; hi = c > hi ? c : hi;
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(mn, lo); atomicMax(mx, hi); }
}

// One warp per label song: lanes stride over the test users, count TP / FP / FN per threshold, lane 0 finishes the AP.
__global__ void __launch_bounds__(128)
eval_ap_kernel(const double* __restrict__ scores, int n_users, int n_songs, const long long* __restrict__ lab_ptr,
               const int* __restrict__ lab_col, const int* __restrict__ new_songs, int n_new, int n_thresholds,
               const unsigned long long* __restrict__ mn_bits, const unsigned long long* __restrict__ mx_bits, double* __restrict__ ap_out) {
  const double TH[11] = {0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0};
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= n_new) return;
  const int song = new_songs[c];
  const double mn = __longlong_as_double(static_cast<long long>(*mn_bits)), mx = __longlong_as_double(static_cast<long long>(*mx_bits));
  const double range = __dsub_rn(mx, mn);
  int tp[11], fp[11], fn[11];
#pragma unroll
  for (int t = 0; t < 11; ++t) { tp[t] = 0; fp[t] = 0; fn[t] = 0; }
  for (int u = lane; u < n_users; u += 32) {
    // testLabels(user).contains(song): label rows are ascending
    long long lo = lab_ptr[u], hi = lab_ptr[u + 1];
    const long long end = hi;
    while (lo < hi) { const long long m = (lo + hi) >> 1; if (lab_col[m] < song) lo = m + 1; else hi = m; }
    const bool labelled = lo < end && lab_col[lo] == song;
    double norm = __longlong_as_double(0x7ff8000000000000LL);
    if (song < n_songs) {
      const double x = scores[static_cast<long long>(u) * n_songs + song];
      if (x == x) norm = __ddiv_rn(__dsub_rn(x, mn), range);                  // (score - min) / (max - min), MR:529
    }
#pragma unroll
    for (int t = 0; t < 11; ++t) {
      if (t < n_thresholds) {
        const bool predicted = norm > TH[t];                                   // NaN compares false
        tp[t] += predicted && labelled; fp[t] += predicted && !labelled; fn[t] += !predicted && labelled;
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 11; ++t)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      tp[t] += __shfl_xor_sync(0xffffffffu, tp[t], o); fp[t] += __shfl_xor_sync(0xffffffffu, fp[t], o); fn[t] += __shfl_xor_sync(0xffffffffu, fn[t], o);
    }
  if (lane == 0) {
    double prec[11], rec[11];
#pragma unroll
    for (int t = 0; t < 11; ++t) {
      prec[t] = (tp[t] + fp[t] > 0) ? __ddiv_rn(static_cast<double>(tp[t]), static_cast<double>(tp[t] + fp[t])) : 0.0;   // MR:561-566
      rec[t] = (tp[t] + fn[t] > 0) ? __ddiv_rn(static_cast<double>(tp[t]), static_cast<double>(tp[t] + fn[t])) : 0.0;    // MR:574-579
    }
    double ap = 0.0;
#pragma unroll
    for (int t = 0; t < 11; ++t) {
      if (t < n_thresholds) {
        double term;
        if (t == n_thresholds - 1) term = 0.0;
        else if (t == n_thresholds - 2) term = __dmul_rn(__dsub_rn(rec[t], 0.0), prec[t]);
        else term = __dmul_rn(__dsub_rn(rec[t], rec[t + 1]), prec[t]);
        ap = __dadd_rn(ap, term);
      }
    }
    ap_out[c] = ap;
  }
}

int launch_evaluate(const double* scores, int n_users, int n_songs, const long long* lab_ptr, const int* lab_col, const int* new_songs,
                    int n_new, int n_thresholds, unsigned long long* minmax, double* ap_out, int num_sms, cudaStream_t st) {
  if (n_new <= 0 || n_thresholds < 2 || n_thresholds > 11) return -2;
  const unsigned long long init[2] = {~0ULL, 0ULL};
  if (cudaMemcpyAsync(minmax, init, sizeof init, cudaMemcpyHostToDevice, st) != cudaSuccess) return -1;
  eval_minmax_kernel<<<num_sms * 8, 256, 0, st>>>(scores, static_cast<long long>(n_users) * n_songs, minmax, minmax + 1);
  eval_ap_kernel<<<(n_new + 3) / 4, 128, 0, st>>>(scores, n_users, n_songs, lab_ptr, lab_col, new_songs, n_new, n_thresholds, minmax, minmax + 1, ap_out);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------------------------------------------------------------
// The same metric streamed over the batches of the scoring pipeline (DESIGN.md §4.5), for models too large to materialise.  Per label
// song c and threshold t it needs only integers: pred_t(c) = #users whose normalised score for c exceeds TH[t], tp_t(c) = the same over
// the users labelled with c, nlab(c) = #users labelled with c; they add exactly over batches, user shards and song windows.  The
// normalisation f(x) = RN(RN(x - mn) / RN(mx - mn)) is monotone in x, so f(x) > TH[t] <=> x >= c_t with host-computed cutoffs
// (mr_eval_cutoffs): the kernels compare bit patterns of non-negative doubles and never divide.  A pair's bucket is the number of
// cutoffs <= its score (it is predicted at exactly the thresholds t < bucket); counts are kept per bucket, the host sums them up.
// ---------------------------------------------------------------------------------------------------------------------
// A launch serves a group of models (EvalGroup, DESIGN.md §4.6): the panel words, the select word and the label entries are read once and
// every model of the group scores them.  AGG needs no select plane here: its pick is "column < split[u]" (launch_agg_split).
constexpr int kEvalThreads = 256;
constexpr int kEvalTile = 4 * kEvalThreads;   // songs per CTA column tile: 4 consecutive songs per thread (two 16-byte loads per panel)
constexpr int kEvalRows = 512;                // at most this many panel rows per eval_count_kernel CTA: its u16 histogram cannot wrap

struct GroupNeeds { bool u, i, sel; };        // which panels / the select plane the group's models read
__device__ __forceinline__ GroupNeeds group_needs(const EvalGroup& g) {
  GroupNeeds r{false, false, false};
#pragma unroll
  for (int m = 0; m < kEvalGroupMax; ++m)
    if (m < g.n) { r.u = r.u || g.model[m] != MODEL_IBM; r.i = r.i || g.model[m] != MODEL_UBM; r.sel = r.sel || g.model[m] == MODEL_STOCH; }
  return r;
}

// Numerators of the songs s .. s+3 of one panel row; ok = emitted (not listened, inside the row), exactly as scan_row (k3_topk.cu).
// Both panels of a set carry the same listened mask, so whichever one is read decides.
__device__ __forceinline__ void eval_load4(const GroupNeeds& nd, const long long* ru, const long long* ri, int s, int n_songs,
                                           long long (&a)[4], long long (&b)[4], bool (&ok)[4]) {
#pragma unroll
  for (int t = 0; t < 4; ++t) { a[t] = 0; b[t] = 0; }
  if (nd.u) {
    const longlong2 x = *reinterpret_cast<const longlong2*>(ru + s), y = *reinterpret_cast<const longlong2*>(ru + s + 2);
    a[0] = x.x; a[1] = x.y; a[2] = y.x; a[3] = y.y;
  }
  if (nd.i) {
    const longlong2 x = *reinterpret_cast<const longlong2*>(ri + s), y = *reinterpret_cast<const longlong2*>(ri + s + 2);
    b[0] = x.x; b[1] = x.y; b[2] = y.x; b[3] = y.y;
  }
#pragma unroll
  for (int t = 0; t < 4; ++t) ok[t] = s + t < n_songs && a[t] >= 0 && b[t] >= 0;
}

// score bits of model m at column c; selbit = the STOCH plane's bit of c, split = the AGG split column of this row
__device__ __forceinline__ unsigned long long eval_key(const EvalGroup& g, int m, long long a, long long b, double rsu, double rd, int c,
                                                       bool selbit, int split) {
  const int model = g.model[m];
  const bool pick = model == MODEL_STOCH ? selbit : (model == MODEL_AGG && c < split);
  return static_cast<unsigned long long>(__double_as_longlong(blend_score(model, a, b, rsu, rd, g.alpha[m], g.oma[m], pick)));
}

__device__ __forceinline__ void eval_rsd4(bool need_i, const double* rsd, int s, int n_songs, double (&rd)[4]) {
#pragma unroll
  for (int t = 0; t < 4; ++t) rd[t] = (need_i && s + t < n_songs) ? rsd[s + t] : 0.0;
}

__device__ __forceinline__ int eval_bucket(const EvalGroup& g, int m, int n_thresholds, unsigned long long kb) {
  int bk = 0;
#pragma unroll
  for (int t = 0; t < 11; ++t) bk += (t < n_thresholds && kb >= g.cut[m][t]) ? 1 : 0;
  return bk;
}

// min / max of each model's emitted scores of a slice: warp shuffles, one pair of atomics per model and warp that saw an emitted pair
__global__ void __launch_bounds__(kEvalThreads)
eval_range_kernel(EvalGroup g, const long long* __restrict__ sint_u, const long long* __restrict__ sint_i, long long spitch,
                  const uint64_t* __restrict__ sel, long long sel_pitch_words, int u0, int n_songs, const double* __restrict__ rsa,
                  const double* __restrict__ rsd, unsigned long long* __restrict__ mm) {
  const GroupNeeds nd = group_needs(g);
  const int b = blockIdx.y;
  const double rsu = nd.u ? rsa[u0 + b] : 0.0;
  const long long* ru = nd.u ? sint_u + static_cast<long long>(b) * spitch : nullptr;
  const long long* ri = nd.i ? sint_i + static_cast<long long>(b) * spitch : nullptr;
  const uint64_t* rsel = nd.sel ? sel + static_cast<long long>(b) * sel_pitch_words : nullptr;
  int split[kEvalGroupMax];
  unsigned long long lo[kEvalGroupMax], hi[kEvalGroupMax];
#pragma unroll
  for (int m = 0; m < kEvalGroupMax; ++m) {
    split[m] = (m < g.n && g.model[m] == MODEL_AGG) ? g.split[m][u0 + b] : 0;
    lo[m] = ~0ULL; hi[m] = 0ULL;
  }
  for (int s = 4 * (blockIdx.x * kEvalThreads + static_cast<int>(threadIdx.x)); s < n_songs; s += 4 * kEvalThreads * gridDim.x) {
    double rd[4]; long long a[4], x[4]; bool ok[4];
    eval_rsd4(nd.i, rsd, s, n_songs, rd);
    eval_load4(nd, ru, ri, s, n_songs, a, x, ok);
    const uint64_t selw = nd.sel ? rsel[s >> 6] >> (s & 63) : 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      if (!ok[t]) continue;
#pragma unroll
      for (int m = 0; m < kEvalGroupMax; ++m) {
        if (m >= g.n) break;
        const unsigned long long kb = eval_key(g, m, a[t], x[t], rsu, rd[t], s + t, (selw >> t) & 1ULL, split[m]);
        lo[m] = kb < lo[m] ? kb : lo[m]; hi[m] = kb > hi[m] ? kb : hi[m];
      }
    }
  }
#pragma unroll
  for (int m = 0; m < kEvalGroupMax; ++m) {
    if (m >= g.n) break;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long p = __shfl_xor_sync(0xffffffffu, lo[m], o), q = __shfl_xor_sync(0xffffffffu, hi[m], o);
      lo[m] = p < lo[m] ? p : lo[m]; hi[m] = q > hi[m] ? q : hi[m];
    }
    if ((threadIdx.x & 31) == 0 && lo[m] != ~0ULL) { atomicMin(mm + 2 * g.out[m], lo[m]); atomicMax(mm + 2 * g.out[m] + 1, hi[m]); }
  }
}

// Prediction counts of the label songs.  A CTA owns a tile of 1024 songs (4 per thread) over `rows` panel rows (<= 512: the flush, one
// global atomic per non-zero (model, song, bucket) per CTA, is paid once per up to 512 rows, and a u16 counter cannot wrap); each thread
// counts its own songs' buckets in a private slice of the shared histogram (no shared atomics), then flushes the non-zero entries with
// global atomics.  Threads whose 4 songs are no label song read nothing: the kernel moves only the panel sectors of label songs.
__global__ void __launch_bounds__(kEvalThreads)
eval_count_kernel(EvalGroup g, const long long* __restrict__ sint_u, const long long* __restrict__ sint_i, long long spitch,
                  const uint64_t* __restrict__ sel, long long sel_pitch_words, int u0, int n_users, int n_songs, const double* __restrict__ rsa,
                  const double* __restrict__ rsd, int rows, EvalCounts ec) {
  extern __shared__ unsigned short hist[];   // [model][bucket - 1][song of the thread][thread]
  const GroupNeeds nd = group_needs(g);
  const int tid = threadIdx.x;
  const int s = blockIdx.x * kEvalTile + 4 * tid;
  const int nth = ec.n_thresholds;
  int li[4];
  bool any = false;
#pragma unroll
  for (int t = 0; t < 4; ++t) { li[t] = s + t < n_songs ? ec.colmap[s + t] : -1; any = any || li[t] >= 0; }
  if (!any) return;
  const int nh = g.n * nth * 4;
  for (int i = 0; i < nh; ++i) hist[i * kEvalThreads + tid] = 0;
  double rd[4];
  eval_rsd4(nd.i, rsd, s, n_songs, rd);
  const int r0 = blockIdx.y * rows, r1 = min(n_users, r0 + rows);
#pragma unroll 2
  for (int b = r0; b < r1; ++b) {
    const long long* ru = nd.u ? sint_u + static_cast<long long>(b) * spitch : nullptr;
    const long long* ri = nd.i ? sint_i + static_cast<long long>(b) * spitch : nullptr;
    long long a[4], x[4]; bool ok[4];
    eval_load4(nd, ru, ri, s, n_songs, a, x, ok);
    const uint64_t selw = nd.sel ? sel[static_cast<long long>(b) * sel_pitch_words + (s >> 6)] >> (s & 63) : 0;
    const double rsu = nd.u ? rsa[u0 + b] : 0.0;
#pragma unroll
    for (int m = 0; m < kEvalGroupMax; ++m) {
      if (m >= g.n) break;
      const int split = g.model[m] == MODEL_AGG ? g.split[m][u0 + b] : 0;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int bk = (ok[t] && li[t] >= 0) ? eval_bucket(g, m, nth, eval_key(g, m, a[t], x[t], rsu, rd[t], s + t, (selw >> t) & 1ULL, split)) : 0;
        if (bk) hist[(((m * nth) + bk - 1) * 4 + t) * kEvalThreads + tid] += 1;
      }
    }
  }
  for (int m = 0; m < g.n; ++m) {
    unsigned long long* pred = ec.pred_b + g.out[m] * ec.model_stride;
    for (int k = 0; k < nth; ++k)
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const unsigned int v = hist[(((m * nth) + k) * 4 + t) * kEvalThreads + tid];
        if (v) atomicAdd(pred + static_cast<long long>(li[t]) * nth + k, static_cast<unsigned long long>(v));
      }
  }
}

// One warp per test user of the slice: its label songs inside the scored columns add to nlab, and to each model's tp in the bucket of
// that model's score
__global__ void __launch_bounds__(128)
eval_label_kernel(EvalGroup g, const long long* __restrict__ sint_u, const long long* __restrict__ sint_i, long long spitch,
                  const uint64_t* __restrict__ sel, long long sel_pitch_words, int u0, int n_users, int n_songs, const double* __restrict__ rsa,
                  const double* __restrict__ rsd, EvalCounts ec) {
  const GroupNeeds nd = group_needs(g);
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= n_users) return;
  const int u = u0 + b;
  for (long long e = ec.lab_ptr[u] + lane; e < ec.lab_ptr[u + 1]; e += 32) {
    const int c = ec.lab_col[e] - ec.col_lo;
    if (c < 0 || c >= n_songs) continue;                  // another song window's label, or a label-only song (id >= S)
    const int li = ec.colmap[c];
    if (li < 0) continue;                                  // cannot happen: mr_eval_counts checks new_songs covers every label
    if (ec.nlab) atomicAdd(ec.nlab + li, 1ULL);
    const long long o = static_cast<long long>(b) * spitch + c;
    const long long a = nd.u ? sint_u[o] : 0, x = nd.i ? sint_i[o] : 0;
    if (a < 0 || x < 0) continue;                          // listened: not emitted, a false negative at every threshold
    const bool selbit = nd.sel && ((sel[static_cast<long long>(b) * sel_pitch_words + (c >> 6)] >> (c & 63)) & 1ULL);
    const double rsu = nd.u ? rsa[u] : 0.0, rd = nd.i ? rsd[c] : 0.0;
#pragma unroll
    for (int m = 0; m < kEvalGroupMax; ++m) {
      if (m >= g.n) break;
      const int split = g.model[m] == MODEL_AGG ? g.split[m][u] : 0;
      const int bk = eval_bucket(g, m, ec.n_thresholds, eval_key(g, m, a, x, rsu, rd, c, selbit, split));
      if (bk) atomicAdd(ec.tp_b + g.out[m] * ec.model_stride + static_cast<long long>(li) * ec.n_thresholds + (bk - 1), 1ULL);
    }
  }
}

int launch_eval_range(const EvalGroup& g, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                      long long sel_pitch_words, int u0, int n_users, int n_songs, const double* rsa, const double* rsd,
                      unsigned long long* mm, cudaStream_t st) {
  if (n_songs <= 0) return 0;
  if (g.n < 1 || g.n > kEvalGroupMax) return -2;
  for (int r0 = 0; r0 < n_users; r0 += 32768) {   // grid.y limit
    const int n = min(32768, n_users - r0);
    const long long off = static_cast<long long>(r0) * spitch;
    const int tiles = (n_songs + kEvalTile - 1) / kEvalTile;
    const int gx = max(1, min(tiles, (2048 + n - 1) / n));   // >= ~2048 CTAs per launch, each sweeping a long stretch of its row
    eval_range_kernel<<<dim3(gx, n), kEvalThreads, 0, st>>>(g, sint_u ? sint_u + off : nullptr, sint_i ? sint_i + off : nullptr, spitch,
                                                            sel ? sel + static_cast<long long>(r0) * sel_pitch_words : nullptr, sel_pitch_words,
                                                            u0 + r0, n_songs, rsa, rsd, mm);
  }
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_eval_count(const EvalGroup& g, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                      long long sel_pitch_words, int u0, int n_users, int n_songs, const double* rsa, const double* rsd,
                      const EvalCounts& ec, cudaStream_t st) {
  if (n_users <= 0 || n_songs <= 0) return 0;
  if (ec.n_thresholds < 1 || ec.n_thresholds > 11 || g.n < 1 || g.n > kEvalGroupMax) return -2;
  const size_t smem = static_cast<size_t>(g.n) * ec.n_thresholds * 4 * kEvalThreads * sizeof(unsigned short);
  // per call, not once per process: the attribute belongs to the current device, and a process may drive several
  if (smem > 48 * 1024 && cudaFuncSetAttribute(eval_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess) return -1;
  const int chunks = (n_users + kEvalRows - 1) / kEvalRows, rows = (n_users + chunks - 1) / chunks;   // equal row chunks
  const dim3 grid((n_songs + kEvalTile - 1) / kEvalTile, chunks);
  eval_count_kernel<<<grid, kEvalThreads, smem, st>>>(g, sint_u, sint_i, spitch, sel, sel_pitch_words, u0, n_users, n_songs, rsa, rsd, rows, ec);
  eval_label_kernel<<<(n_users + 3) / 4, 128, 0, st>>>(g, sint_u, sint_i, spitch, sel, sel_pitch_words, u0, n_users, n_songs, rsa, rsd, ec);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------------------------------------------------------------
// mAP@k of the ranked lists (north_star's "mAP@500"; the reference has no ranking, so this is the Million Song Dataset Challenge
// definition, stated in include/mrscore.h at mr_map_at_k):  AP@k(u) = (sum_i [r_i in L_u] * hits_i / i) / min(|L_u|, k).
// One warp per test user: the lanes test 32 ranks at a time against the user's ascending label row (binary search), lane 0 adds the
// terms of the relevant ranks in rank order with explicit round-to-nearest operations, so the per-user AP is bit-identical to the CPU
// restatement; the mean over users is taken on the host in ascending user order.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
map_at_k_kernel(const int* __restrict__ top_song, const int* __restrict__ top_len, int n_users, int k, const long long* __restrict__ lab_ptr,
                const int* __restrict__ lab_col, double* __restrict__ ap_out) {
  const int lane = threadIdx.x & 31;
  const int u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= n_users) return;
  const long long l0 = lab_ptr[u], l1 = lab_ptr[u + 1];
  const long long nl = l1 - l0;
  if (nl <= 0) { if (lane == 0) ap_out[u] = 0.0; return; }
  const int n = min(top_len[u], k);
  const int* row = top_song + static_cast<long long>(u) * k;
  int hits = 0;
  double ap = 0.0;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    bool rel = false;
    if (i < n) {
      const int s = row[i];
      long long lo = l0, hi = l1;
      while (lo < hi) { const long long m = (lo + hi) >> 1; if (lab_col[m] < s) lo = m + 1; else hi = m; }
      rel = lo < l1 && lab_col[lo] == s;
    }
    uint32_t m = __ballot_sync(0xffffffffu, rel);
    if (lane == 0) {
      while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        ++hits;
        ap = __dadd_rn(ap, __ddiv_rn(static_cast<double>(hits), static_cast<double>(base + b + 1)));
      }
    }
  }
  if (lane == 0) ap_out[u] = __ddiv_rn(ap, static_cast<double>(nl < k ? nl : static_cast<long long>(k)));
}

int launch_map_at_k(const int* top_song, const int* top_len, int n_users, int k, const long long* lab_ptr, const int* lab_col,
                    double* ap_out, cudaStream_t st) {
  if (n_users <= 0) return 0;
  map_at_k_kernel<<<(n_users + 3) / 4, 128, 0, st>>>(top_song, top_len, n_users, k, lab_ptr, lab_col, ap_out);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mr
