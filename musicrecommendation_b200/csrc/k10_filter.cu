// k10_filter.cu — filtered top-k, candidate path (DESIGN.md §4.11): the exact top-k of each test user over a small allowed song set.
// The full-row select (topk_kernel) streams S x 8 bytes per user and panel whatever the filter keeps; this kernel reads the ascending list
// of allowed columns (coalesced) and gathers only their panel entries, select words and rsd values.  The ranking is row_select, the exact
// select the similar, explain and audience kernels share, so the lists and score bits are those of topk_kernel over the same candidates.
#include "mr_common.cuh"
#include "mr_kernels.h"

namespace mr {

__global__ void __launch_bounds__(kTopkThreads)
candidate_topk_kernel(BlendParams bp, const long long* __restrict__ sint_u, const long long* __restrict__ sint_i, long long spitch,
                      const uint64_t* __restrict__ sel, long long sel_pitch_words, int u0, const int* __restrict__ cols, int n_cols,
                      const double* __restrict__ rsa, const double* __restrict__ rsd, int k, int* __restrict__ out_song,
                      double* __restrict__ out_score, int* __restrict__ out_len) {
  __shared__ RowSelect sm;
  const int b = blockIdx.x, u = u0 + b;
  const long long* su = sint_u ? sint_u + static_cast<long long>(b) * spitch : nullptr;
  const long long* si = sint_i ? sint_i + static_cast<long long>(b) * spitch : nullptr;
  const uint64_t* sw = sel ? sel + static_cast<long long>(b) * sel_pitch_words : nullptr;
  const double rsu = rsa[u];
  // every thread calls f the same number of times (row_select's passes use warp collectives); a sentinel entry (listened or excluded)
  // is no candidate
  auto scan = [&](auto&& f) {
    for (int base = 0; base < n_cols; base += kTopkThreads) {
      const int i = base + static_cast<int>(threadIdx.x);
      int c = 0; bool ok = false; unsigned long long kb = 0;
      if (i < n_cols) {
        c = cols[i];
        const long long a = su ? su[c] : 0, e = si ? si[c] : 0;
        ok = a >= 0 && e >= 0;
        if (ok) {
          const bool pick = sw && ((sw[c >> 6] >> (c & 63)) & 1ULL);
          kb = key_bits(blend_score(bp.model, a, e, rsu, si ? rsd[c] : 0.0, bp.alpha, bp.one_minus_alpha, pick));
        }
      }
      f(c + bp.song_off, kb, ok);   // the rotation keeps window order equal to global id order, so ids tie-break like columns
    }
  };
  row_select(scan, scan, k, sm, out_song + static_cast<long long>(u) * k, out_score + static_cast<long long>(u) * k, out_len + u,
             bp.stats ? bp.stats + 2 : nullptr);
}

int launch_candidate_topk(const BlendParams& bp, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                          long long sel_pitch_words, int u0, int n_users, const int* cols, int n_cols, const double* rsa, const double* rsd, int k,
                          int* out_song, double* out_score, int* out_len, cudaStream_t st) {
  if (n_users <= 0) return 0;
  if (k <= 0 || k > kTopkCap / 2) return -2;
  candidate_topk_kernel<<<n_users, kTopkThreads, 0, st>>>(bp, sint_u, sint_i, spitch, sel, sel_pitch_words, u0, cols, n_cols, rsa, rsd, k,
                                                          out_song, out_score, out_len);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mr
