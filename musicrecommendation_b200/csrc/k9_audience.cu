// k9_audience.cu — song audiences (mr_song_audience, DESIGN.md §4.10): per query song, the k test users of highest score under one model,
// ranked by column from the masked score panels of the batch pipeline.
//
// One CTA per query column and batch.  Its scan streams the column's running list from the earlier batches (user id, stored score: the key
// is the stored double's bits, so scores round-trip exactly), then the batch's rows of the column: (u0 + r, blend_score of the panels'
// numerators), the getTopK bits of the pair; a listened pair (kListened in the panels) is no candidate.  row_select (mr_common.cuh) ranks
// that stream and write_list stores the new top-k over the running list: every scan of the CTA ends before its sort, and each CTA owns its
// list.  The user ids of different batches are disjoint, so the union "running top-k ∪ this batch's column" contains the new top-k and the
// lists are exact for any batching, slicing or pipelining.
// Query columns arrive sorted, so CTAs of adjacent columns are scheduled together and their 8-byte loads of one panel row share 32-byte
// sectors in L2.
#include "mr_common.cuh"
#include "mr_kernels.h"

namespace mr {

constexpr int kAudRowsPerThread = 4;   // panel loads in flight per thread and step

__global__ void __launch_bounds__(kTopkThreads, 2)
audience_kernel(const AudienceArgs a, int n_q, int u0, int nb, int k) {
  __shared__ RowSelect sm;
  const int q = blockIdx.x;
  if (q >= n_q) return;
  const int2 cq = a.q[q];
  const int c = cq.x;
  int* const l_user = a.user + static_cast<long long>(cq.y) * k;
  double* const l_score = a.score + static_cast<long long>(cq.y) * k;
  const int len = a.len[cq.y];     // read by every thread before row_select's first barrier; thread 0 rewrites it at the very end
  const double rds = a.rsd[c];
  const int model = a.model;
  const uint64_t sel_bit = 1ULL << (c & 63);
  auto scan = [&](auto&& f) {
    const int n = len + nb;
    for (int base = 0; base < n; base += kAudRowsPerThread * kTopkThreads) {
      long long pu[kAudRowsPerThread], pi[kAudRowsPerThread];
      bool pick[kAudRowsPerThread];
#pragma unroll
      for (int t = 0; t < kAudRowsPerThread; ++t) {
        const int r = base + t * kTopkThreads + static_cast<int>(threadIdx.x) - len;   // batch row, < 0 inside the running list
        pu[t] = -1; pi[t] = -1; pick[t] = false;
        if (r >= 0 && r < nb) {
          const long long o = static_cast<long long>(r) * a.spitch + c;
          if (model != MODEL_IBM) pu[t] = __ldcg(a.su + o);
          if (model != MODEL_UBM) pi[t] = __ldcg(a.si + o);
          if (model >= MODEL_AGG) pick[t] = (__ldg(a.sel + static_cast<long long>(r) * a.sel_pitch + (c >> 6)) & sel_bit) != 0;
        }
      }
#pragma unroll
      for (int t = 0; t < kAudRowsPerThread; ++t) {
        const int j = base + t * kTopkThreads + static_cast<int>(threadIdx.x), r = j - len;
        int id = 0; unsigned long long kb = 0; bool ok = false;
        if (j < len) {
          id = l_user[j]; kb = key_bits(l_score[j]); ok = true;
        } else if (r < nb) {
          id = u0 + r;
          ok = (model == MODEL_IBM || pu[t] >= 0) && (model == MODEL_UBM || pi[t] >= 0);
          if (ok) kb = key_bits(blend_score(model, pu[t], pi[t], model != MODEL_IBM ? __ldg(a.rsa + id) : 0.0, rds, a.alpha, a.oma, pick[t]));
        }
        f(id, kb, ok);
      }
    }
  };
  row_select(scan, scan, k, sm, l_user, l_score, a.len + cq.y, a.radix_rows);
}

int launch_audience(const AudienceArgs& a, int n_q, int u0, int nb, int k, cudaStream_t st) {
  if (n_q <= 0 || nb <= 0) return 0;
  if (k <= 0 || k > kTopkCap / 2) return -2;
  audience_kernel<<<n_q, kTopkThreads, 0, st>>>(a, n_q, u0, nb, k);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mr
