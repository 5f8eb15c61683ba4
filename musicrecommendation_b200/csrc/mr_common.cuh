// mr_common.cuh — shared device helpers for the sm_100a kernels of libmrscore.
// Hand-written PTX wrappers for mbarrier / TMA / tcgen05 (no CUTLASS dependency).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <climits>

#include "mr_kernels.h"

namespace mr {

// Fixed-point scales of the canonical arithmetic (see DESIGN.md §3): q(deg) = rint(scale / sqrt(deg)).
//   UBM: 2^24 — the weighted co-occurrence sum_{v in U_j ∩ U_s} q(|I_v|) of the item-space head rows fits a u32 for all but a few
//               thousand pairs of very popular songs (those are kept exactly in an exception list).
//   IBM: 2^26 — the user-space weighted count sum_{j in I_u ∩ I_v} q(d_j) stays below 2^32 for up to 90 shared songs, so the
//               gathered panel holds u32 entries (wrap-arounds are recorded as carry events and repaired exactly).
constexpr double kQScaleUbm = 16777216.0;         // 2^24
constexpr double kQInvUbm = 1.0 / 16777216.0;
constexpr double kQScaleIbm = 67108864.0;         // 2^26
constexpr double kQInvIbm = 1.0 / 67108864.0;
constexpr long long kListened = -1;               // sentinel written into Sint at listened (u, s) pairs

// fp64 score of one (user, song) pair from its Sint numerators (DESIGN.md §3), shared by the top-k select and the evaluator:
// ubm = (double)Sint_u * rsa[u], ibm = (double)Sint_i * rsd[s], blends as in k3_topk.cu's header
__device__ __forceinline__ double blend_score(int model, long long su, long long si, double rsu, double rds, double alpha,
                                              double oma, bool pick_ibm) {
  switch (model) {
    case MODEL_UBM: return __dmul_rn(__ll2double_rn(su), rsu);
    case MODEL_IBM: return __dmul_rn(__ll2double_rn(si), rds);
    case MODEL_LC:
      return __dadd_rn(__dmul_rn(__dmul_rn(__ll2double_rn(su), rsu), alpha), __dmul_rn(__dmul_rn(__ll2double_rn(si), rds), oma));
    default: return pick_ibm ? __dmul_rn(__ll2double_rn(si), rds) : __dmul_rn(__ll2double_rn(su), rsu);
  }
}

// ---------------------------------------------------------------- exact top-k select helpers (k3_topk.cu, k8_similar.cu)
// Keys are the composite (score bits : 64, ~song : 32): "larger key" == "better", ties broken by the smaller song id.
// The one exact select of topk_kernel and similar_row_topk_kernel: after the caller's linear histogram of a row (kTopkBins bins of a bin
// map bin_of that is monotone in the key), find_bin picks the bin holding the need-th best key, radix_refine narrows a bin too crowded
// for the candidate buffer, collect_keys gathers the keys at or above the result, sort_keys orders them and write_list stores the list.
// The row is streamed by the caller's scan(f): f(song, key bits, valid) called the same number of times by every thread of the CTA.
constexpr int kTopkThreads = 512;   // per CTA = per row, 2 CTAs per SM (64 registers); 256 x 4 measured the same on whole rows and on 48 k-song rows
constexpr int kTopkCap = 2048;      // candidate buffer (>= 2 * k); bitonic-sorted in shared memory
constexpr int kTopkBins = 2048;

// digit d (0 = most significant) of the 96-bit composite (kb : 64, ~song : 32), 8 bits each
__device__ __forceinline__ uint32_t key_digit(unsigned long long kb, uint32_t inv_song, int d) {
  return d < 8 ? static_cast<uint32_t>(kb >> (56 - 8 * d)) & 255u : (inv_song >> (24 - 8 * (d - 8))) & 255u;
}
// compare the first nd digits of (kb, inv) against the prefix: -1 below, 0 equal, +1 above
__device__ __forceinline__ int prefix_cmp(unsigned long long kb, uint32_t inv, unsigned long long phi, uint32_t plo, int nd) {
  if (nd == 0) return 0;
  if (nd <= 8) {
    const int sh = 64 - 8 * nd;
    const unsigned long long a = kb >> sh, b = phi >> sh;
    return a < b ? -1 : (a > b ? 1 : 0);
  }
  if (kb != phi) return kb < phi ? -1 : 1;
  const int sh = 32 - 8 * (nd - 8);
  const uint32_t a = inv >> sh, b = plo >> sh;
  return a < b ? -1 : (a > b ? 1 : 0);
}

// warp-aggregated shared-memory histogram increment: peel the two most common bins of the warp with ballots
__device__ __forceinline__ void hist_add(int* hist, uint32_t bin, bool ok, int lane) {
  uint32_t pending = __ballot_sync(0xffffffffu, ok);
#pragma unroll 1
  for (int round = 0; round < 2 && pending; ++round) {
    const int leader = __ffs(pending) - 1;
    const uint32_t lb = __shfl_sync(0xffffffffu, bin, leader);
    const uint32_t same = __ballot_sync(0xffffffffu, ok && bin == lb) & pending;
    if (lane == leader) atomicAdd(&hist[lb], __popc(same));
    pending &= ~same;
  }
  if ((pending >> lane) & 1u) atomicAdd(&hist[bin], 1);
}

// Suffix search by warp 0 over the kTopkBins-bin histogram: the highest bin with at least `want` keys in it or above (want first clamped
// to the histogram's total when clamp_to_total).  s_ctl[0] = that bin, s_ctl[1] = keys strictly above it, s_ctl[2] = keys in it; bin 0
// when want exceeds the total or is <= 0.  Returns the (clamped) want.
__device__ __forceinline__ int find_bin(const int* hist, int want, bool clamp_to_total, int* s_ctl) {
  const int lane = threadIdx.x & 31;
  int part = 0;
  for (int i = 0; i < kTopkBins / 32; ++i) part += hist[lane * (kTopkBins / 32) + i];
  int above_lane = 0;   // keys in bins owned by higher lanes; lane 0's above_lane + part is the total
  for (int l = 0; l < 32; ++l) { const int pp = __shfl_sync(0xffffffffu, part, l); if (l > lane) above_lane += pp; }
  if (clamp_to_total) want = min(want, __shfl_sync(0xffffffffu, above_lane + part, 0));
  if (lane == 0) { s_ctl[0] = 0; s_ctl[1] = above_lane + part - hist[0]; s_ctl[2] = hist[0]; }   // unless a lane owns the answer
  __syncwarp();
  if (want > 0 && above_lane < want && above_lane + part >= want) {
    int cum = above_lane, chosen = lane * (kTopkBins / 32);
    for (int i = kTopkBins / 32 - 1; i >= 0; --i) {
      const int bin = lane * (kTopkBins / 32) + i;
      if (cum + hist[bin] >= want) { chosen = bin; break; }
      cum += hist[bin];
    }
    s_ctl[0] = chosen; s_ctl[1] = cum; s_ctl[2] = hist[chosen];
  }
  return want;
}

// Crowded bin (thousands of exact ties): exact most-significant-digit radix select of the (need - above) best keys inside bin cbin, 8 bits
// of the 96-bit key per pass.  On return the keys better than the prefix (phi : plo, nd digits) number `above`, and they plus the keys on
// the prefix fit the candidate buffer, or the prefix is the whole key.  Called by every thread when the bin does not fit.
template <class Scan, class BinOf>
__device__ __forceinline__ void radix_refine(Scan&& scan, BinOf&& bin_of, uint32_t cbin, int need, int& above, unsigned long long& phi,
                                             uint32_t& plo, int& nd, int* s_hist, int* s_ctl) {
  const int tid = threadIdx.x, lane = tid & 31;
  for (;;) {
    __syncthreads();
    for (int i = tid; i < 256; i += kTopkThreads) s_hist[i] = 0;
    __syncthreads();
    scan([&](int s, unsigned long long kb, bool ok) {
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
    if (above + s_ctl[2] <= kTopkCap || nd == 12) break;
  }
}

// Collect every key in a higher bin than cbin, plus the keys of bin cbin at or above the radix prefix (nd = 0: all of them), one ballot
// and one shared-memory atomic per warp.  *s_count ends as the number of such keys; the buffer holds the first kTopkCap.
template <class Scan, class BinOf>
__device__ __forceinline__ void collect_keys(Scan&& scan, BinOf&& bin_of, uint32_t cbin, unsigned long long phi, uint32_t plo, int nd,
                                             unsigned long long* s_key, int* s_song, int* s_count) {
  const int lane = threadIdx.x & 31;
  __syncthreads();
  if (threadIdx.x == 0) *s_count = 0;
  __syncthreads();
  scan([&](int s, unsigned long long kb, bool ok) {
    if (ok) {
      const uint32_t bn = bin_of(kb);
      ok = bn > cbin || (bn == cbin && prefix_cmp(kb, ~static_cast<uint32_t>(s), phi, plo, nd) >= 0);
    }
    const uint32_t m = __ballot_sync(0xffffffffu, ok);
    if (m) {
      int base = 0;
      if (lane == 0) base = atomicAdd(s_count, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (ok) {
        const int pos = base + __popc(m & ((1u << lane) - 1));
        if (pos < kTopkCap) { s_key[pos] = kb; s_song[pos] = s; }
      }
    }
  });
}

// bitonic sort of n_pad (a power of two) (key, song) pairs, "better first": key descending, then song ascending; every thread of the CTA
// calls it
__device__ __forceinline__ void bitonic_keys(unsigned long long* key, int* song, int n_pad) {
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

// pad the n collected keys to a power of two with entries that sort last, then sort
__device__ __forceinline__ void sort_keys(unsigned long long* s_key, int* s_song, int n) {
  int n_sort = 1;
  while (n_sort < n) n_sort <<= 1;
  for (int i = n + threadIdx.x; i < n_sort; i += kTopkThreads) { s_key[i] = 0; s_song[i] = INT_MAX; }
  bitonic_keys(s_key, s_song, n_sort);
}

// the list of one row: the first `need` sorted keys (song ids + song_off), then (-1, 0.0) up to k
__device__ __forceinline__ void write_list(const unsigned long long* s_key, const int* s_song, int need, int k, int song_off, int* o_song,
                                           double* o_score, int* o_len) {
  for (int i = threadIdx.x; i < k; i += kTopkThreads) {
    if (i < need) { o_song[i] = s_song[i] + song_off; o_score[i] = __longlong_as_double(static_cast<long long>(s_key[i])); }
    else { o_song[i] = -1; o_score[i] = 0.0; }
  }
  if (threadIdx.x == 0) *o_len = need;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must trap (-> cudaErrorLaunchFailure) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}

// ---------------------------------------------------------------- TMA (cp.async.bulk.tensor)
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tile load global -> shared, completion signalled on `bar` (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, 8-bit integer operands, int32 accumulate.
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on `bar` once every previously issued tcgen05.mma of this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread t of the warp receives lane (base_lane + t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// UMMA shared-memory matrix descriptor, K-major operand tile stored as rows of 128 bytes with the
// 128-byte swizzle TMA produces (8-row x 128 B atoms, 1024 B apart):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (unused for swizzled K-major, 1)
//   [32,46) stride byte offset >> 4 (= 1024 >> 4) | [46,48) descriptor version = 1 (sm_100)
//   [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// tcgen05 instruction descriptor for kind::i8: unsigned 8-bit A and B (both K-major), int32 accumulator.
//   [4,6) c_format = 2 (S32) | [7,10) a_format = 0 (U8) | [10,13) b_format = 0 (U8)
//   [15] a_major = 0 (K) | [16] b_major = 0 (K) | [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ constexpr uint32_t umma_idesc_u8(uint32_t M, uint32_t N) {
  return (2u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

}  // namespace mr
