// k1_count_gemm.cu — kernel K1: intersection counts as a dense 0/1 contraction on the 5th-gen tensor cores.
//
//   C[m][n] = sum_k A[m][k] * B[n][k]        A, B: unsigned 8-bit 0/1, K-major;  C: int32 (exact)
//
// replaces the reference's hot loops
//   UBM  |I_u ∩ I_v|  — MusicRecommender.scala:142-145 (songs.map(both contain ? 1 : 0).sum):  A = A_test (U x S), B = A_train (T x S)
//   IBM  |U_i ∩ U_j|  — MusicRecommender.scala:232-235 (trainUsers.map(both contain ? 1 : 0).sum): A = A_train^T rows J, B = A_train^T (S x T)
//
// Structure (one persistent CTA per SM, 256 threads, warp-specialised):
//   warp 0   TMA producer : cp.async.bulk.tensor 2-D tiles (128 B swizzle) into a kStages-deep smem ring
//   warp 1   MMA issuer   : one elected lane issues tcgen05.mma.kind::i8 (M=128, N=BN, K=32), int32 accumulators in TMEM
//   warp 2   TMEM allocator (2 accumulator stages x BN columns, so the epilogue of tile i overlaps the MMAs of tile i+1)
//   warps 4-7 epilogue    : tcgen05.ld 32x32b -> registers -> fused output transform -> global
// Epilogue modes:
//   EPI_I32      int32 C row-major                      (count rows: IBM aggregation, similar songs / users, explanations, parity probes)
//   EPI_U16_T    uint16 C^T  (Ct[n][m], m contiguous)   (UBM: train-user-major count panel consumed by the K2 gather)
//   EPI_I32_SCATTER  int32 rows stored into per-owner receive slots (local or NVLink peer memory): the reduce-scatter of the K-split
//                item-item sweep fused into the epilogue (coalesced 128-byte row segments via a shared-memory transpose)
//   EPI_ACC_U64  u64 out (+)= C << shift                         byte-plane accumulation of the weighted Gram Gq (item-space head rows)
#include "mr_common.cuh"
#include "mr_kernels.h"

#include <cuda.h>
#include <stdio.h>

namespace mr {

constexpr int kBM = 128;        // UMMA M (cta_group::1)
constexpr int kBK = 128;        // bytes (= u8 elements) of K per smem stage = one 128 B swizzle row
constexpr int kUmmaK = 32;      // K per tcgen05.mma for 8-bit operands
constexpr int kGemmThreads = 256;

template <int BN>
struct GemmCfg {
  static constexpr int kStageBytesA = kBM * kBK;
  static constexpr int kStageBytesB = BN * kBK;
  static constexpr int kStageBytes = kStageBytesA + kStageBytesB;
  static constexpr int kStages = (BN == 256) ? 4 : 6;
  static constexpr int kTmemCols = 2 * BN;  // double-buffered accumulator (power of two: 256 or 512)
  static constexpr int kTransposeBytes = 4 * 32 * 33 * 4;   // per epilogue warp a padded 32x32 int32 tile (EPI_I32_SCATTER)
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/ + kTransposeBytes;
};

struct GemmParams {
  int M, N;            // logical output extent (rows of A / rows of B that are real)
  int num_k_blocks;    // K_pad / 128
  int num_m_tiles, num_n_tiles;
  void* out;           // int32* / uint16_t* / unsigned long long*
  long long ld;        // leading dimension of `out` in elements
  int32_t* slots[8];   // EPI_I32_SCATTER: row m goes to slots[m / rows_per_owner] + (m % rows_per_owner) * ld  (peer or local memory)
  int rows_per_owner;
  int shift;           // EPI_ACC_U64: out = (plane 0 ? 0 : out) + (u64(acc) << shift)  (byte-plane weighted Gram)
  int accumulate;
};

// p is __grid_constant__ so that the run-time index into p.slots reads the parameter bank in place instead of a per-thread local copy of p
template <int BN, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
count_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ GemmParams p) {
  using Cfg = GemmCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  // 128 B swizzle atoms need 1024 B alignment
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::kStages * Cfg::kStageBytesA;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* full_bar = bars;                       // [kStages]  TMA -> MMA
  uint64_t* empty_bar = bars + Cfg::kStages;       // [kStages]  MMA -> TMA
  uint64_t* tmem_full = bars + 2 * Cfg::kStages;   // [2]        MMA -> epilogue
  uint64_t* tmem_empty = tmem_full + 2;            // [2]        epilogue -> MMA
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  int32_t* tr_smem = reinterpret_cast<int32_t*>(smem + Cfg::kStages * Cfg::kStageBytes + 256);   // [4 warps][32][33]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_tiles = p.num_m_tiles * p.num_n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_base_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_tile = tile % p.num_m_tiles, n_tile = tile / p.num_m_tiles;
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
          tma_load_2d(smem_a + stage * Cfg::kStageBytesA, &tmap_a, &full_bar[stage], kb * kBK, m_tile * kBM);
          tma_load_2d(smem_b + stage * Cfg::kStageBytesB, &tmap_b, &full_bar[stage], kb * kBK, n_tile * BN);
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_u8(kBM, BN);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BN);
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t adesc = umma_desc_k_sw128(smem_u32(smem_a + stage * Cfg::kStageBytesA));
          const uint64_t bdesc = umma_desc_k_sw128(smem_u32(smem_b + stage * Cfg::kStageBytesB));
#pragma unroll
          for (int k = 0; k < kBK / kUmmaK; ++k) {
            // advance 32 bytes of K inside the 128 B swizzle row: +2 in the (addr >> 4) start-address field
            umma_i8(d_tmem, adesc + static_cast<uint64_t>(k * (kUmmaK >> 4)), bdesc + static_cast<uint64_t>(k * (kUmmaK >> 4)),
                    idesc, static_cast<uint32_t>((kb | k) != 0));
          }
          umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs have read it
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[acc]);      // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (warps 4..7 own TMEM lane quadrants 0..3) =====================
    const int q = warp & 3;
    int acc = 0; uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m_tile = tile % p.num_m_tiles, n_tile = tile / p.num_m_tiles;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const int m = m_tile * kBM + q * 32 + lane;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BN);
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(taddr + static_cast<uint32_t>(c * 32), r);
        tmem_ld_wait();
        const int n0 = n_tile * BN + c * 32;
        if (n0 >= p.N) continue;
        if constexpr (EPI == EPI_I32) {
          if (m < p.M) {
            int32_t* dst = reinterpret_cast<int32_t*>(p.out) + static_cast<long long>(m) * p.ld + n0;
            if (n0 + 32 <= p.N) {
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<int4*>(dst + j) = make_int4((int)r[j], (int)r[j + 1], (int)r[j + 2], (int)r[j + 3]);
            } else {
              for (int j = 0; j < 32 && n0 + j < p.N; ++j) dst[j] = (int)r[j];
            }
          }
        } else if constexpr (EPI == EPI_I32_SCATTER) {
          // Reduce-scatter fused into the GEMM: every output row is stored straight into the receive slot of the rank that owns
          // it (its own HBM or a peer's over NVLink, IPC-mapped).  The 32x32 block is transposed through shared memory so that
          // each store instruction writes 128 contiguous bytes of ONE row — full NVLink / HBM packets instead of 32 slivers.
          int32_t* tile = tr_smem + q * (32 * 33);
#pragma unroll
          for (int j = 0; j < 32; ++j) tile[lane * 33 + j] = static_cast<int32_t>(r[j]);
          __syncwarp();
          const int m_base = m_tile * kBM + q * 32;
          if (n0 + lane < p.N) {
#pragma unroll 4
            for (int rr = 0; rr < 32; ++rr) {
              const int mm = m_base + rr;
              if (mm < p.M) {
                const int o = mm / p.rows_per_owner;
                p.slots[o][static_cast<long long>(mm - o * p.rows_per_owner) * p.ld + n0 + lane] = tile[rr * 33 + lane];
              }
            }
          }
          __syncwarp();
        } else if constexpr (EPI == EPI_U16_T) {
          // Ct[n][m] (p.ld = 128): the 32 lanes of a warp hold 32 consecutive m -> one 64-byte store per column n
          if (m < kUserBatch) {
            uint16_t* dst = reinterpret_cast<uint16_t*>(p.out) + static_cast<long long>(n0) * kUserBatch + m;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + j < p.N) dst[j * kUserBatch] = static_cast<uint16_t>(r[j] > 65535u ? 65535u : r[j]);
          }
        } else if constexpr (EPI == EPI_ACC_U64) {
          // byte-plane accumulation of a weighted contraction: the B operand held byte `shift/8` of a 32-bit weight
          if (m < p.M) {
            unsigned long long* dst = reinterpret_cast<unsigned long long*>(p.out) + static_cast<long long>(m) * p.ld + n0;
            if (n0 + 32 <= p.N) {
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                ulonglong2 v = p.accumulate ? *reinterpret_cast<ulonglong2*>(dst + j) : make_ulonglong2(0, 0);
                v.x += static_cast<unsigned long long>(r[j]) << p.shift;
                v.y += static_cast<unsigned long long>(r[j + 1]) << p.shift;
                *reinterpret_cast<ulonglong2*>(dst + j) = v;
              }
            } else {
              for (int j = 0; j < 32 && n0 + j < p.N; ++j)
                dst[j] = (p.accumulate ? dst[j] : 0ULL) + (static_cast<unsigned long long>(r[j]) << p.shift);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

// ------------------------------------------------------------------------------------------------
// CSR -> dense 0/1 u8 operand rows (K-major).  One warp per output row: zero the row, then scatter ones.
//   out[r][col] = 1 for col in idx[ptr[row_id(r)] .. ptr[row_id(r)+1]),  row_id(r) = rows ? rows[r] : row0 + r
// Rows r >= n_rows (padding up to n_rows_pad) are zeroed.  pitch is a multiple of 128 bytes.
// ------------------------------------------------------------------------------------------------
__global__ void expand_rows_kernel(const long long* __restrict__ ptr, const int* __restrict__ idx,
                                   const int* __restrict__ rows, int row0, int n_rows, int n_rows_pad,
                                   long long pitch, uint8_t* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  for (long long r = static_cast<long long>(blockIdx.x) * warps_per_block + (threadIdx.x >> 5); r < n_rows_pad;
       r += static_cast<long long>(gridDim.x) * warps_per_block) {
    uint8_t* dst = out + r * pitch;
    int4* d4 = reinterpret_cast<int4*>(dst);
    for (long long i = lane; i < pitch / 16; i += 32) d4[i] = make_int4(0, 0, 0, 0);
    __syncwarp();
    if (r < n_rows) {
      const int rid = rows ? rows[r] : row0 + static_cast<int>(r);
      const long long b = ptr[rid], e = ptr[rid + 1];
      for (long long i = b + lane; i < e; i += 32) dst[idx[i]] = 1;
    }
  }
}

// Weighted variant for the byte-plane GEMMs: out[r][col] = byte `plane` of weight[col] (instead of 1).
__global__ void expand_rows_weighted_kernel(const long long* __restrict__ ptr, const int* __restrict__ idx,
                                            const uint32_t* __restrict__ weight, int plane, int n_rows, long long pitch,
                                            uint8_t* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  for (long long r = static_cast<long long>(blockIdx.x) * warps_per_block + (threadIdx.x >> 5); r < n_rows;
       r += static_cast<long long>(gridDim.x) * warps_per_block) {
    uint8_t* dst = out + r * pitch;
    int4* d4 = reinterpret_cast<int4*>(dst);
    for (long long i = lane; i < pitch / 16; i += 32) d4[i] = make_int4(0, 0, 0, 0);
    __syncwarp();
    const long long b = ptr[r], e = ptr[r + 1];
    for (long long i = b + lane; i < e; i += 32) {
      const int c = idx[i];
      dst[c] = static_cast<uint8_t>((weight[c] >> (8 * plane)) & 255u);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || !p) return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 2-D u8 tensor [rows][pitch] -> box [box_rows][128 B], 128 B swizzle, zero fill out of bounds.
static int make_tmap_u8(CUtensorMap* tm, const uint8_t* base, long long rows, long long pitch, int box_rows) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return -1;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(pitch), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(pitch)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kBK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -2;
}

template <int BN, int EPI>
static cudaError_t launch_gemm_t(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, int num_sms, cudaStream_t st) {
  using Cfg = GemmCfg<BN>;
  {  // the attribute is per device (handles may live on several GPUs of one process); setting it is cheap, so no caching
    cudaError_t e = cudaFuncSetAttribute(count_gemm_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) return e;
  }
  const int tiles = p.num_m_tiles * p.num_n_tiles;
  const int grid = tiles < num_sms ? tiles : num_sms;
  count_gemm_kernel<BN, EPI><<<grid, kGemmThreads, Cfg::kSmemBytes, st>>>(ta, tb, p);
  return cudaGetLastError();
}

int launch_count_gemm(const uint8_t* A, long long a_rows, const uint8_t* B, long long b_rows, long long pitch, int M, int N,
                      int epi, void* out, long long ld, int num_sms, cudaStream_t st,
                      int shift, int accumulate, int32_t* const* slots, int n_slots, int rows_per_owner) {
  if (pitch % kBK != 0 || M <= 0 || N <= 0) return -3;
  const int bn = (N > 128) ? 256 : 128;
  CUtensorMap ta, tb;
  int rc = make_tmap_u8(&ta, A, a_rows, pitch, kBM);
  if (rc) return rc;
  rc = make_tmap_u8(&tb, B, b_rows, pitch, bn);
  if (rc) return rc;
  GemmParams p;
  p.M = M; p.N = N;
  p.num_k_blocks = static_cast<int>(pitch / kBK);
  p.num_m_tiles = (M + kBM - 1) / kBM;
  p.num_n_tiles = (N + bn - 1) / bn;
  p.out = out; p.ld = ld; p.shift = shift; p.accumulate = accumulate;
  for (int i = 0; i < 8; ++i) p.slots[i] = (slots && i < n_slots) ? slots[i] : nullptr;
  p.rows_per_owner = rows_per_owner > 0 ? rows_per_owner : 1;
  if (epi == EPI_I32_SCATTER && (!slots || n_slots < 1 || n_slots > 8 || static_cast<long long>(n_slots) * p.rows_per_owner < M)) return -4;
  cudaError_t e;
  if (bn == 256) {
    e = epi == EPI_I32 ? launch_gemm_t<256, EPI_I32>(ta, tb, p, num_sms, st)
      : epi == EPI_U16_T ? launch_gemm_t<256, EPI_U16_T>(ta, tb, p, num_sms, st)
      : epi == EPI_ACC_U64 ? launch_gemm_t<256, EPI_ACC_U64>(ta, tb, p, num_sms, st)
                         : launch_gemm_t<256, EPI_I32_SCATTER>(ta, tb, p, num_sms, st);
  } else {
    e = epi == EPI_I32 ? launch_gemm_t<128, EPI_I32>(ta, tb, p, num_sms, st)
      : epi == EPI_U16_T ? launch_gemm_t<128, EPI_U16_T>(ta, tb, p, num_sms, st)
      : epi == EPI_ACC_U64 ? launch_gemm_t<128, EPI_ACC_U64>(ta, tb, p, num_sms, st)
                         : launch_gemm_t<128, EPI_I32_SCATTER>(ta, tb, p, num_sms, st);
  }
  return e == cudaSuccess ? 0 : -100 - static_cast<int>(e);
}

int launch_expand_rows(const long long* ptr, const int* idx, const int* rows, int row0, int n_rows, int n_rows_pad,
                       long long pitch, uint8_t* out, cudaStream_t st) {
  if (n_rows_pad <= 0) return 0;
  const int threads = 256, wpb = threads / 32;
  long long blocks = (static_cast<long long>(n_rows_pad) + wpb - 1) / wpb;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  expand_rows_kernel<<<static_cast<int>(blocks), threads, 0, st>>>(ptr, idx, rows, row0, n_rows, n_rows_pad, pitch, out);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_expand_rows_weighted(const long long* ptr, const int* idx, const uint32_t* weight, int plane, int n_rows, long long pitch,
                                uint8_t* out, cudaStream_t st) {
  if (n_rows <= 0) return 0;
  const int threads = 256, wpb = threads / 32;
  long long blocks = (static_cast<long long>(n_rows) + wpb - 1) / wpb;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  expand_rows_weighted_kernel<<<static_cast<int>(blocks), threads, 0, st>>>(ptr, idx, weight, plane, n_rows, pitch, out);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------------------------------------------------------------
// Completion flags of the fused K-split exchange (EPI_I32_SCATTER): no host round trip per panel.  A sender's signal kernel runs on
// the library stream right after its scatter GEMM (stream order = its tiles have been issued and the kernel has drained), fences at
// system scope and raises a 64-bit counter in every owner's flag block with a release store — local HBM or a peer's over NVLink.
// The owner's wait kernel spins with acquire loads on its own flag block until every sender has reached the panel's sequence number,
// so whatever follows on that stream (the sum of the slots, the normalisation) sees complete data.  Waits are bounded (trap, no hang).
// ---------------------------------------------------------------------------------------------------------------------
__global__ void peer_signal_kernel(PeerFlags flags, int n, unsigned long long value) {
  if (static_cast<int>(threadIdx.x) < n) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flags.p[threadIdx.x]), "l"(value) : "memory");
  }
}

__global__ void peer_wait_kernel(const unsigned long long* flags, int n, unsigned long long value) {
  if (static_cast<int>(threadIdx.x) < n) {
    const long long t0 = clock64();
    for (;;) {
      unsigned long long v;
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + threadIdx.x) : "memory");
      if (v >= value) break;
      if (clock64() - t0 > 40000000000LL) __trap();     // ~20 s: a peer died or the protocol is broken
      __nanosleep(200);
    }
  }
  __syncthreads();
  __threadfence_system();
}

int launch_peer_signal(PeerFlags flags, int n, unsigned long long value, cudaStream_t st) {
  if (n < 1 || n > 8) return -2;
  peer_signal_kernel<<<1, 32, 0, st>>>(flags, n, value);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_peer_wait(const unsigned long long* flags, int n, unsigned long long value, cudaStream_t st) {
  if (n < 1 || n > 8) return -2;
  peer_wait_kernel<<<1, 32, 0, st>>>(flags, n, value);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mr
