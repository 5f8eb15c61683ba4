// mr_kernels.h — launcher prototypes shared between the kernel translation units and the C-ABI (mrscore.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mr {

constexpr int kUserBatch = 128;   // test users per batch of the user-space engine = UMMA M
constexpr int kHeadCtasPerSm = 8;  // head_rowsum: resident 256-thread CTAs per SM the UBM pass is compiled for (32 registers per thread)
constexpr int kDenseChunk = 1184;  // rows per device->host chunk of mr_score_dense
constexpr int kTailSubBatch = 592; // tail scatter runs per 592 users so its atomics stay within a ~1.8 GB slice of a Sint panel
// Count panels K1 hands to K2, train-user-major so that one gathered row serves the whole 128-user batch in one coalesced read:
//   UBM  u16 Ct[T][128]   256-byte rows     IBM (user space)  u32 Wi[T][128]   512-byte rows
// (A sub-panel-major variant with 32-byte, L2-resident rows was measured 1.7-1.9x slower on B200: random 32-byte sector
//  gathers out of L2 lose more than the saved HBM traffic gains — profiles/r01_notes.md.)
__host__ __device__ inline long long ct_index(long long T, int v, int b) { (void)T; return static_cast<long long>(v) * kUserBatch + b; }
__host__ __device__ inline long long wi_index(long long T, int v, int b) { (void)T; return static_cast<long long>(v) * kUserBatch + b; }

enum { EPI_I32 = 0, EPI_U16_T = 1, EPI_ACC_U64 = 3, EPI_I32_SCATTER = 4 };
enum { MODEL_UBM = 0, MODEL_IBM = 1, MODEL_LC = 2, MODEL_AGG = 3, MODEL_STOCH = 4 };

// ---- K1 (k1_count_gemm.cu)
int launch_count_gemm(const uint8_t* A, long long a_rows, const uint8_t* B, long long b_rows, long long pitch, int M, int N,
                      int epi, void* out, long long ld, int num_sms, cudaStream_t st,
                      int shift = 0, int accumulate = 0, int32_t* const* slots = nullptr, int n_slots = 0, int rows_per_owner = 0);
int launch_expand_rows_weighted(const long long* ptr, const int* idx, const uint32_t* weight, int plane, int n_rows, long long pitch,
                                uint8_t* out, cudaStream_t st);
int launch_expand_rows(const long long* ptr, const int* idx, const int* rows, int row0, int n_rows, int n_rows_pad,
                       long long pitch, uint8_t* out, cudaStream_t st);

// stream-ordered completion flags of the fused K-split exchange (k1_count_gemm.cu): a sender raises a 64-bit counter in every owner's
// memory (local or NVLink peer) after its tiles have landed; the owner spins on its own flags before it sums its slots
struct PeerFlags { unsigned long long* p[8]; };
int launch_peer_signal(PeerFlags flags, int n, unsigned long long value, cudaStream_t st);
int launch_peer_wait(const unsigned long long* flags, int n, unsigned long long value, cudaStream_t st);

// ---- K1s (k1_sparse_count.cu): the same counts from the inverted index, for shapes whose dense operands do not fit
int launch_sparse_count_u16t(const long long* te_ptr, const int* te_col, int u0, int n_users, const long long* csc_ptr,
                             const int* csc_idx, uint16_t* ct, long long n_train, cudaStream_t st);
struct CarryList {            // wrap-arounds of the u32 weighted-count panel: (v, b) pairs, repaired by launch_carry_fixup
  unsigned int* count;        // [1]
  uint2* events;              // [capacity]
  unsigned int capacity;
};
int launch_sparse_wcount_u32(const long long* te_ptr, const int* te_col, int u0, int n_users, const long long* csc_ptr,
                             const int* csc_idx, const uint32_t* qd, uint32_t* wi, long long n_train, CarryList carry, cudaStream_t st);
int launch_carry_fixup(CarryList carry, const long long* tr_ptr, const int* tr_col, long long* sint, long long spitch, cudaStream_t st);
int launch_sparse_gram_rows(const int* rows, int n_rows, const long long* csc_ptr, const int* csc_idx, const long long* tr_ptr,
                            const int* tr_col, int32_t* g, long long ldg, cudaStream_t st);

// ---- K2 (k2_aggregate.cu)
struct AggItems {            // work list over the train inverted index: one warp per item
  const int* song;           // [n_items]
  const long long* begin;    // [n_items] offset into csc_idx
  const int* len;            // [n_items]
  const uint8_t* split;      // [n_items] 1 -> the song is covered by several items (accumulate atomically)
  int n_items;
};
int launch_aggregate_ubm(const AggItems& items, const int* csc_idx, const uint32_t* qv, const uint16_t* ct, long long n_train,
                         long long* sint, long long spitch, int num_sms, cudaStream_t st);
int launch_aggregate_w32(const AggItems& items, const int* csc_idx, const uint32_t* wi, long long n_train, long long* sint,
                         long long spitch, int num_sms, cudaStream_t st);
int launch_aggregate_ibm(const long long* te_ptr, const int* te_col, const int* te_grow, const uint32_t* qd, int u0, int n_users,
                         const int32_t* g, long long ldg, int n_songs, long long* sint, long long spitch, cudaStream_t st);

// ---- item-space engine (k4_itemspace.cu)
struct HeadExceptions {      // entries of the packed head rows whose count exceeds 16 bits or whose weighted sum exceeds 32 bits
  unsigned int* count; unsigned int capacity;
  int* row; int* song; uint32_t* g_extra; unsigned long long* gq_extra;
};
int launch_gram_head_scatter(const int* head_song, const long long* lst_ptr, int r0, int r1, const long long* csc_ptr, const int* csc_idx,
                             const long long* tr_ptr, const long long* tr_end, const int* tr_col, const uint32_t* qv, uint32_t* g,
                             unsigned long long* gq, long long pitch, int packed, int num_sms, cudaStream_t st);
int launch_gram_head_direct(const int* head_song, const long long* lst_ptr, int r0, int r1, const long long* csc_ptr, const int* csc_idx,
                            const long long* tr_ptr, const long long* tr_end, const int* tr_col, const uint32_t* qv, uint16_t* g16,
                            uint32_t* gq32, long long pitch, int num_sms, cudaStream_t st);
int launch_pack_head_rows(const uint32_t* g, const unsigned long long* gq, int packed, int r0, int n_rows, long long pitch, int n_songs,
                          uint16_t* g16, uint32_t* gq32, HeadExceptions ex, int num_sms, cudaStream_t st);
// model: 1 = UBM pass over Gq32, 2 = IBM pass over G16; words = 32-bit words per row load (1, 2 or 4); threads per CTA (a CTA covers
// threads * songs-per-thread songs); groups / segments: see k4_itemspace.cu
int launch_head_rowsum(int model, int words, int threads, const int4* grp_hdr, int n_groups, const int4* seg, const int* ge_row,
                       const uint32_t* ge_q, int seg_cap, int ent_cap, const uint16_t* g16, const uint32_t* gq32, long long pitch,
                       int n_songs, long long* sint, long long spitch, cudaStream_t st);
int launch_zero_rows(const int* rows, int n_rows, long long* sint, long long spitch, cudaStream_t st);
int launch_head_fixup(int models, const long long* hu_ptr, const int* hu_row, const int* hu_song, const uint32_t* hu_q, int u0, int n_users,
                      const long long* ex_ptr, const int* ex_song, const uint32_t* ex_g, const unsigned long long* ex_gq,
                      long long* sint_u, long long* sint_i, long long spitch, cudaStream_t st);
int launch_tail_scatter(int models, const int* tu_user, const int* tu_song, const long long* tu_lptr, long long e0, long long e1,
                        const long long* csc_ptr, const int* csc_idx, const long long* tr_ptr, const long long* tr_end, const int* tr_col,
                        const uint32_t* qv, const uint32_t* qd, int u0, long long* sint_u, long long* sint_i, long long spitch, long long n_pairs,
                        int lanes, cudaStream_t st);

// ---- per-shard work lists of the item-space engine, built on the device (k7_testlists.cu)
size_t test_lists_temp_bytes(long long nnz);
int launch_build_test_lists(const long long* te_ptr, const int* te_col, int n_users, long long nnz, const int2* song_info, int* flag,
                            int* head_pos, long long* deg, long long* lsum, void* cub_tmp, size_t cub_tmp_bytes, int* hu_row, int* hu_song,
                            uint32_t* hu_q, long long* hu_ptr, int* tu_user, int* tu_song, long long* tu_lptr, long long* tu_ptr,
                            cudaStream_t st);
int launch_gather_group_entries(const int4* desc, int n_desc, const int* hu_row, const uint32_t* hu_q, int* ge_row, uint32_t* ge_q,
                                cudaStream_t st);

// ---- K3 (k3_topk.cu)
int launch_mask_listened(const long long* te_ptr, const long long* te_end, const int* te_col, int u0, int n_users, long long* sint_u,
                         long long* sint_i, long long spitch, cudaStream_t st);
int launch_dense_scores(int model, const long long* sint, long long spitch, int u0, int n_users, int n_songs, const double* rsa,
                        const double* rsd, double* out, cudaStream_t st);
struct BlendParams {
  int model;                 // MODEL_*
  double alpha, one_minus_alpha;   // LC (MusicRecommender.scala:328)
  long long agg_threshold;   // AGG: (pct * N).toInt (MR:372)
  double prob;               // STOCH (MR:447)
  unsigned long long seed;   // STOCH: java.util.Random seed
  const long long* pair_base;  // [U+1] exclusive prefix of per-user scored-pair counts (index in MAIN:57-59 order)
  const float* rsd_up;       // [S] rsd rounded up to fp32 (upper bounds for the IBM pre-filter of the top-k select), or null
  int ubm_int_ok;            // every UBM numerator of the shard is < 2^52: (double)Sint * rsu is strictly monotone in Sint, top-k may compare integers
  const long long* te_end;   // [U] end of each test row's scored columns: te_ptr + 1, or the in-window prefix ends (song window)
  int song_off;              // added to the ranked column ids: first song of the window (0 without one)
  unsigned int* stats;       // [3] or null: rows the fast path of the select handed to the exact path, short rows (exact path by design), degenerate rows (radix select)
  const uint32_t* allow;     // filtered top-k, full-row path (DESIGN.md §4.11): bitmap of the allowed columns (bit c % 32 of word c / 32), or null
};
int launch_select_bits(const BlendParams& bp, const long long* te_ptr, const int* te_col, int u0, int n_users, int n_songs,
                       uint64_t* sel, long long sel_pitch_words, cudaStream_t st);
int launch_topk(const BlendParams& bp, const long long* te_ptr, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                long long sel_pitch_words, int u0, int n_users, int n_songs, const double* rsa, const double* rsd, int k,
                int* out_song, double* out_score, int* out_len, cudaStream_t st);
constexpr int kMergeMaxParts = 16;   // song partitions whose ranked lists one launch_merge_topk joins
struct MergeParts { const int* song[kMergeMaxParts]; const double* score[kMergeMaxParts]; const int* len[kMergeMaxParts]; int n; };
int launch_merge_topk(const MergeParts& p, int k, int n_users, int* out_song, double* out_score, int* out_len, cudaStream_t st);
int launch_gather_columns(const double* dense, int n_rows, int n_songs, const int* songs, int n_sel, double* out, long long out_ld, int u_base,
                          cudaStream_t st);
int launch_blend_arrays(const BlendParams& bp, const double* ubm, const double* ibm, double* out, long long n, long long first_index,
                        cudaStream_t st);

// ---- evaluation (k5_evaluate.cu)
int launch_evaluate(const double* scores, int n_users, int n_songs, const long long* lab_ptr, const int* lab_col, const int* new_songs,
                    int n_new, int n_thresholds, unsigned long long* minmax, double* ap_out, int num_sms, cudaStream_t st);

// Streamed evaluateModel (DESIGN.md §4.5, §4.6): per slice of a batch's score panels (masked; the STOCH select plane built), the consumers
// of a GROUP of models in one launch, reading each panel sector, select word and label entry once: either the min / max of each model's
// emitted scores (bit patterns, mm[2 * out] / mm[2 * out + 1]) or each model's confusion counts of the label songs by threshold bucket.
// kEvalGroupMax: eval_count_kernel keeps 4 songs x n_thresholds u16 counters per thread and model (22 KB per model at 11 thresholds);
// five models take 110 KB, two CTAs per SM (sm_100a: 228 KB of shared memory per SM), so the five models of main.scala take one launch.
constexpr int kEvalGroupMax = 5;
struct EvalGroup {
  int n;                                        // models in the group, 1..kEvalGroupMax; at most one MODEL_STOCH (it reads the select plane)
  int model[kEvalGroupMax];
  double alpha[kEvalGroupMax], oma[kEvalGroupMax];   // LC
  const int* split[kEvalGroupMax];              // AGG: [U] per test user of the shard, the first column whose pair index reaches (pct * N).toInt
  int out[kEvalGroupMax];                       // index of the model in its set: min / max pair mm[2 * out], count block pred_b + out * model_stride
  unsigned long long cut[kEvalGroupMax][11];    // count pass: bit patterns of the model's cutoffs c_t (predicted at t <=> score >= c_t)
};
int launch_eval_range(const EvalGroup& g, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                      long long sel_pitch_words, int u0, int n_users, int n_songs, const double* rsa, const double* rsd,
                      unsigned long long* mm, cudaStream_t st);
struct EvalCounts {
  int n_thresholds;
  const int* colmap;             // [n_songs] scored column -> label-song index, -1 for columns that are no label song
  unsigned long long* pred_b;    // [n_new][n_thresholds] emitted pairs whose bucket (number of cutoffs <= score) is b + 1 (model 0 of the set)
  unsigned long long* tp_b;      // [n_new][n_thresholds] the same, restricted to labelled pairs
  long long model_stride;        // elements from one model's pred_b / tp_b block to the next model's
  unsigned long long* nlab;      // [n_new] labelled pairs of the scored columns (counted by the launch that gets it non-null)
  const long long* lab_ptr;      // [U + 1] label CSR of the shard (global song ids)
  const int* lab_col;
  int col_lo;                    // first song of the scored columns (song window); column = song - col_lo
};
int launch_eval_count(const EvalGroup& g, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                      long long sel_pitch_words, int u0, int n_users, int n_songs, const double* rsa, const double* rsd,
                      const EvalCounts& ec, cudaStream_t st);
// AGG's pick as one split column per test user (k3_topk.cu): split[u] for u in [0, n_users) of the shard
int launch_agg_split(const BlendParams& bp, const long long* te_ptr, const int* te_col, int n_users, int n_songs, int* split, cudaStream_t st);

int launch_map_at_k(const int* top_song, const int* top_len, int n_users, int k, const long long* lab_ptr, const int* lab_col,
                    double* ap_out, cudaStream_t st);

// ---- similar songs and similar users (k8_similar.cu, DESIGN.md §4.7, §4.8)
// kSimShortMax: events E_q (candidate ids with repeats) a short row gathers into shared memory: 12 bytes each (id + sort key),
// 96 KB at the limit, two CTAs per SM
constexpr int kSimShortMax = 8192;
// A query kind: query q -> items q_idx[q_ptr[q] .. q_ptr[q + 1]) -> candidates c_idx[c_ptr[j] .. c_ptr[j + 1]) of each item j; the score of
// (q, c) with count n is n / (sq_q[q] * sq_c[c]); self: c == q is no candidate (similar songs)
struct SimLists {
  const long long* q_ptr; const int* q_idx;
  const long long* c_ptr; const int* c_idx;
  const double* sq_q; const double* sq_c;
  bool self;
};
int launch_sqrt_deg(const int* deg, int n, double* out, cudaStream_t st);
int launch_sim_events(const int* ids, int n, const SimLists& l, long long* events, cudaStream_t st);
// cap: a power of two in [64, kSimShortMax], >= E_q of every query of the launch; query q writes row q_row[q] of the outputs ([row][k])
int launch_similar_short(const int* q_ids, const int* q_row, int n_q, int cap, const SimLists& l, int k, int* out_song, double* out_score,
                         int* out_len, cudaStream_t st);
// row r of g (count row of query rows[r] over n_cols candidates, ldg apart, padded to 32) -> row r of the outputs
int launch_similar_rows(const int* rows, int n_rows, const int32_t* g, long long ldg, int n_cols, const SimLists& l, int k, int* out_song,
                        double* out_score, int* out_len, cudaStream_t st);

// ---- explanations (k8_similar.cu, DESIGN.md §4.9): the contributors of (test user, song) scores of UBM or IBM from the count rows of a chunk
struct ExplainArgs {
  const int* keys;                                   // [rows] key of each count row: test user (UBM) or song (IBM)
  const int2* pairs;                                 // [n] (count row in the chunk, other id: song (UBM) or test user (IBM))
  const int32_t* g; long long ld;                    // count rows c(u, .) over the train users (UBM) or g(s, .) over the songs (IBM)
  const long long* list_ptr; const int* list_idx;    // contributor lists: the inverted index by song (UBM), the test rows (IBM)
  const long long* te_ptr; const int* te_col;        // test rows (ascending): the listened check
  const double* sq_key; const double* sq_other;      // sqrt of the degrees: deg_test, deg_train (UBM); deg_song_all, deg_song_all (IBM)
  const uint32_t* q;                                 // q_24(deg_train) (UBM), q_26(deg_song_all) (IBM)
  const double* rs;                                  // the score factor: rsa per test user (UBM), rsd per song (IBM)
};
struct ExplainOut { int* id; double* term; long long* num; int* len; int* count; long long* total; double* score; };   // [n][m] x 3, [n] x 4
int launch_explain_pairs(int model, const ExplainArgs& a, int n, int m, const ExplainOut& o, cudaStream_t st);

// ---- song audiences (k9_audience.cu, DESIGN.md §4.10): the column select of one masked batch into the running per-song lists
struct AudienceArgs {
  int model; double alpha, oma;                      // MODEL_*, LC weights
  const long long* su; const long long* si;          // the batch's masked panels, row r = test user u0 + r (null where the model reads none)
  long long spitch;
  const uint64_t* sel; long long sel_pitch;          // AGG / STOCH select plane of the batch (words per row)
  const double* rsa; const double* rsd;
  const int2* q;                                     // [n_q] (column, list row), ascending column
  int* user; double* score; int* len;                // running lists: [rows][k], [rows][k], [rows]
  unsigned int* radix_rows;                          // columns that took the radix select, or null
};
int launch_audience(const AudienceArgs& a, int n_q, int u0, int nb, int k, cudaStream_t st);

// ---- filtered top-k, candidate path (k10_filter.cu, DESIGN.md §4.11): per test user u0 + r the exact top-k of the masked panel rows r over
// the ascending allowed columns cols[0 .. n_cols); ids are reported as column + bp.song_off; bp.stats[2] counts the rows through the radix select
int launch_candidate_topk(const BlendParams& bp, const long long* sint_u, const long long* sint_i, long long spitch, const uint64_t* sel,
                          long long sel_pitch_words, int u0, int n_users, const int* cols, int n_cols, const double* rsa, const double* rsd, int k,
                          int* out_song, double* out_score, int* out_len, cudaStream_t st);

}  // namespace mr
