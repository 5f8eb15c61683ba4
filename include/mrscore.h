/*
 * mrscore.h — C-ABI of libmrscore.so: the B200-native drop-in for MusicRecommendation's scoring hot path.
 *
 * The reference (alberto-paparella/MusicRecommendation, Scala) has no FFI of its own; the boundary is the public method
 * surface of `MusicRecommender` (reference file src/main/scala/music_recommandation/MusicRecommender.scala, "MR" below)
 * and the per-partition objects of distributed.scala ("DIST").  Each entry point names the reference interface whose body
 * it replaces.  Plain C: pointers and sizes only, so that JNI, JNA, Panama and ctypes all bind it directly
 * (INTEGRATION.md shows the Scala/JNI stub).
 *
 * Conventions
 *  - One handle = one GPU = one process-local scorer ("one process per GPU"); handles are not thread-safe, use one per
 *    calling thread (Spark executor task threads, DIST:451-478).
 *  - Users and songs are dense int32 ids assigned in ascending String.compareTo order, so int order == Ordering.String
 *    (main.scala:57) and dense outputs are already in the order of the alignment sort main.scala:57-59.
 *  - Every function returns MR_OK or an error code; mr_last_error() gives the message.  Nothing exits or throws across
 *    the boundary (the reference calls System.exit(2) / System.exit(-1), MR:326, 366-369: the host wrapper maps
 *    MR_ERR_KEY_MISMATCH -> exit(2) and MR_ERR_PARAM_RANGE -> stderr message + exit(-1)).
 *  - Outputs are copied into caller-allocated host buffers; the library owns only device memory behind the handle.
 *  - There is no CPU fallback: without a CUDA device mr_create fails with MR_ERR_CUDA.
 */
#ifndef MRSCORE_H
#define MRSCORE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mr_handle mr_handle;

enum {
  MR_OK = 0,
  MR_ERR_PARAM_RANGE = 1,   /* blend parameter outside [0,1]            (System.exit(-1), MR:366-369, 434-437) */
  MR_ERR_KEY_MISMATCH = 2,  /* ubm / ibm arrays not aligned             (System.exit(2),  MR:326, 379, 445)    */
  MR_ERR_CUDA = 3,
  MR_ERR_NCCL = 4,
  MR_ERR_OOM = 5,
  MR_ERR_BAD_ARG = 6,
  MR_ERR_STATE = 7          /* call order: nothing loaded, no test users, no top-k computed ... */
};

/* model selectors */
enum {
  MR_UBM = 0,    /* getUserBasedModel[P]                MR:132, 177; DIST UserBasedModel  DIST:172-239 */
  MR_IBM = 1,    /* getItemBasedModel[P]                MR:222, 268; DIST ItemBasedModel  DIST:244-310 */
  MR_LC = 2,     /* getLinearCombinationModel[P]        MR:317, 340   param = alpha                     */
  MR_AGG = 3,    /* getAggregationModel[P]              MR:361, 396   param = itemBasedPercentage       */
  MR_STOCH = 4   /* getStochasticCombinationModel[P]    MR:429, 461   param = itemBasedProbability, seed = java.util.Random seed */
};

/* mr_create flags */
enum {
  MR_ENGINE_AUTO = 0,     /* tensor-core count GEMM when the dense 0/1 operands fit in HBM, else inverted-index counts */
  MR_ENGINE_TENSOR = 1,   /* force K1 = tcgen05 int8 GEMM */
  MR_ENGINE_SPARSE = 2,   /* force K1s = inverted-index counts */
  MR_ENGINE_MASK = 3,
  MR_PROFILE = 4,         /* record CUDA events around every kernel phase (mr_get_timing) */
  /* scoring formulation (bit-identical results; DESIGN.md §4) */
  MR_SPACE_AUTO = 0,      /* item space when the test shard has >= 1024 users, else user space */
  MR_SPACE_USER = 8,      /* K1 counts |I_u ∩ I_v| per test-user batch, K2 gathers them through the inverted index */
  MR_SPACE_ITEM = 16,     /* rows of the (weighted) song-song co-occurrence matrices: head rows precomputed once per train set */
  MR_SPACE_MASK = 24
};

/* Create a scorer on CUDA device device_ids[0] (n_devices must be 1: one process per GPU).  Replaces nothing in the
 * reference; it is the native half of `new MusicRecommender(...)` (MR:12). */
int mr_create(mr_handle** out, const int* device_ids, int n_devices, unsigned flags);
void mr_destroy(mr_handle* h);
const char* mr_last_error(const mr_handle* h);

/* Hand over the data model the constructor builds (MR:26-62): CSR of the binary train matrix (T x S) and of the visible
 * half of the test users (U x S), column ids ascending and unique within a row, plus the `.length` values the cosine
 * denominators use (MR:147: per-user song counts; MR:237: per-song listener counts over train AND test-visible rows).
 * n_test may be 0 (train replica only; test users follow through mr_set_test_users). */
int mr_load(mr_handle* h, int n_train, int n_test, int n_songs,
            const int64_t* tr_rowptr, const int32_t* tr_col,
            const int64_t* te_rowptr, const int32_t* te_col,
            const int32_t* deg_train, const int32_t* deg_test, const int32_t* deg_song_all);

/* Replace the current test users by a shard — the unit DIST's getRanks1(user) works on (DIST:198-205, 269-276), i.e.
 * `ctx.parallelize(testUsers, slices)` (DIST:451).  pair_index_base = number of scored pairs of all test users that sort
 * before this shard and n_pairs_total = ubm.length of the whole model; both only matter for MR_AGG / MR_STOCH (MR:372,
 * 381, 447).  Pass n_pairs_total = 0 for "this shard is the whole test set". */
int mr_set_test_users(mr_handle* h, int n_test, const int64_t* te_rowptr, const int32_t* te_col, const int32_t* deg_test,
                      int64_t pair_index_base, int64_t n_pairs_total);

/* Tunables.  MR_OPT_HEAD_MIN_DEG (before mr_load): a song gets a precomputed dense head row when it has at least this many train
 * listeners (0 = default max(2, S / 6000), the optimum when the rows are reused by many shards; a one-shot job over few test users is
 * faster with a smaller head, bench.py picks it from the number of shards per GPU).  MR_OPT_ITEM_BATCH: upper bound on the test users
 * per item-space batch (0 = as many as fit in HBM).  Results never depend on either. */
enum { MR_OPT_HEAD_MIN_DEG = 1, MR_OPT_ITEM_BATCH = 2, MR_OPT_SONG_WINDOW_LO = 3, MR_OPT_SONG_WINDOW_HI = 4 };
/* Song window (both before mr_load): the handle scores only the songs [LO, HI) of every test user — the reference's second
 * partitioning, `ctx.parallelize(songs, 4).map(getRanks2)` (DIST:214-221, 285-292, 459-461, 477-479): one partition of songs against ALL
 * test users.  Everything that is indexed by a scored column shrinks to HI - LO entries (head rows, score panels, mr_score_dense /
 * mr_score_users rows, the valid ids of mr_score_songs); the train set, the test histories and every degree are still the whole data
 * set's, so each score has the same bits as without a window.  mr_topk then ranks inside the window (ids are global song ids); the lists
 * of the partitions of one test user are joined by mr_topk_merge.  Needs MR_ENGINE_SPARSE and MR_SPACE_ITEM (AUTO selects them). */
int mr_set_option(mr_handle* h, int option, int64_t value);

/* Build the item-space head rows (G, Gq of the popular songs; DESIGN.md §4.2) now instead of lazily on the first scoring call
 * that uses them.  One-off per train set: tensor-core GEMMs on the tensor engine, inverted-index scatter otherwise. */
int mr_prepare(mr_handle* h);
/* The same build started on a stream of its own: returns as soon as the kernels are queued, so that the caller's next host work
 * (typically mr_set_test_users of the shard that is about to be scored) overlaps it; the first call that needs the rows completes
 * the build.  mr_prepare after mr_prepare_async waits for it. */
int mr_prepare_async(mr_handle* h);
/* Forget the head rows (their HBM stays allocated): the next mr_prepare / scoring call rebuilds them.  bench.py uses it to put the
 * whole of getUserBasedModel / getItemBasedModel (MR:132-170, 222-261 — they have no amortisable half) inside every timed step. */
int mr_invalidate_prepared(mr_handle* h);

/* Parity probes for kernel K1: out[u*T + v] = |I_u ∩ I_v| (numerator of MR:142-145), and rows [s0,s1) of the train
 * co-occurrence matrix out[(i-s0)*S + j] = |U_i ∩ U_j| over train users (numerator of MR:232-235). */
int mr_counts_ubm(mr_handle* h, int32_t* out_UxT);
int mr_counts_ibm(mr_handle* h, int s0, int s1, int32_t* out_rows);

/* Device-resident variant for the K-split item-item sweep (BASELINE configs[4], DIST:459-461 song partitioning): rows [s0,s1) of
 * this handle's PARTIAL co-occurrence matrix (its train-user shard only) stay in HBM as int32 [s1-s0][*ld]; the caller sums the
 * partial panels of all ranks with one NCCL reduce-scatter.  The pointer is valid until the next call on the handle. */
int mr_gram_rows_device(mr_handle* h, int s0, int s1, int32_t** dev_out, int64_t* ld);

/* The same with the reduce-scatter FUSED into the count GEMM: the epilogue stores every output row straight into the receive slot of
 * the rank that owns it — slot_ptrs[m / rows_per_owner] + (m % rows_per_owner) * ld, int32 — which may be this GPU's memory or a
 * peer's HBM mapped over NVLink (mr_peer_alloc / mr_peer_open, CUDA IPC), in coalesced 128-byte row segments, tile by tile while the
 * tensor cores work on the next tile.  The owner then sums its `world` slots locally (integers: exact).  Tensor engine only. */
int mr_gram_rows_scatter(mr_handle* h, int s0, int s1, void* const* slot_ptrs, int n_owners, int rows_per_owner, int64_t ld);
/* Stream-ordered variant for a pipelined exchange without host synchronisation: mr_gram_rows_scatter_async only enqueues; mr_peer_signal
 * enqueues "raise the 64-bit counters at flag_ptrs[0..n) (local or peer memory) to `value` once everything enqueued before has completed"
 * (system-scope release); mr_peer_wait enqueues "hold this handle's stream until the n consecutive 64-bit counters at `flags` (local
 * memory) are all >= value" (system-scope acquire, bounded: a dead peer traps instead of hanging).  mr_sync drains the handle's stream.
 * musicrecommendation_b200/ksplit.py shows the double-buffered protocol built from them. */
int mr_gram_rows_scatter_async(mr_handle* h, int s0, int s1, void* const* slot_ptrs, int n_owners, int rows_per_owner, int64_t ld);
int mr_peer_signal(mr_handle* h, void* const* flag_ptrs, int n, uint64_t value);
int mr_peer_wait(mr_handle* h, const void* flags, int n, uint64_t value);
int mr_sync(mr_handle* h);
int mr_peer_alloc(mr_handle* h, uint64_t bytes, void** dev_ptr, unsigned char* handle_out_64);   /* zeroed device buffer + its IPC handle */
int mr_peer_open(mr_handle* h, const unsigned char* handle_64, void** dev_ptr);                  /* map a peer's buffer into this process */
int mr_peer_close(mr_handle* h, void* dev_ptr);

/* Cosine similarities in fp32: user-user MR:140-149 and rows [s0,s1) of item-item MR:230-239 (denominator uses the train+test
 * listener counts, MR:237).  Each entry is float(c) * (rs(a) * rs(b)) for the count c and the degrees a, b of its row and column, with
 * rs(d) = float(1.0 / sqrt((double) d)) and rs(0) = 0. */
int mr_similarity_ubm(mr_handle* h, float* out_UxT);
int mr_similarity_ibm(mr_handle* h, int s0, int s1, float* out_rows);

/* Whole model as the dense row-major U x S matrix of fp64 scores in main.scala:57-59 order; NaN marks the listened pairs
 * the reference does not emit (MR:109).  model = MR_UBM | MR_IBM.  Small configurations only (U*S*8 bytes). */
int mr_score_dense(mr_handle* h, int model, double* out_UxS);

/* The per-partition granularities of distributed.scala: UserBasedModel / ItemBasedModel.getRanks1(user) (DIST:198-205, 269-276) — every
 * unlistened song of the listed test users, out[i*S + s] (NaN at listened pairs) — and getRanks2(song) (DIST:214-221, 285-292) — every
 * test user that has not listened to the listed songs, out[i*U + u] (NaN where user u listened to song_ids[i]).  model = MR_UBM | MR_IBM;
 * ids index the current test shard / the songs.  Same values as the corresponding entries of mr_score_dense. */
int mr_score_users(mr_handle* h, int model, const int32_t* user_idx, int n, double* out_nxS);
int mr_score_songs(mr_handle* h, int model, const int32_t* song_ids, int n, double* out_nxU);

/* Blends on materialised, aligned model arrays (MR:317-481): kind = MR_LC | MR_AGG | MR_STOCH.  first_index / n_total as in
 * mr_set_test_users (0 / 0 for whole models). */
int mr_blend_dense(mr_handle* h, int kind, double param, uint64_t seed, const double* ubm, const double* ibm, double* out,
                   int64_t n_pairs, int64_t first_index, int64_t n_total);

/* evaluateModel(model) — the reference's threshold-sweep mAP (MR:521-639, 62-75 s per model on the JVM at 2000 / 100 users,
 * README:940-944) on a materialised model: scores_UxS as mr_score_dense / mr_blend_dense produce it (NaN = pair not emitted), labels as
 * a CSR over the same test users (rows ascending; song ids >= n_songs are label songs that occur nowhere else).  n_thresholds = 10
 * (MR:590) or 11 (DIST:395).  Bit-identical to the CPU restatement. */
int mr_evaluate_dense(mr_handle* h, const double* scores_UxS, int n_users, int n_songs, const int64_t* lab_rowptr, const int32_t* lab_col,
                      int n_thresholds, double* out_map);

/* evaluateModel(model) (MR:521-639) for models too large to materialise: the same metric, streamed over the batches of the scoring
 * pipeline, with the same bits as mr_evaluate_dense on the materialised model.  It decomposes into integers that add exactly over batches,
 * user shards and song windows (DESIGN.md §4.5): per label song c and threshold t, pred_t(c) = test users whose normalised score for c
 * exceeds TH[t] (MR:541-553), tp_t(c) = the same among the users labelled with c, nlab(c) = users labelled with c; only the global min /
 * max (MR:524-529) must be known first.  A distributed caller runs range -> all-reduce(min, max) -> counts -> all-reduce(sum) -> finish
 * (INTEGRATION.md).  model / param / seed as in mr_topk; the LC alpha must be in [0, 1] (MR_ERR_PARAM_RANGE), as for getTopK.
 *
 * Range pass: min and max over the pairs this handle scores (its shard, its song window) that the model emits (listened pairs are not
 * emitted, MR:109); +inf / -inf when it emits none. */
int mr_eval_range(mr_handle* h, int model, double param, uint64_t seed, double* out_min, double* out_max);
/* Count pass, with the global mn / mx.  lab_rowptr [U + 1] / lab_col: the labels of the CURRENT shard's test users, rows ascending and
 * unique (song ids >= n_songs are label-only songs).  new_songs [n_new]: the distinct label songs of ALL test users (newSongs, MR:72, 79),
 * strictly ascending, containing every label song of this shard (MR_ERR_BAD_ARG naming the first one missing).  Outputs, row c for
 * new_songs[c]: out_pred / out_tp [n_new][n_thresholds], out_nlab [n_new].  A label entry (u, c) is counted by the handle whose shard holds
 * u and whose song window holds c, a label-only song by none (its AP is 0 whatever its counts), so the sums over any partitioning of
 * users and songs are the counts of the whole model.  n_thresholds = 10 (MR:590) or 11 (DIST:395).  On a single-batch item-space shard
 * the count pass reuses the score panels of an mr_eval_range of the same (model, param, seed) just before it: one scoring pass, not two. */
int mr_eval_counts(mr_handle* h, int model, double param, uint64_t seed, double mn, double mx, int n_thresholds,
                   const int64_t* lab_rowptr, const int32_t* lab_col, const int32_t* new_songs, int n_new,
                   int64_t* out_pred, int64_t* out_tp, int64_t* out_nlab);
/* Host only (no handle, no GPU): precision tp / pred and recall tp / nlab per threshold (MR:561-579), the per-song AP (MR:600-610,
 * out_ap [n_new], may be NULL) and the mean over the n_new songs (MR:626), in the operation order of mr_evaluate_dense. */
int mr_eval_finish(const int64_t* pred, const int64_t* tp, const int64_t* nlab, int n_new, int n_thresholds, double* out_ap, double* out_map);
/* Host only: out[t] = the least double x with RN(RN(x - mn) / RN(mx - mn)) > TH[t], TH = 0.0, 0.1, ..., 1.0, or +inf when no x in
 * [mn, mx] qualifies (always when mx - mn is not > 0).  The count pass predicts a pair at t iff its score >= out[t]. */
int mr_eval_cutoffs(double mn, double mx, int n_thresholds, double* out);

/* ---- model sets: several models from one scoring of the shard (DESIGN.md §4.6) ------------------------------------------------------
 * A model set is 1..16 entries (models[i], params[i], seeds[i]), each with the meaning it has in mr_topk; duplicates are allowed (a
 * parameter sweep is a set).  The calls score the shard and song window once per batch (one head pass per panel the set needs, one tail
 * scatter, one listened mask) and run every entry's consumer on the masked panels; entry i's outputs have exactly the bits of the
 * single-model call for entry i.  Every entry is checked before any GPU work: an LC alpha or an AGG / STOCH parameter outside [0, 1] or NaN
 * is MR_ERR_PARAM_RANGE, an unknown selector MR_ERR_BAD_ARG, and the message names the first bad entry ("entry i: ...").  The ownership
 * rule and the partition sums of the single-model calls hold per entry.  A set call leaves the single-model results (mr_topk_fetch,
 * mr_topk_device_ptrs, mr_map_at_k with NULL lists) untouched.
 *
 * getTopK for every entry: out_song[i] / out_score[i] / out_len[i] as mr_topk's for entry i (host arrays). */
int mr_topk_multi(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k,
                  int32_t* const* out_song, double* const* out_score, int32_t* const* out_len);
/* The same with the results kept in HBM, n_models x U x k x 12 bytes in a grow-only block of their own.  It must fit in the device memory
 * the batch plan leaves free (MR_ERR_OOM stating the bytes otherwise; the plan is not changed for it).  mr_topk_multi_ptrs gives entry i's
 * device arrays (int32 [U,k], double [U,k], int32 [U]), valid until the next set call or mr_set_test_users. */
int mr_topk_multi_device(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k);
int mr_topk_multi_ptrs(mr_handle* h, int i, int k, void** song, void** score, void** len);
/* Streamed evaluateModel for a set: out_min / out_max [n_models] as mr_eval_range's per entry; then the counts under per-entry global
 * (mn[i], mx[i]): out_pred / out_tp [n_models][n_new][n_thresholds], out_nlab [n_new] (label counts do not depend on the model).  Labels
 * and new_songs are checked as in mr_eval_counts, once per call.  On a single-batch item-space shard, mr_eval_counts_multi right after
 * mr_eval_range_multi of the same set reuses the score panels. */
int mr_eval_range_multi(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds,
                        double* out_min, double* out_max);
int mr_eval_counts_multi(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds,
                         const double* mn, const double* mx, int n_thresholds, const int64_t* lab_rowptr, const int32_t* lab_col,
                         const int32_t* new_songs, int n_new, int64_t* out_pred, int64_t* out_tp, int64_t* out_nlab);

/* ---- similar songs: the reference's item-item cosine ranked per song (DESIGN.md §4.7) -------------------------------------------------
 * For each query song i = song_ids[r] (any ids in [0, S), any order, duplicates allowed), the k songs s with the highest
 *   sim(i, s) = g(i, s) / (sqrt((double) d_i) * sqrt((double) d_s))      (cosineSimilarity, MR:230-239)
 * with g(i, s) = |U_i^train ∩ U_s^train| over train listeners only (MR:232) and d = deg_song_all as handed to mr_load (train plus test-visible
 * listeners, MR:237), evaluated in that operation order with correctly rounded steps: every score has the bits of the CPU formula.
 * Candidates are the co-listened songs only (s != i, g(i, s) > 0) — unlike getTopK, which ranks every unlistened song and so lists 0.0 scores,
 * a song that shares no train listener with i is never listed.  Order: score descending, then song id ascending (as mr_topk).
 * Outputs (host arrays): out_song / out_score [n][k], out_len [n]; row r belongs to song_ids[r]; out_len[r] = min(k, #candidates), song -1 /
 * score 0.0 past it.  A song without train listeners gets out_len 0.  1 <= k <= 1024.  Needs mr_load only (n_test may be 0; the test shard
 * plays no part).  MR_ERR_BAD_ARG names the first query id out of range; MR_ERR_STATE before mr_load and on a handle with a song window.
 * Rows whose work E_i = sum over the train listeners v of i of |I_v^train| is small are answered in shared memory (short path, timed as
 * MR_T_OTHER together with the E_i count); the others from exact count rows of the count engine in chunks of up to 1024 rows (MR_T_COUNT,
 * MR_T_EXPAND on the tensor engine) and a select over each chunk (MR_T_TOPK).  mr_get_info values 21 / 22 count the rows each path answered.
 * The call leaves every result and resident state of the scoring calls as it was (top-k results, score panels, head rows, the resident
 * reuse of mr_eval_counts) and returns with all its work complete.  MR_ERR_OOM, stating the bytes, when not even one chunk of count rows
 * fits in the free device memory. */
int mr_similar_songs(mr_handle* h, const int32_t* song_ids, int n, int k, int32_t* out_song, double* out_score, int32_t* out_len);

/* ---- similar users: the reference's user-user cosine ranked per test user (DESIGN.md §4.8) -----------------------------------------------
 * For each query u = user_idx[r] (indices into the CURRENT test shard, as mr_score_users: any order, duplicates allowed), the k train users v
 * with the highest
 *   w(u, v) = c / (sqrt((double) deg_test[u]) * sqrt((double) deg_train[v]))      (cosineSimilarity, MR:140-149)
 * with c = |I_u ∩ I_v| over u's visible test row and v's train row, and the degrees as handed to mr_load / mr_set_test_users (MR:147),
 * evaluated in that operation order with correctly rounded steps: every score has the bits of the CPU formula (the weight UBM sums, MR:159-166).
 * Candidates are the train users with c > 0 only: a train user who shares no song with u is never listed.  Order: score descending, then
 * train-user id ascending.  Outputs (host arrays): out_user / out_score [n][k], out_len [n]; row r belongs to user_idx[r]; out_len[r] =
 * min(k, #candidates), user -1 / score 0.0 past it.  A test user with an empty visible row gets out_len 0.  1 <= k <= 1024; n = 0 returns
 * MR_OK.  MR_ERR_BAD_ARG names the first query index outside [0, U); MR_ERR_STATE before mr_load and without test users.
 * Works on a handle with a song window and gives the same lists there (user ids are not rotated; the handle keeps whole rows).
 * Paths, phase timers and chunking as mr_similar_songs; mr_get_info values 23 / 24 count the rows each path answered.  The call leaves
 * every result and resident state of the scoring calls as it was and returns with all its work complete.  MR_ERR_OOM, stating the bytes,
 * when not even one chunk of count rows fits in the free device memory. */
int mr_similar_users(mr_handle* h, const int32_t* user_idx, int n, int k, int32_t* out_user, double* out_score, int32_t* out_len);

/* ---- explanations: why a song scores what it scores for a test user (DESIGN.md §4.9) --------------------------------------------------
 * Pair r is (u = user_idx[r], an index into the CURRENT test shard as in mr_score_users; s = song_ids[r] in [0, S)); any order, duplicates
 * allowed.  model = MR_UBM or MR_IBM (blends: MR_ERR_BAD_ARG).  The score of DESIGN.md §3 is one integer numerator times one factor, and
 * each term of the numerator is one contributor:
 *   MR_UBM: the train listeners v of s with c(u, v) = |I_u ∩ I_v| > 0;
 *           term = c / (sqrt((double) deg_test[u]) * sqrt((double) deg_train[v]))   (the score mr_similar_users gives (u, v)),
 *           num = c * q_24(deg_train[v]);
 *   MR_IBM: u's visible songs j != s with g(s, j) = |U_s^train ∩ U_j^train| > 0;
 *           term = g / (sqrt((double) d_s) * sqrt((double) d_j)), d = deg_song_all  (the score mr_similar_songs gives (s, j)),
 *           num = g * q_26(d_j);
 * each term evaluated in that operation order, correctly rounded.  Contributors are ordered by term descending, then id ascending.
 * Outputs (host arrays): out_id / out_term / out_num [n][m] hold the first out_len[r] = min(m, out_count[r]) contributors of pair r, then
 * id -1, term 0.0, num 0; out_count[r] = the number of all contributors; out_total[r] = the sum of num over ALL of them, whatever m;
 * out_score[r] = (double) out_total[r] * (2^-24 / sqrt(deg_test[u]) for UBM, 2^-26 / sqrt(d_s) for IBM), with the bits mr_topk and
 * mr_score_users give the pair.  Two exactness statements:
 *   1. out_total is the library's score numerator Sint[u, s], bit for bit;
 *   2. the sum of term over all contributors in ascending id is the as-written score of the reference's loops (MR:159-166, 249-257),
 *      bit for bit.
 * The two scores (the sum of the terms and out_score) differ within the quantisation bound of DESIGN.md §3: that is expected, not a bug.
 * A listened pair (s in I_u; the reference emits none, MR:109) gets score NaN, len 0, count 0, total 0; an unlistened pair without
 * contributors score 0.0 and len 0.  1 <= m <= 1024; n = 0 returns MR_OK.  MR_ERR_BAD_ARG names the first pair with an id out of range, and
 * covers a bad m or model and null arrays; MR_ERR_STATE before mr_load, without test users and on a handle with a song window.  One count
 * row serves all pairs of its key (UBM: c(u, .) over the train users, IBM: g(s, .) over the songs), built by the count engine in chunks of up
 * to 1024 rows (MR_T_COUNT, MR_T_EXPAND on the tensor engine); the contributors of each pair are ranked by one select (MR_T_TOPK).
 * mr_get_info value 25 counts the count rows built since mr_load.  The call leaves every result and resident state of the scoring calls as it
 * was and returns with all its work complete.  MR_ERR_OOM, stating the bytes, when not even one chunk of count rows fits. */
int mr_explain(mr_handle* h, int model, const int32_t* user_idx, const int32_t* song_ids, int n, int m, int32_t* out_id, double* out_term,
               int64_t* out_num, int32_t* out_len, int32_t* out_count, int64_t* out_total, double* out_score);

/* ---- song audiences: the test users who score a song highest (DESIGN.md §4.10) ----------------------------------------------------------
 * For each query song s = song_ids[r] (any order, duplicates allowed), the k test users u of the CURRENT shard with the highest score of
 * (u, s) under model / param / seed, which mean what they mean in mr_topk (any MR_* selector, blends fused).  Candidates are the test users
 * who have not listened to s (the reference emits no listened pair, MR:109); a 0.0 score is a candidate, as in mr_topk.  Order: score
 * descending, then user index ascending.  Every listed score has the bits mr_score_songs (getRanks2) and mr_topk give the pair, AGG and
 * STOCH under the global pair index of mr_set_test_users included.  User ids are indices into the current shard, as in mr_score_users.
 * Outputs (host arrays): out_user / out_score [n][k], out_len [n]; out_len[r] = min(k, test users who have not listened to s), user -1 /
 * score 0.0 past it.  On a handle with a song window the ids must lie in the window; such a handle sees every test user, so its lists are
 * the global ones.  1 <= k <= 1024; n = 0 returns MR_OK.  MR_ERR_BAD_ARG names the first id outside [0, S) or the window, and covers a bad
 * k or model and null arrays; MR_ERR_PARAM_RANGE as in mr_topk (LC alpha, AGG / STOCH parameter outside [0, 1] or NaN); MR_ERR_STATE
 * before mr_load and without test users.  A scoring call: it scores the shard once per batch (mr_get_info value 20 grows by the batches),
 * ranks each batch's panels by column (MR_T_TOPK) into running per-song lists of n x k x 12 bytes in a grow-only block of their own, and
 * returns with all its work complete.  The lists must fit in the device memory the batch plan leaves free (MR_ERR_OOM stating the bytes
 * otherwise; the plan is not changed for it).  It leaves the single-model top-k result and the model-set results untouched.
 * mr_get_info value 26 counts the query rows answered since mr_load, value 27 the (column, batch) selects that took the radix select. */
int mr_song_audience(mr_handle* h, int model, double param, uint64_t seed, const int32_t* song_ids, int n, int k, int32_t* out_user,
                     double* out_score, int32_t* out_len);

/* ---- filtered top-k: an allowed song set and per-user exclusions (DESIGN.md §4.11) -------------------------------------------------------
 * The filter belongs to the handle's CURRENT test shard: an allowed song set A (allow_songs [n_allow], global ids in [0, S), any order,
 * duplicates ignored; n_allow = -1: every song, 0: the empty set) and exclusion rows E_u (ex_rowptr [U + 1] with ex_rowptr[0] = 0,
 * non-decreasing, one row per test user of the shard; ex_col ids in [0, S), strictly ascending within a row; ex_rowptr = NULL: none).
 * The candidates of test user u are the songs of the handle's window that lie in A, that u has not listened to (MR:109) and that are not in
 * E_u (an excluded listened song changes nothing).  A handle with a song window keeps the in-window part of A and E: ids outside it are no
 * error, so every rank of a song-partitioned job sets the same global filter.  mr_set_topk_filter(h, NULL, -1, NULL, NULL) clears it;
 * mr_set_test_users drops it.  MR_ERR_BAD_ARG names the first allowed id out of range or the first bad exclusion row; MR_ERR_STATE before
 * mr_load and without test users; MR_ERR_OOM (stating the bytes) when the filter's device copy does not fit in the caller's reserve the
 * batch plan leaves free.  The filter changes no other call: every unfiltered call gives what it gives without one. */
int mr_set_topk_filter(mr_handle* h, const int32_t* allow_songs, int n_allow, const int64_t* ex_rowptr, const int32_t* ex_col);
/* The filtered top-k of a model set (arguments, checks and outputs as mr_topk_multi): for every entry, each test user's unfiltered ranking
 * (score descending, song id ascending) with every non-candidate removed, truncated to k.  Every listed score has the bits mr_topk and
 * mr_score_users give the pair, AGG and STOCH under the global pair index of mr_set_test_users (a filter removes pairs from the output,
 * it never renumbers the model).  out_len[u] = min(k, candidates of u), song -1 / score 0.0 past it.  MR_ERR_STATE without a filter.  A
 * scoring call: the exclusions are written into the score panels as listened pairs (MR_T_TOPK), after which the lists come from the
 * full-row select with the allowed-column bitmap, or, for an allowed set below 3 % of the window, from a select over the allowed
 * columns only; mr_get_info values 28 / 29 count the rows (test users x entries) each path answered since mr_load. */
int mr_topk_filtered(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k,
                     int32_t* const* out_song, double* const* out_score, int32_t* const* out_len);
/* The same with the lists kept in HBM as the result of a set call (mr_topk_multi_device, read with mr_topk_multi_ptrs); it replaces the
 * last set result and leaves the single-model result untouched. */
int mr_topk_filtered_device(mr_handle* h, int n_models, const int* models, const double* params, const uint64_t* seeds, int k);

/* mAP@k of ranked lists against the hidden (label) half of the test users — north_star's "mAP@500".  The reference has no ranking and
 * no such metric (its evaluateModel is the threshold sweep above); this is the Million Song Dataset Challenge definition:
 * AP@k(u) = (sum_{i<=n} [r_i in L_u] * hits_i / i) / min(|L_u|, k), mean over the test users with at least one label row.
 * top_song [n_users x k] / top_len [n_users] as mr_topk returns them, or both NULL to rank the device-resident result of the last
 * mr_topk / mr_topk_device of this handle (n_users must then be the shard size).  out_ap (optional) receives the per-user AP.
 * Users are folded in ascending id order, terms in rank order (fp64), so the CPU restatement the tests hold gives the same bits. */
int mr_map_at_k(mr_handle* h, int k, const int32_t* top_song, const int32_t* top_len, int n_users, const int64_t* lab_rowptr,
                const int32_t* lab_col, double* out_map, double* out_ap);

/* getTopK(model, k): per test user the k best unlistened songs, score descending then song id ascending (new derived
 * output named by north_star; the reference has no ranking step).  out_song / out_score are U x k (song -1 / score 0.0 past
 * out_len[u] = min(k, S - |I_u|)).  1 <= k <= 1024.  model = any MR_* selector; blends are fused into the select. */
int mr_topk(mr_handle* h, int model, double param, uint64_t seed, int k, int32_t* out_song, double* out_score, int32_t* out_len);

/* The same, split for callers that keep results on the device between steps: compute only (results stay in HBM), then fetch. */
int mr_topk_device(mr_handle* h, int model, double param, uint64_t seed, int k);
int mr_topk_fetch(mr_handle* h, int k, int32_t* out_song, double* out_score, int32_t* out_len);
/* Device addresses of the last mr_topk_device result (int32 [U,k], double [U,k], int32 [U]) for callers that gather it over
 * NCCL without a host round trip (the reference's `.collect`, DIST:451-478).  Valid until the next call on the handle. */
int mr_topk_device_ptrs(mr_handle* h, int k, void** song, void** score, void** len);
/* The three arrays live in ONE device block (song | score | len at the returned byte offsets), so the whole result of a shard travels
 * in a single transfer — one NCCL gather to the rank that plays the Spark driver instead of three collectives. */
int mr_topk_packed(mr_handle* h, int k, void** base, uint64_t* bytes, uint64_t* score_offset, uint64_t* len_offset);
/* Join the ranked lists that n_parts song partitions produced for the same n_users test users (the driver-side `.collect` of DIST:461, 479
 * followed by the ranking): part_song[p] / part_score[p] / part_len[p] are DEVICE arrays ([n_users, k] int32, [n_users, k] double,
 * [n_users] int32, each list ordered by (score descending, song id ascending) as mr_topk leaves it); out_* are device arrays of the same
 * shapes and receive the first min(k, sum of lengths) entries of the merged order.  Exact: the global top-k is contained in the union of
 * the partitions' top-k.  Runs on the handle's stream (mr_stream); the pointer tables themselves are host memory. */
int mr_topk_merge(mr_handle* h, int k, int n_parts, int n_users, const int32_t* const* part_song, const double* const* part_score,
                  const int32_t* const* part_len, int32_t* out_song, double* out_score, int32_t* out_len);

/* ---- ingest: `new MusicRecommender(trainFile, testFile, testLabelsFile)` (MR:12, 26-91) on the GPU ----------------------------------
 * The three TSV files as byte buffers (`user \t song \t count` per line, third field ignored, MR:35) become the int-id data model
 * mr_load takes: ids assigned in ascending String.compareTo order per id space (train users; test users; songs of the train and the test
 * file, MR:38, 51, 58), sorted de-duplicated CSR rows, and the `.length` degrees that count duplicate rows (MR:40-41, 147, 237).  Label
 * rows of users outside the test file are dropped; label songs that occur nowhere else get ids >= n_songs (they score 0 in MR:521-639).
 * A line without exactly 3 fields (after Java's split dropped trailing empty ones) is the reference's scala.MatchError -> MR_ERR_BAD_ARG
 * naming the line.  The result lives in host memory owned by the library until mr_ingest_free.  No CPU fallback. */
typedef struct mr_ingest mr_ingest;
enum { MR_ING_TR_PTR = 0, MR_ING_TR_COL, MR_ING_TE_PTR, MR_ING_TE_COL, MR_ING_LAB_PTR, MR_ING_LAB_COL,      /* int64 [rows+1] / int32 [nnz] */
       MR_ING_DEG_TRAIN, MR_ING_DEG_TEST, MR_ING_DEG_SONG,                                                   /* int32 */
       MR_ING_TRAIN_USER_CHARS, MR_ING_TRAIN_USER_OFF, MR_ING_TEST_USER_CHARS, MR_ING_TEST_USER_OFF,           /* id -> string tables: bytes + int64 [n+1] */
       MR_ING_SONG_CHARS, MR_ING_SONG_OFF,                                                                   /* n_songs + n_label_only entries */
       MR_ING_TIMING_MS };                                                                                   /* double [8]: h2d, lines+parse, users, songs, host sort, csr, -, total */
int mr_ingest_tsv(int device, const char* train, uint64_t train_len, const char* test, uint64_t test_len, const char* labels,
                  uint64_t labels_len, mr_ingest** out);
const char* mr_ingest_error(const mr_ingest* g);
int mr_ingest_dims(const mr_ingest* g, int32_t* n_train, int32_t* n_test, int32_t* n_songs, int32_t* n_label_only_songs);
int mr_ingest_get(const mr_ingest* g, int which, const void** ptr, int64_t* n_elems);
void mr_ingest_free(mr_ingest* g);

/* ---- model file writer: writeModelOnFile (MR:489-496), host code ------------------------------------------------------------------------
 * One line `user \t song \t Double.toString(score) \n` per emitted pair of a materialised model (scores_UxS as mr_score_dense /
 * mr_blend_dense produce it, NaN = not emitted), in main.scala:57-59 order, with the ids turned back into the reference's strings through
 * the id -> string tables (bytes + int64 offsets [n+1], as mr_ingest_get returns them).  Scores are laid out by java.lang.Double.toString's
 * rules (shortest round-tripping digits; plain decimal in [1e-3, 1e7), d.dddE-n otherwise) so importModelFromFile (MR:505-512) reads
 * them back bit for bit.  mr_format_double exposes the formatter (out32: >= 32 bytes, NUL-terminated; returns the length). */
int mr_write_model(const char* path, const double* scores_UxS, int n_users, int n_songs, const char* user_chars, const int64_t* user_off,
                   const char* song_chars, const int64_t* song_off, int append, int64_t* rows_written);
int mr_format_double(double x, char* out32);

/* Introspection used by bench.py / tests. */
enum { MR_T_EXPAND = 0, MR_T_COUNT = 1, MR_T_AGG_UBM = 2, MR_T_AGG_IBM = 3, MR_T_TOPK = 4, MR_T_OTHER = 5,
       MR_T_PRECOMPUTE = 6, MR_T_HEAD_ROWSUM = 7, MR_T_TAIL_SCATTER = 8, MR_T_N = 9 };
int mr_get_timing(mr_handle* h, double* ms_out, int n);      /* accumulated CUDA-event ms per phase since the last reset */
int mr_reset_timing(mr_handle* h);
int mr_set_profile(mr_handle* h, int on);                   /* toggle MR_PROFILE at run time (it synchronises after every phase) */
int mr_get_info(mr_handle* h, int64_t* out, int n);          /* [engine, kernel launches so far, dense operand bytes, n_items, num_sms, device bytes the handle holds now, space, n_head songs,
                                                                 test entries on head songs, test entries on tail songs, head-row exceptions,
                                                                 test users per batch, head_rowsum work groups per batch, users split over groups,
                                                                 scored columns (= songs of the window), first song of the window,
                                                                 top-k select since mr_load: rows its sampled fast path handed to the exact path, short rows
                                                                 (exact path by design), degenerate rows (radix select),
                                                                 scoring passes since mr_load (batches whose score panels were built),
                                                                 mr_similar_songs rows since mr_load: answered by the short path, by the long path,
                                                                 mr_similar_users rows since mr_load: answered by the short path, by the long path,
                                                                 mr_explain count rows built since mr_load,
                                                                 mr_song_audience since mr_load: query rows answered, column selects through the radix select,
                                                                 mr_topk_filtered rows since mr_load: answered by the full-row path, by the candidate path,
                                                                 carry events of the u32 weighted-count panel in the last scoring call (sparse
                                                                 user-space IBM; 0 after any other call), staged head rows (the rest are built
                                                                 in place), whether the last head-row build used the packed 64-bit accumulator,
                                                                 byte planes of the weights in the last tensor-engine head-row build (0 = none),
                                                                 whether the top-k select may rank the UBM integers of the current shard] */
void* mr_stream(mr_handle* h);                               /* cudaStream_t every call's work is ordered on: what a caller enqueues on it
                                                                 after a call returns runs behind that call's results (internally the
                                                                 batches of a top-k call also use a second stream, joined back before
                                                                 the call returns) */

#ifdef __cplusplus
}
#endif
#endif /* MRSCORE_H */
