"""ctypes binding of libmrscore.so (include/mrscore.h).  No fallback: a missing library or GPU raises."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
SO = PKG / "libmrscore.so"

MR_OK, MR_ERR_PARAM_RANGE, MR_ERR_KEY_MISMATCH, MR_ERR_CUDA, MR_ERR_NCCL, MR_ERR_OOM, MR_ERR_BAD_ARG, MR_ERR_STATE = range(8)
MR_UBM, MR_IBM, MR_LC, MR_AGG, MR_STOCH = range(5)
MR_ENGINE_AUTO, MR_ENGINE_TENSOR, MR_ENGINE_SPARSE = 0, 1, 2
MR_PROFILE = 4
MR_SPACE_AUTO, MR_SPACE_USER, MR_SPACE_ITEM = 0, 8, 16
MR_OPT_HEAD_MIN_DEG, MR_OPT_ITEM_BATCH, MR_OPT_SONG_WINDOW_LO, MR_OPT_SONG_WINDOW_HI = 1, 2, 3, 4
(MR_ING_TR_PTR, MR_ING_TR_COL, MR_ING_TE_PTR, MR_ING_TE_COL, MR_ING_LAB_PTR, MR_ING_LAB_COL, MR_ING_DEG_TRAIN, MR_ING_DEG_TEST, MR_ING_DEG_SONG,
 MR_ING_TRAIN_USER_CHARS, MR_ING_TRAIN_USER_OFF, MR_ING_TEST_USER_CHARS, MR_ING_TEST_USER_OFF, MR_ING_SONG_CHARS, MR_ING_SONG_OFF, MR_ING_TIMING_MS) = range(16)
TIMING_NAMES = ["expand", "count", "agg_ubm", "agg_ibm", "topk", "other", "precompute", "head_rowsum", "tail_scatter"]

# every symbol include/mrscore.h declares
SYMBOLS = ["mr_create", "mr_destroy", "mr_last_error", "mr_load", "mr_set_test_users", "mr_prepare", "mr_prepare_async", "mr_counts_ubm", "mr_counts_ibm", "mr_gram_rows_device", "mr_gram_rows_scatter", "mr_peer_alloc", "mr_peer_open", "mr_peer_close",
           "mr_similarity_ubm", "mr_similarity_ibm", "mr_score_dense", "mr_blend_dense", "mr_evaluate_dense", "mr_topk", "mr_topk_device",
           "mr_topk_fetch", "mr_topk_device_ptrs", "mr_set_option", "mr_invalidate_prepared", "mr_score_users", "mr_score_songs", "mr_map_at_k", "mr_write_model", "mr_format_double", "mr_topk_packed", "mr_topk_merge", "mr_gram_rows_scatter_async", "mr_peer_signal", "mr_peer_wait", "mr_sync", "mr_get_timing", "mr_reset_timing", "mr_set_profile", "mr_get_info", "mr_stream",
           "mr_ingest_tsv", "mr_ingest_error", "mr_ingest_dims", "mr_ingest_get", "mr_ingest_free",
           "mr_eval_range", "mr_eval_counts", "mr_eval_finish", "mr_eval_cutoffs",
           "mr_topk_multi", "mr_topk_multi_device", "mr_topk_multi_ptrs", "mr_eval_range_multi", "mr_eval_counts_multi",
           "mr_similar_songs", "mr_similar_users", "mr_explain", "mr_song_audience",
           "mr_set_topk_filter", "mr_topk_filtered", "mr_topk_filtered_device"]

_lib = None


class MrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libmrscore error {code}: {msg}")
        self.code = code
        self.msg = msg


def load():
    """dlopen libmrscore.so.  Raises if it has not been built — the product path never substitutes a CPU implementation."""
    global _lib
    if _lib is not None:
        return _lib
    so = Path(os.environ.get("MRSCORE_SO", SO))      # developer aid: an alternative build of the same library (kernel tuning experiments)
    if not so.exists():
        raise ImportError(f"{so} is missing: build it with `python -m musicrecommendation_b200.build` (needs nvcc). "
                          "There is no CPU fallback for the scoring path.")
    lib = C.CDLL(str(so))
    vp, i32, i64, u64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_double
    lib.mr_create.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), i32, C.c_uint]
    lib.mr_destroy.argtypes = [vp]
    lib.mr_destroy.restype = None
    lib.mr_last_error.argtypes = [vp]
    lib.mr_last_error.restype = C.c_char_p
    lib.mr_load.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.mr_set_test_users.argtypes = [vp, i32, vp, vp, vp, i64, i64]
    lib.mr_prepare.argtypes = [vp]
    lib.mr_prepare_async.argtypes = [vp]
    lib.mr_counts_ubm.argtypes = [vp, vp]
    lib.mr_counts_ibm.argtypes = [vp, i32, i32, vp]
    lib.mr_gram_rows_device.argtypes = [vp, i32, i32, C.POINTER(vp), C.POINTER(i64)]
    lib.mr_gram_rows_scatter.argtypes = [vp, i32, i32, C.POINTER(vp), i32, i32, i64]
    lib.mr_peer_alloc.argtypes = [vp, u64, C.POINTER(vp), vp]
    lib.mr_peer_open.argtypes = [vp, vp, C.POINTER(vp)]
    lib.mr_peer_close.argtypes = [vp, vp]
    lib.mr_similarity_ubm.argtypes = [vp, vp]
    lib.mr_similarity_ibm.argtypes = [vp, i32, i32, vp]
    lib.mr_score_dense.argtypes = [vp, i32, vp]
    lib.mr_blend_dense.argtypes = [vp, i32, dbl, u64, vp, vp, vp, i64, i64, i64]
    lib.mr_evaluate_dense.argtypes = [vp, vp, i32, i32, vp, vp, i32, C.POINTER(dbl)]
    lib.mr_topk.argtypes = [vp, i32, dbl, u64, i32, vp, vp, vp]
    lib.mr_topk_device.argtypes = [vp, i32, dbl, u64, i32]
    lib.mr_topk_fetch.argtypes = [vp, i32, vp, vp, vp]
    lib.mr_topk_device_ptrs.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.mr_set_option.argtypes = [vp, i32, i64]
    lib.mr_invalidate_prepared.argtypes = [vp]
    lib.mr_score_users.argtypes = [vp, i32, vp, i32, vp]
    lib.mr_score_songs.argtypes = [vp, i32, vp, i32, vp]
    lib.mr_map_at_k.argtypes = [vp, i32, vp, vp, i32, vp, vp, C.POINTER(dbl), vp]
    lib.mr_write_model.argtypes = [C.c_char_p, vp, i32, i32, vp, vp, vp, vp, i32, C.POINTER(i64)]
    lib.mr_format_double.argtypes = [dbl, C.c_char_p]
    lib.mr_topk_packed.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
    lib.mr_topk_merge.argtypes = [vp, i32, i32, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), vp, vp, vp]
    lib.mr_gram_rows_scatter_async.argtypes = [vp, i32, i32, C.POINTER(vp), i32, i32, i64]
    lib.mr_peer_signal.argtypes = [vp, C.POINTER(vp), i32, u64]
    lib.mr_peer_wait.argtypes = [vp, vp, i32, u64]
    lib.mr_sync.argtypes = [vp]
    lib.mr_get_timing.argtypes = [vp, vp, i32]
    lib.mr_reset_timing.argtypes = [vp]
    lib.mr_set_profile.argtypes = [vp, i32]
    lib.mr_get_info.argtypes = [vp, vp, i32]
    lib.mr_stream.argtypes = [vp]
    lib.mr_stream.restype = vp
    lib.mr_ingest_tsv.argtypes = [i32, vp, u64, vp, u64, vp, u64, C.POINTER(vp)]
    lib.mr_ingest_error.argtypes = [vp]
    lib.mr_ingest_error.restype = C.c_char_p
    lib.mr_ingest_dims.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.mr_ingest_get.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(i64)]
    lib.mr_ingest_free.argtypes = [vp]
    lib.mr_ingest_free.restype = None
    lib.mr_eval_range.argtypes = [vp, i32, dbl, u64, C.POINTER(dbl), C.POINTER(dbl)]
    lib.mr_eval_counts.argtypes = [vp, i32, dbl, u64, dbl, dbl, i32, vp, vp, vp, i32, vp, vp, vp]
    lib.mr_eval_finish.argtypes = [vp, vp, vp, i32, i32, vp, C.POINTER(dbl)]
    lib.mr_eval_cutoffs.argtypes = [dbl, dbl, i32, vp]
    lib.mr_topk_multi.argtypes = [vp, i32, vp, vp, vp, i32, vp, vp, vp]
    lib.mr_topk_multi_device.argtypes = [vp, i32, vp, vp, vp, i32]
    lib.mr_topk_multi_ptrs.argtypes = [vp, i32, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.mr_eval_range_multi.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.mr_eval_counts_multi.argtypes = [vp, i32, vp, vp, vp, vp, vp, i32, vp, vp, vp, i32, vp, vp, vp]
    lib.mr_similar_songs.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.mr_similar_users.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.mr_explain.argtypes = [vp, i32, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.mr_song_audience.argtypes = [vp, i32, dbl, u64, vp, i32, i32, vp, vp, vp]
    lib.mr_set_topk_filter.argtypes = [vp, vp, i32, vp, vp]
    lib.mr_topk_filtered.argtypes = [vp, i32, vp, vp, vp, i32, vp, vp, vp]
    lib.mr_topk_filtered_device.argtypes = [vp, i32, vp, vp, vp, i32]
    _lib = lib
    return lib
