"""Host-side mirror of the reference's `MusicRecommender` class (MusicRecommender.scala:12-640) over libmrscore.so.

Same method names, argument meaning and error behaviour as the Scala class, so a caller of the reference finds
`getUserBasedModel`, `getItemBasedModel`, the three blends, `writeModelOnFile`, `importModelFromFile` and `evaluateModel`
where they expect them; every scoring method is one call through the C-ABI (include/mrscore.h) into the sm_100a kernels.
The JVM is absent from this image, so this mirror is Python; INTEGRATION.md shows the Scala/JNI binding of the same ABI.

Differences a caller can observe (all documented in DESIGN.md):
  * models come back already in the order of the alignment sort main.scala:57-59 (user asc, song asc), as a `Model`
    holding the dense U x S score matrix (NaN = pair not emitted, MR:109); `Model.tuples()` yields the reference's
    `(user, (song, score))` elements;
  * where the reference calls System.exit(2) / System.exit(-1) this raises `KeyMismatch` / `ParameterRange` (the Scala
    wrapper maps the error codes back to the exits);
  * `getStochasticCombinationModel` takes an explicit `seed` (the reference uses an unseeded `new Random`, MR:439);
  * `getTopK` is new (north_star): the only output that exists at MSD scale.
"""
from __future__ import annotations

import ctypes as C
import io
import sys
from dataclasses import dataclass
from typing import NamedTuple

import numpy as np

from . import _lib
from .dataset import Dataset, _csr_from_pairs
from .javafmt import double_to_string


class KeyMismatch(RuntimeError):
    """ubm / ibm not aligned — the reference calls System.exit(2) (MR:326, 347, 379, 413, 445, 476)."""
    exit_code = 2


class ParameterRange(ValueError):
    """blend parameter outside [0,1] — the reference prints to stderr and calls System.exit(-1) (MR:366-369, 434-437)."""
    exit_code = -1


@dataclass
class Model:
    """A scored model in main.scala:57-59 order.  scores[u, s] is NaN where the reference emits no element (MR:109)."""
    scores: np.ndarray            # [U, S] float64
    test_users: list | None = None
    songs: list | None = None
    name: str = ""

    def __len__(self) -> int:
        return int(np.count_nonzero(~np.isnan(self.scores)))

    def compact(self) -> np.ndarray:
        """The score column of the sorted `Array[(String, (String, Double))]`."""
        return self.scores[~np.isnan(self.scores)]

    def keys(self):
        u, s = np.nonzero(~np.isnan(self.scores))
        return u.astype(np.int32), s.astype(np.int32)

    def tuples(self):
        u, s = self.keys()
        v = self.scores[u, s]
        un = self.test_users if self.test_users is not None else list(range(self.scores.shape[0]))
        sn = self.songs if self.songs is not None else list(range(self.scores.shape[1]))
        for a, b, c in zip(u.tolist(), s.tolist(), v.tolist()):
            yield un[a], (sn[b], c)


class Explanation(NamedTuple):
    """The contributors of (test user, song) scores (mr_explain, DESIGN.md §4.9), row r for pair r: the first len[r] of count[r]
    contributors by term descending then id ascending (id -1, term 0.0, num 0 past len[r]); total[r] = the sum of num over all of them, the
    score's exact numerator; score[r] = the library's score of the pair (NaN for a listened pair)."""
    id: np.ndarray        # [n, m] int32: train users (UBM) or the user's visible songs (IBM)
    term: np.ndarray      # [n, m] float64: the cosine weight of the contributor, as the reference computes it
    num: np.ndarray       # [n, m] int64: the contributor's term of the fixed-point numerator (DESIGN.md §3)
    len: np.ndarray       # [n] int32
    count: np.ndarray     # [n] int32
    total: np.ndarray     # [n] int64
    score: np.ndarray     # [n] float64


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


def _cuda_view(ptr, shape, typestr):
    """A torch view (no copy) of device memory the library owns."""
    import torch

    class _Arr:
        __cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2}
    return torch.as_tensor(_Arr(), device="cuda")


def parse_triplets(stream):
    """One TSV stream -> (users list, songs list) exactly as MR:32-42 accepts it: 3 tab-separated fields, third ignored.
    Java's String.split drops trailing empty strings; a line without exactly 3 fields raises (scala.MatchError, MR:34-35)."""
    users, songs = [], []
    for line in stream:
        line = line.rstrip("\n").rstrip("\r")
        parts = line.split("\t")
        while parts and parts[-1] == "":
            parts.pop()
        if len(parts) != 3:
            raise ValueError(f"scala.MatchError: line does not have 3 tab-separated fields: {line!r}")
        users.append(parts[0])
        songs.append(parts[1])
    return users, songs


def dataset_from_streams(train, test, labels) -> Dataset:
    """The constructor's ingest (MR:26-91) with ids assigned in ascending string order.  Degrees are the `.length` of the
    reference's non-deduplicated lists (MR:40-41), so duplicate rows inflate denominators exactly as they do there."""
    tr_u, tr_s = parse_triplets(train)
    te_u, te_s = parse_triplets(test)
    lb_u, lb_s = parse_triplets(labels)
    train_users = sorted(set(tr_u))
    test_users = sorted(set(te_u))
    songs = sorted(set(tr_s) | set(te_s))                    # mutSongs: train ∪ test-visible (MR:38, 51, 58)
    label_only = sorted(set(lb_s) - set(songs))              # label songs that occur nowhere else get ids >= S
    tix = {u: i for i, u in enumerate(train_users)}
    uix = {u: i for i, u in enumerate(test_users)}
    six = {s: i for i, s in enumerate(songs + label_only)}
    T, U, S = len(train_users), len(test_users), len(songs)
    tr_rows = np.fromiter((tix[u] for u in tr_u), np.int64, len(tr_u))
    tr_cols = np.fromiter((six[s] for s in tr_s), np.int64, len(tr_s))
    te_rows = np.fromiter((uix[u] for u in te_u), np.int64, len(te_u))
    te_cols = np.fromiter((six[s] for s in te_s), np.int64, len(te_s))
    lb_keep = [(uix[u], six[s]) for u, s in zip(lb_u, lb_s) if u in uix]
    lb_rows = np.array([a for a, _ in lb_keep], np.int64)
    lb_cols = np.array([b for _, b in lb_keep], np.int64)
    tr_ptr, tr_col = _csr_from_pairs(tr_rows, tr_cols, T)
    te_ptr, te_col = _csr_from_pairs(te_rows, te_cols, U)
    lab_ptr, lab_col = _csr_from_pairs(lb_rows, lb_cols, U)
    deg_tr = np.bincount(tr_rows, minlength=T).astype(np.int32)           # .length incl. duplicates (MR:147)
    deg_te = np.bincount(te_rows, minlength=U).astype(np.int32)
    deg_song = (np.bincount(tr_cols, minlength=S) + np.bincount(te_cols, minlength=S)).astype(np.int32)   # MR:237
    return Dataset(T, U, S, tr_ptr, tr_col, te_ptr, te_col, lab_ptr, lab_col, deg_tr, deg_te, deg_song,
                   train_users, test_users, songs + label_only, {"source": "tsv"})


def _read_bytes(f) -> bytes:
    if isinstance(f, (bytes, bytearray, memoryview)):
        return bytes(f)
    if isinstance(f, str) or hasattr(f, "__fspath__"):
        with open(f, "rb") as fh:
            return fh.read()
    data = f.read()
    return data.encode("utf-8") if isinstance(data, str) else bytes(data)


def dataset_from_streams_native(train, test, labels, device: int = 0, with_strings: bool = True) -> Dataset:
    """The same ingest on the GPU (`mr_ingest_tsv`, csrc/k6_ingest.cu): the three TSV files as bytes -> int-id CSR, ids in ascending
    string order, `.length` degrees.  Same result as dataset_from_streams (tests/test_gpu_parity.py compares them field by field);
    a malformed line raises ValueError like the host path.  `timing_ms` of the stages is kept in Dataset.meta."""
    lib = _lib.load()
    bufs = [_read_bytes(f) for f in (train, test, labels)]
    g = C.c_void_p()
    rc = lib.mr_ingest_tsv(device, bufs[0], len(bufs[0]), bufs[1], len(bufs[1]), bufs[2], len(bufs[2]), C.byref(g))
    try:
        if rc != _lib.MR_OK:
            msg = (lib.mr_ingest_error(g) or b"").decode()
            if rc == _lib.MR_ERR_BAD_ARG and msg.startswith("scala.MatchError"):
                raise ValueError(msg)
            raise _lib.MrError(rc, msg)
        dims = [C.c_int32() for _ in range(4)]
        lib.mr_ingest_dims(g, *[C.byref(d) for d in dims])
        T, U, S, n_extra = (d.value for d in dims)

        def get(which, dtype):
            ptr, n = C.c_void_p(), C.c_int64()
            lib.mr_ingest_get(g, which, C.byref(ptr), C.byref(n))
            if n.value == 0:
                return np.zeros(0, dtype)
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(np.ctypeslib.as_ctypes_type(dtype))), shape=(n.value,)).copy()

        def table(chars_id, off_id):
            if not with_strings:
                return None
            chars = get(chars_id, np.uint8).tobytes()
            off = get(off_id, np.int64)
            return [chars[off[i]:off[i + 1]].decode("utf-8") for i in range(len(off) - 1)]

        return Dataset(T, U, S, get(_lib.MR_ING_TR_PTR, np.int64), get(_lib.MR_ING_TR_COL, np.int32), get(_lib.MR_ING_TE_PTR, np.int64),
                       get(_lib.MR_ING_TE_COL, np.int32), get(_lib.MR_ING_LAB_PTR, np.int64), get(_lib.MR_ING_LAB_COL, np.int32),
                       get(_lib.MR_ING_DEG_TRAIN, np.int32), get(_lib.MR_ING_DEG_TEST, np.int32), get(_lib.MR_ING_DEG_SONG, np.int32),
                       table(_lib.MR_ING_TRAIN_USER_CHARS, _lib.MR_ING_TRAIN_USER_OFF), table(_lib.MR_ING_TEST_USER_CHARS, _lib.MR_ING_TEST_USER_OFF),
                       table(_lib.MR_ING_SONG_CHARS, _lib.MR_ING_SONG_OFF),
                       {"source": "tsv-native", "label_only_songs": n_extra, "timing_ms": dict(zip(
                           ["h2d", "lines_parse", "unique_users", "unique_songs", "host_sort", "csr", "unused", "total"], get(_lib.MR_ING_TIMING_MS, np.float64).tolist()))})
    finally:
        lib.mr_ingest_free(g)


class MusicRecommender:
    """`new MusicRecommender(trainFile, testFile, testLabelsFile)` (MR:12).  Also accepts a ready `Dataset`."""

    def __init__(self, trainFile, testFile=None, testLabelsFile=None, device: int = 0, engine: int = _lib.MR_ENGINE_AUTO,
                 profile: bool = False, space: int = _lib.MR_SPACE_AUTO, ingest: str = "host", head_min_deg: int = 0,
                 item_batch: int = 0, song_window=None):
        """song_window = (lo, hi): score only the songs [lo, hi) of every test user — one song partition of distributed.scala:459-461
        (MR_OPT_SONG_WINDOW_*): dense models become [U, hi - lo], getTopK ranks inside the window (global song ids)."""
        if isinstance(trainFile, Dataset):
            ds = trainFile
        elif ingest == "native":
            ds = dataset_from_streams_native(trainFile, testFile, testLabelsFile, device=device)
        else:
            def op(f):
                return open(f, "r", encoding="utf-8") if isinstance(f, (str, bytes)) or hasattr(f, "__fspath__") else f
            ds = dataset_from_streams(op(trainFile), op(testFile), op(testLabelsFile))
        self.ds = ds
        self._lib = _lib.load()
        self._h = C.c_void_p()
        dev = (C.c_int * 1)(device)
        rc = self._lib.mr_create(C.byref(self._h), dev, 1, engine | space | (_lib.MR_PROFILE if profile else 0))
        self._check(rc)
        if head_min_deg:
            self._check(self._lib.mr_set_option(self._h, _lib.MR_OPT_HEAD_MIN_DEG, int(head_min_deg)))
        if item_batch:
            self._check(self._lib.mr_set_option(self._h, _lib.MR_OPT_ITEM_BATCH, int(item_batch)))
        self.song_window = (0, ds.S) if song_window is None else (int(song_window[0]), int(song_window[1]))
        self._whole_test_set = True      # the test users are the whole test set (not a shard of it): evaluateOnDevice is the model's mAP
        if song_window is not None:
            self._check(self._lib.mr_set_option(self._h, _lib.MR_OPT_SONG_WINDOW_LO, self.song_window[0]))
            self._check(self._lib.mr_set_option(self._h, _lib.MR_OPT_SONG_WINDOW_HI, self.song_window[1]))
        a = self._arrs = dict(
            tr_ptr=np.ascontiguousarray(ds.tr_ptr, np.int64), tr_col=np.ascontiguousarray(ds.tr_col, np.int32),
            te_ptr=np.ascontiguousarray(ds.te_ptr, np.int64), te_col=np.ascontiguousarray(ds.te_col, np.int32),
            deg_tr=np.ascontiguousarray(ds.deg_tr, np.int32), deg_te=np.ascontiguousarray(ds.deg_te, np.int32),
            deg_song=np.ascontiguousarray(ds.deg_song, np.int32))
        rc = self._lib.mr_load(self._h, ds.T, ds.U, ds.S, _p(a["tr_ptr"]), _p(a["tr_col"]), _p(a["te_ptr"]), _p(a["te_col"]),
                               _p(a["deg_tr"]), _p(a["deg_te"]), _p(a["deg_song"]))
        self._check(rc)

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc: int):
        if rc == _lib.MR_OK:
            return
        msg = self._lib.mr_last_error(self._h).decode(errors="replace") if self._h else "mr_create failed"
        if rc == _lib.MR_ERR_PARAM_RANGE:
            sys.stderr.write(msg + "\n\n")            # System.err.println("... must be between 0 and 1\n"), MR:367, 435
            raise ParameterRange(msg)
        if rc == _lib.MR_ERR_KEY_MISMATCH:
            raise KeyMismatch(msg)
        raise _lib.MrError(rc, msg)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.mr_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_test_users(self, ds_shard: Dataset, pair_index_base: int = 0, n_pairs_total: int = 0):
        """Score another shard of test users against the resident train replica (DIST:450-452 partitioning)."""
        a = self._arrs
        a["te_ptr"] = np.ascontiguousarray(ds_shard.te_ptr, np.int64)
        a["te_col"] = np.ascontiguousarray(ds_shard.te_col, np.int32)
        a["deg_te"] = np.ascontiguousarray(ds_shard.deg_te, np.int32)
        self._check(self._lib.mr_set_test_users(self._h, ds_shard.U, _p(a["te_ptr"]), _p(a["te_col"]), _p(a["deg_te"]),
                                                pair_index_base, n_pairs_total))
        self.ds = ds_shard
        self._whole_test_set = pair_index_base == 0 and n_pairs_total == 0   # the ABI's "this shard is the whole test set"

    def _model(self, kind: int, name: str) -> Model:
        lo, hi = self.song_window
        out = np.empty((self.ds.U, hi - lo), np.float64)
        self._check(self._lib.mr_score_dense(self._h, kind, _p(out)))
        songs = self.ds.songs if (lo, hi) == (0, self.ds.S) or self.ds.songs is None else self.ds.songs[lo:hi]
        return Model(out, self.ds.test_users, songs, name)

    # ------------------------------------------------------------------ reference method surface
    def getUserBasedModel(self) -> Model:                    # MR:132
        return self._model(_lib.MR_UBM, "userBasedModel")

    getUserBasedModelP = getUserBasedModel                   # MR:177 (.par twin: same values)

    def getItemBasedModel(self) -> Model:                    # MR:222
        return self._model(_lib.MR_IBM, "itemBasedModel")

    getItemBasedModelP = getItemBasedModel                   # MR:268

    def _blend(self, kind: int, ubm: Model, ibm: Model, param: float, seed: int, name: str) -> Model:
        mu, mi = ~np.isnan(ubm.scores), ~np.isnan(ibm.scores)
        cu, ci = ubm.scores[mu], ibm.scores[mi]
        n = min(len(cu), len(ci))                            # zip truncates (MR:322)
        ku, ki = np.flatnonzero(mu.ravel())[:n], np.flatnonzero(mi.ravel())[:n]
        # parameter range first (MR:366-369 precedes the zip), then the per-element key check (MR:326)
        out = np.empty(n, np.float64)
        rc = self._lib.mr_blend_dense(self._h, kind, float(param), C.c_uint64(seed & (2**64 - 1)), _p(cu), _p(ci), _p(out), n, 0,
                                      len(cu))
        self._check(rc)
        if not np.array_equal(ku, ki):
            raise KeyMismatch("(user, song) keys of ubm and ibm differ")
        res = np.full(ubm.scores.shape, np.nan)
        res.ravel()[ku] = out
        return Model(res, ubm.test_users, ubm.songs, name)

    def getLinearCombinationModel(self, ubm: Model, ibm: Model, alpha: float) -> Model:                    # MR:317
        return self._blend(_lib.MR_LC, ubm, ibm, alpha, 0, "linearCombinationModel")

    getLinearCombinationModelP = getLinearCombinationModel                                                  # MR:340

    def getAggregationModel(self, ubm: Model, ibm: Model, itemBasedPercentage: float = 0.5) -> Model:      # MR:361
        return self._blend(_lib.MR_AGG, ubm, ibm, itemBasedPercentage, 0, "aggregationModel")

    getAggregationModelP = getAggregationModel                                                              # MR:396

    def getStochasticCombinationModel(self, ubm: Model, ibm: Model, itemBasedProbability: float = 0.5,
                                      seed: int = 0) -> Model:                                              # MR:429
        return self._blend(_lib.MR_STOCH, ubm, ibm, itemBasedProbability, seed, "stochasticCombinationModel")

    getStochasticCombinationModelP = getStochasticCombinationModel                                          # MR:461

    def getTopK(self, model: int = _lib.MR_UBM, k: int = 500, param: float = 0.5, seed: int = 0):
        """Per test user the k best unlistened songs (score desc, song id asc): (song [U,k] int32, score [U,k] f64, len [U])."""
        U = self.ds.U
        song = np.empty((U, k), np.int32)
        score = np.empty((U, k), np.float64)
        ln = np.empty(U, np.int32)
        self._check(self._lib.mr_topk(self._h, model, float(param), C.c_uint64(seed & (2**64 - 1)), k, _p(song), _p(score), _p(ln)))
        return song, score, ln

    def getSimilarSongs(self, songs=None, k: int = 100):
        """Songs like each of `songs` (default: all S songs): the k co-listened songs of highest item-item cosine (MR:230-239), score
        descending then song id ascending (mr_similar_songs, DESIGN.md §4.7).  Returns (song [n, k] int32, score [n, k] float64,
        len [n] int32); row r belongs to songs[r], song -1 / score 0.0 past len[r]."""
        ids = np.arange(self.ds.S, dtype=np.int32) if songs is None else np.ascontiguousarray(songs, np.int32).reshape(-1)
        n = len(ids)
        song = np.empty((n, k), np.int32)
        score = np.empty((n, k), np.float64)
        ln = np.empty(n, np.int32)
        self._check(self._lib.mr_similar_songs(self._h, _p(ids), n, k, _p(song), _p(score), _p(ln)))
        return song, score, ln

    def getSimilarUsers(self, users=None, k: int = 100):
        """Listeners like each of `users` (indices into the current test shard, default: all of them): the k train users of highest
        user-user cosine (MR:140-149), score descending then train-user id ascending (mr_similar_users, DESIGN.md §4.8).  Returns
        (user [n, k] int32, score [n, k] float64, len [n] int32); row r belongs to users[r], user -1 / score 0.0 past len[r]."""
        ids = np.arange(self.ds.U, dtype=np.int32) if users is None else np.ascontiguousarray(users, np.int32).reshape(-1)
        n = len(ids)
        user = np.empty((n, k), np.int32)
        score = np.empty((n, k), np.float64)
        ln = np.empty(n, np.int32)
        self._check(self._lib.mr_similar_users(self._h, _p(ids), n, k, _p(user), _p(score), _p(ln)))
        return user, score, ln

    def explain(self, model: int, users, songs, m: int = 10) -> Explanation:
        """Why song songs[r] scores what it does for test user users[r] (indices into the current test shard): the contributors of the
        UBM score (train listeners of the song who share songs with the user) or of the IBM score (the user's visible songs co-listened
        with it), each with its cosine weight and its exact fixed-point term, the m largest weights listed (mr_explain, DESIGN.md §4.9)."""
        u = np.ascontiguousarray(users, np.int32).reshape(-1)
        s = np.ascontiguousarray(songs, np.int32).reshape(-1)
        if len(u) != len(s):
            raise ValueError(f"{len(u)} users but {len(s)} songs")
        n = len(u)
        out = Explanation(np.empty((n, m), np.int32), np.empty((n, m), np.float64), np.empty((n, m), np.int64), np.empty(n, np.int32),
                          np.empty(n, np.int32), np.empty(n, np.int64), np.empty(n, np.float64))
        self._check(self._lib.mr_explain(self._h, model, _p(u), _p(s), n, m, *[_p(a) for a in out]))
        return out

    def getSongAudience(self, model: int = _lib.MR_UBM, songs=None, k: int = 100, param: float = 0.5, seed: int = 0):
        """Who scores each of `songs` highest (default: every song of the handle's window, ascending): the k test users of the current
        shard with the best score of (user, song) under model / param / seed as in getTopK, score descending then user index ascending
        (mr_song_audience, DESIGN.md §4.10).  Returns (user [n, k] int32, score [n, k] float64, len [n] int32); row r belongs to
        songs[r], user -1 / score 0.0 past len[r]."""
        lo, hi = self.song_window
        ids = np.arange(lo, hi, dtype=np.int32) if songs is None else np.ascontiguousarray(songs, np.int32).reshape(-1)
        n = len(ids)
        kk = max(int(k), 0)                 # a k outside 1..1024 is refused by the library (MR_ERR_BAD_ARG), not by numpy
        user = np.empty((n, kk), np.int32)
        score = np.empty((n, kk), np.float64)
        ln = np.empty(n, np.int32)
        self._check(self._lib.mr_song_audience(self._h, model, float(param), C.c_uint64(seed & (2**64 - 1)), _p(ids), n, k, _p(user),
                                               _p(score), _p(ln)))
        return user, score, ln

    def getTopKMulti(self, specs, k: int = 500):
        """getTopK for every entry of a model set (model, param, seed) from one scoring of the shard (mr_topk_multi, DESIGN.md §4.6):
        one (song [U,k] int32, score [U,k] f64, len [U]) per entry, each equal to getTopK(model, k, param, seed)."""
        models, params, seeds = model_set_arrays(specs)
        U, n = self.ds.U, len(models)
        out = [(np.empty((U, k), np.int32), np.empty((U, k), np.float64), np.empty(U, np.int32)) for _ in range(n)]
        tab = lambda j: (C.c_void_p * n)(*[o[j].ctypes.data for o in out])      # noqa: E731
        self._check(self._lib.mr_topk_multi(self._h, n, _p(models), _p(params), _p(seeds), k, tab(0), tab(1), tab(2)))
        return out

    def topk_multi_device(self, specs, k: int = 500):
        """mr_topk_multi_device: the set's lists stay in HBM (topk_multi_device_tensors reads them)."""
        models, params, seeds = model_set_arrays(specs)
        self._check(self._lib.mr_topk_multi_device(self._h, len(models), _p(models), _p(params), _p(seeds), k))

    def setTopKFilter(self, allowed=None, exclude=None):
        """The filter of getTopKFiltered for the current shard (mr_set_topk_filter, DESIGN.md §4.11): `allowed` global song ids (any order,
        duplicates ignored; None = every song), `exclude` a CSR (rowptr [U + 1], col) of songs not to recommend per test user of the shard,
        ids ascending within a row (exclusions_from_topk turns a previous page into one).  set_test_users drops the filter."""
        a = None if allowed is None else np.ascontiguousarray(allowed, np.int32).reshape(-1)
        ep = ec = None
        if exclude is not None:
            ep = np.ascontiguousarray(exclude[0], np.int64).reshape(-1)
            ec = np.ascontiguousarray(exclude[1], np.int32).reshape(-1)
            if len(ep) != self.ds.U + 1:
                raise ValueError(f"exclusion rowptr has {len(ep)} entries, the shard has {self.ds.U} test users")
        self._check(self._lib.mr_set_topk_filter(self._h, None if a is None else _p(a), -1 if a is None else len(a),
                                                 None if ep is None else _p(ep), None if ec is None else _p(ec)))

    def clearTopKFilter(self):
        self._check(self._lib.mr_set_topk_filter(self._h, None, -1, None, None))

    def getTopKMultiFiltered(self, specs, k: int = 500):
        """getTopKMulti under the filter of setTopKFilter (mr_topk_filtered): per entry each user's ranking without the songs the filter
        removes, truncated to k, one (song [U,k] int32, score [U,k] f64, len [U]) per entry."""
        models, params, seeds = model_set_arrays(specs)
        U, n = self.ds.U, len(models)
        kk = max(int(k), 0)                 # a k outside 1..1024 is refused by the library (MR_ERR_BAD_ARG), not by numpy
        out = [(np.empty((U, kk), np.int32), np.empty((U, kk), np.float64), np.empty(U, np.int32)) for _ in range(n)]
        tab = lambda j: (C.c_void_p * n)(*[o[j].ctypes.data for o in out])      # noqa: E731
        self._check(self._lib.mr_topk_filtered(self._h, n, _p(models), _p(params), _p(seeds), k, tab(0), tab(1), tab(2)))
        return out

    def getTopKFiltered(self, model: int = _lib.MR_UBM, k: int = 500, param: float = 0.5, seed: int = 0):
        """getTopK under the filter of setTopKFilter: (song [U,k] int32, score [U,k] f64, len [U])."""
        return self.getTopKMultiFiltered([(model, param, seed)], k)[0]

    def topk_filtered_device(self, specs, k: int = 500):
        """mr_topk_filtered_device: the filtered lists stay in HBM as the last set result (topk_multi_device_tensors reads them)."""
        models, params, seeds = model_set_arrays(specs)
        self._check(self._lib.mr_topk_filtered_device(self._h, len(models), _p(models), _p(params), _p(seeds), k))

    def topk_multi_device_tensors(self, i: int, k: int):
        """torch views (no copy) of entry i of the last set top-k on the device: (song int32 [U,k], score f64 [U,k], len int32 [U])."""
        ps, pv, pl = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(self._lib.mr_topk_multi_ptrs(self._h, i, k, C.byref(ps), C.byref(pv), C.byref(pl)))
        U = self.ds.U
        return _cuda_view(ps.value, (U, k), "<i4"), _cuda_view(pv.value, (U, k), "<f8"), _cuda_view(pl.value, (U,), "<i4")

    def prepare(self):
        """Build the item-space head rows now (one-off per train set) instead of lazily."""
        self._check(self._lib.mr_prepare(self._h))

    def prepare_async(self):
        """Start the head-row build on its own stream and return; the next scoring call completes it (overlaps set_test_users)."""
        self._check(self._lib.mr_prepare_async(self._h))

    def invalidate_prepared(self):
        """Forget the head rows so that the next prepare() / scoring call rebuilds them (bench.py: the whole model build inside a step)."""
        self._check(self._lib.mr_invalidate_prepared(self._h))

    def getRanks1(self, model: int, users) -> np.ndarray:
        """DIST UserBasedModel/ItemBasedModel.getRanks1(user) (DIST:198-205, 269-276) for the listed test users of the current shard:
        [len(users), S] fp64, NaN at listened pairs."""
        ids = np.ascontiguousarray(users, np.int32)
        out = np.empty((len(ids), self.song_window[1] - self.song_window[0]), np.float64)
        self._check(self._lib.mr_score_users(self._h, model, _p(ids), len(ids), _p(out)))
        return out

    def getRanks2(self, model: int, songs) -> np.ndarray:
        """DIST getRanks2(song) (DIST:214-221, 285-292) for the listed songs: [len(songs), U] fp64, NaN where the user listened."""
        ids = np.ascontiguousarray(songs, np.int32)
        out = np.empty((len(ids), self.ds.U), np.float64)
        self._check(self._lib.mr_score_songs(self._h, model, _p(ids), len(ids), _p(out)))
        return out

    def mapAtK(self, k: int = 500, top=None, per_user: bool = False, labels: Dataset | None = None):
        """mAP@k (north_star's mAP@500; MSD-challenge definition, include/mrscore.h) of ranked lists against this data set's label rows.
        top = (song [U,k], len [U]) as getTopK returns them, or None for the device-resident result of the last getTopK / mr_topk_device."""
        lab = labels if labels is not None else self.ds      # labels: the data set whose label rows match explicit lists of other users
        lp = np.ascontiguousarray(lab.lab_ptr, np.int64)
        lc = np.ascontiguousarray(lab.lab_col, np.int32)
        out = C.c_double(0.0)
        ap = np.zeros(lab.U, np.float64)
        if top is None:
            self._check(self._lib.mr_map_at_k(self._h, k, None, None, self.ds.U, _p(lp), _p(lc), C.byref(out), _p(ap)))
        else:
            song = np.ascontiguousarray(top[0], np.int32)
            ln = np.ascontiguousarray(top[1], np.int32)
            self._check(self._lib.mr_map_at_k(self._h, song.shape[1], _p(song), _p(ln), song.shape[0], _p(lp), _p(lc), C.byref(out), _p(ap)))
        return (float(out.value), ap) if per_user else float(out.value)

    def topk_device_tensors(self, k: int):
        """torch views (no copy) of the last mr_topk_device result in this GPU's HBM: (song int32 [U,k], score f64 [U,k], len int32 [U])."""
        ps, pv, pl = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(self._lib.mr_topk_device_ptrs(self._h, k, C.byref(ps), C.byref(pv), C.byref(pl)))
        U = self.ds.U
        return _cuda_view(ps.value, (U, k), "<i4"), _cuda_view(pv.value, (U, k), "<f8"), _cuda_view(pl.value, (U,), "<i4")

    def mergeTopK(self, parts_song, parts_score, parts_len, out_song, out_score, out_len):
        """Join the ranked lists of several song partitions for the same users (mr_topk_merge; the `.collect` + ranking of
        distributed.scala:459-461).  All arguments are CUDA torch tensors: parts_* [P, n, k] / [P, n], out_* [n, k] / [n]; the join runs
        on the library stream."""
        P, n, k = parts_song.shape
        tab = lambda t: (C.c_void_p * P)(*[t[i].data_ptr() for i in range(P)])      # noqa: E731
        self._check(self._lib.mr_topk_merge(self._h, k, P, n, tab(parts_song), tab(parts_score), tab(parts_len), C.c_void_p(out_song.data_ptr()),
                                            C.c_void_p(out_score.data_ptr()), C.c_void_p(out_len.data_ptr())))

    def topk_packed_tensor(self, k: int):
        """The last top-k result as ONE uint8 torch view of device memory plus the byte offsets of its parts:
        (block, score_offset, len_offset); song int32 [U,k] starts at 0."""
        base, nbytes, so, lo = C.c_void_p(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self._lib.mr_topk_packed(self._h, k, C.byref(base), C.byref(nbytes), C.byref(so), C.byref(lo)))
        return _cuda_view(base.value, (int(nbytes.value),), "|u1"), int(so.value), int(lo.value)

    # ------------------------------------------------------------------ parity probes / similarity products
    def counts_ubm(self) -> np.ndarray:
        out = np.empty((self.ds.U, self.ds.T), np.int32)
        self._check(self._lib.mr_counts_ubm(self._h, _p(out)))
        return out

    def counts_ibm(self, s0: int, s1: int) -> np.ndarray:
        out = np.empty((s1 - s0, self.ds.S), np.int32)
        self._check(self._lib.mr_counts_ibm(self._h, s0, s1, _p(out)))
        return out

    def gram_rows_device(self, s0: int, s1: int):
        """Rows [s0,s1) of this handle's (partial) train co-occurrence matrix as a torch int32 view [s1-s0, ld] of device memory."""
        ptr, ld = C.c_void_p(), C.c_int64()
        self._check(self._lib.mr_gram_rows_device(self._h, s0, s1, C.byref(ptr), C.byref(ld)))
        return _cuda_view(ptr.value, (s1 - s0, ld.value), "<i4")

    # ---- fused K-split reduce-scatter (GEMM epilogue stores into the owners' receive slots, local or NVLink peer memory)
    def peer_alloc(self, nbytes: int):
        """(device pointer, 64-byte CUDA IPC handle) of a zeroed buffer other ranks can map with peer_open."""
        ptr = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        self._check(self._lib.mr_peer_alloc(self._h, nbytes, C.byref(ptr), handle))
        return int(ptr.value), bytes(handle)

    def peer_open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        buf = (C.c_ubyte * 64).from_buffer_copy(handle)
        self._check(self._lib.mr_peer_open(self._h, buf, C.byref(ptr)))
        return int(ptr.value)

    def peer_close(self, ptr: int):
        self._check(self._lib.mr_peer_close(self._h, C.c_void_p(ptr)))

    def gram_rows_scatter(self, s0: int, s1: int, slot_ptrs, rows_per_owner: int, ld: int, sync: bool = True):
        arr = (C.c_void_p * len(slot_ptrs))(*slot_ptrs)
        fn = self._lib.mr_gram_rows_scatter if sync else self._lib.mr_gram_rows_scatter_async
        self._check(fn(self._h, s0, s1, arr, len(slot_ptrs), rows_per_owner, ld))

    def peer_signal(self, flag_ptrs, value: int):
        arr = (C.c_void_p * len(flag_ptrs))(*flag_ptrs)
        self._check(self._lib.mr_peer_signal(self._h, arr, len(flag_ptrs), value))

    def peer_wait(self, flags_ptr: int, n: int, value: int):
        self._check(self._lib.mr_peer_wait(self._h, C.c_void_p(flags_ptr), n, value))

    def sync(self):
        self._check(self._lib.mr_sync(self._h))

    def similarity_ubm(self) -> np.ndarray:
        out = np.empty((self.ds.U, self.ds.T), np.float32)
        self._check(self._lib.mr_similarity_ubm(self._h, _p(out)))
        return out

    def similarity_ibm(self, s0: int, s1: int) -> np.ndarray:
        out = np.empty((s1 - s0, self.ds.S), np.float32)
        self._check(self._lib.mr_similarity_ibm(self._h, s0, s1, _p(out)))
        return out

    def timing(self, reset: bool = False) -> dict:
        t = (C.c_double * 9)()
        self._lib.mr_get_timing(self._h, t, 9)
        if reset:
            self._lib.mr_reset_timing(self._h)
        return dict(zip(_lib.TIMING_NAMES, list(t)))

    def info(self) -> dict:
        v = (C.c_int64 * 34)()
        self._lib.mr_get_info(self._h, v, 34)
        return dict(zip(["engine", "launches", "dense_bytes", "n_items", "num_sms", "device_bytes", "space", "n_head", "head_entries",
                         "tail_entries", "head_exceptions", "batch_rows", "head_groups", "split_users", "n_cols", "win_lo", "topk_fast_rejects",
                         "topk_short_rows", "topk_degenerate_rows", "scoring_passes", "similar_short_rows", "similar_long_rows",
                         "similar_user_short_rows", "similar_user_long_rows", "explain_rows", "audience_rows",
                         "audience_radix_selects", "filter_full_rows", "filter_candidate_rows", "carry_events", "head_staged_rows",
                         "head_packed", "head_planes", "ubm_int_ok"], list(v)))

    # ------------------------------------------------------------------ model file I/O (MR:489-512)
    def writeModelOnFile(self, model: Model, outputFileName: str = "") -> int:
        """`user \\t song \\t Double.toString(score) \\n` per element, in model order (MR:492-494), through the native writer
        `mr_write_model` (csrc/modelio.cu).  Returns the number of lines written."""
        return write_model_file(model, outputFileName, self._lib)

    def importModelFromFile(self, pathToModel: str):
        """Array[(String, String, Double)] sorted by (user, song, score desc) (MR:505-512)."""
        return import_model_file(pathToModel)

    # ------------------------------------------------------------------ evaluation (MR:521-639), host-side like the reference
    def evaluateModel(self, model: Model, parallel: bool = False, n_thresholds: int = 10) -> float:
        """The reference's threshold-sweep mAP (MR:521-639; 10 thresholds MR:590, 11 in distributed.scala:395) on the GPU
        (`mr_evaluate_dense`).  `evaluate_map` below is the same computation in numpy for hosts without a GPU handle."""
        sc = np.ascontiguousarray(model.scores, np.float64)
        lp = np.ascontiguousarray(self.ds.lab_ptr, np.int64)
        lc = np.ascontiguousarray(self.ds.lab_col, np.int32)
        out = C.c_double(0.0)
        self._check(self._lib.mr_evaluate_dense(self._h, _p(sc), sc.shape[0], sc.shape[1], _p(lp), _p(lc), n_thresholds, C.byref(out)))
        return float(out.value)

    # ---- the same metric streamed over the scoring batches: no materialised model (include/mrscore.h mr_eval_*, DESIGN.md §4.5)
    def eval_range(self, model: int = _lib.MR_UBM, param: float = 0.5, seed: int = 0) -> tuple[float, float]:
        """(min, max) of the scores this handle's shard and song window emit (MR:524-529); (inf, -inf) when it emits none."""
        mn, mx = C.c_double(), C.c_double()
        self._check(self._lib.mr_eval_range(self._h, model, float(param), C.c_uint64(seed & (2**64 - 1)), C.byref(mn), C.byref(mx)))
        return float(mn.value), float(mx.value)

    def _label_csr(self, labels: Dataset | None):
        """The label CSR (row offsets int64, songs int32) of labels (default: the handle's data set) for the count pass, whose rows must be
        the current shard's users."""
        lab = labels if labels is not None else self.ds
        lp = np.ascontiguousarray(lab.lab_ptr, np.int64)
        lc = np.ascontiguousarray(lab.lab_col, np.int32)
        if len(lp) != self.ds.U + 1 or len(lc) < (lp[-1] if len(lp) else 0):   # mr_eval_counts reads U + 1 row offsets
            raise ValueError(f"labels must hold {self.ds.U} label rows (the current shard's users), got {len(lp) - 1}")
        return lp, lc

    def _require_whole_model(self, caller: str, combine: str):
        """caller evaluates the whole model: no song window, and test users that are the whole test set; a partitioned job combines
        its handles' parts with distributed.<combine> instead."""
        if self.song_window != (0, self.ds.S):
            raise ValueError(f"{caller} needs the whole model: this handle scores a song window (use distributed.{combine})")
        if not self._whole_test_set:
            raise ValueError(f"{caller} needs the whole model: this handle holds a shard of the test users (set_test_users with a "
                             f"pair index base / total); use distributed.{combine}")

    def eval_counts(self, model: int, mn: float, mx: float, new_songs, param: float = 0.5, seed: int = 0, n_thresholds: int = 10,
                    labels: Dataset | None = None):
        """Confusion counts of this handle's part of the model under the global (mn, mx): (pred [n_new, n_thr], tp [n_new, n_thr],
        nlab [n_new]) int64, row c for new_songs[c] (all test users' distinct label songs, ascending).  labels: the data set whose
        label rows belong to the current shard's users (default: the handle's)."""
        lp, lc = self._label_csr(labels)
        ns = np.ascontiguousarray(new_songs, np.int32)
        pred = np.zeros((len(ns), n_thresholds), np.int64)
        tp = np.zeros((len(ns), n_thresholds), np.int64)
        nlab = np.zeros(len(ns), np.int64)
        self._check(self._lib.mr_eval_counts(self._h, model, float(param), C.c_uint64(seed & (2**64 - 1)), float(mn), float(mx), n_thresholds,
                                             _p(lp), _p(lc), _p(ns), len(ns), _p(pred), _p(tp), _p(nlab)))
        return pred, tp, nlab

    def evaluateOnDevice(self, model: int = _lib.MR_UBM, param: float = 0.5, seed: int = 0, n_thresholds: int = 10,
                         labels: Dataset | None = None) -> float:
        """evaluateModel (MR:521-639) of the model this handle scores, without materialising it: range pass, count pass, finish.
        Same bits as evaluateModel(getXxxModel()) on shapes where that fits.  The handle must hold the whole model: no song window, and
        test users that are the whole test set (ValueError otherwise); a partitioned job combines its handles' parts with
        distributed.evaluate_reference_map."""
        self._require_whole_model("evaluateOnDevice", "evaluate_reference_map")
        lab = labels if labels is not None else self.ds
        mn, mx = self.eval_range(model, param, seed)
        new_songs = np.unique(np.asarray(lab.lab_col, np.int32))
        pred, tp, nlab = self.eval_counts(model, mn, mx, new_songs, param, seed, n_thresholds, lab)
        return eval_finish(pred, tp, nlab, n_thresholds)

    # ---- a model set from one scoring per batch (include/mrscore.h mr_eval_*_multi, DESIGN.md §4.6)
    def eval_range_multi(self, specs) -> tuple[np.ndarray, np.ndarray]:
        """(min [M], max [M]) of each entry of the model set, as eval_range per entry, from one scoring of the shard."""
        models, params, seeds = model_set_arrays(specs)
        mn, mx = np.empty(len(models), np.float64), np.empty(len(models), np.float64)
        self._check(self._lib.mr_eval_range_multi(self._h, len(models), _p(models), _p(params), _p(seeds), _p(mn), _p(mx)))
        return mn, mx

    def eval_counts_multi(self, specs, mn, mx, new_songs, n_thresholds: int = 10, labels: Dataset | None = None):
        """eval_counts for every entry of the model set under its global (mn[i], mx[i]): (pred [M, n_new, n_thr], tp [M, n_new, n_thr],
        nlab [n_new]) int64."""
        models, params, seeds = model_set_arrays(specs)
        n = len(models)
        mn = np.ascontiguousarray(mn, np.float64)
        mx = np.ascontiguousarray(mx, np.float64)
        if mn.shape != (n,) or mx.shape != (n,):
            raise ValueError(f"mn and mx must hold one value per entry of the set ({n})")
        lp, lc = self._label_csr(labels)
        ns = np.ascontiguousarray(new_songs, np.int32)
        pred = np.zeros((n, len(ns), n_thresholds), np.int64)
        tp = np.zeros((n, len(ns), n_thresholds), np.int64)
        nlab = np.zeros(len(ns), np.int64)
        self._check(self._lib.mr_eval_counts_multi(self._h, n, _p(models), _p(params), _p(seeds), _p(mn), _p(mx), n_thresholds, _p(lp), _p(lc),
                                                   _p(ns), len(ns), _p(pred), _p(tp), _p(nlab)))
        return pred, tp, nlab

    def evaluateAllOnDevice(self, specs, n_thresholds: int = 10, labels: Dataset | None = None) -> list[float]:
        """evaluateOnDevice for every entry of a model set, from two scorings of the shard (one on a single-batch item-space shard): one
        mAP per entry, each with the bits of evaluateOnDevice(model, param, seed).  The same whole-model guards as evaluateOnDevice."""
        self._require_whole_model("evaluateAllOnDevice", "evaluate_reference_map_multi")
        lab = labels if labels is not None else self.ds
        mn, mx = self.eval_range_multi(specs)
        new_songs = np.unique(np.asarray(lab.lab_col, np.int32))
        pred, tp, nlab = self.eval_counts_multi(specs, mn, mx, new_songs, n_thresholds, lab)
        return [eval_finish(pred[i], tp[i], nlab, n_thresholds) for i in range(len(pred))]


MAX_MODEL_SET = 16


def model_set_arrays(specs):
    """A model set [(model, param, seed), ...] of 1..16 entries as the parallel arrays of the C-ABI (int32, float64, uint64).  The shape
    is checked here; parameter ranges are checked by the library, which names the first bad entry."""
    specs = list(specs)
    if not 1 <= len(specs) <= MAX_MODEL_SET:
        raise ValueError(f"a model set holds 1..{MAX_MODEL_SET} entries, got {len(specs)}")
    for i, e in enumerate(specs):
        if len(e) != 3:
            raise ValueError(f"entry {i}: expected (model, param, seed), got {e!r}")
        if int(e[0]) != e[0] or not 0 <= int(e[0]) <= _lib.MR_STOCH:
            raise ValueError(f"entry {i}: unknown model selector {e[0]!r}")
    models = np.array([int(e[0]) for e in specs], np.int32)
    params = np.array([float(e[1]) for e in specs], np.float64)
    seeds = np.array([int(e[2]) & (2**64 - 1) for e in specs], np.uint64)
    return models, params, seeds


def _string_table(names, n):
    """id -> string list as (uint8 chars, int64 offsets [n+1]); ints stand in for missing tables."""
    enc = [(str(i) if names is None else names[i]).encode("utf-8") for i in range(n)]
    off = np.zeros(n + 1, np.int64)
    np.cumsum([len(b) for b in enc], out=off[1:])
    chars = np.frombuffer(b"".join(enc) or b"\0", np.uint8)
    return np.ascontiguousarray(chars), off


def write_model_file(model: Model, path: str, lib=None) -> int:
    """writeModelOnFile (MR:489-496) natively: one `user\\tsong\\tDouble.toString(score)\\n` line per emitted pair."""
    lib = lib or _lib.load()
    sc = np.ascontiguousarray(model.scores, np.float64)
    U, S = sc.shape
    uc, uo = _string_table(model.test_users, U)
    scs, so = _string_table(model.songs, S)
    rows = C.c_int64(0)
    rc = lib.mr_write_model(str(path).encode(), _p(sc), U, S, _p(uc), _p(uo), _p(scs), _p(so), 0, C.byref(rows))
    if rc != _lib.MR_OK:
        raise OSError(f"mr_write_model({path!r}) failed with code {rc}")
    return int(rows.value)


def write_model_file_py(model: Model, path: str) -> None:
    """The same file from pure Python (javafmt.double_to_string): the independent check of the native formatter in tests."""
    with open(path, "w", encoding="utf-8", newline="") as out:
        buf = io.StringIO()
        for user, (song, score) in model.tuples():
            buf.write(f"{user}\t{song}\t{double_to_string(score)}\n")
        out.write(buf.getvalue())


def import_model_file(path: str):
    """importModelFromFile (MR:505-512): Array[(String, String, Double)] sorted by (user, song, score desc)."""
    rows = []
    with open(path, "r", encoding="utf-8") as f:
        for line in f:
            parts = line.rstrip("\n").split("\t")
            if len(parts) != 3:
                raise ValueError(f"scala.MatchError: {line!r}")
            rows.append((parts[0], parts[1], float(parts[2])))
    rows.sort(key=lambda r: (r[0], r[1], -r[2]))
    return rows


def eval_finish(pred, tp, nlab, n_thresholds: int = 10, per_song: bool = False):
    """mr_eval_finish (host code, no GPU): the mAP of summed confusion counts, bit for bit as mr_evaluate_dense; per_song=True also
    returns the per-label-song AP."""
    pred = np.ascontiguousarray(pred, np.int64)
    tp = np.ascontiguousarray(tp, np.int64)
    nlab = np.ascontiguousarray(nlab, np.int64)
    n_new = len(nlab)
    if pred.shape != (n_new, n_thresholds) or tp.shape != (n_new, n_thresholds):
        raise ValueError("pred / tp must be [n_new, n_thresholds]")
    ap = np.zeros(n_new, np.float64)
    out = C.c_double(0.0)
    rc = _lib.load().mr_eval_finish(_p(pred), _p(tp), _p(nlab), n_new, n_thresholds, _p(ap), C.byref(out))
    if rc != _lib.MR_OK:
        raise _lib.MrError(rc, "mr_eval_finish: bad counts or sizes")
    return (float(out.value), ap) if per_song else float(out.value)


def eval_cutoffs(mn: float, mx: float, n_thresholds: int = 10) -> np.ndarray:
    """mr_eval_cutoffs: per threshold the least score the count pass predicts (+inf: none)."""
    out = np.zeros(n_thresholds, np.float64)
    rc = _lib.load().mr_eval_cutoffs(float(mn), float(mx), n_thresholds, _p(out))
    if rc != _lib.MR_OK:
        raise _lib.MrError(rc, "mr_eval_cutoffs: n_thresholds must be 10 or 11")
    return out


def eval_counts_host(scores: np.ndarray, ds: Dataset, lo: int, mn: float, mx: float, n_thresholds: int, new_songs):
    """numpy mirror of mr_eval_counts over a dense block of a model: scores [U, W] are the songs [lo, lo + W) of ds's test users (NaN =
    not emitted), normalised with the given global (mn, mx) as MR:529 does; labels of ds outside those songs are not counted (the
    ownership rule).  Returns (pred, tp, nlab) like MusicRecommender.eval_counts."""
    scores = np.asarray(scores, np.float64)
    U, W = scores.shape
    new_songs = np.asarray(new_songs, np.int64)
    th = [0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0][:n_thresholds]
    pred = np.zeros((len(new_songs), n_thresholds), np.int64)
    tp = np.zeros((len(new_songs), n_thresholds), np.int64)
    nlab = np.zeros(len(new_songs), np.int64)
    idx = np.flatnonzero((new_songs >= lo) & (new_songs < lo + W))
    if len(idx) == 0:
        return pred, tp, nlab
    rows = np.repeat(np.arange(U), np.diff(ds.lab_ptr))
    cols = np.asarray(ds.lab_col, np.int64)
    keep = (cols >= lo) & (cols < lo + W)
    pos = np.searchsorted(new_songs[idx], cols[keep])
    lab = np.zeros((U, len(idx)), bool)
    lab[rows[keep], pos] = True
    with np.errstate(invalid="ignore", divide="ignore"):
        norm = (scores[:, new_songs[idx] - lo] - mn) / (mx - mn)
    for t, thr in enumerate(th):
        with np.errstate(invalid="ignore"):
            p = norm > thr                              # NaN compares false (not emitted, max == min)
        pred[idx, t] = p.sum(0)
        tp[idx, t] = (p & lab).sum(0)
    nlab[idx] = lab.sum(0)
    return pred, tp, nlab


def similar_songs_host(ds: Dataset, songs, k: int):
    """numpy mirror of mr_similar_songs: per query song i, the train histories of i's train listeners concatenated, their distinct songs
    s != i with counts g (np.unique), sim = g / (sqrt(d_i) * sqrt(d_s)) in that operation order (0 where the denominator is 0, as the
    reference's cosineSimilarity), ranked by score descending then song id ascending.  Returns (song [n, k], score [n, k], len [n])."""
    songs = np.asarray(songs, np.int64).reshape(-1)
    n = len(songs)
    out_song = np.full((n, k), -1, np.int32)
    out_score = np.zeros((n, k), np.float64)
    out_len = np.zeros(n, np.int32)
    tr_ptr = np.asarray(ds.tr_ptr, np.int64)
    tr_col = np.asarray(ds.tr_col, np.int64)
    owner = np.repeat(np.arange(ds.T), np.diff(tr_ptr))                    # train user of every train entry
    order = np.argsort(tr_col, kind="stable")                              # inverted index: listeners of a song, ascending
    csc_ptr = np.concatenate([[0], np.cumsum(np.bincount(tr_col, minlength=ds.S))])
    listeners = owner[order]
    deg = np.asarray(ds.deg_song, np.int64)
    for r, i in enumerate(songs):
        users = listeners[csc_ptr[i]:csc_ptr[i + 1]]
        if len(users) == 0:
            continue
        hist = np.concatenate([tr_col[tr_ptr[v]:tr_ptr[v + 1]] for v in users])
        s, g = np.unique(hist, return_counts=True)
        keep = s != i
        s, g = s[keep], g[keep]
        den = np.sqrt(np.float64(deg[i])) * np.sqrt(deg[s].astype(np.float64))
        with np.errstate(divide="ignore", invalid="ignore"):
            sim = np.where(den != 0, g.astype(np.float64) / den, 0.0)
        rank = np.lexsort((s, -sim))
        m = min(k, len(rank))
        out_song[r, :m] = s[rank[:m]]
        out_score[r, :m] = sim[rank[:m]]
        out_len[r] = m
    return out_song, out_score, out_len


def similar_users_host(ds: Dataset, users, k: int):
    """numpy mirror of mr_similar_users: per query test user u, the train listeners of u's visible songs concatenated, their distinct
    train users v with counts c (np.unique), w = c / (sqrt(deg_te[u]) * sqrt(deg_tr[v])) in that operation order (0 where the
    denominator is 0, as the reference's cosineSimilarity), ranked by score descending then train-user id ascending.
    Returns (user [n, k], score [n, k], len [n])."""
    users = np.asarray(users, np.int64).reshape(-1)
    n = len(users)
    out_user = np.full((n, k), -1, np.int32)
    out_score = np.zeros((n, k), np.float64)
    out_len = np.zeros(n, np.int32)
    tr_ptr = np.asarray(ds.tr_ptr, np.int64)
    tr_col = np.asarray(ds.tr_col, np.int64)
    te_ptr = np.asarray(ds.te_ptr, np.int64)
    te_col = np.asarray(ds.te_col, np.int64)
    owner = np.repeat(np.arange(ds.T), np.diff(tr_ptr))                    # train user of every train entry
    order = np.argsort(tr_col, kind="stable")                              # inverted index: listeners of a song, ascending
    csc_ptr = np.concatenate([[0], np.cumsum(np.bincount(tr_col, minlength=ds.S))])
    listeners = owner[order]
    deg_tr = np.asarray(ds.deg_tr, np.int64)
    deg_te = np.asarray(ds.deg_te, np.int64)
    for r, u in enumerate(users):
        songs = te_col[te_ptr[u]:te_ptr[u + 1]]
        if len(songs) == 0:
            continue
        hist = np.concatenate([listeners[csc_ptr[j]:csc_ptr[j + 1]] for j in songs])
        if len(hist) == 0:
            continue
        v, c = np.unique(hist, return_counts=True)
        den = np.sqrt(np.float64(deg_te[u])) * np.sqrt(deg_tr[v].astype(np.float64))
        with np.errstate(divide="ignore", invalid="ignore"):
            w = np.where(den != 0, c.astype(np.float64) / den, 0.0)
        rank = np.lexsort((v, -w))
        m = min(k, len(rank))
        out_user[r, :m] = v[rank[:m]]
        out_score[r, :m] = w[rank[:m]]
        out_len[r] = m
    return out_user, out_score, out_len


def song_audience_host(scores: np.ndarray, songs, k: int):
    """numpy mirror of mr_song_audience over a dense model [U, S] (NaN at listened pairs, as mr_score_dense and the oracle give it): per
    query song, its column's non-NaN entries ordered by (-score, user), the first k.  Returns (user [n, k] int32, score [n, k] f64,
    len [n] int32), user -1 / score 0.0 past len."""
    ids = np.asarray(songs, np.int64).reshape(-1)
    n = len(ids)
    cols = np.asarray(scores, np.float64)[:, ids]                      # [U, n]
    order = np.argsort(-cols, axis=0, kind="stable")[:k].T             # NaN sorts last; equal scores keep user order
    ln = np.minimum(k, (~np.isnan(cols)).sum(axis=0)).astype(np.int32)
    user = np.full((n, k), -1, np.int32)
    score = np.zeros((n, k), np.float64)
    for r in range(n):
        user[r, :ln[r]] = order[r, :ln[r]]
        score[r, :ln[r]] = cols[order[r, :ln[r]], r]
    return user, score, ln


def exclusions_from_topk(song, ln):
    """Exclusion rows (rowptr [U + 1] int64, col int32) holding each user's listed songs of a previous top-k (song [U, k], len [U]), for
    setTopKFilter: the next page is the top-k with this page excluded."""
    song = np.asarray(song)
    ln = np.asarray(ln, np.int64).reshape(-1)
    ptr = np.zeros(len(ln) + 1, np.int64)
    np.cumsum(ln, out=ptr[1:])
    keep = np.arange(song.shape[1])[None, :] < ln[:, None]
    rows = np.sort(np.where(keep, song, np.iinfo(np.int32).max), axis=1)   # each row's listed songs first, ascending
    return ptr, np.ascontiguousarray(rows[keep], np.int32)


def topk_filtered_host(scores: np.ndarray, allowed, ex_ptr, ex_col, k: int):
    """numpy mirror of mr_topk_filtered over a dense model [U, S] (NaN at listened pairs, as mr_score_dense and the oracle give it):
    per user the non-NaN entries of the allowed songs (None = all) outside the user's exclusion row (ex_ptr None = none), ordered by
    (-score, song), the first k.  Returns (song [U, k] int32, score [U, k] f64, len [U] int32), song -1 / score 0.0 past len."""
    sc = np.array(scores, np.float64)
    U, S = sc.shape
    if allowed is not None:
        keep = np.zeros(S, bool)
        keep[np.asarray(allowed, np.int64)] = True
        sc[:, ~keep] = np.nan
    if ex_ptr is not None:
        ex_ptr = np.asarray(ex_ptr, np.int64)
        rows = np.repeat(np.arange(U), np.diff(ex_ptr))
        sc[rows, np.asarray(ex_col, np.int64)[:ex_ptr[-1]]] = np.nan
    order = np.argsort(-sc, axis=1, kind="stable")[:, :k]             # NaN sorts last; equal scores keep song order
    ln = np.minimum(k, (~np.isnan(sc)).sum(axis=1)).astype(np.int32)
    song = np.full((U, k), -1, np.int32)
    score = np.zeros((U, k), np.float64)
    for u in range(U):
        song[u, :ln[u]] = order[u, :ln[u]]
        score[u, :ln[u]] = sc[u, order[u, :ln[u]]]
    return song, score, ln


def explain_host(ds: Dataset, model: int, users, songs, m: int) -> Explanation:
    """numpy mirror of mr_explain.  UBM: the train listeners v of s with c = |I_u ∩ I_v| > 0, term = c / (sqrt(deg_te[u]) * sqrt(deg_tr[v])),
    num = c * q_24(deg_tr[v]); IBM: u's visible songs j with g = |U_s^train ∩ U_j^train| > 0, term = g / (sqrt(d_s) * sqrt(d_j)),
    num = g * q_26(d_j), d = deg_song; each term in that operation order (0 where the denominator is 0), ranked by term descending then id
    ascending.  q_k(x) = rint(2^k / sqrt(x)) (0 for x = 0) as the oracle's mro_q; score = float(total) * 2^-k / sqrt(deg_te[u] or d_s)."""
    users = np.asarray(users, np.int64).reshape(-1)
    songs = np.asarray(songs, np.int64).reshape(-1)
    n = len(users)
    out = Explanation(np.full((n, m), -1, np.int32), np.zeros((n, m), np.float64), np.zeros((n, m), np.int64), np.zeros(n, np.int32),
                      np.zeros(n, np.int32), np.zeros(n, np.int64), np.zeros(n, np.float64))
    tr_ptr = np.asarray(ds.tr_ptr, np.int64)
    tr_col = np.asarray(ds.tr_col, np.int64)
    te_ptr = np.asarray(ds.te_ptr, np.int64)
    te_col = np.asarray(ds.te_col, np.int64)
    owner = np.repeat(np.arange(ds.T), np.diff(tr_ptr))                    # train user of every train entry
    order = np.argsort(tr_col, kind="stable")                              # inverted index: listeners of a song, ascending
    csc_ptr = np.concatenate([[0], np.cumsum(np.bincount(tr_col, minlength=ds.S))])
    listeners = owner[order]
    deg_tr = np.asarray(ds.deg_tr, np.int64)
    deg_te = np.asarray(ds.deg_te, np.int64)
    deg = np.asarray(ds.deg_song, np.int64)
    kq = 24 if model == _lib.MR_UBM else 26

    def q(d):
        with np.errstate(divide="ignore"):
            return np.where(d > 0, np.rint(2.0 ** kq / np.sqrt(d.astype(np.float64))), 0).astype(np.int64)

    def rs(d):
        return (1.0 / 2.0 ** kq) / np.sqrt(np.float64(d)) if d > 0 else 0.0

    for r, (u, s) in enumerate(zip(users, songs)):
        iu = te_col[te_ptr[u]:te_ptr[u + 1]]
        if s in iu:                                                        # a listened pair: no element of the model (MR:109)
            out.score[r] = np.nan
            continue
        if model == _lib.MR_UBM:
            seen = [listeners[csc_ptr[j]:csc_ptr[j + 1]] for j in iu]
            cnt = np.bincount(np.concatenate(seen) if seen else np.zeros(0, np.int64), minlength=ds.T)
            ids = listeners[csc_ptr[s]:csc_ptr[s + 1]]
            c = cnt[ids]
            den = np.sqrt(np.float64(deg_te[u])) * np.sqrt(deg_tr[ids].astype(np.float64))
            dq = deg_tr[ids]
            factor = rs(deg_te[u])
        else:
            hist = [tr_col[tr_ptr[v]:tr_ptr[v + 1]] for v in listeners[csc_ptr[s]:csc_ptr[s + 1]]]
            gram = np.bincount(np.concatenate(hist) if hist else np.zeros(0, np.int64), minlength=ds.S)
            ids = iu
            c = gram[ids]
            den = np.sqrt(np.float64(deg[s])) * np.sqrt(deg[ids].astype(np.float64))
            dq = deg[ids]
            factor = rs(deg[s])
        keep = c > 0
        ids, c, den, dq = ids[keep], c[keep], den[keep], dq[keep]
        with np.errstate(divide="ignore", invalid="ignore"):
            term = np.where(den != 0, c.astype(np.float64) / den, 0.0)
        num = c.astype(np.int64) * q(dq)
        rank = np.lexsort((ids, -term))
        k = min(m, len(rank))
        out.id[r, :k] = ids[rank[:k]]
        out.term[r, :k] = term[rank[:k]]
        out.num[r, :k] = num[rank[:k]]
        out.len[r] = k
        out.count[r] = len(ids)
        out.total[r] = int(num.sum())
        out.score[r] = np.float64(out.total[r]) * factor
    return out


def evaluate_map(scores: np.ndarray, ds: Dataset, n_thresholds: int = 10) -> float:
    """MR:521-639 vectorised over label songs: global min/max normalisation (MR:524-529), per-song confusion counts over
    test users (MR:541-553), AP = sum_i (R_i - R_{i+1}) P_i with the last two terms as in MR:601-609, mean over the
    distinct label songs (MR:626)."""
    U, S = scores.shape
    valid = ~np.isnan(scores)
    mn, mx = scores[valid].min(), scores[valid].max()
    with np.errstate(invalid="ignore", divide="ignore"):
        norm = (scores - mn) / (mx - mn)
    new_songs = np.unique(ds.lab_col)
    labelled = np.zeros((U, int(max(S, new_songs.max() + 1))), bool)
    rows = np.repeat(np.arange(U), np.diff(ds.lab_ptr))
    labelled[rows, ds.lab_col] = True
    th = [0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0][:n_thresholds]
    in_model = new_songs[new_songs < S]
    prec = np.zeros((len(th), len(new_songs)))
    rec = np.zeros((len(th), len(new_songs)))
    lab = labelled[:, new_songs]                       # [U, n_new]
    pos = np.flatnonzero(new_songs < S)
    for t, thr in enumerate(th):
        pred = np.zeros((U, len(new_songs)), bool)
        with np.errstate(invalid="ignore"):
            pred[:, pos] = norm[:, in_model] > thr     # NaN compares false (listened pairs, max == min)
        tp = (pred & lab).sum(0).astype(np.float64)
        fp = (pred & ~lab).sum(0)
        fn = (~pred & lab).sum(0)
        with np.errstate(invalid="ignore", divide="ignore"):
            prec[t] = np.where(tp + fp > 0, tp / (tp + fp), 0.0)
            rec[t] = np.where(tp + fn > 0, tp / (tp + fn), 0.0)
    n = len(th)
    ap = np.zeros(len(new_songs))
    for t in range(n):                                  # List.sum: left fold from 0.0 in threshold order
        if t == n - 1:
            term = 0.0
        elif t == n - 2:
            term = (rec[t] - 0.0) * prec[t]
        else:
            term = (rec[t] - rec[t + 1]) * prec[t]
        ap = ap + term
    total = 0.0
    for x in ap.tolist():                               # foldLeft(0.0)(_+_) (MR:626)
        total += x
    return total / len(new_songs)
