"""GPU tests (-m gpu) of mr_similar_songs (DESIGN.md §4.7): ids, score bits and lengths equal the numpy mirror similar_songs_host and the
oracle's exact count rows on both count engines and spaces, through the short and the long row path; ranking edge cases; the call leaves
the scoring state alone; argument guards; the MSD shape."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import from_triplets, synth, synth_config
from musicrecommendation_b200.recommender import MusicRecommender, _p, eval_finish, similar_songs_host

ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
ENGINES = {"tensor_user": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER),
           "sparse_user": dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER),
           "sparse_item": ITEM,
           "tensor_item": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_ITEM)}
MIXED = dict(T=3000, U=60, S=4000, seed=7)      # about 200 songs above the short-path limit
SHORT = dict(T=120, U=15, S=300, seed=1)        # every row short
ITEMDS = dict(T=800, U=300, S=3001, seed=5)
SHORT_MAX = 8192                                # kSimShortMax


def events(ds):
    """E_i = sum over the train listeners v of song i of |I_v^train|: the work that picks a row's path."""
    deg = np.diff(ds.tr_ptr)
    return np.bincount(ds.tr_col, weights=deg[np.repeat(np.arange(ds.T), deg)], minlength=ds.S).astype(np.int64)


def from_gram(oracle, ds, songs, k):
    """The ranked lists from the oracle's exact count rows g(i, :)."""
    songs = np.asarray(songs, np.int64)
    G = oracle.gram_rows(ds, songs)
    sq = np.sqrt(np.asarray(ds.deg_song, np.float64))
    out = np.full((len(songs), k), -1, np.int32), np.zeros((len(songs), k)), np.zeros(len(songs), np.int32)
    for r, i in enumerate(songs):
        s = np.flatnonzero(G[r] > 0)
        s = s[s != i]
        den = sq[i] * sq[s]
        with np.errstate(divide="ignore", invalid="ignore"):
            sim = np.where(den != 0, G[r, s].astype(np.float64) / den, 0.0)
        o = np.lexsort((s, -sim))[:k]
        out[0][r, :len(o)], out[1][r, :len(o)], out[2][r] = s[o], sim[o], len(o)
    return out


def assert_same(got, want):
    np.testing.assert_array_equal(got[2], want[2])
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1].view(np.int64), want[1].view(np.int64))


def run_paths(mr, ds, songs, k):
    """getSimilarSongs and the path counters it moved: (result, short rows, long rows)."""
    i0 = mr.info()
    got = mr.getSimilarSongs(songs, k)
    i1 = mr.info()
    return got, i1["similar_short_rows"] - i0["similar_short_rows"], i1["similar_long_rows"] - i0["similar_long_rows"]


@pytest.mark.parametrize("cfg", list(ENGINES))
@pytest.mark.parametrize("path", ["mixed", "all_long"])
def test_engines_and_paths(mrlib, oracle_lib, monkeypatch, cfg, path):
    ds = synth(**MIXED)
    e = events(ds)
    n_long = int((e > SHORT_MAX).sum())
    assert 0 < n_long < ds.S
    if path == "all_long":
        monkeypatch.setenv("MRSCORE_SIM_SHORT_MAX", "0")
        n_long = ds.S
    songs = np.arange(ds.S)
    want = similar_songs_host(ds, songs, 50)
    assert_same(want, from_gram(oracle_lib, ds, songs, 50))
    with MusicRecommender(ds, **ENGINES[cfg]) as mr:
        got, n_s, n_l = run_paths(mr, ds, songs, 50)
        assert (n_s, n_l) == (ds.S - n_long, n_long)
        assert_same(got, want)


def test_every_row_short(mrlib, oracle_lib):
    ds = synth(**SHORT)
    assert events(ds).max() <= SHORT_MAX
    for kw in (ITEM, ENGINES["tensor_user"]):
        with MusicRecommender(ds, **kw) as mr:
            got, n_s, n_l = run_paths(mr, ds, None, 20)
            assert (n_s, n_l) == (ds.S, 0)
            assert_same(got, similar_songs_host(ds, np.arange(ds.S), 20))
            assert_same(got, from_gram(oracle_lib, ds, np.arange(ds.S), 20))


def test_multi_chunk_long_path(mrlib, monkeypatch):
    """Chunks of 64 count rows: 4000 long rows take 63 chunks, on both engines."""
    ds = synth(**MIXED)
    monkeypatch.setenv("MRSCORE_SIM_SHORT_MAX", "0")
    monkeypatch.setenv("MRSCORE_SIM_CHUNK", "64")
    want = similar_songs_host(ds, np.arange(ds.S), 30)
    for kw in (ITEM, ENGINES["tensor_user"]):
        with MusicRecommender(ds, **kw) as mr:
            got, n_s, n_l = run_paths(mr, ds, None, 30)
            assert (n_s, n_l) == (0, ds.S)
            assert_same(got, want)


def test_many_short_path_windows(mrlib, monkeypatch):
    """Short-path results in windows of 97 query rows (the last one partial), long rows in chunks of 50 written over their rows of those
    windows; the first window holds long rows only.  Shuffled queries with duplicates, so most windows mix both paths."""
    ds = synth(**MIXED)
    e = events(ds)
    monkeypatch.setenv("MRSCORE_SIM_WINDOW", "97")
    monkeypatch.setenv("MRSCORE_SIM_CHUNK", "50")
    rng = np.random.default_rng(5)
    long_songs = np.flatnonzero(e > SHORT_MAX)
    assert len(long_songs) >= 97
    songs = np.concatenate([long_songs[:97], rng.permutation(ds.S), rng.integers(0, ds.S, 500)])
    want = similar_songs_host(ds, songs, 25)
    for kw in (ITEM, ENGINES["tensor_user"]):
        with MusicRecommender(ds, **kw) as mr:
            got, n_s, n_l = run_paths(mr, ds, songs, 25)
            assert (n_s, n_l) == (int((e[songs] <= SHORT_MAX).sum()), int((e[songs] > SHORT_MAX).sum()))
            assert_same(got, want)


def ties_dataset(n=3000):
    """Train user v listens to song 0 and song v + 1 (g = 1 with song 0 for every other song, all of train degree 1); test users give songs
    1..100 a second, test-visible listener (d_s = 2 > train degree) and are the only listeners of song n + 1."""
    tr_u = np.repeat(np.arange(n), 2)
    tr_s = np.stack([np.zeros(n, np.int64), np.arange(1, n + 1)], 1).reshape(-1)
    te_u = np.concatenate([np.arange(100), np.arange(100)])
    te_s = np.concatenate([np.arange(1, 101), np.full(100, n + 1)])
    return from_triplets((tr_u, tr_s), (te_u, te_s), ([], []), T=n, U=100, S=n + 2)


@pytest.mark.parametrize("path", ["default", "all_long"])
def test_ranking_edge_cases(mrlib, oracle_lib, monkeypatch, path):
    ds = ties_dataset()
    n = ds.T
    if path == "all_long":
        monkeypatch.setenv("MRSCORE_SIM_SHORT_MAX", "0")
    assert ds.deg_song[5] == 2 and ds.deg_song[500] == 1 and ds.deg_song[n + 1] == 100
    queries = [0, n + 1, 7, 500, 0, 3, n, 7, 1]                   # duplicates, unsorted, a song heard only by test users
    with MusicRecommender(ds, **ITEM) as mr:
        for k in (1, 5, 1024):
            got = mr.getSimilarSongs(queries, k)
            want = similar_songs_host(ds, queries, k)
            assert_same(got, want)
            assert_same(got, from_gram(oracle_lib, ds, queries, k))
            assert got[2][0] == min(k, n) and got[2][1] == 0 and got[2][2] == 1   # k above the candidates of song 7: one entry
        song, score, ln = mr.getSimilarSongs([0], 1024)
        # the 2900 songs with d_s = 1 tie at 1 / sqrt(3000) and come first, by id; the songs of d_s = 2 follow
        assert list(song[0, :3]) == [101, 102, 103] and score[0, 0] == score[0, 1023]


def test_train_only_handle(mrlib):
    """A handle loaded with n_test = 0 (train replica only)."""
    ds = synth(**MIXED)
    train = from_triplets((np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr)), ds.tr_col), ([], []), ([], []), T=ds.T, U=0, S=ds.S)
    songs = np.random.default_rng(2).integers(0, ds.S, 400)
    with MusicRecommender(train, **ITEM) as mr:
        assert_same(mr.getSimilarSongs(songs, 40), similar_songs_host(train, songs, 40))


def test_scoring_state_is_left_alone(mrlib):
    """Single-batch item-space shard: device-resident top-k results of both kinds survive the call and the parity probes, host top-k results
    are unchanged, and range -> similar + probes -> counts still reuses the panels (one scoring pass) with the same mAP bits."""
    import torch
    ds = synth(**ITEMDS)
    new = np.unique(ds.lab_col)
    specs = [(_lib.MR_UBM, 0.5, 0), (_lib.MR_IBM, 0.5, 0), (_lib.MR_LC, 0.3, 0)]
    with MusicRecommender(ds, **ITEM) as mr:
        assert mr.info()["batch_rows"] >= ds.U
        top = mr.getTopK(_lib.MR_UBM, 50)
        multi = mr.getTopKMulti(specs, 30)
        mr._check(mr._lib.mr_topk_device(mr._h, _lib.MR_AGG, 0.5, C.c_uint64(0), 50))
        dev = [t.clone() for t in mr.topk_device_tensors(50)]
        mr.topk_multi_device(specs, 30)
        devm = [[t.clone() for t in mr.topk_multi_device_tensors(i, 30)] for i in range(len(specs))]
        mn, mx = mr.eval_range(_lib.MR_IBM)
        p0 = mr.info()["scoring_passes"]
        got, n_s, n_l = run_paths(mr, ds, None, 100)
        assert n_s > 0 and n_l > 0
        mr.counts_ubm()
        mr.similarity_ibm(0, 50)
        cnt = mr.eval_counts(_lib.MR_IBM, mn, mx, new)
        assert mr.info()["scoring_passes"] == p0                    # the count pass reused the panels of the range pass
        for a, b in zip(dev, mr.topk_device_tensors(50)):
            assert torch.equal(a.view(torch.uint8), b.view(torch.uint8))
        for i in range(len(specs)):
            for a, b in zip(devm[i], mr.topk_multi_device_tensors(i, 30)):
                assert torch.equal(a.view(torch.uint8), b.view(torch.uint8))
        assert_same(mr.getTopK(_lib.MR_UBM, 50), top)
        for a, b in zip(mr.getTopKMulti(specs, 30), multi):
            assert_same(a, b)
        mn2, mx2 = mr.eval_range(_lib.MR_IBM)
        cnt2 = mr.eval_counts(_lib.MR_IBM, mn2, mx2, new)
        assert (mn, mx) == (mn2, mx2)
        for a, b in zip(cnt, cnt2):
            np.testing.assert_array_equal(a, b)
        assert float(eval_finish(*cnt, 10)).hex() == float(eval_finish(*cnt2, 10)).hex()
        assert_same(got, similar_songs_host(ds, np.arange(ds.S), 100))


def test_guards(mrlib):
    ds = synth(**SHORT)
    with MusicRecommender(ds, **ITEM) as mr:
        for k in (0, 1025):
            with pytest.raises(_lib.MrError) as e:
                mr.getSimilarSongs([1, 2], k)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        for bad in (-1, ds.S):
            with pytest.raises(_lib.MrError, match=f"song id {bad} ") as e:
                mr.getSimilarSongs([3, bad, ds.S + 7], 10)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        n0 = np.empty(0, np.int32)
        assert mr._lib.mr_similar_songs(mr._h, _p(n0), 0, 10, None, None, None) == _lib.MR_OK
        assert mr._lib.mr_similar_songs(mr._h, None, 3, 10, None, None, None) == _lib.MR_ERR_BAD_ARG
    with MusicRecommender(ds, song_window=(0, ds.S // 2)) as mr:
        with pytest.raises(_lib.MrError) as e:
            mr.getSimilarSongs([1], 10)
        assert e.value.code == _lib.MR_ERR_STATE
    lib = mrlib
    h = C.c_void_p()
    assert lib.mr_create(C.byref(h), (C.c_int * 1)(0), 1, 0) == _lib.MR_OK
    try:
        ids, song, score, ln = np.zeros(1, np.int32), np.zeros(10, np.int32), np.zeros(10), np.zeros(1, np.int32)
        assert lib.mr_similar_songs(h, _p(ids), 1, 10, _p(song), _p(score), _p(ln)) == _lib.MR_ERR_STATE
    finally:
        lib.mr_destroy(h)


def test_msd_shape(mrlib, oracle_lib):
    """configs[3] (MSD) shape, default engine: 200 query songs over the popularity range (the most popular, around the head boundary, the
    tail, the least popular) against the oracle's count rows, through both paths."""
    ds = synth_config("c4").shard_test_users(0, 2560)
    deg_tr = np.bincount(ds.tr_col, minlength=ds.S)
    order = np.argsort(-deg_tr, kind="stable")
    rng = np.random.default_rng(4)
    boundary = int(np.searchsorted(-deg_tr[order], -max(2, ds.S // 6000)))   # default head: train degree >= S / 6000
    songs = np.concatenate([order[:40], order[boundary - 40:boundary + 40], rng.choice(order[boundary + 40:], 60, replace=False),
                            order[-20:]])
    e = events(ds)[songs]
    assert (e > SHORT_MAX).sum() >= 40 and (e <= SHORT_MAX).sum() >= 100
    want = from_gram(oracle_lib, ds, songs, 500)
    with MusicRecommender(ds) as mr:
        for k in (100, 500):
            got, n_s, n_l = run_paths(mr, ds, songs, k)
            assert (n_s, n_l) == (int((e <= SHORT_MAX).sum()), int((e > SHORT_MAX).sum()))
            assert_same(got, tuple(w[:, :k] if w.ndim == 2 else np.minimum(w, k) for w in want))
    assert_same(tuple(w[80:100] for w in want), similar_songs_host(ds, songs[80:100], 500))
