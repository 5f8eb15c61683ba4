"""GPU tests (-m gpu) of mr_similar_users (DESIGN.md §4.8): ids, score bits and lengths equal the numpy mirror similar_users_host on both
count engines and spaces, through the short and the long row path; chunks, windows, ties and k edge cases; test-user shards and song
windows; the call leaves the scoring state alone; argument guards; the MSD shape."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import Dataset, from_triplets, synth, synth_config
from musicrecommendation_b200.recommender import MusicRecommender, _p, eval_finish, similar_users_host

ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
ENGINES = {"tensor_user": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER),
           "sparse_user": dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER),
           "sparse_item": ITEM,
           "tensor_item": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_ITEM)}
MIXED = dict(T=3000, U=300, S=4000, seed=7)     # about a third of the test users above the short-path limit
SHORT = dict(T=120, U=15, S=300, seed=1)        # every row short
ITEMDS = dict(T=800, U=300, S=3001, seed=5)
SHORT_MAX = 8192                                # kSimShortMax
EMPTY = [3, 77, 299]                            # test users of the mixed set whose visible rows are emptied


def events(ds):
    """E_u = sum over the visible songs j of test user u of |U_j^train|: the work that picks a row's path."""
    deg = np.bincount(ds.tr_col, minlength=ds.S)
    owner = np.repeat(np.arange(ds.U), np.diff(ds.te_ptr))
    return np.bincount(owner, weights=deg[ds.te_col], minlength=ds.U).astype(np.int64)


def with_empty_rows(ds, rows):
    """ds with the visible test rows of `rows` emptied (their test degree 0, as the reference's .length)."""
    te_ptr = np.asarray(ds.te_ptr, np.int64)
    keep = np.ones(len(ds.te_col), bool)
    for u in rows:
        keep[te_ptr[u]:te_ptr[u + 1]] = False
    lens = np.diff(te_ptr)
    lens[list(rows)] = 0
    return Dataset(ds.T, ds.U, ds.S, ds.tr_ptr, ds.tr_col, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64),
                   np.asarray(ds.te_col, np.int32)[keep], ds.lab_ptr, ds.lab_col, ds.deg_tr, lens.astype(np.int32), ds.deg_song)


def mixed():
    return with_empty_rows(synth(**MIXED), EMPTY)


def assert_same(got, want):
    np.testing.assert_array_equal(got[2], want[2])
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1].view(np.int64), want[1].view(np.int64))


def run_paths(mr, users, k):
    """getSimilarUsers and the path counters it moved: (result, short rows, long rows)."""
    i0 = mr.info()
    got = mr.getSimilarUsers(users, k)
    i1 = mr.info()
    return got, i1["similar_user_short_rows"] - i0["similar_user_short_rows"], i1["similar_user_long_rows"] - i0["similar_user_long_rows"]


@pytest.mark.parametrize("cfg", list(ENGINES))
@pytest.mark.parametrize("path", ["mixed", "all_long"])
def test_engines_and_paths(mrlib, monkeypatch, cfg, path):
    ds = mixed()
    e = events(ds)
    n_long = int((e > SHORT_MAX).sum())
    assert 0 < n_long < ds.U and (e[EMPTY] == 0).all()
    if path == "all_long":
        monkeypatch.setenv("MRSCORE_SIM_SHORT_MAX", "0")
        n_long = ds.U - len(EMPTY)                       # E_u = 0 is never above the limit
    want = similar_users_host(ds, np.arange(ds.U), 60)
    assert (want[2][EMPTY] == 0).all() and (want[0][EMPTY] == -1).all()
    with MusicRecommender(ds, **ENGINES[cfg]) as mr:
        got, n_s, n_l = run_paths(mr, None, 60)
        assert (n_s, n_l) == (ds.U - n_long, n_long)
        assert_same(got, want)


def test_every_row_short(mrlib):
    ds = synth(**SHORT)
    assert events(ds).max() <= SHORT_MAX
    want = similar_users_host(ds, np.arange(ds.U), 20)
    for kw in (ITEM, ENGINES["tensor_user"]):
        with MusicRecommender(ds, **kw) as mr:
            got, n_s, n_l = run_paths(mr, None, 20)
            assert (n_s, n_l) == (ds.U, 0)
            assert_same(got, want)


def test_chunks_and_windows(mrlib, monkeypatch):
    """Short-path results in windows of 37 query rows, long rows in chunks of 16 written over their rows of those windows; shuffled
    queries with duplicates.  Then every row long in chunks of 16."""
    ds = mixed()
    e = events(ds)
    rng = np.random.default_rng(5)
    users = np.concatenate([rng.permutation(ds.U), rng.integers(0, ds.U, 200), EMPTY])
    want = similar_users_host(ds, users, 25)
    monkeypatch.setenv("MRSCORE_SIM_WINDOW", "37")
    monkeypatch.setenv("MRSCORE_SIM_CHUNK", "16")
    for kw in (ITEM, ENGINES["tensor_user"]):
        with MusicRecommender(ds, **kw) as mr:
            got, n_s, n_l = run_paths(mr, users, 25)
            assert (n_s, n_l) == (int((e[users] <= SHORT_MAX).sum()), int((e[users] > SHORT_MAX).sum()))
            assert_same(got, want)
            monkeypatch.setenv("MRSCORE_SIM_SHORT_MAX", "0")
            got, n_s, n_l = run_paths(mr, users, 25)
            assert n_l == int((e[users] > 0).sum())
            assert_same(got, want)
            monkeypatch.delenv("MRSCORE_SIM_SHORT_MAX")


def ties_dataset(n=3000):
    """Train users 0..n-1 listen to song 0 only (w = 1 / (sqrt(1) * 1) for test user 0 = {0}: n exact ties, a crowded bin); train users
    n..n+99 listen to songs 0 and 1 (degree 2, lower weight for test user 0, higher for test user 1 = {0, 1}).  Test user 2 hears song 2,
    which no train user heard; test user 3 has an empty visible row."""
    tr_u = np.concatenate([np.arange(n), np.repeat(np.arange(n, n + 100), 2)])
    tr_s = np.concatenate([np.zeros(n, np.int64), np.tile([0, 1], 100)])
    te_u = np.array([0, 1, 1, 2])
    te_s = np.array([0, 0, 1, 2])
    return from_triplets((tr_u, tr_s), (te_u, te_s), ([], []), T=n + 100, U=4, S=3)


@pytest.mark.parametrize("path", ["default", "all_long"])
def test_ranking_edge_cases(mrlib, monkeypatch, path):
    ds = ties_dataset()
    n = ds.T - 100
    if path == "all_long":
        monkeypatch.setenv("MRSCORE_SIM_SHORT_MAX", "0")     # E_0 = 3100 stays under the limit: the radix select needs this
    queries = [0, 1, 2, 3, 0, 1]
    for kw in (ITEM, ENGINES["tensor_user"]):
        with MusicRecommender(ds, **kw) as mr:
            for k in (1, 5, 1024):
                got = mr.getSimilarUsers(queries, k)
                assert_same(got, similar_users_host(ds, queries, k))
                assert list(got[2]) == [k, k, 0, 0, k, k]
            (user, score, ln), n_s, n_l = run_paths(mr, [0, 1, 2, 3], 1024)
            assert (n_s, n_l) == ((2, 2) if path == "all_long" else (4, 0))   # E_u = 0 (users 2, 3) is never above the limit
            assert list(user[0, :3]) == [0, 1, 2] and score[0, 0] == score[0, 1023] == 1.0    # the n ties, by id
            assert list(user[1, :3]) == [n, n + 1, n + 2]                                      # two shared songs rank first


def test_test_user_shards(mrlib):
    """After mr_set_test_users with a shard, the shard-local indices give the whole set's rows (and the sqrt of the test degrees follows)."""
    ds = mixed()
    want = similar_users_host(ds, np.arange(ds.U), 40)
    with MusicRecommender(ds, **ITEM) as mr:
        assert_same(mr.getSimilarUsers(None, 40), want)
        for u0, u1 in ((0, 100), (100, 300), (250, 260)):
            mr.set_test_users(ds.shard_test_users(u0, u1))
            assert_same(mr.getSimilarUsers(None, 40), tuple(w[u0:u1] for w in want))
            assert_same(mr.getSimilarUsers([u1 - u0 - 1, 0], 40), tuple(w[[u1 - 1, u0]] for w in want))


def test_song_window(mrlib):
    """A handle with a song window (its song ids rotated) gives the un-windowed handle's lists, on both paths."""
    ds = mixed()
    rng = np.random.default_rng(9)
    users = np.concatenate([rng.permutation(ds.U), EMPTY])
    with MusicRecommender(ds, **ITEM) as mr:
        want = mr.getSimilarUsers(users, 80)
    assert_same(want, similar_users_host(ds, users, 80))
    for lo, hi in ((ds.S // 3, ds.S), (0, ds.S // 2), (1000, 2500)):
        with MusicRecommender(ds, song_window=(lo, hi)) as mr:
            got, n_s, n_l = run_paths(mr, users, 80)
            assert n_s > 0 and n_l > 0
            assert_same(got, want)


def test_scoring_state_is_left_alone(mrlib):
    """Single-batch item-space shard: range -> similar users -> counts still costs one scoring pass with the same mAP bits; the device
    top-k result fetched afterwards is unchanged; device_bytes is the same over repeated calls."""
    import torch
    ds = synth(**ITEMDS)
    new = np.unique(ds.lab_col)
    e = events(ds)
    with MusicRecommender(ds, **ITEM) as mr:
        assert mr.info()["batch_rows"] >= ds.U
        top = mr.getTopK(_lib.MR_UBM, 50)
        mr._check(mr._lib.mr_topk_device(mr._h, _lib.MR_AGG, 0.5, C.c_uint64(0), 50))
        dev = [t.clone() for t in mr.topk_device_tensors(50)]
        mn, mx = mr.eval_range(_lib.MR_IBM)
        p0 = mr.info()["scoring_passes"]
        got, n_s, n_l = run_paths(mr, None, 100)
        assert n_s > 0 and n_l == int((e > SHORT_MAX).sum()) > 0
        cnt = mr.eval_counts(_lib.MR_IBM, mn, mx, new)
        assert mr.info()["scoring_passes"] == p0                    # the count pass reused the panels of the range pass
        for a, b in zip(dev, mr.topk_device_tensors(50)):
            assert torch.equal(a.view(torch.uint8), b.view(torch.uint8))
        assert_same(mr.getTopK(_lib.MR_UBM, 50), top)
        mn2, mx2 = mr.eval_range(_lib.MR_IBM)
        cnt2 = mr.eval_counts(_lib.MR_IBM, mn2, mx2, new)
        assert (mn, mx) == (mn2, mx2)
        assert float(eval_finish(*cnt, 10)).hex() == float(eval_finish(*cnt2, 10)).hex()
        assert_same(got, similar_users_host(ds, np.arange(ds.U), 100))
        b0 = mr.info()["device_bytes"]
        for _ in range(3):
            assert_same(mr.getSimilarUsers(None, 100), got)
            assert mr.info()["device_bytes"] == b0


def test_guards(mrlib):
    ds = synth(**SHORT)
    with MusicRecommender(ds, **ITEM) as mr:
        for k in (0, 1025):
            with pytest.raises(_lib.MrError) as e:
                mr.getSimilarUsers([1, 2], k)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        for bad in (-1, ds.U):
            with pytest.raises(_lib.MrError, match=f"test user index {bad} ") as e:
                mr.getSimilarUsers([3, bad, ds.U + 7], 10)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        n0 = np.empty(0, np.int32)
        assert mr._lib.mr_similar_users(mr._h, _p(n0), 0, 10, None, None, None) == _lib.MR_OK
        assert mr._lib.mr_similar_users(mr._h, None, 3, 10, None, None, None) == _lib.MR_ERR_BAD_ARG
    train = from_triplets((np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr)), ds.tr_col), ([], []), ([], []), T=ds.T, U=0, S=ds.S)
    with MusicRecommender(train, **ITEM) as mr:                # no test users
        with pytest.raises(_lib.MrError) as e:
            mr.getSimilarUsers([0], 10)
        assert e.value.code == _lib.MR_ERR_STATE
    lib = mrlib
    h = C.c_void_p()
    assert lib.mr_create(C.byref(h), (C.c_int * 1)(0), 1, 0) == _lib.MR_OK
    try:
        ids, user, score, ln = np.zeros(1, np.int32), np.zeros(10, np.int32), np.zeros(10), np.zeros(1, np.int32)
        assert lib.mr_similar_users(h, _p(ids), 1, 10, _p(user), _p(score), _p(ln)) == _lib.MR_ERR_STATE
    finally:
        lib.mr_destroy(h)


def test_msd_shape(mrlib):
    """configs[3] (MSD) shape, default engine: 256 test users, the 32 heaviest by E_u among them, against the mirror, through both paths."""
    ds = synth_config("c4")
    e = events(ds)
    order = np.argsort(-e, kind="stable")
    rng = np.random.default_rng(4)
    users = np.concatenate([order[:32], rng.choice(order[32:], 200, replace=False), order[-24:]])
    eu = e[users]
    assert (eu <= SHORT_MAX).sum() >= 20 and (eu > SHORT_MAX).sum() >= 200
    want = similar_users_host(ds, users, 500)
    with MusicRecommender(ds) as mr:
        for k in (100, 500):
            got, n_s, n_l = run_paths(mr, users, k)
            assert (n_s, n_l) == (int((eu <= SHORT_MAX).sum()), int((eu > SHORT_MAX).sum()))
            assert_same(got, tuple(w[:, :k] if w.ndim == 2 else np.minimum(w, k) for w in want))
