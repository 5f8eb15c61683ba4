"""GPU tests (-m gpu) of mr_explain (DESIGN.md §4.9): ids, term bits, nums, lengths, counts and totals equal the numpy mirror explain_host
on both count engines and spaces; scores with the bits of getRanks1 and getTopK; chunks and the count rows they build; duplicate, unordered,
listened and empty pairs; m edge cases; a tie too crowded for the collect buffer (radix select); guards; device memory; the scoring state
left alone; the MSD shape."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import Dataset, from_triplets, synth, synth_config
from musicrecommendation_b200.recommender import Explanation, MusicRecommender, _p, eval_finish, explain_host

UBM, IBM = _lib.MR_UBM, _lib.MR_IBM
ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
ENGINES = {"tensor_user": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER),
           "sparse_user": dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER),
           "sparse_item": ITEM,
           "tensor_item": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_ITEM)}
EMPTY = [3, 77, 299]                            # test users whose visible rows are emptied: their pairs have no contributors


def with_empty_rows(ds, rows):
    te_ptr = np.asarray(ds.te_ptr, np.int64)
    keep = np.ones(len(ds.te_col), bool)
    for u in rows:
        keep[te_ptr[u]:te_ptr[u + 1]] = False
    lens = np.diff(te_ptr)
    lens[list(rows)] = 0
    return Dataset(ds.T, ds.U, ds.S, ds.tr_ptr, ds.tr_col, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64),
                   np.asarray(ds.te_col, np.int32)[keep], ds.lab_ptr, ds.lab_col, ds.deg_tr, lens.astype(np.int32), ds.deg_song)


def mixed():
    return with_empty_rows(synth(T=3000, U=300, S=4000, seed=7), EMPTY)


def pairs_of(ds, seed, n=400):
    """Random pairs (duplicates, any order), listened pairs, pairs of the emptied users and a few repeated keys."""
    rng = np.random.default_rng(seed)
    u = rng.integers(0, ds.U, n)
    s = rng.integers(0, ds.S, n)
    lu = rng.integers(0, ds.U, 20)
    lu = lu[np.diff(ds.te_ptr)[lu] > 0]
    ls = np.asarray(ds.te_col)[ds.te_ptr[lu]]                       # the first visible song of each: listened
    eu = np.repeat(EMPTY, 3)
    es = rng.integers(0, ds.S, len(eu))
    u = np.concatenate([u, lu, eu, u[:30], np.full(40, u[0])])
    s = np.concatenate([s, ls, es, s[:30], rng.integers(0, ds.S, 40)])
    p = rng.permutation(len(u))
    return u[p].astype(np.int32), s[p].astype(np.int32)


def assert_same(got, want):
    for name in Explanation._fields:
        a, b = getattr(got, name), getattr(want, name)
        if a.dtype == np.float64:
            a, b = a.view(np.int64), b.view(np.int64)
        np.testing.assert_array_equal(a, b, err_msg=name)


def run(mr, model, u, s, m):
    """explain and the count rows it built."""
    r0 = mr.info()["explain_rows"]
    got = mr.explain(model, u, s, m)
    return got, mr.info()["explain_rows"] - r0


def n_keys(model, u, s):
    return len(np.unique(u if model == UBM else s))


@pytest.mark.parametrize("cfg", list(ENGINES))
def test_engines_and_spaces(mrlib, cfg):
    ds = mixed()
    u, s = pairs_of(ds, 1)
    with MusicRecommender(ds, **ENGINES[cfg]) as mr:
        for model in (UBM, IBM):
            want = explain_host(ds, model, u, s, 20)
            assert np.isnan(want.score).sum() >= 10 and ((want.count == 0) & ~np.isnan(want.score)).sum() >= 9
            assert (want.count > 20).sum() >= 20
            got, rows = run(mr, model, u, s, 20)
            assert rows == n_keys(model, u, s)
            assert_same(got, want)
            ranks = mr.getRanks1(model, u)[np.arange(len(u)), s]
            np.testing.assert_array_equal(np.isnan(got.score), np.isnan(ranks))
            np.testing.assert_array_equal(np.nan_to_num(got.score).view(np.int64), np.nan_to_num(ranks).view(np.int64))


@pytest.mark.parametrize("model", [UBM, IBM])
def test_scores_of_the_top_k(mrlib, model):
    ds = mixed()
    with MusicRecommender(ds, **ITEM) as mr:
        song, score, ln = mr.getTopK(model, 10)
        u = np.repeat(np.arange(ds.U), ln).astype(np.int32)
        s = np.concatenate([song[i, :ln[i]] for i in range(ds.U)]).astype(np.int32)
        sc = np.concatenate([score[i, :ln[i]] for i in range(ds.U)])
        got = mr.explain(model, u, s, 5)
        np.testing.assert_array_equal(got.score.view(np.int64), sc.view(np.int64))
        assert_same(got, explain_host(ds, model, u, s, 5))


def test_chunks(mrlib, monkeypatch):
    """Count rows in chunks of 16 keys; every key's row built once however many pairs it serves."""
    ds = mixed()
    u, s = pairs_of(ds, 2, 900)
    monkeypatch.setenv("MRSCORE_SIM_CHUNK", "16")
    for kw in (ITEM, ENGINES["tensor_user"]):
        with MusicRecommender(ds, **kw) as mr:
            for model in (UBM, IBM):
                got, rows = run(mr, model, u, s, 7)
                assert rows == n_keys(model, u, s) > 16 * 4
                assert_same(got, explain_host(ds, model, u, s, 7))


def test_m_edges(mrlib):
    ds = mixed()
    u, s = pairs_of(ds, 3, 200)
    with MusicRecommender(ds, **ITEM) as mr:
        for model in (UBM, IBM):
            full = explain_host(ds, model, u, s, 1024)
            assert full.count.max() < 1024 and (full.len == full.count).all()
            for m in (1, int(full.count.max()), 1024):
                got = mr.explain(model, u, s, m)
                assert_same(got, explain_host(ds, model, u, s, m))
                assert (got.total == full.total).all() and (got.len == np.minimum(full.count, m)).all()


def ties_dataset(n=3000):
    """UBM: test user 0 hears songs 1 and 2; train users 0..n-1 hear {0, 1} (c = 1, degree 2: n equal terms for the pair (0, song 0), a
    crowded bin) and train users n..n+9 hear {0, 1, 2} (c = 2, higher terms).  IBM: test user 1 hears songs 3 .. n+2, and train user
    n+10+i hears {0, 3+i}: g(0, 3+i) = 1 against songs of one degree, n equal terms for the pair (1, song 0)."""
    tr_u = np.concatenate([np.repeat(np.arange(n), 2), np.repeat(np.arange(n, n + 10), 3), np.repeat(np.arange(n + 10, 2 * n + 10), 2)])
    tr_s = np.concatenate([np.tile([0, 1], n), np.tile([0, 1, 2], 10), np.stack([np.zeros(n, np.int64), 3 + np.arange(n)], 1).ravel()])
    te_u = np.concatenate([[0, 0], np.ones(n, np.int64)])
    te_s = np.concatenate([[1, 2], 3 + np.arange(n)])
    return from_triplets((tr_u, tr_s), (te_u, te_s), ([], []), T=2 * n + 10, U=2, S=n + 3)


def test_crowded_tie_takes_the_radix_select(mrlib):
    ds = ties_dataset()
    n = 3000
    with MusicRecommender(ds, **ITEM) as mr:
        for model, u, ids in ((UBM, 0, list(range(n, n + 10)) + list(range(1014))), (IBM, 1, [3 + i for i in range(1024)])):
            want = explain_host(ds, model, [u, u], [0, 0], 1024)
            assert want.count[0] >= n and want.len[0] == 1024
            assert len(set(want.term[0, 10 if model == UBM else 0:].tolist())) == 1        # one tied term past the head
            got = mr.explain(model, [u, u], [0, 0], 1024)
            assert_same(got, want)
            assert list(got.id[0]) == ids


def test_guards(mrlib):
    ds = synth(T=120, U=15, S=300, seed=1)
    with MusicRecommender(ds, **ITEM) as mr:
        for m in (0, 1025):
            with pytest.raises(_lib.MrError) as e:
                mr.explain(UBM, [1, 2], [3, 4], m)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        for model in (_lib.MR_LC, _lib.MR_AGG, _lib.MR_STOCH, 7):
            with pytest.raises(_lib.MrError) as e:
                mr.explain(model, [1], [3], 5)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        for bad in (-1, ds.U):
            with pytest.raises(_lib.MrError, match=f"pair 1: test user index {bad} ") as e:
                mr.explain(IBM, [3, bad, ds.U + 7], [0, 0, 0], 10)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        for bad in (-1, ds.S):
            with pytest.raises(_lib.MrError, match=f"pair 2: song id {bad} ") as e:
                mr.explain(UBM, [3, 4, 5], [0, 1, bad], 10)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        n0 = np.empty(0, np.int32)
        assert mr._lib.mr_explain(mr._h, UBM, _p(n0), _p(n0), 0, 10, *([None] * 7)) == _lib.MR_OK
        assert mr._lib.mr_explain(mr._h, UBM, None, None, 3, 10, *([None] * 7)) == _lib.MR_ERR_BAD_ARG
    train = from_triplets((np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr)), ds.tr_col), ([], []), ([], []), T=ds.T, U=0, S=ds.S)
    with MusicRecommender(train, **ITEM) as mr:                # no test users
        with pytest.raises(_lib.MrError) as e:
            mr.explain(UBM, [0], [0], 10)
        assert e.value.code == _lib.MR_ERR_STATE
    with MusicRecommender(ds, song_window=(0, 150)) as mr:     # a song window
        with pytest.raises(_lib.MrError, match="song window") as e:
            mr.explain(IBM, [0], [0], 10)
        assert e.value.code == _lib.MR_ERR_STATE
    lib = mrlib
    h = C.c_void_p()
    assert lib.mr_create(C.byref(h), (C.c_int * 1)(0), 1, 0) == _lib.MR_OK
    try:
        one = np.zeros(1, np.int32)
        out = [np.zeros(10, np.int32), np.zeros(10), np.zeros(10, np.int64), np.zeros(1, np.int32), np.zeros(1, np.int32),
               np.zeros(1, np.int64), np.zeros(1)]
        assert lib.mr_explain(h, UBM, _p(one), _p(one), 1, 10, *[_p(a) for a in out]) == _lib.MR_ERR_STATE
    finally:
        lib.mr_destroy(h)


def test_scoring_state_is_left_alone(mrlib):
    """Single-batch item-space shard: range -> explain -> counts still costs one scoring pass with the same mAP bits; the device top-k
    result fetched afterwards is unchanged; device_bytes is the same over repeated calls."""
    import torch
    ds = synth(T=800, U=300, S=3001, seed=5)
    new = np.unique(ds.lab_col)
    u, s = pairs_of(ds, 6, 300)
    with MusicRecommender(ds, **ITEM) as mr:
        assert mr.info()["batch_rows"] >= ds.U
        top = mr.getTopK(_lib.MR_UBM, 50)
        mr._check(mr._lib.mr_topk_device(mr._h, _lib.MR_AGG, 0.5, C.c_uint64(0), 50))
        dev = [t.clone() for t in mr.topk_device_tensors(50)]
        mn, mx = mr.eval_range(_lib.MR_IBM)
        p0 = mr.info()["scoring_passes"]
        got = [mr.explain(model, u, s, 30) for model in (UBM, IBM)]
        cnt = mr.eval_counts(_lib.MR_IBM, mn, mx, new)
        assert mr.info()["scoring_passes"] == p0                    # the count pass reused the panels of the range pass
        for a, b in zip(dev, mr.topk_device_tensors(50)):
            assert torch.equal(a.view(torch.uint8), b.view(torch.uint8))
        for a, b in zip(mr.getTopK(_lib.MR_UBM, 50), top):
            np.testing.assert_array_equal(a.view(np.uint8), b.view(np.uint8))
        mn2, mx2 = mr.eval_range(_lib.MR_IBM)
        cnt2 = mr.eval_counts(_lib.MR_IBM, mn2, mx2, new)
        assert (mn, mx) == (mn2, mx2)
        assert float(eval_finish(*cnt, 10)).hex() == float(eval_finish(*cnt2, 10)).hex()
        for model, g in zip((UBM, IBM), got):
            assert_same(g, explain_host(ds, model, u, s, 30))
        b0 = mr.info()["device_bytes"]
        for _ in range(3):
            for model, g in zip((UBM, IBM), got):
                assert_same(mr.explain(model, u, s, 30), g)
            assert mr.info()["device_bytes"] == b0


def test_msd_shape(mrlib):
    """configs[3] (MSD) shape, default engine: the explanations of the top-10 of 64 test users reproduce getTopK's score bits, and 24 of
    those pairs equal the mirror."""
    ds = synth_config("c4")
    rng = np.random.default_rng(8)
    users = rng.choice(ds.U, 64, replace=False)
    with MusicRecommender(ds) as mr:
        for model in (UBM, IBM):
            song, score, ln = mr.getTopK(model, 10)
            u = np.repeat(users, ln[users]).astype(np.int32)
            s = np.concatenate([song[i, :ln[i]] for i in users]).astype(np.int32)
            sc = np.concatenate([score[i, :ln[i]] for i in users])
            got = mr.explain(model, u, s, 10)
            np.testing.assert_array_equal(got.score.view(np.int64), sc.view(np.int64))
            assert (got.count > 0).mean() > 0.9 and (got.len == np.minimum(got.count, 10)).all()
            pick = rng.choice(len(u), 24, replace=False)
            assert_same(Explanation(*[a[pick] for a in got]), explain_host(ds, model, u[pick], s[pick], 10))
