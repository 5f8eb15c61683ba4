"""GPU tests (-m gpu) of song audiences (mr_song_audience, DESIGN.md §4.10): per song, the k test users of highest score under a model, ranked
by column from the score panels.  Every list must equal the numpy mirror over the oracle's dense model in ids, score bits and lengths, on
every engine, space and batching, across song windows and user shards, and agree with getRanks2 / getRanks1 of the same handle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import from_triplets, synth, synth_config
from musicrecommendation_b200.distributed import pair_index_bases, shard_range, song_window
from musicrecommendation_b200.recommender import MusicRecommender, ParameterRange, _p, song_audience_host

ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
MODELS = [(_lib.MR_UBM, 0.5, 0), (_lib.MR_IBM, 0.5, 0), (_lib.MR_LC, 0.3, 0), (_lib.MR_AGG, 0.5, 0), (_lib.MR_STOCH, 0.5, 42)]
SMALL = dict(T=300, U=40, S=2000, seed=3)
ITEMDS = dict(T=800, U=300, S=3001, seed=5)


def dense_models(oracle, ds):
    ubm, ibm = oracle.canon_scores(ds, oracle.UBM), oracle.canon_scores(ds, oracle.IBM)
    kinds = {_lib.MR_LC: oracle.LC, _lib.MR_AGG: oracle.AGG, _lib.MR_STOCH: oracle.STOCH}
    return [ubm if m == _lib.MR_UBM else ibm if m == _lib.MR_IBM else oracle.blend_dense(kinds[m], p, ubm, ibm, seed=s) for m, p, s in MODELS]


def assert_lists_equal(got, want, what=""):
    np.testing.assert_array_equal(got[2], want[2], err_msg=what)
    np.testing.assert_array_equal(got[0], want[0], err_msg=what)
    np.testing.assert_array_equal(np.ascontiguousarray(got[1]).view(np.int64), np.ascontiguousarray(want[1]).view(np.int64), err_msg=what)


def check_consistency(mr, songs, k):
    """The lists of UBM and IBM are the ranked getRanks2 columns, and every listed pair scores the same bits in getRanks1."""
    lo = mr.song_window[0]
    for m in (_lib.MR_UBM, _lib.MR_IBM):
        got = mr.getSongAudience(m, songs, k)
        cols = mr.getRanks2(m, songs)
        assert_lists_equal(got, song_audience_host(cols.T, np.arange(len(songs)), k), f"model {m} against getRanks2")
        users = np.unique(got[0][got[0] >= 0])
        rows = mr.getRanks1(m, users)
        pos = {u: i for i, u in enumerate(users)}
        for r, s in enumerate(songs):
            for i in range(got[2][r]):
                assert rows[pos[got[0][r, i]], s - lo].tobytes() == got[1][r, i].tobytes()


@pytest.mark.parametrize("cfg", ["tensor_user", "sparse_user", "item_one_batch", "item_batches", "item_batches_serial", "head_exceptions", "c3"])
def test_audience_equals_the_oracle(mrlib, oracle_lib, monkeypatch, cfg):
    kw = {}
    if cfg == "tensor_user":
        ds, kw = synth(**SMALL), dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER)
    elif cfg == "sparse_user":
        ds, kw = synth(**SMALL), dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER)
    elif cfg == "item_one_batch":
        ds, kw = synth(**ITEMDS), ITEM
    elif cfg.startswith("item_batches"):
        if cfg.endswith("serial"):
            monkeypatch.setenv("MRSCORE_NO_PIPELINE", "1")
        ds, kw = synth(**ITEMDS), dict(ITEM, item_batch=128)
    elif cfg == "head_exceptions":
        ds, kw = synth(T=12000, U=1040, S=30000, seed=6), dict(ITEM, head_min_deg=8)
    else:
        ds = synth_config("c3")
    songs = np.arange(ds.S, dtype=np.int32)
    with MusicRecommender(ds, **kw) as mr:
        if cfg.startswith("item_batches"):
            assert mr.info()["batch_rows"] == 128
        for (m, p, s), dense in zip(MODELS, dense_models(oracle_lib, ds)):
            assert_lists_equal(mr.getSongAudience(m, None, 50, p, s), song_audience_host(dense, songs, 50), f"model {m}")
        if cfg == "head_exceptions":
            assert mr.info()["head_exceptions"] > 0
        pick = np.random.default_rng(1).choice(ds.S, 12, replace=False).astype(np.int32)
        check_consistency(mr, pick, 50)


def test_song_windows(mrlib, oracle_lib):
    """Three song windows: each windowed handle's lists for its songs equal the unwindowed handle's (and the mirror's) for all five models;
    an id outside the window is refused."""
    ds = synth(**ITEMDS)
    dense = dense_models(oracle_lib, ds)
    with MusicRecommender(ds, **ITEM) as whole:
        want = [whole.getSongAudience(m, None, 50, p, s) for m, p, s in MODELS]
    for d, w in zip(dense, want):
        assert_lists_equal(w, song_audience_host(d, np.arange(ds.S), 50))
    for r in range(3):
        lo, hi = song_window(ds.S, r, 3)
        with MusicRecommender(ds, song_window=(lo, hi), **ITEM) as mr:
            for (m, p, s), w in zip(MODELS, want):
                assert_lists_equal(mr.getSongAudience(m, None, 50, p, s), tuple(a[lo:hi] for a in w), f"window {r} model {m}")
            check_consistency(mr, np.array([lo, hi - 1, (lo + hi) // 2], np.int32), 50)
            for bad in (lo - 1 if lo else hi, hi if hi < ds.S else lo - 1, ds.S):
                with pytest.raises(_lib.MrError, match=f"song id {bad} ") as e:
                    mr.getSongAudience(_lib.MR_UBM, [lo, bad], 10)
                assert e.value.code == _lib.MR_ERR_BAD_ARG


def test_user_shards(mrlib, oracle_lib):
    """Two test-user shards with their global pair bases: the lists with globalised ids, joined with mergeTopK, equal the whole shard's."""
    import torch
    ds = synth(T=800, U=61, S=3001, seed=5)
    starts, n_total = pair_index_bases(ds, 2)
    songs = np.arange(ds.S, dtype=np.int32)
    with MusicRecommender(ds, **ITEM) as mr:
        want = [mr.getSongAudience(m, songs, 40, p, s) for m, p, s in MODELS]
        for d, w in zip(dense_models(oracle_lib, ds), want):
            assert_lists_equal(w, song_audience_host(d, songs, 40))
        for (m, p, s), w in zip(MODELS, want):
            parts = []
            for r in range(2):
                u0, u1 = shard_range(ds.U, r, 2)
                mr.set_test_users(ds.shard_test_users(u0, u1), int(starts[r]), n_total)
                user, score, ln = mr.getSongAudience(m, songs, 40, p, s)
                parts.append((np.where(user >= 0, user + u0, -1).astype(np.int32), score, ln))
            ps, pv, pl = (torch.from_numpy(np.stack([q[i] for q in parts])).cuda() for i in range(3))
            out = (torch.empty_like(ps[0]), torch.empty_like(pv[0]), torch.empty_like(pl[0]))
            mr.mergeTopK(ps, pv, pl, *out)
            mr.sync()
            assert_lists_equal(tuple(t.cpu().numpy() for t in out), w, f"model {m}")


def edge_dataset():
    """SMALL with song 0 listened by every test user and song S - 1 without train listeners."""
    ds = synth(**SMALL)
    tu, ts = np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr)), ds.tr_col
    keep = ts != ds.S - 1
    eu, es = np.repeat(np.arange(ds.U), np.diff(ds.te_ptr)), ds.te_col
    eu, es = np.concatenate([eu, np.arange(ds.U)]), np.concatenate([es, np.zeros(ds.U, es.dtype)])
    lu, ls = np.repeat(np.arange(ds.U), np.diff(ds.lab_ptr)), ds.lab_col
    return from_triplets((tu[keep], ts[keep]), (eu, es), (lu, ls), T=ds.T, U=ds.U, S=ds.S)


def test_edges(mrlib, oracle_lib):
    ds = edge_dataset()
    dense = dense_models(oracle_lib, ds)
    S, U = ds.S, ds.U
    unheard = S - 1
    assert unheard not in ds.tr_col
    with MusicRecommender(ds, **ITEM) as mr:
        for (m, p, s), d in zip(MODELS, dense):
            user, score, ln = mr.getSongAudience(m, [0, unheard], 100, p, s)
            assert ln[0] == 0 and (user[0] == -1).all() and (score[0] == 0.0).all()         # listened by every test user
            listeners = {u for u in range(U) if unheard in ds.te_col[ds.te_ptr[u]:ds.te_ptr[u + 1]]}
            rest = [u for u in range(U) if u not in listeners]
            assert ln[1] == len(rest) and list(user[1, :ln[1]]) == rest and (score[1] == 0.0).all()   # zeros, in id order; k > U
            for k in (1, 100, 1024):
                q = np.array([5, 3, 5, 0, S - 2, 3, 1999], np.int32)                       # duplicates, unordered
                assert_lists_equal(mr.getSongAudience(m, q, k, p, s), song_audience_host(d, q, k), f"model {m} k {k}")
        for k in (-1, 0, 1025):
            with pytest.raises(_lib.MrError) as e:
                mr.getSongAudience(_lib.MR_UBM, [1], k)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        with pytest.raises(_lib.MrError, match="song id -1 ") as e:
            mr.getSongAudience(_lib.MR_UBM, [1, -1, S + 3], 10)
        assert e.value.code == _lib.MR_ERR_BAD_ARG
        with pytest.raises(_lib.MrError) as e:
            mr.getSongAudience(7, [1], 10)
        assert e.value.code == _lib.MR_ERR_BAD_ARG
        for alpha in (1.5, float("nan")):
            with pytest.raises(ParameterRange, match="alpha of the linear combination must be between 0 and 1"):
                mr.getSongAudience(_lib.MR_LC, [1], 10, alpha)
        for m, msg in ((_lib.MR_AGG, "Percentage"), (_lib.MR_STOCH, "Probability")):
            with pytest.raises(ParameterRange, match=msg):
                mr.getSongAudience(m, [1], 10, 1.5)
        n0 = np.empty(0, np.int32)
        assert mr._lib.mr_song_audience(mr._h, _lib.MR_UBM, 0.5, 0, _p(n0), 0, 10, None, None, None) == _lib.MR_OK
        assert mr._lib.mr_song_audience(mr._h, _lib.MR_UBM, 0.5, 0, None, 3, 10, None, None, None) == _lib.MR_ERR_BAD_ARG
    train = from_triplets((np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr)), ds.tr_col), ([], []), ([], []), T=ds.T, U=0, S=ds.S)
    with MusicRecommender(train, **ITEM) as mr:                # no test users
        with pytest.raises(_lib.MrError) as e:
            mr.getSongAudience(_lib.MR_UBM, [0], 10)
        assert e.value.code == _lib.MR_ERR_STATE


@pytest.mark.parametrize("space", [_lib.MR_SPACE_USER, _lib.MR_SPACE_ITEM])
def test_profiled_calls(mrlib, oracle_lib, space):
    """Under MR_PROFILE (serial batches, a CUDA-event timer per phase) the lists are the same, and the column select is timed as topk."""
    ds = synth(**ITEMDS)
    ubm = oracle_lib.canon_scores(ds, oracle_lib.UBM)
    songs = np.arange(0, ds.S, 2, dtype=np.int32)
    with MusicRecommender(ds, engine=_lib.MR_ENGINE_SPARSE, space=space, profile=True) as mr:
        mr.timing(reset=True)
        assert_lists_equal(mr.getSongAudience(_lib.MR_UBM, songs, 50), song_audience_host(ubm, songs, 50))
        assert mr.timing()["topk"] > 0


def test_radix_path(mrlib, oracle_lib):
    """3 200 test users with one history: each column holds thousands of exact ties, more than the candidate buffer, so the bin of the
    k-th key is refined by the radix select (counted in audience_radix_selects)."""
    base = synth(T=300, U=4, S=2000, seed=7)
    hist = base.te_col[base.te_ptr[0]:base.te_ptr[1]]
    assert len(hist) > 0
    U = 3200
    tr = (np.repeat(np.arange(base.T), np.diff(base.tr_ptr)), base.tr_col)
    te = (np.repeat(np.arange(U), len(hist)), np.tile(hist, U))
    ds = from_triplets(tr, te, ([], []), T=base.T, U=U, S=base.S)
    songs = np.arange(0, ds.S, 5, dtype=np.int32)
    with MusicRecommender(ds, **ITEM) as mr:
        for (m, p, s), d in zip(MODELS, dense_models(oracle_lib, ds)):
            r0 = mr.info()["audience_radix_selects"]
            assert_lists_equal(mr.getSongAudience(m, songs, 50, p, s), song_audience_host(d, songs, 50), f"model {m}")
            if m in (_lib.MR_UBM, _lib.MR_IBM, _lib.MR_LC):     # every user scores a column alike: every column ties
                assert mr.info()["audience_radix_selects"] - r0 >= len(songs) - int(np.isin(songs, hist).sum())


def test_scoring_state(mrlib):
    """The single-model top-k and a model-set block survive an audience call; device memory is stable; the shard is scored once per batch
    and the query rows are counted."""
    ds = synth(**ITEMDS)
    songs = np.arange(0, ds.S, 3, dtype=np.int32)
    with MusicRecommender(ds, **dict(ITEM, item_batch=128)) as mr:
        n_batches = -(-ds.U // 128)
        top = mr.getTopK(_lib.MR_IBM, 30)
        mr.topk_multi_device([(_lib.MR_AGG, 0.5, 0), (_lib.MR_UBM, 0.5, 0)], 20)
        before = [t.clone() for t in mr.topk_multi_device_tensors(0, 20)]
        first = mr.getSongAudience(_lib.MR_STOCH, songs, 60, 0.5, 42)
        b0 = mr.info()["device_bytes"]
        for _ in range(3):
            i0 = mr.info()
            assert_lists_equal(mr.getSongAudience(_lib.MR_STOCH, songs, 60, 0.5, 42), first)
            i1 = mr.info()
            assert i1["device_bytes"] == b0
            assert i1["scoring_passes"] - i0["scoring_passes"] == n_batches
            assert i1["audience_rows"] - i0["audience_rows"] == len(songs)
        fetched = (np.empty((ds.U, 30), np.int32), np.empty((ds.U, 30)), np.empty(ds.U, np.int32))
        assert mr._lib.mr_topk_fetch(mr._h, 30, *[_p(a) for a in fetched]) == _lib.MR_OK
        assert_lists_equal(fetched, top)
        for a, b in zip(mr.topk_multi_device_tensors(0, 20), before):
            assert bool((a == b).all())


def test_msd_shape_shard(mrlib):
    """configs[3] (MSD) shape, a 2 560-user shard on the default engine: the lists of the 150 most popular songs and 150 random ones equal
    the ranked getRanks2 columns, for UBM and IBM at k = 100 and 500."""
    ds = synth_config("c4").shard_test_users(0, 2560)
    pop = np.argsort(-np.asarray(ds.deg_song), kind="stable")
    rng = np.random.default_rng(3)
    songs = np.concatenate([pop[:150], rng.choice(pop[150:], 150, replace=False)]).astype(np.int32)
    with MusicRecommender(ds) as mr:
        assert mr.info()["space"] == _lib.MR_SPACE_ITEM
        for m in (_lib.MR_UBM, _lib.MR_IBM):
            cols = mr.getRanks2(m, songs)
            for k in (100, 500):
                assert_lists_equal(mr.getSongAudience(m, songs, k), song_audience_host(cols.T, np.arange(len(songs)), k), f"model {m} k {k}")
