"""GPU tests (-m gpu) of the filtered top-k (mr_set_topk_filter / mr_topk_filtered, DESIGN.md §4.11): each user's ranking without the songs
outside an allowed set and without the user's excluded songs.  Every list must equal the numpy mirror over the oracle's dense model in ids,
score bits and lengths, on every engine, space and batching, through both select paths, across song windows and user shards; paging must
give the second page of getTopK; and no unfiltered call may see the filter."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import from_triplets, synth, synth_config
from musicrecommendation_b200.distributed import pair_index_bases, shard_exclusions, shard_range, song_window
from musicrecommendation_b200.recommender import MusicRecommender, ParameterRange, _p, exclusions_from_topk, topk_filtered_host

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


def random_exclusions(ds, rng, n=25, empty_every=5):
    """Per test user about n random songs plus three of its listened songs (an excluded listened song changes nothing); every
    empty_every-th row is empty."""
    rows = []
    for u in range(ds.U):
        heard = ds.te_col[ds.te_ptr[u]:ds.te_ptr[u + 1]]
        r = np.concatenate([rng.choice(ds.S, n, replace=False), heard[:3]]) if u % empty_every else np.empty(0, np.int64)
        rows.append(np.unique(r))
    ptr = np.zeros(ds.U + 1, np.int64)
    ptr[1:] = np.cumsum([len(r) for r in rows])
    return ptr, np.concatenate(rows).astype(np.int32)


def filters(ds, rng):
    """exclusions only; about 1 % of the songs allowed (candidate path) with exclusions; about 90 % allowed (full-row path) with exclusions"""
    ex = random_exclusions(ds, rng)
    few = rng.choice(ds.S, max(8, ds.S // 100), replace=False)
    many = rng.choice(ds.S, ds.S * 9 // 10, replace=False)
    return {"exclusions": (None, ex), "allow_1pct": (few, ex), "allow_90pct": (many, ex)}


def config(cfg, monkeypatch):
    if cfg == "tensor_user":
        return synth(**SMALL), dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER)
    if cfg == "sparse_user":
        return synth(**SMALL), dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER)
    if cfg == "item_one_batch":
        return synth(**ITEMDS), ITEM
    if cfg.startswith("item_batches"):
        if cfg.endswith("serial"):
            monkeypatch.setenv("MRSCORE_NO_PIPELINE", "1")
        return synth(**ITEMDS), dict(ITEM, item_batch=128)
    if cfg == "head_exceptions":
        return synth(T=12000, U=1040, S=30000, seed=6), dict(ITEM, head_min_deg=8)
    return synth_config("c3"), {}


@pytest.mark.parametrize("cfg", ["tensor_user", "sparse_user", "item_one_batch", "item_batches", "item_batches_serial", "head_exceptions", "c3"])
def test_filtered_equals_the_oracle(mrlib, oracle_lib, monkeypatch, cfg):
    ds, kw = config(cfg, monkeypatch)
    rng = np.random.default_rng(11)
    dense = dense_models(oracle_lib, ds)
    with MusicRecommender(ds, **kw) as mr:
        i0 = mr.info()
        for name, (allowed, ex) in filters(ds, rng).items():
            mr.setTopKFilter(allowed, ex)
            for (m, p, s), d in zip(MODELS, dense):
                assert_lists_equal(mr.getTopKFiltered(m, 50, p, s), topk_filtered_host(d, allowed, *ex, 50), f"{name} model {m}")
        i1 = mr.info()
        assert i1["filter_full_rows"] - i0["filter_full_rows"] == 2 * len(MODELS) * ds.U
        assert i1["filter_candidate_rows"] - i0["filter_candidate_rows"] == len(MODELS) * ds.U
        # identity: every song allowed and no exclusions gives getTopK's lists
        mr.setTopKFilter(np.arange(ds.S)[::-1], None)
        for m, p, s in MODELS:
            assert_lists_equal(mr.getTopKFiltered(m, 50, p, s), mr.getTopK(m, 50, p, s), f"identity model {m}")


def page_two(mr, m, k, p=0.5, s=0):
    song, score, ln = mr.getTopK(m, 2 * k, p, s)
    mr.setTopKFilter(None, exclusions_from_topk(*mr.getTopK(m, k, p, s)[::2]))
    got = mr.getTopKFiltered(m, k, p, s)
    mr.clearTopKFilter()
    return got, (song[:, k:], score[:, k:], np.maximum(ln - k, 0).astype(np.int32))


def test_paging_item_batches(mrlib):
    """Page 2 with page 1 excluded is entries [k, 2k) of getTopK(2k), for every model."""
    with MusicRecommender(synth(**ITEMDS), **dict(ITEM, item_batch=128)) as mr:
        for m, p, s in MODELS:
            got, want = page_two(mr, m, 500, p, s)
            assert_lists_equal(got, want, f"model {m}")


def test_paging_msd_shape_shard(mrlib):
    """configs[3] (MSD) shape, a 2 560-user shard on the default engine: page 2 of 500 for UBM and IBM; a popular allowed set of 1 000 songs
    (candidate path) and 90 % of the songs (full-row path) against the filtered getRanks1 rows."""
    ds = synth_config("c4").shard_test_users(0, 2560)
    with MusicRecommender(ds) as mr:
        assert mr.info()["space"] == _lib.MR_SPACE_ITEM
        for m in (_lib.MR_UBM, _lib.MR_IBM):
            got, want = page_two(mr, m, 500)
            assert_lists_equal(got, want, f"model {m}")
        rng = np.random.default_rng(4)
        users = rng.choice(ds.U, 40, replace=False).astype(np.int32)
        pop = np.argsort(-np.asarray(ds.deg_song), kind="stable")
        for allowed in (pop[:1000], rng.choice(ds.S, ds.S * 9 // 10, replace=False)):
            mr.setTopKFilter(allowed, None)
            rows = mr.getRanks1(_lib.MR_UBM, users)
            got = mr.getTopKFiltered(_lib.MR_UBM, 500)
            assert_lists_equal(tuple(a[users] for a in got), topk_filtered_host(rows, allowed, None, None, 500))
        assert mr.info()["filter_full_rows"] > 0 and mr.info()["filter_candidate_rows"] > 0


def test_model_sets(mrlib):
    """getTopKMultiFiltered equals getTopKFiltered per entry, through both paths; the device variant is read with topk_multi_device_tensors."""
    ds = synth(**ITEMDS)
    rng = np.random.default_rng(2)
    with MusicRecommender(ds, **ITEM) as mr:
        for allowed, ex in filters(ds, rng).values():
            mr.setTopKFilter(allowed, ex)
            multi = mr.getTopKMultiFiltered(MODELS + [(_lib.MR_AGG, 0.25, 0)], 40)
            for (m, p, s), got in zip(MODELS + [(_lib.MR_AGG, 0.25, 0)], multi):
                assert_lists_equal(got, mr.getTopKFiltered(m, 40, p, s), f"model {m}")
            mr.topk_filtered_device(MODELS, 40)
            for i, got in enumerate(multi[:len(MODELS)]):
                assert_lists_equal(tuple(t.cpu().numpy() for t in mr.topk_multi_device_tensors(i, 40)), got)


def test_song_windows_and_user_shards(mrlib, oracle_lib):
    """Three song windows joined with mergeTopK, and two user shards with their pair bases, give the unwindowed filtered lists."""
    import torch
    ds = synth(T=800, U=61, S=3001, seed=5)
    rng = np.random.default_rng(5)
    dense = dense_models(oracle_lib, ds)
    for allowed, ex in filters(ds, rng).values():
        want = [topk_filtered_host(d, allowed, *ex, 40) for d in dense]
        parts = []
        for r in range(3):
            with MusicRecommender(ds, song_window=song_window(ds.S, r, 3), **ITEM) as mr:
                mr.setTopKFilter(allowed, ex)
                parts.append(mr.getTopKMultiFiltered(MODELS, 40))
        with MusicRecommender(ds, **ITEM) as mr:
            for e, w in enumerate(want):
                ps, pv, pl = (torch.from_numpy(np.stack([q[e][i] for q in parts])).cuda() for i in range(3))
                out = (torch.empty_like(ps[0]), torch.empty_like(pv[0]), torch.empty_like(pl[0]))
                mr.mergeTopK(ps, pv, pl, *out)
                mr.sync()
                assert_lists_equal(tuple(t.cpu().numpy() for t in out), w, f"windows, entry {e}")
            starts, n_total = pair_index_bases(ds, 2)
            got = []
            for r in range(2):
                u0, u1 = shard_range(ds.U, r, 2)
                mr.set_test_users(ds.shard_test_users(u0, u1), int(starts[r]), n_total)
                mr.setTopKFilter(allowed, shard_exclusions(*ex, u0, u1))
                got.append(mr.getTopKMultiFiltered(MODELS, 40))
            for e, w in enumerate(want):
                assert_lists_equal(tuple(np.concatenate([g[e][i] for g in got]) for i in range(3)), w, f"shards, entry {e}")


def test_distributed_one_process(mrlib, oracle_lib, tmp_path):
    """distributed.topk_filtered in a gloo world of one: a song-window handle goes through the exchange and the join, a whole handle
    through the shard rows."""
    import torch.distributed as dist
    from musicrecommendation_b200.distributed import topk_filtered
    ds = synth(**ITEMDS)
    rng = np.random.default_rng(8)
    allowed, ex = filters(ds, rng)["allow_1pct"]
    dense = dense_models(oracle_lib, ds)
    dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1)
    try:
        with MusicRecommender(ds, **ITEM) as mr:
            for (m, p, s), d, got in zip(MODELS, dense, topk_filtered(mr, MODELS, 30, allowed, ex)):
                assert_lists_equal(got, topk_filtered_host(d, allowed, *ex, 30), f"model {m}")
        lo, hi = 0, ds.S // 2
        with MusicRecommender(ds, song_window=(lo, hi), **ITEM) as mr:
            for (m, p, s), d, got in zip(MODELS, dense, topk_filtered(mr, MODELS, 30, allowed, ex)):
                sub = np.full_like(d, np.nan)
                sub[:, lo:hi] = d[:, lo:hi]
                assert_lists_equal(got, topk_filtered_host(sub, allowed, *ex, 30), f"window model {m}")
    finally:
        dist.destroy_process_group()


def edge_dataset():
    """SMALL with song 0 listened by every test user."""
    ds = synth(**SMALL)
    eu, es = np.repeat(np.arange(ds.U), np.diff(ds.te_ptr)), ds.te_col
    eu, es = np.concatenate([eu, np.arange(ds.U)]), np.concatenate([es, np.zeros(ds.U, es.dtype)])
    return from_triplets((np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr)), ds.tr_col), (eu, es),
                         (np.repeat(np.arange(ds.U), np.diff(ds.lab_ptr)), ds.lab_col), T=ds.T, U=ds.U, S=ds.S)


def test_edges(mrlib, oracle_lib):
    ds = edge_dataset()
    dense = dense_models(oracle_lib, ds)
    S, U = ds.S, ds.U
    rng = np.random.default_rng(3)
    with MusicRecommender(ds, **ITEM) as mr:
        small = np.array([7, 3, 7, 0, S - 2, 3, 1999, 11], np.int32)              # unordered, duplicates, a listened-by-all song
        cover = np.unique(small).astype(np.int32)
        ex_ptr = np.zeros(U + 1, np.int64)
        ex_ptr[1:] = len(cover)                                                    # user 0 excludes every allowed song, the rest nothing
        for allowed, ex in ((np.empty(0, np.int32), (None, None)), (np.zeros(3, np.int32), (None, None)), (small, (ex_ptr, cover)),
                            (rng.choice(S, S * 9 // 10, replace=False), random_exclusions(ds, rng, n=40, empty_every=2))):
            mr.setTopKFilter(allowed, None if ex[0] is None else ex)
            for (m, p, s), d in zip(MODELS, dense):
                for k in (1, 50, 1024):
                    got = mr.getTopKFiltered(m, k, p, s)
                    assert_lists_equal(got, topk_filtered_host(d, allowed, *ex, k), f"model {m} k {k} n_allow {len(allowed)}")
                    if len(allowed) <= len(small):
                        assert (got[2] <= len(cover) - 1).all()                    # song 0 is listened by everyone
                    if ex[1] is cover:
                        assert got[2][0] == 0 and (got[0][0] == -1).all() and (got[1][0] == 0.0).all()


def test_radix_ties_both_paths(mrlib, oracle_lib):
    """Test users whose one history is a song without train listeners: every score is 0.0, so each row is thousands of exact ties, more
    than the candidate buffer, and both paths (2 200 allowed songs, under 3 % of the catalogue; 90 %) refine the bin of the k-th key by the
    radix select.  Both give the mirror's lists."""
    base = synth(T=300, U=4, S=80000, seed=7)
    U, S = 400, base.S + 1
    ds = from_triplets((np.repeat(np.arange(base.T), np.diff(base.tr_ptr)), base.tr_col), (np.arange(U), np.full(U, S - 1)), ([], []),
                       T=base.T, U=U, S=S)
    rng = np.random.default_rng(9)
    dense = dense_models(oracle_lib, ds)
    with MusicRecommender(ds, **ITEM) as mr:
        for allowed, path in ((np.append(rng.choice(S, 2200, replace=False), S - 1), "filter_candidate_rows"),
                              (rng.choice(S, S * 9 // 10, replace=False), "filter_full_rows")):
            i0 = mr.info()
            mr.setTopKFilter(allowed, None)
            for (m, p, s), d in zip(MODELS, dense):
                assert_lists_equal(mr.getTopKFiltered(m, 300, p, s), topk_filtered_host(d, allowed, None, None, 300), f"model {m}")
            i1 = mr.info()
            assert i1[path] - i0[path] == len(MODELS) * U
            assert i1["topk_degenerate_rows"] - i0["topk_degenerate_rows"] == len(MODELS) * U


def test_guards(mrlib):
    ds = synth(**ITEMDS)
    U, S = ds.U, ds.S
    with MusicRecommender(ds, **ITEM) as mr:
        with pytest.raises(_lib.MrError) as e:
            mr.getTopKFiltered(_lib.MR_UBM, 10)
        assert e.value.code == _lib.MR_ERR_STATE
        with pytest.raises(_lib.MrError, match=r"allowed song -4 \(entry 2\)") as e:
            mr.setTopKFilter([1, 2, -4, S], None)
        assert e.value.code == _lib.MR_ERR_BAD_ARG
        ptr = np.arange(U + 1, dtype=np.int64) * 2
        col = np.tile(np.array([3, 9], np.int32), U)
        col[2 * 7: 2 * 7 + 2] = [9, 3]
        col[2 * 11] = S
        with pytest.raises(_lib.MrError, match="exclusions row 7 not ascending") as e:
            mr.setTopKFilter(None, (ptr, col))
        assert e.value.code == _lib.MR_ERR_BAD_ARG
        col[2 * 7: 2 * 7 + 2] = [3, 9]
        with pytest.raises(_lib.MrError, match=f"column id {S} out of range at row 11"):
            mr.setTopKFilter(None, (ptr, col))
        bad = ptr.copy()
        bad[5] = bad[6] + 1
        with pytest.raises(_lib.MrError, match="rowptr not monotone at row 5"):
            mr.setTopKFilter(None, (bad, col))
        assert mr._lib.mr_set_topk_filter(mr._h, None, -2, None, None) == _lib.MR_ERR_BAD_ARG
        assert mr._lib.mr_set_topk_filter(mr._h, None, 3, None, None) == _lib.MR_ERR_BAD_ARG
        mr.setTopKFilter([5], None)
        for k in (0, 1025):
            with pytest.raises(_lib.MrError) as e:
                mr.getTopKFiltered(_lib.MR_UBM, k)
            assert e.value.code == _lib.MR_ERR_BAD_ARG
        with pytest.raises(ParameterRange, match="entry 0: Percentage must be between 0 and 1"):
            mr.getTopKFiltered(_lib.MR_AGG, 10, 1.5)
        mr.clearTopKFilter()
        with pytest.raises(_lib.MrError) as e:
            mr.getTopKFiltered(_lib.MR_UBM, 10)
        assert e.value.code == _lib.MR_ERR_STATE
        mr.setTopKFilter([5], None)
        mr.set_test_users(ds)
        with pytest.raises(_lib.MrError) as e:
            mr.getTopKFiltered(_lib.MR_UBM, 10)
        assert e.value.code == _lib.MR_ERR_STATE
    train = from_triplets((np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr)), ds.tr_col), ([], []), ([], []), T=ds.T, U=0, S=ds.S)
    with MusicRecommender(train, **ITEM) as mr:                # no test users
        assert mr._lib.mr_set_topk_filter(mr._h, None, -1, None, None) == _lib.MR_ERR_STATE


def test_unfiltered_calls_ignore_the_filter(mrlib):
    """With a filter set, and right after a filtered call, every unfiltered call gives exactly its unfiltered output; the single-model
    result and its mAP survive a filtered call."""
    ds = synth(**ITEMDS)
    rng = np.random.default_rng(6)
    allowed, ex = filters(ds, rng)["allow_1pct"]
    songs = np.arange(0, ds.S, 7, dtype=np.int32)

    def outputs(mr):
        return dict(top=mr.getTopK(_lib.MR_LC, 40, 0.3), map=mr.mapAtK(40), multi=mr.getTopKMulti(MODELS, 30),
                    ev=mr.evaluateOnDevice(_lib.MR_UBM), evs=mr.evaluateOnDevice(_lib.MR_STOCH, 0.5, 42),
                    aud=mr.getSongAudience(_lib.MR_IBM, songs, 20))

    def same(a, b):
        assert_lists_equal(a["top"], b["top"])
        assert a["map"] == b["map"] and a["ev"] == b["ev"] and a["evs"] == b["evs"]
        for x, y in zip(a["multi"], b["multi"]):
            assert_lists_equal(x, y)
        assert_lists_equal(a["aud"], b["aud"])

    with MusicRecommender(ds, **ITEM) as mr:          # one batch: evaluateOnDevice takes the range -> counts resident reuse
        base = outputs(mr)
        mr.setTopKFilter(allowed, ex)
        same(outputs(mr), base)
        top = mr.getTopK(_lib.MR_IBM, 30)
        mr.getTopKFiltered(_lib.MR_UBM, 30)
        fetched = (np.empty((ds.U, 30), np.int32), np.empty((ds.U, 30)), np.empty(ds.U, np.int32))
        assert mr._lib.mr_topk_fetch(mr._h, 30, *[_p(a) for a in fetched]) == _lib.MR_OK
        assert_lists_equal(fetched, top)
        mr.getTopKFiltered(_lib.MR_STOCH, 30, 0.5, 42)
        same(outputs(mr), base)


@pytest.mark.parametrize("space", [_lib.MR_SPACE_USER, _lib.MR_SPACE_ITEM])
def test_profiled_calls(mrlib, oracle_lib, space):
    """Under MR_PROFILE (serial batches, a CUDA-event timer per phase) the filtered lists are the same and the select is timed as topk."""
    ds = synth(**ITEMDS)
    ubm = oracle_lib.canon_scores(ds, oracle_lib.UBM)
    rng = np.random.default_rng(7)
    with MusicRecommender(ds, engine=_lib.MR_ENGINE_SPARSE, space=space, profile=True) as mr:
        for allowed, ex in filters(ds, rng).values():
            mr.timing(reset=True)
            mr.setTopKFilter(allowed, ex)
            assert_lists_equal(mr.getTopKFiltered(_lib.MR_UBM, 50), topk_filtered_host(ubm, allowed, *ex, 50))
            assert mr.timing()["topk"] > 0
