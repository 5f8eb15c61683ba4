"""GPU parity tests (-m gpu): the CUDA path, called through the C-ABI (via the host mirror), against the oracle."""
import dataclasses
import json
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import fixture_4_3, synth, synth_config
from musicrecommendation_b200.recommender import MusicRecommender, ParameterRange, KeyMismatch, Model, evaluate_map

GOLD = Path(__file__).resolve().parent / "golden"
# count engine x scoring formulation: every combination must give the oracle's bits
ENGINES = [dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER), dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER),
           dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM), dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_ITEM)]
KINDS = {"ubm": _lib.MR_UBM, "ibm": _lib.MR_IBM}


def compact(a):
    return a[~np.isnan(a)]


def assert_bits_equal(a, b):
    """fp64 arrays identical bit for bit (NaN pattern included)."""
    a = np.ascontiguousarray(a, np.float64)
    b = np.ascontiguousarray(b, np.float64)
    np.testing.assert_array_equal(np.isnan(a), np.isnan(b))
    np.testing.assert_array_equal(np.where(np.isnan(a), 0, a).view(np.int64), np.where(np.isnan(b), 0, b).view(np.int64))


@pytest.fixture(scope="module", params=ENGINES, ids=["tensor-userspace", "sparse-userspace", "sparse-itemspace", "tensor-itemspace"])
def engine(request, mrlib):
    return request.param


def test_fixture_4_3(engine, oracle_lib):
    fx = json.loads((GOLD / "fixture_4_3.json").read_text())
    ds = fixture_4_3()
    with MusicRecommender(ds, **engine) as mr:
        assert mr.counts_ubm().tolist() == [fx["ubm_counts"]["X"], fx["ubm_counts"]["Y"]]
        g = mr.counts_ibm(0, 4)
        assert g[0, 1] == 1 and g[1, 2] == 1 and g[0, 2] == 0 and g[1, 1] == 2
        ubm, ibm = mr.getUserBasedModel(), mr.getItemBasedModel()
        assert [(u, s) for u, (s, _) in ubm.tuples()] == [tuple(p) for p in fx["pairs"]]
        np.testing.assert_allclose(ubm.compact(), fx["ubm"], rtol=1e-5, atol=0)      # tolerance named by north_star
        np.testing.assert_allclose(ibm.compact(), fx["ibm"], rtol=1e-5, atol=0)
        assert_bits_equal(ubm.scores, oracle_lib.canon_scores(ds, oracle_lib.UBM))
        assert_bits_equal(ibm.scores, oracle_lib.canon_scores(ds, oracle_lib.IBM))
        np.testing.assert_allclose(mr.getLinearCombinationModel(ubm, ibm, 0.5).compact(), fx["lc_0.5"], rtol=1e-5)
        np.testing.assert_allclose(mr.getAggregationModel(ubm, ibm, 0.5).compact(), fx["agg_0.5"], rtol=1e-5)
        for m in (ubm, ibm):
            assert round(mr.evaluateModel(m), 10) == fx["map_rounded"]
        names = ds.songs
        for key in ("ubm", "ibm"):
            song, score, ln = mr.getTopK(KINDS[key], k=2)
            assert ln.tolist() == [2, 2]
            assert [[names[s] for s in row] for row in song] == [fx["top2"][key]["X"], fx["top2"][key]["Y"]]


def check_dataset(ds, oracle_lib, engine, k=500, blends=True):
    with MusicRecommender(ds, **engine) as mr:
        # K1: intersection counts, bit-exact
        np.testing.assert_array_equal(mr.counts_ubm(), oracle_lib.counts_ubm(ds))
        rows = np.unique(np.concatenate([[0, ds.S - 1], np.random.default_rng(0).integers(0, ds.S, 30)])).astype(np.int32)
        s0 = int(rows[len(rows) // 2]); s1 = min(ds.S, s0 + 70)
        np.testing.assert_array_equal(mr.counts_ibm(s0, s1), oracle_lib.gram_rows(ds, np.arange(s0, s1)))
        # K2: scores — bit-identical to the canonical oracle, hence within 1e-5 of the as-written fp64 maths
        want = {"ubm": oracle_lib.canon_scores(ds, oracle_lib.UBM), "ibm": oracle_lib.canon_scores(ds, oracle_lib.IBM)}
        ubm, ibm = mr.getUserBasedModel(), mr.getItemBasedModel()
        assert_bits_equal(ubm.scores, want["ubm"])
        assert_bits_equal(ibm.scores, want["ibm"])
        assert len(ubm) == ds.n_pairs
        # K3: top-k, ranked ids bit-exact with ties broken by song id
        for key, kind in KINDS.items():
            song, score, ln = mr.getTopK(kind, k=k)
            ws, wv, wl = oracle_lib.topk(want[key], k)
            np.testing.assert_array_equal(ln, wl)
            np.testing.assert_array_equal(song, ws)
            assert_bits_equal(score, wv)
        if blends:
            for kind, okind, param, seed in ((_lib.MR_LC, oracle_lib.LC, 0.5, 0), (_lib.MR_LC, oracle_lib.LC, 0.3, 0),
                                             (_lib.MR_AGG, oracle_lib.AGG, 0.5, 0), (_lib.MR_AGG, oracle_lib.AGG, 0.37, 0),
                                             (_lib.MR_STOCH, oracle_lib.STOCH, 0.5, 42), (_lib.MR_STOCH, oracle_lib.STOCH, 0.8, 7)):
                wb = oracle_lib.blend_dense(okind, param, want["ubm"], want["ibm"], seed)
                song, score, ln = mr.getTopK(kind, k=k, param=param, seed=seed)
                ws, wv, wl = oracle_lib.topk(wb, k)
                np.testing.assert_array_equal(song, ws)
                assert_bits_equal(score, wv)
                # the materialised blend (MR:317-481) too
                if kind == _lib.MR_LC:
                    got = mr.getLinearCombinationModel(ubm, ibm, param)
                elif kind == _lib.MR_AGG:
                    got = mr.getAggregationModel(ubm, ibm, param)
                else:
                    got = mr.getStochasticCombinationModel(ubm, ibm, param, seed=seed)
                assert_bits_equal(got.scores, wb)
        # reference mAP on the GPU (MR:521-639): bit-identical to the CPU restatement, for both threshold lists
        for nt in (10, 11):
            assert mr.evaluateModel(ubm, n_thresholds=nt) == oracle_lib.evaluate(want["ubm"], ds, nt)
            assert mr.evaluateModel(ibm, n_thresholds=nt) == oracle_lib.evaluate(want["ibm"], ds, nt)
        return mr.info()


def test_golden_small_seed11(engine, oracle_lib):
    """The committed golden vectors (as-written restatement) against the CUDA path."""
    g = np.load(GOLD / "small_seed11.npz")
    ds = synth(T=40, U=6, S=500, seed=11)
    with MusicRecommender(ds, **engine) as mr:
        np.testing.assert_array_equal(mr.counts_ubm(), g["counts_ubm"])
        np.testing.assert_array_equal(mr.counts_ibm(0, 64), g["gram_0_64"])
        ubm, ibm = mr.getUserBasedModel(), mr.getItemBasedModel()
        for got, key in ((ubm, "ubm"), (ibm, "ibm")):
            assert_bits_equal(got.scores, g[f"canon_{key}"])
            m = ~np.isnan(g[f"naive_{key}"])
            np.testing.assert_allclose(got.scores[m], g[f"naive_{key}"][m], rtol=1e-5, atol=0)
        song, score, ln = mr.getTopK(_lib.MR_UBM, k=50)
        np.testing.assert_array_equal(song, g["top50_ubm_song"])
        assert_bits_equal(score, g["top50_ubm_score"])
        assert_bits_equal(mr.getStochasticCombinationModel(ubm, ibm, 0.5, seed=42).scores, g["stoch_seed42"])
        assert round(mr.evaluateModel(ubm), 10) == round(float(g["map_ubm"]), 10)


@pytest.mark.parametrize("T,U,S,seed", [(300, 20, 2000, 1), (64, 3, 130, 2), (1000, 130, 5000, 3), (257, 129, 1025, 4)])
def test_synthetic_parity(engine, oracle_lib, T, U, S, seed):
    check_dataset(synth(T=T, U=U, S=S, seed=seed), oracle_lib, engine, k=min(500, S))


def test_popular_songs_split_across_warps(engine, oracle_lib):
    """Songs with more than 4096 train listeners are aggregated by several warps with 64-bit integer atomics: still exact."""
    ds = synth(T=12000, U=200, S=30000, seed=6)
    assert np.bincount(ds.tr_col).max() > 4096
    info = check_dataset(ds, oracle_lib, engine, blends=False)
    if engine["space"] == _lib.MR_SPACE_ITEM:
        # pairs of very popular songs overflow the packed 16 / 32-bit head-row entries and live in the exact exception list
        assert info["head_exceptions"] > 0


def test_long_rows_take_the_sampled_topk_path(oracle_lib):
    """Rows longer than 65536 songs use the sampled-cut single-pass select; it must still equal the exact ranking."""
    ds = synth(T=3000, U=40, S=70000, seed=8)
    for cfg in (dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM), dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER)):
        check_dataset(ds, oracle_lib, cfg, blends=True)


def test_item_space_balanced_groups_and_batches(oracle_lib, monkeypatch):
    """More test users than head_rowsum work groups (148 SMs x 8): groups hold several segments, heavy users are split over groups
    and accumulate atomically, and a capped batch size makes the shard span several batches — all still the oracle's bits.
    Every row-load width of the head pass is covered."""
    ds = synth(T=2500, U=2700, S=3100, seed=12)
    want = {"ubm": oracle_lib.canon_scores(ds, oracle_lib.UBM), "ibm": oracle_lib.canon_scores(ds, oracle_lib.IBM)}
    for cap, words in (("", "4"), ("1000", "2"), ("128", "1")):
        if cap:
            monkeypatch.setenv("MRSCORE_ITEM_BATCH", cap)
        monkeypatch.setenv("MRSCORE_HEAD_WORDS_U", words)
        monkeypatch.setenv("MRSCORE_HEAD_WORDS_I", words)
        if words == "1":   # the two-atomics fallback of the head-row precompute (data sets whose sums could overflow the packed accumulator)
            monkeypatch.setenv("MRSCORE_PRECOMPUTE_UNPACKED", "1")
        with MusicRecommender(ds, engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM) as mr:
            info = mr.info()
            assert info["batch_rows"] == (ds.U if not cap else max(128, -(-ds.U // -(-ds.U // int(cap)))))
            assert info["split_users"] > 0
            assert_bits_equal(mr.getUserBasedModel().scores, want["ubm"])
            assert_bits_equal(mr.getItemBasedModel().scores, want["ibm"])
            for key, kind in KINDS.items():
                song, score, ln = mr.getTopK(kind, k=100)
                ws, wv, wl = oracle_lib.topk(want[key], 100)
                np.testing.assert_array_equal(song, ws)
                assert_bits_equal(score, wv)
            song, score, ln = mr.getTopK(_lib.MR_LC, k=100, param=0.25)
            ws, wv, wl = oracle_lib.topk(oracle_lib.blend_dense(oracle_lib.LC, 0.25, want["ubm"], want["ibm"], 0), 100)
            np.testing.assert_array_equal(song, ws)
            assert_bits_equal(score, wv)


def test_long_rows_with_grouped_head_pass(oracle_lib, monkeypatch):
    """Rows longer than 65536 songs (sampled-cut top-k: integer select for UBM, fp32-bounded collect for IBM, fp64 for the blends) on a
    shard whose head pass packs several users per work group and spans three batches."""
    monkeypatch.setenv("MRSCORE_HEAD_GROUPS", "48")
    monkeypatch.setenv("MRSCORE_ITEM_BATCH", "128")
    ds = synth(T=3000, U=300, S=70000, seed=21)
    want = {"ubm": oracle_lib.canon_scores(ds, oracle_lib.UBM), "ibm": oracle_lib.canon_scores(ds, oracle_lib.IBM)}
    with MusicRecommender(ds, engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM) as mr:
        info = mr.info()
        assert info["batch_rows"] == 128 and info["head_groups"] == 48
        for key, kind in KINDS.items():
            song, score, ln = mr.getTopK(kind, k=500)
            ws, wv, wl = oracle_lib.topk(want[key], 500)
            np.testing.assert_array_equal(ln, wl)
            np.testing.assert_array_equal(song, ws)
            assert_bits_equal(score, wv)
        for kind, okind, param, seed in ((_lib.MR_LC, oracle_lib.LC, 0.4, 0), (_lib.MR_AGG, oracle_lib.AGG, 0.5, 0), (_lib.MR_STOCH, oracle_lib.STOCH, 0.6, 9)):
            song, score, ln = mr.getTopK(kind, k=500, param=param, seed=seed)
            ws, wv, wl = oracle_lib.topk(oracle_lib.blend_dense(okind, param, want["ubm"], want["ibm"], seed), 500)
            np.testing.assert_array_equal(song, ws)
            assert_bits_equal(score, wv)


def test_config_c1(engine, oracle_lib):
    ds = synth_config("c1")
    info = check_dataset(ds, oracle_lib, engine)
    assert info["engine"] == engine["engine"] and info["space"] == engine["space"]


def test_config_c2_and_c3_topk(oracle_lib):
    """BASELINE.json configs[1] and configs[2] shapes on the default (auto) engine: rankings and blends bit-exact."""
    for name in ("c2", "c3"):
        ds = synth_config(name)
        info = check_dataset(ds, oracle_lib, dict(engine=_lib.MR_ENGINE_AUTO), blends=(name == "c3"))
        assert info["engine"] == _lib.MR_ENGINE_TENSOR and info["space"] == _lib.MR_SPACE_USER


def test_edge_cases(engine, oracle_lib):
    """Songs with no train listener still get 0.0 and are emitted; users overlapping nobody get all zeros; k > S - |I_u|;
    max degree users; U not a multiple of the 128-user batch."""
    rng = np.random.default_rng(5)
    T, U, S = 50, 5, 40
    tr = (np.repeat(np.arange(T), 3), rng.integers(0, 20, T * 3))          # songs 20..39 have no train listener
    te = (np.array([0, 0, 1, 2, 2, 2, 3, 4]), np.array([1, 2, 30, 5, 31, 39, 25, 0]))   # user 1 and 3 overlap nobody
    lab = (np.arange(U), np.array([3, 4, 5, 6, 7]))
    from musicrecommendation_b200.dataset import from_triplets
    ds = from_triplets(tr, te, lab, T, U, S)
    with MusicRecommender(ds, **engine) as mr:
        ubm = mr.getUserBasedModel()
        assert_bits_equal(ubm.scores, oracle_lib.canon_scores(ds, oracle_lib.UBM))
        assert np.all(compact(ubm.scores[1]) == 0.0) and np.all(compact(ubm.scores[3]) == 0.0)
        assert np.all(ubm.scores[0, 20:] == 0.0)
        for kind, m in ((_lib.MR_UBM, oracle_lib.UBM), (_lib.MR_IBM, oracle_lib.IBM)):
            song, score, ln = mr.getTopK(kind, k=64)
            ws, wv, wl = oracle_lib.topk(oracle_lib.canon_scores(ds, m), 64)
            np.testing.assert_array_equal(ln, wl)
            assert ln.tolist() == [S - 2, S - 1, S - 3, S - 1, S - 1]
            np.testing.assert_array_equal(song, ws)
            assert_bits_equal(score, wv)
        # an all-zero row ranks purely by song id
        song, _, _ = mr.getTopK(_lib.MR_UBM, k=10)
        assert song[1].tolist() == [s for s in range(11) if s != 30][:10]


def test_evaluate_degenerate_and_blends(mrlib, oracle_lib):
    ds = synth(T=300, U=20, S=2000, seed=1)
    with MusicRecommender(ds) as mr:
        ubm, ibm = mr.getUserBasedModel(), mr.getItemBasedModel()
        for got in (mr.getLinearCombinationModel(ubm, ibm, 0.5), mr.getAggregationModel(ubm, ibm, 0.5), mr.getStochasticCombinationModel(ubm, ibm, 0.5, seed=3)):
            assert mr.evaluateModel(got) == oracle_lib.evaluate(got.scores, ds)
            assert mr.evaluateModel(got) == pytest.approx(evaluate_map(got.scores, ds), abs=1e-15)
        flat = Model(np.where(ds.listened_mask(), np.nan, 0.25))          # max == min -> NaN comparisons -> no predictions -> mAP 0
        assert mr.evaluateModel(flat) == 0.0


def test_error_behaviour(mrlib, oracle_lib):
    ds = synth(T=64, U=3, S=130, seed=2)
    with MusicRecommender(ds) as mr:
        ubm, ibm = mr.getUserBasedModel(), mr.getItemBasedModel()
        for bad in (-0.1, 1.5):
            with pytest.raises(ParameterRange, match="Percentage must be between 0 and 1"):
                mr.getAggregationModel(ubm, ibm, bad)
            with pytest.raises(ParameterRange, match="Probability must be between 0 and 1"):
                mr.getStochasticCombinationModel(ubm, ibm, bad)
            with pytest.raises(ParameterRange):
                mr.getTopK(_lib.MR_AGG, k=10, param=bad)
        mr.getLinearCombinationModel(ubm, ibm, 1.5)                 # no range check on alpha (MR:317-330)
        shifted = Model(np.roll(ibm.scores, 1, axis=1))
        with pytest.raises(KeyMismatch):
            mr.getLinearCombinationModel(ubm, shifted, 0.5)
        with pytest.raises(_lib.MrError):
            mr.getTopK(_lib.MR_UBM, k=0)
        with pytest.raises(_lib.MrError):
            mr.counts_ibm(5, ds.S + 1)
    bad = synth(T=64, U=3, S=130, seed=2)
    bad.tr_col = bad.tr_col[::-1].copy()
    with pytest.raises(_lib.MrError, match="ascending"):
        MusicRecommender(bad)


def with_empty_test_user(ds):
    """ds with one more test user, last, whose visible row is empty (degree 0)."""
    return dataclasses.replace(ds, U=ds.U + 1, te_ptr=np.append(ds.te_ptr, ds.te_ptr[-1]), lab_ptr=np.append(ds.lab_ptr, ds.lab_ptr[-1]),
                               deg_te=np.append(ds.deg_te, 0).astype(np.int32))


def rs32(deg):
    """float(1 / sqrt(deg)) rounded from fp64, 0 for degree 0: the fp32 factor of the similarity products."""
    d = np.asarray(deg, np.float64)
    with np.errstate(divide="ignore"):
        return np.where(d > 0, 1.0 / np.sqrt(d), 0.0).astype(np.float32)


def check_probes(ds, oracle_lib, engine):
    """The parity probes: counts bit for bit; cosines user-user MR:140-149 and item-item MR:230-239 within 1e-5 of the fp64 formula and
    bit for bit float(c) * (rs(a) * rs(b)) in fp32."""
    with MusicRecommender(ds, **engine) as mr:
        c = oracle_lib.counts_ubm(ds)
        np.testing.assert_array_equal(mr.counts_ubm(), c)
        g = oracle_lib.gram_rows(ds, np.arange(100, 300))
        np.testing.assert_array_equal(mr.counts_ibm(100, 300), g)
        sim_u, sim_i = mr.similarity_ubm(), mr.similarity_ibm(100, 300)
        du, dv = ds.deg_te.astype(np.float64), ds.deg_tr.astype(np.float64)
        with np.errstate(invalid="ignore"):
            want = np.where(du[:, None] > 0, c / (np.sqrt(du)[:, None] * np.sqrt(dv)[None, :]), 0.0)
        np.testing.assert_allclose(sim_u, want, rtol=1e-5, atol=0)
        d = np.sqrt(ds.deg_song.astype(np.float64))
        np.testing.assert_allclose(sim_i, g / (d[100:300, None] * d[None, :]), rtol=1e-5, atol=0)
        exact_u = c.astype(np.float32) * (rs32(ds.deg_te)[:, None] * rs32(ds.deg_tr)[None, :])
        rd = rs32(ds.deg_song)
        exact_i = g.astype(np.float32) * (rd[100:300, None] * rd[None, :])
        np.testing.assert_array_equal(sim_u.view(np.int32), exact_u.view(np.int32))
        np.testing.assert_array_equal(sim_i.view(np.int32), exact_i.view(np.int32))


def test_similarity_products(engine, oracle_lib):
    check_probes(with_empty_test_user(synth(T=300, U=20, S=2000, seed=1)), oracle_lib, engine)


def test_probes_across_chunks(engine, oracle_lib, monkeypatch):
    """The same with chunks of 7 count rows (MRSCORE_SIM_CHUNK): every probe crosses chunk boundaries."""
    monkeypatch.setenv("MRSCORE_SIM_CHUNK", "7")
    check_probes(with_empty_test_user(synth(T=300, U=20, S=2000, seed=1)), oracle_lib, engine)


def test_shard_invariance(oracle_lib):
    """Test users sharded as distributed.scala:450-452 does: every shard reproduces its rows of the whole-model result,
    including the index-dependent Aggregation / Stochastic blends (global pair index, SURVEY A.4)."""
    ds = synth(T=400, U=37, S=3000, seed=9)
    with MusicRecommender(ds) as mr:
        full = {kind: mr.getTopK(kind, k=100, param=0.5, seed=11) for kind in (_lib.MR_UBM, _lib.MR_IBM, _lib.MR_AGG, _lib.MR_STOCH)}
        base = np.concatenate([[0], np.cumsum(ds.S - np.diff(ds.te_ptr))])
        for u0, u1 in ((0, 10), (10, 29), (29, 37)):
            mr.set_test_users(ds.shard_test_users(u0, u1), int(base[u0]), int(base[-1]))
            for kind, (fs, fv, fl) in full.items():
                s, v, l = mr.getTopK(kind, k=100, param=0.5, seed=11)
                np.testing.assert_array_equal(s, fs[u0:u1])
                assert_bits_equal(v, fv[u0:u1])
