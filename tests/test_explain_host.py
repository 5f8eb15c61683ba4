"""CPU tests of the explanation checker (explain_host, the numpy mirror of mr_explain): the known answers of the SURVEY §4.3 fixture,
brute force from the oracle's dense count rows, the exact numerator of the canonical restatement, the as-written scores rebuilt from the
terms bit for bit, and an explanation as the similar-users / similar-songs list of the pair's key filtered to the pair's contributors."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import fixture_4_3, synth
from musicrecommendation_b200.recommender import explain_host, similar_songs_host, similar_users_host

UBM, IBM = _lib.MR_UBM, _lib.MR_IBM


def golden():
    return synth(T=40, U=6, S=500, seed=11), np.load(ROOT / "tests" / "golden" / "small_seed11.npz")


def all_pairs(ds):
    u, s = np.meshgrid(np.arange(ds.U), np.arange(ds.S), indexing="ij")
    return u.ravel(), s.ravel()


def listened(ds, u, s):
    return s in np.asarray(ds.te_col)[ds.te_ptr[u]:ds.te_ptr[u + 1]]


def brute_explain(oracle, ds, model, users, songs, m):
    """Contributors from the dense count rows: oracle.counts_ubm (c(u, v)) or oracle.gram_rows (g(s, j)), terms and nums entry by entry."""
    tr_ptr, tr_col = np.asarray(ds.tr_ptr), np.asarray(ds.tr_col)
    cu = oracle.counts_ubm(ds) if model == UBM else None
    rows = []
    for u, s in zip(users, songs):
        if listened(ds, u, s):
            rows.append(None)
            continue
        if model == UBM:
            cand = [(v, int(cu[u, v])) for v in range(ds.T) if s in tr_col[tr_ptr[v]:tr_ptr[v + 1]] and cu[u, v] > 0]
            sq_k, sq_o, q = np.sqrt(float(ds.deg_te[u])), lambda v: np.sqrt(float(ds.deg_tr[v])), lambda v: oracle.q(ds.deg_tr[v], oracle.UBM)
        else:
            g = oracle.gram_rows(ds, [s])[0]
            iu = np.asarray(ds.te_col)[ds.te_ptr[u]:ds.te_ptr[u + 1]]
            cand = [(int(j), int(g[j])) for j in iu if g[j] > 0]
            sq_k, sq_o, q = np.sqrt(float(ds.deg_song[s])), lambda j: np.sqrt(float(ds.deg_song[j])), lambda j: oracle.q(ds.deg_song[j], oracle.IBM)
        ent = [(i, c / (sq_k * sq_o(i)), c * q(i)) for i, c in cand]
        rows.append((sorted(ent, key=lambda e: (-e[1], e[0])), sum(e[2] for e in ent)))
    return rows


def assert_rows(got, brute, m):
    for r, want in enumerate(brute):
        if want is None:
            assert np.isnan(got.score[r]) and got.len[r] == 0 and got.count[r] == 0 and got.total[r] == 0
            assert (got.id[r] == -1).all()
            continue
        ent, total = want
        k = min(m, len(ent))
        assert (got.len[r], got.count[r], got.total[r]) == (k, len(ent), total)
        assert list(got.id[r, :k]) == [e[0] for e in ent[:k]] and (got.id[r, k:] == -1).all()
        assert [float(t).hex() for t in got.term[r, :k]] == [float(e[1]).hex() for e in ent[:k]] and (got.term[r, k:] == 0).all()
        assert list(got.num[r, :k]) == [e[2] for e in ent[:k]] and (got.num[r, k:] == 0).all()


def test_fixture_known_answers():
    ds = fixture_4_3()
    X, Y, A, B = 0, 1, 0, 1
    s1, s2, s3 = 0, 1, 2
    e = explain_host(ds, UBM, [X, Y, X], [s2, s3, s1], 3)
    assert e.len[0] == 1 and e.id[0, 0] == A and e.term[0, 0] == 0.4999999999999999
    assert e.len[1] == 1 and e.id[1, 0] == B and e.term[1, 0] == 0.7071067811865475
    assert np.isnan(e.score[2]) and e.len[2] == 0 and e.count[2] == 0 and e.total[2] == 0 and (e.id[2] == -1).all()
    e = explain_host(ds, IBM, [X, Y], [s2, s2], 3)
    assert e.len[0] == 1 and e.id[0, 0] == s1 and e.term[0, 0] == 0.40824829046386296
    assert np.isnan(e.score[1]) and e.len[1] == 0
    e = explain_host(ds, UBM, [X], [s3], 3)            # s3's train listeners B and C share no song with X: no contributor, score 0.0
    assert e.len[0] == 0 and e.count[0] == 0 and e.score[0] == 0.0 and not np.signbit(e.score[0])


@pytest.mark.parametrize("model", [UBM, IBM])
@pytest.mark.parametrize("shape,m", [(dict(T=60, U=10, S=200, seed=2), 4), (dict(T=120, U=15, S=300, seed=1), 1000)])
def test_host_mirror_equals_brute_force(oracle_lib, model, shape, m):
    ds = synth(**shape)
    rng = np.random.default_rng(shape["seed"])
    users = rng.integers(0, ds.U, 60)
    songs = rng.integers(0, ds.S, 60)
    users = np.concatenate([users, [0, 0]])
    songs = np.concatenate([songs, [ds.te_col[ds.te_ptr[0]], ds.S - 1]])      # a listened pair
    got = explain_host(ds, model, users, songs, m)
    assert_rows(got, brute_explain(oracle_lib, ds, model, users, songs, m), m)
    assert (got.count > 0).sum() >= 10


@pytest.mark.parametrize("model", [UBM, IBM])
def test_total_is_the_canonical_numerator(oracle_lib, model):
    ds, z = golden()
    u, s = all_pairs(ds)
    sint = z["sint_ubm" if model == UBM else "sint_ibm"]
    np.testing.assert_array_equal(sint, oracle_lib.canon_sint(ds, oracle_lib.UBM if model == UBM else oracle_lib.IBM))
    canon = z["canon_ubm" if model == UBM else "canon_ibm"]
    e = explain_host(ds, model, u, s, 5)
    open_ = ~np.isnan(canon.ravel())
    assert open_.sum() > 0 and (e.count[open_] > 0).sum() > 100
    np.testing.assert_array_equal(e.total[open_], sint.ravel()[open_])
    np.testing.assert_array_equal(e.score[open_].view(np.int64), canon.ravel()[open_].view(np.int64))
    assert np.isnan(e.score[~open_]).all() and (e.len[~open_] == 0).all()


@pytest.mark.parametrize("model", [UBM, IBM])
@pytest.mark.parametrize("case", ["golden_seed11", "fixture_4_3"])
def test_terms_in_id_order_sum_to_the_as_written_score(oracle_lib, model, case):
    if case == "golden_seed11":
        ds, z = golden()
        want = z["naive_ubm" if model == UBM else "naive_ibm"]
    else:
        ds = fixture_4_3()
        want = oracle_lib.naive_scores(ds, oracle_lib.UBM if model == UBM else oracle_lib.IBM)
    u, s = all_pairs(ds)
    m = max(ds.T, ds.S)
    e = explain_host(ds, model, u, s, m)
    assert (e.len == e.count).all()
    got = np.zeros(len(u))
    for r in range(len(u)):
        k = e.len[r]
        order = np.argsort(e.id[r, :k], kind="stable")
        acc = 0.0
        for t in e.term[r, :k][order]:
            acc += t
        got[r] = acc
    open_ = ~np.isnan(want.ravel())
    np.testing.assert_array_equal(got[open_].view(np.int64), want.ravel()[open_].view(np.int64))


def test_explanation_is_the_filtered_neighbour_list():
    ds = synth(T=120, U=15, S=300, seed=4)
    tr_ptr, tr_col, te_ptr, te_col = np.asarray(ds.tr_ptr), np.asarray(ds.tr_col), np.asarray(ds.te_ptr), np.asarray(ds.te_col)
    rng = np.random.default_rng(4)
    users, songs = rng.integers(0, ds.U, 80), rng.integers(0, ds.S, 80)
    nu = similar_users_host(ds, np.arange(ds.U), ds.T)
    ns = similar_songs_host(ds, np.arange(ds.S), ds.S)
    for model in (UBM, IBM):
        e = explain_host(ds, model, users, songs, ds.T)
        for r, (u, s) in enumerate(zip(users, songs)):
            if listened(ds, u, s):
                continue
            if model == UBM:     # similar users of u whose train row holds s
                ids, w, n = nu[0][u], nu[1][u], nu[2][u]
                keep = [i for i in range(n) if s in tr_col[tr_ptr[ids[i]]:tr_ptr[ids[i] + 1]]]
            else:                # similar songs of s that u listened to
                ids, w, n = ns[0][s], ns[1][s], ns[2][s]
                keep = [i for i in range(n) if ids[i] in te_col[te_ptr[u]:te_ptr[u + 1]]]
            k = e.len[r]
            assert k == len(keep)
            assert list(e.id[r, :k]) == [ids[i] for i in keep]
            np.testing.assert_array_equal(e.term[r, :k].view(np.int64), w[keep].view(np.int64))
