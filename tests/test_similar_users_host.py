"""CPU tests of the similar-users checker (similar_users_host, the numpy mirror of mr_similar_users): brute force from the oracle's dense
test x train count rows, the reference's user-based model rebuilt from the neighbour lists bit for bit, and the operation order of the
cosine on the SURVEY §4.3 fixture."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200.dataset import Dataset, fixture_4_3, from_triplets, synth
from musicrecommendation_b200.recommender import similar_users_host


def brute_similar_users(oracle, ds, users, k):
    """Ranked train neighbours from the dense count rows c(u, :) = |I_u ∩ I_v| (oracle.counts_ubm)."""
    users = np.asarray(users, np.int64)
    C = oracle.counts_ubm(ds)
    deg_tr = np.asarray(ds.deg_tr, np.int64)
    deg_te = np.asarray(ds.deg_te, np.int64)
    out_user = np.full((len(users), k), -1, np.int32)
    out_score = np.zeros((len(users), k), np.float64)
    out_len = np.zeros(len(users), np.int32)
    for r, u in enumerate(users):
        v = np.flatnonzero(C[u] > 0)
        w = []
        for j in v:
            den = np.sqrt(float(deg_te[u])) * np.sqrt(float(deg_tr[j]))
            w.append(float(C[u, j]) / den if den != 0 else 0.0)
        order = sorted(range(len(v)), key=lambda t: (-w[t], v[t]))[:k]
        out_user[r, :len(order)] = v[order]
        out_score[r, :len(order)] = np.asarray(w, np.float64)[order] if order else []
        out_len[r] = len(order)
    return out_user, out_score, out_len


def assert_same(got, want):
    np.testing.assert_array_equal(got[2], want[2])
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1].view(np.int64), want[1].view(np.int64))


def with_empty_rows(ds, rows):
    """ds with the visible test rows of `rows` emptied (degrees follow the rows, as the reference's .length)."""
    te_ptr = np.asarray(ds.te_ptr, np.int64)
    keep = np.ones(len(ds.te_col), bool)
    for u in rows:
        keep[te_ptr[u]:te_ptr[u + 1]] = False
    lens = np.diff(te_ptr)
    lens[list(rows)] = 0
    return Dataset(ds.T, ds.U, ds.S, ds.tr_ptr, ds.tr_col, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64),
                   np.asarray(ds.te_col)[keep], ds.lab_ptr, ds.lab_col, ds.deg_tr, lens.astype(np.int32), ds.deg_song)


@pytest.mark.parametrize("shape,k", [(dict(T=120, U=15, S=300, seed=1), 7), (dict(T=300, U=40, S=2000, seed=3), 50),
                                     (dict(T=50, U=30, S=900, seed=9), 1000)])
def test_host_mirror_equals_brute_force(oracle_lib, shape, k):
    ds = with_empty_rows(synth(**shape), [0, 5])
    rng = np.random.default_rng(shape["seed"])
    users = np.concatenate([rng.integers(0, ds.U, 40), [0, ds.U - 1, 5, 0]])
    got = similar_users_host(ds, users, k)
    assert_same(got, brute_similar_users(oracle_lib, ds, users, k))
    assert got[2][-1] == 0 and got[2][-2] == 0 and (got[0][-1] == -1).all()   # empty visible rows list nobody


def test_ties_order_by_train_id():
    # train users 0..5 share the one song of test user 0 and all have degree 2: six equal weights, listed by ascending id
    tr = ([v for v in range(6) for _ in range(2)], [s for v in range(6) for s in (0, 1 + v)])
    ds = from_triplets(tr, ([0], [0]), ([], []), T=6, U=1, S=7)
    user, score, ln = similar_users_host(ds, [0], 4)
    assert ln[0] == 4 and list(user[0]) == [0, 1, 2, 3]
    assert len(set(score[0].tolist())) == 1 and score[0, 0] == 1.0 / (np.sqrt(1.0) * np.sqrt(2.0))


def _ubm_from_neighbours(ds, k_all):
    """UBM(u, s) = sum over the listed neighbours v with s in I_v of w(u, v), added in ascending train id (naive_ubm_rank's order)."""
    user, score, ln = similar_users_host(ds, np.arange(ds.U), k_all)
    tr_ptr = np.asarray(ds.tr_ptr, np.int64)
    tr_col = np.asarray(ds.tr_col)
    out = np.zeros((ds.U, ds.S), np.float64)
    for u in range(ds.U):
        m = ln[u]
        order = np.argsort(user[u, :m], kind="stable")
        for v, w in zip(user[u, :m][order], score[u, :m][order]):
            for s in tr_col[tr_ptr[v]:tr_ptr[v + 1]]:
                out[u, s] += w
    return out


@pytest.mark.parametrize("case", ["golden_seed11", "fixture_4_3"])
def test_neighbour_lists_rebuild_the_user_based_model(oracle_lib, case):
    if case == "golden_seed11":
        ds = synth(T=40, U=6, S=500, seed=11)
        want = np.load(ROOT / "tests" / "golden" / "small_seed11.npz")["naive_ubm"]
    else:
        ds = fixture_4_3()
        want = oracle_lib.naive_scores(ds, oracle_lib.UBM)
    got = _ubm_from_neighbours(ds, max(ds.T, 1))
    unlistened = ~np.isnan(want)
    assert unlistened.sum() > 0
    np.testing.assert_array_equal(got[unlistened].view(np.int64), want[unlistened].view(np.int64))


def test_fixture_operation_order():
    # test user 0 (2 visible songs) and train user 0 (2 songs) share one song: 1 / (sqrt(2) * sqrt(2)), not 1 / 2
    ds = fixture_4_3()
    user, score, ln = similar_users_host(ds, [0, 1], 3)
    assert list(ln) == [1, 2]
    assert user[0, 0] == 0 and score[0, 0] == 0.4999999999999999 == 1.0 / (np.sqrt(2.0) * np.sqrt(2.0))
    assert list(user[1, :2]) == [0, 1] and score[1, 0] == score[1, 1]           # equal scores: the lower id first
