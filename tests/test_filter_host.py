"""CPU tests of the filtered top-k host code (DESIGN.md §4.11): the numpy mirror topk_filtered_host against a brute-force ranking,
exclusions_from_topk (paging), and shard_exclusions, the host step of distributed.topk_filtered under test-user sharding."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200.dataset import fixture_4_3
from musicrecommendation_b200.distributed import shard_exclusions
from musicrecommendation_b200.recommender import exclusions_from_topk, topk_filtered_host


def brute_force(scores, allowed, ex_ptr, ex_col, k):
    """Per user: every allowed, unexcluded song with a non-NaN score, as (score, song) pairs sorted by hand with a Python comparison."""
    U, S = scores.shape
    allow = set(range(S)) if allowed is None else {int(s) for s in allowed}
    out = []
    for u in range(U):
        ex = set() if ex_ptr is None else {int(s) for s in ex_col[ex_ptr[u]:ex_ptr[u + 1]]}
        cand = [(float(scores[u, s]), s) for s in range(S) if s in allow and s not in ex and not np.isnan(scores[u, s])]
        cand.sort(key=lambda t: (-t[0], t[1]))
        out.append(cand[:k])
    return out


def check(scores, allowed, ex_ptr, ex_col, k):
    song, score, ln = topk_filtered_host(scores, allowed, ex_ptr, ex_col, k)
    for u, w in enumerate(brute_force(scores, allowed, ex_ptr, ex_col, k)):
        assert ln[u] == len(w)
        assert list(song[u, :ln[u]]) == [s for _, s in w]
        np.testing.assert_array_equal(score[u, :ln[u]].view(np.int64), np.array([x for x, _ in w], np.float64).view(np.int64))
        assert (song[u, ln[u]:] == -1).all() and (score[u, ln[u]:] == 0.0).all()
    return song, score, ln


def csr(rows):
    ptr = np.zeros(len(rows) + 1, np.int64)
    ptr[1:] = np.cumsum([len(r) for r in rows])
    return ptr, np.concatenate([np.asarray(r, np.int32) for r in rows] + [np.empty(0, np.int32)])


@pytest.mark.parametrize("case", ["golden_seed11", "fixture_4_3"])
def test_mirror_equals_brute_force(oracle_lib, case):
    if case == "golden_seed11":
        g = np.load(ROOT / "tests" / "golden" / "small_seed11.npz")
        models = [g["canon_ubm"], g["canon_ibm"], g["lc"], g["agg"], g["stoch_seed42"]]
    else:
        ds = fixture_4_3()
        models = [oracle_lib.canon_scores(ds, oracle_lib.UBM), oracle_lib.canon_scores(ds, oracle_lib.IBM)]
    rng = np.random.default_rng(0)
    for sc in models:
        U, S = sc.shape
        ex = csr([np.unique(rng.choice(S, min(S, 3), replace=False)) if u % 3 else [] for u in range(U)])
        allowed = [S - 1, 0, S // 2, 0, S - 1]                               # unordered, with duplicates
        for a, e in ((None, (None, None)), (allowed, (None, None)), (None, ex), (allowed, ex), ([], ex)):
            for k in (1, 3, S + 2):                                            # k past the candidates
                check(sc, a, *e, k)


def test_mirror_ties_and_listened_pairs():
    sc = np.array([[0.5, np.nan, 0.0, 0.5], [0.5, 0.25, 0.0, 0.0], [np.nan, np.nan, np.nan, 0.75]])
    song, score, ln = check(sc, [0, 2, 3, 1], *csr([[3], [], [3]]), 4)
    assert list(ln) == [2, 4, 0]
    assert list(song[0, :2]) == [0, 2] and list(song[1]) == [0, 1, 2, 3]


def test_exclusions_from_topk_pages():
    """The exclusion rows of a page hold its listed songs ascending; excluding them leaves the next page of the unfiltered ranking."""
    rng = np.random.default_rng(1)
    sc = rng.integers(0, 5, size=(6, 30)).astype(np.float64) / 4         # many ties
    sc[rng.random(sc.shape) < 0.3] = np.nan
    sc[5] = np.nan                                                       # a user with no candidate
    full = topk_filtered_host(sc, None, None, None, 20)
    first = topk_filtered_host(sc, None, None, None, 10)
    ptr, col = exclusions_from_topk(first[0], first[2])
    assert list(np.diff(ptr)) == list(first[2])
    for u in range(sc.shape[0]):
        row = col[ptr[u]:ptr[u + 1]]
        assert list(row) == sorted(first[0][u, :first[2][u]])
    song, score, ln = topk_filtered_host(sc, None, ptr, col, 10)
    np.testing.assert_array_equal(song, full[0][:, 10:])
    np.testing.assert_array_equal(score, full[1][:, 10:])
    np.testing.assert_array_equal(ln, np.maximum(full[2] - 10, 0))


def test_shard_exclusions():
    ptr, col = csr([[1, 4], [], [0, 2, 3], [5], []])
    sp, sc = shard_exclusions(ptr, col, 2, 4)
    assert list(sp) == [0, 3, 4] and list(sc) == [0, 2, 3, 5] and sc.dtype == np.int32
    sp, sc = shard_exclusions(ptr, col, 4, 5)
    assert list(sp) == [0, 0] and len(sc) == 0
