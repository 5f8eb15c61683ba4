"""CPU tests of the similar-songs checker (similar_songs_host, the numpy mirror of mr_similar_songs): brute force from the dense train
co-occurrence rows of the oracle, the SURVEY §4.3 fixture as known answers, and the operation order of the cosine."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200.dataset import fixture_4_3, from_triplets, synth
from musicrecommendation_b200.recommender import similar_songs_host


def brute_similar(oracle, ds, songs, k):
    """Ranked co-listened songs from the dense count rows g(i, :) = |U_i ∩ U_s| over train users (oracle.gram_rows)."""
    songs = np.asarray(songs, np.int32)
    G = oracle.gram_rows(ds, songs)
    deg = np.asarray(ds.deg_song, np.int64)
    out_song = np.full((len(songs), k), -1, np.int32)
    out_score = np.zeros((len(songs), k), np.float64)
    out_len = np.zeros(len(songs), np.int32)
    for r, i in enumerate(songs):
        s = np.flatnonzero(G[r] > 0)
        s = s[s != i]
        sim = np.array([float(G[r, j]) / (np.sqrt(float(deg[i])) * np.sqrt(float(deg[j]))) for j in s], np.float64)
        order = sorted(range(len(s)), key=lambda t: (-sim[t], s[t]))[:k]
        out_song[r, :len(order)] = s[order]
        out_score[r, :len(order)] = sim[order]
        out_len[r] = len(order)
    return out_song, out_score, out_len


def assert_same(got, want):
    np.testing.assert_array_equal(got[2], want[2])
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1].view(np.int64), want[1].view(np.int64))


@pytest.mark.parametrize("shape,k", [(dict(T=120, U=15, S=300, seed=1), 7), (dict(T=300, U=40, S=2000, seed=3), 50),
                                     (dict(T=50, U=30, S=900, seed=9), 1000)])
def test_host_mirror_equals_brute_force(oracle_lib, shape, k):
    ds = synth(**shape)
    rng = np.random.default_rng(shape["seed"])
    songs = np.concatenate([rng.integers(0, ds.S, 60), np.argsort(-np.asarray(ds.deg_song))[:10], [0, ds.S - 1, 0]])
    assert_same(similar_songs_host(ds, songs, k), brute_similar(oracle_lib, ds, songs, k))


def test_fixture_known_answers():
    ds = fixture_4_3()
    s1, s2, s3, s4 = 0, 1, 2, 3
    song, score, ln = similar_songs_host(ds, [s1, s2, s3, s4], 3)
    assert list(ln) == [1, 2, 1, 0]
    assert list(song[0]) == [s2, -1, -1] and score[0, 0] == 0.40824829046386296
    assert list(song[1]) == [s1, s3, -1] and score[1, 0] == score[1, 1]       # equal scores: the lower id first
    assert list(song[2]) == [s2, -1, -1]
    assert list(song[3]) == [-1, -1, -1] and not score[3].any()               # s4 has no train listeners


def test_operation_order_of_the_cosine():
    # songs a, b: one shared train listener, two listeners each (train + test-visible): 1 / (sqrt(2) * sqrt(2)), not 1 / 2
    ds = from_triplets(([0, 0], [0, 1]), ([0, 1], [0, 1]), ([], []), T=1, U=2, S=2)
    assert list(ds.deg_song) == [2, 2]
    song, score, ln = similar_songs_host(ds, [0, 1], 2)
    assert list(ln) == [1, 1] and song[0, 0] == 1 and song[1, 0] == 0
    assert score[0, 0] == 0.4999999999999999 == 1.0 / (np.sqrt(2.0) * np.sqrt(2.0))
