"""CPU tests of the song-audience host code (DESIGN.md §4.10): the numpy mirror song_audience_host against a brute-force ranking, and the
user-shard exchange and join of distributed.song_audience over a gloo world of 2, with the oracle standing in for the GPU."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200.dataset import fixture_4_3, synth
from musicrecommendation_b200.distributed import audience_shard_parts, shard_range
from musicrecommendation_b200.recommender import song_audience_host


def brute_force(scores, songs, k):
    """Per song: every user with a non-NaN score, as (score, user) pairs sorted by hand with a Python comparison."""
    out = []
    for s in songs:
        cand = [(float(scores[u, s]), u) for u in range(scores.shape[0]) if not np.isnan(scores[u, s])]
        cand.sort(key=lambda t: (-t[0], t[1]))
        out.append(cand[:k])
    return out


def check_against_brute_force(scores, songs, k):
    user, score, ln = song_audience_host(scores, songs, k)
    want = brute_force(scores, songs, k)
    for r, w in enumerate(want):
        assert ln[r] == len(w)
        assert list(user[r, :ln[r]]) == [u for _, u in w]
        np.testing.assert_array_equal(score[r, :ln[r]].view(np.int64), np.array([x for x, _ in w], np.float64).view(np.int64))
        assert (user[r, ln[r]:] == -1).all() and (score[r, ln[r]:] == 0.0).all()
    return user, score, ln


@pytest.mark.parametrize("case", ["golden_seed11", "fixture_4_3"])
def test_mirror_equals_brute_force(oracle_lib, case):
    if case == "golden_seed11":
        g = np.load(ROOT / "tests" / "golden" / "small_seed11.npz")
        models = [g["canon_ubm"], g["canon_ibm"], g["lc"], g["agg"], g["stoch_seed42"]]
    else:
        ds = fixture_4_3()
        models = [oracle_lib.canon_scores(ds, oracle_lib.UBM), oracle_lib.canon_scores(ds, oracle_lib.IBM)]
    for sc in models:
        S = sc.shape[1]
        songs = list(range(S)) + [S - 1, 0, S // 2]                       # every song, then duplicates out of order
        for k in (1, 3, sc.shape[0] + 2):                                  # k past the candidates
            check_against_brute_force(sc, songs, k)


def test_mirror_ties_and_listened_pairs():
    sc = np.array([[0.5, np.nan, 0.0], [0.5, 0.25, 0.0], [0.75, np.nan, np.nan], [0.5, np.nan, 0.0]])
    user, score, ln = check_against_brute_force(sc, [0, 1, 2], 4)
    assert list(ln) == [4, 1, 3]
    assert list(user[0]) == [2, 0, 1, 3]                                   # ties in user order
    assert list(user[1]) == [1, -1, -1, -1]                                # listened pairs (NaN) are no candidates
    assert list(user[2, :3]) == [0, 1, 3] and (score[2, :3] == 0.0).all()  # zero scores are candidates


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _join(parts_user, parts_score, parts_len, k):
    """Checker for the join of the parts (on the GPU: mr_topk_merge)."""
    P, n, _ = parts_user.shape
    user = np.full((n, k), -1, np.int32); score = np.zeros((n, k)); ln = np.zeros(n, np.int32)
    for r in range(n):
        cand = sorted((-float(parts_score[p, r, i]), int(parts_user[p, r, i])) for p in range(P) for i in range(int(parts_len[p, r])))
        ln[r] = min(k, len(cand))
        for i, (neg, u) in enumerate(cand[:k]):
            user[r, i], score[r, i] = u, -neg
    return user, score, ln


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import oracle
    ds = synth(T=120, U=11, S=700, seed=33)
    u0, u1 = shard_range(ds.U, rank, world)
    shard = ds.shard_test_users(u0, u1)
    songs = np.r_[0:ds.S:7, 3, 3, 699].astype(np.int32)
    for name, model in (("ubm", oracle.UBM), ("ibm", oracle.IBM)):
        user, score, ln = song_audience_host(oracle.canon_scores(shard, model), songs, 4)   # the shard's lists, shard-local user ids
        ps, pv, pl = audience_shard_parts(user, score, ln, shard.meta["shard"][0], world, rank)
        np.savez(os.path.join(out_dir, f"{name}_rank{rank}.npz"), **dict(zip(("user", "score", "len"), _join(ps.numpy(), pv.numpy(), pl.numpy(), 4))))
    dist.barrier()
    dist.destroy_process_group()


def test_two_process_user_shard_join(tmp_path, oracle_lib):
    world = 2
    mp.start_processes(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True, start_method="spawn")
    ds = synth(T=120, U=11, S=700, seed=33)
    songs = np.r_[0:ds.S:7, 3, 3, 699].astype(np.int32)
    for name, model in (("ubm", oracle_lib.UBM), ("ibm", oracle_lib.IBM)):
        want = song_audience_host(oracle_lib.canon_scores(ds, model), songs, 4)
        assert want[2].min() == 4                                      # every list is full: the join had to choose across the shards
        for r in range(world):
            r0, r1 = shard_range(len(songs), r, world)
            got = np.load(tmp_path / f"{name}_rank{r}.npz")
            np.testing.assert_array_equal(got["user"], want[0][r0:r1])
            np.testing.assert_array_equal(got["score"].view(np.int64), want[1][r0:r1].view(np.int64))
            np.testing.assert_array_equal(got["len"], want[2][r0:r1])
