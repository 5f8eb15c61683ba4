"""CPU tests of the streamed evaluateModel's host half (mr_eval_cutoffs, mr_eval_finish, the numpy count mirror) and of
distributed.evaluate_reference_map on two gloo ranks, with the oracle standing in for the GPU handles."""
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
from musicrecommendation_b200.distributed import evaluate_reference_map, shard_range, song_window
from musicrecommendation_b200.recommender import eval_counts_host, eval_cutoffs, eval_finish

TH = [0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0]


def _f(x, mn, mx):
    with np.errstate(all="ignore"):
        return (np.float64(x) - np.float64(mn)) / (np.float64(mx) - np.float64(mn))


def _check_cutoffs(mn, mx, rng):
    for n in (10, 11):
        cut = eval_cutoffs(mn, mx, n)
        assert np.all(cut[1:] >= cut[:-1])
        for t in range(n):
            c = cut[t]
            if np.isinf(c):
                assert not (_f(mx, mn, mx) > TH[t])
                continue
            assert mn < c <= mx
            assert _f(c, mn, mx) > TH[t]                                   # the prediction flips exactly at c_t
            assert not (_f(np.nextafter(c, -np.inf), mn, mx) > TH[t])
            # brute force over random doubles of [mn, mx], and over the bit patterns next to c_t
            xs = np.concatenate([mn + (mx - mn) * rng.random(2000), [mn, mx],
                                 (np.float64(c).view(np.int64) + np.arange(-8, 9)).view(np.float64)])
            xs = xs[(xs >= mn) & (xs <= mx)]
            np.testing.assert_array_equal(xs >= c, _f(xs, mn, mx) > TH[t])


@pytest.mark.parametrize("mn,mx", [(0.0, 1.0), (0.0, 0.37), (2.5e-7, 3.1e-2), (1.0, 1.0), (0.0, 0.0),
                                   (1.0, float(np.nextafter(1.0, 2.0))), (0.0, 5e-324), (0.0, 7 * 5e-324), (3e-320, 9e-318),
                                   (1e-300, 1e300), (0.0, 1e308), (4.0, 4.000000000000001)])
def test_cutoffs_adversarial(mn, mx, mrlib):
    _check_cutoffs(mn, mx, np.random.default_rng(0))


def test_cutoffs_random(mrlib):
    rng = np.random.default_rng(7)
    for _ in range(40):
        a, b = np.sort(rng.random(2) * 10.0 ** rng.integers(-12, 6))
        _check_cutoffs(float(a), float(b), rng)
    cut = eval_cutoffs(np.inf, -np.inf, 10)                    # a part that emits nothing: no prediction anywhere
    assert np.all(np.isinf(cut))


def _cases(oracle_lib):
    ds = synth(T=40, U=6, S=500, seed=11)
    g = np.load(ROOT / "tests" / "golden" / "small_seed11.npz")
    u, i = g["canon_ubm"], g["canon_ibm"]
    yield "seed11_ubm", ds, u
    yield "seed11_ibm", ds, i
    yield "seed11_lc", ds, oracle_lib.blend_dense(oracle_lib.LC, 0.3, u, i)
    yield "seed11_stoch", ds, oracle_lib.blend_dense(oracle_lib.STOCH, 0.5, u, i, seed=42)
    fx = fixture_4_3()
    yield "fixture_ubm", fx, oracle_lib.naive_scores(fx, oracle_lib.UBM)
    yield "fixture_ibm", fx, oracle_lib.naive_scores(fx, oracle_lib.IBM)


def _range(scores):
    v = scores[~np.isnan(scores)]
    return (float(v.min()), float(v.max())) if len(v) else (np.inf, -np.inf)


@pytest.mark.parametrize("n_thr", [10, 11])
def test_finish_of_host_counts_equals_oracle(oracle_lib, mrlib, n_thr):
    for name, ds, scores in _cases(oracle_lib):
        new = np.unique(ds.lab_col)
        mn, mx = _range(scores)
        got = eval_finish(*eval_counts_host(scores, ds, 0, mn, mx, n_thr, new), n_thr)
        assert got == oracle_lib.evaluate(scores, ds, n_thr), name


def test_host_counts_add_over_partitions(oracle_lib, mrlib):
    """3 song windows x 2 user shards: the summed counts are the whole model's, so the mAP keeps its bits."""
    for name, ds, scores in _cases(oracle_lib):
        new = np.unique(ds.lab_col)
        mn, mx = _range(scores)
        whole = eval_counts_host(scores, ds, 0, mn, mx, 10, new)
        tot = [np.zeros_like(a) for a in whole]
        for r in range(2):
            u0, u1 = shard_range(ds.U, r, 2)
            sh = ds.shard_test_users(u0, u1)
            for w in range(3):
                lo, hi = song_window(ds.S, w, 3)
                for acc, part in zip(tot, eval_counts_host(scores[u0:u1, lo:hi], sh, lo, mn, mx, 10, new)):
                    acc += part
        for a, b in zip(tot, whole):
            np.testing.assert_array_equal(a, b, err_msg=name)
        assert eval_finish(*tot, 10) == oracle_lib.evaluate(scores, ds, 10)


def test_finish_rejects_inconsistent_counts(mrlib):
    from musicrecommendation_b200 import _lib
    pred = np.zeros((1, 10), np.int64); tp = np.ones((1, 10), np.int64); nlab = np.ones(1, np.int64)
    with pytest.raises(_lib.MrError):
        eval_finish(pred, tp, nlab, 10)        # more true positives than predictions
    with pytest.raises(ValueError):
        eval_finish(np.zeros((1, 9), np.int64), np.zeros((1, 9), np.int64), nlab, 10)


class OracleHandle:
    """Numpy stand-in for a MusicRecommender handle that scores the users of `shard` against the songs [lo, hi)."""

    def __init__(self, full_scores, shard, u0, u1, lo, hi):
        self.ds = shard
        self.scores = full_scores[u0:u1, lo:hi]
        self.lo = lo

    def eval_range(self, model, param, seed):
        return _range(self.scores)

    def eval_counts(self, model, mn, mx, new_songs, param, seed, n_thresholds, labels):
        return eval_counts_host(self.scores, labels, self.lo, mn, mx, n_thresholds, new_songs)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import oracle
    ds = synth(T=120, U=11, S=700, seed=33)
    ubm = oracle.canon_scores(ds, oracle.UBM)
    res = []
    for n_thr in (10, 11):
        # user shards: each rank holds only its own users' labels, the label-song union is gathered
        u0, u1 = shard_range(ds.U, rank, world)
        sh = ds.shard_test_users(u0, u1)
        res.append(evaluate_reference_map(OracleHandle(ubm, sh, u0, u1, 0, ds.S), 0, 0.5, 0, n_thr))
        # song partitions: every rank scores all users against its window
        lo, hi = song_window(ds.S, rank, world)
        res.append(evaluate_reference_map(OracleHandle(ubm, ds, 0, ds.U, lo, hi), 0, 0.5, 0, n_thr))
    np.save(os.path.join(out_dir, f"map_rank{rank}.npy"), np.array(res))
    dist.barrier()
    dist.destroy_process_group()


def test_reference_map_two_gloo_ranks(tmp_path, oracle_lib, mrlib):
    world = 2
    mp.start_processes(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True, start_method="spawn")
    ds = synth(T=120, U=11, S=700, seed=33)
    ubm = oracle_lib.canon_scores(ds, oracle_lib.UBM)
    want = [oracle_lib.evaluate(ubm, ds, 10)] * 2 + [oracle_lib.evaluate(ubm, ds, 11)] * 2
    assert want[0] > 0
    for r in range(world):
        assert np.load(tmp_path / f"map_rank{r}.npy").tolist() == want
