"""CPU tests of the model-set evaluation's host half: distributed.evaluate_reference_map_multi on two gloo ranks, with the oracle standing in
for the GPU handles, equals evaluate_reference_map per entry; and the Python checks of a model set's shape."""
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

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import synth
from musicrecommendation_b200.distributed import evaluate_reference_map, evaluate_reference_map_multi, shard_range, song_window
from musicrecommendation_b200.recommender import eval_counts_host, model_set_arrays

SPECS = [(_lib.MR_UBM, 0.5, 0), (_lib.MR_IBM, 0.5, 0), (_lib.MR_LC, 0.3, 0), (_lib.MR_AGG, 0.5, 0), (_lib.MR_STOCH, 0.5, 42),
         (_lib.MR_LC, 0.0, 0), (_lib.MR_LC, 1.0, 0), (_lib.MR_STOCH, 0.5, 7)]


def _range(scores):
    v = scores[~np.isnan(scores)]
    return (float(v.min()), float(v.max())) if len(v) else (np.inf, -np.inf)


def dense_set(oracle, ds, specs):
    """The dense model of every entry, as the oracle computes it."""
    ubm, ibm = oracle.canon_scores(ds, oracle.UBM), oracle.canon_scores(ds, oracle.IBM)
    out = []
    for model, param, seed in specs:
        if model == _lib.MR_UBM:
            out.append(ubm)
        elif model == _lib.MR_IBM:
            out.append(ibm)
        else:
            kind = {_lib.MR_LC: oracle.LC, _lib.MR_AGG: oracle.AGG, _lib.MR_STOCH: oracle.STOCH}[model]
            out.append(oracle.blend_dense(kind, param, ubm, ibm, seed=seed))
    return out


class OracleSetHandle:
    """Numpy stand-in for a MusicRecommender handle scoring a model set for the users of `shard` against the songs [lo, hi)."""

    def __init__(self, models, specs, shard, u0, u1, lo, hi):
        self.ds = shard
        self.specs = list(specs)
        self.scores = [m[u0:u1, lo:hi] for m in models]
        self.lo = lo

    def _entry(self, model, param, seed):
        return self.scores[self.specs.index((model, param, seed))]

    def eval_range(self, model, param, seed):
        return _range(self._entry(model, param, seed))

    def eval_counts(self, model, mn, mx, new_songs, param, seed, n_thresholds, labels):
        return eval_counts_host(self._entry(model, param, seed), labels, self.lo, mn, mx, n_thresholds, new_songs)

    def eval_range_multi(self, specs):
        assert list(specs) == self.specs
        r = [_range(s) for s in self.scores]
        return np.array([a for a, _ in r]), np.array([b for _, b in r])

    def eval_counts_multi(self, specs, mn, mx, new_songs, n_thresholds, labels):
        assert list(specs) == self.specs
        c = [eval_counts_host(s, labels, self.lo, a, b, n_thresholds, new_songs) for s, a, b in zip(self.scores, mn, mx)]
        return np.stack([x[0] for x in c]), np.stack([x[1] for x in c]), c[0][2]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import oracle
    ds = synth(T=120, U=11, S=700, seed=33)
    models = dense_set(oracle, ds, SPECS)
    multi, single = [], []
    for n_thr in (10, 11):
        u0, u1 = shard_range(ds.U, rank, world)       # user shards: each rank holds its own users' labels
        sh = ds.shard_test_users(u0, u1)
        lo, hi = song_window(ds.S, rank, world)        # song partitions: every rank scores all users against its window
        for h in (OracleSetHandle(models, SPECS, sh, u0, u1, 0, ds.S), OracleSetHandle(models, SPECS, ds, 0, ds.U, lo, hi)):
            multi.append(evaluate_reference_map_multi(h, SPECS, n_thr))
            single.append([evaluate_reference_map(h, m, p, s, n_thr) for m, p, s in SPECS])
    np.save(os.path.join(out_dir, f"multi_rank{rank}.npy"), np.array(multi))
    np.save(os.path.join(out_dir, f"single_rank{rank}.npy"), np.array(single))
    dist.barrier()
    dist.destroy_process_group()


def test_reference_map_multi_two_gloo_ranks(tmp_path, oracle_lib, mrlib):
    world = 2
    mp.start_processes(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True, start_method="spawn")
    ds = synth(T=120, U=11, S=700, seed=33)
    models = dense_set(oracle_lib, ds, SPECS)
    want = [[oracle_lib.evaluate(m, ds, n) for m in models] for n in (10, 10, 11, 11)]
    assert all(w > 0 for w in want[0])
    for r in range(world):
        multi, single = np.load(tmp_path / f"multi_rank{r}.npy"), np.load(tmp_path / f"single_rank{r}.npy")
        assert [[float(x).hex() for x in row] for row in multi] == [[float(x).hex() for x in row] for row in single]
        assert multi.tolist() == want


def test_model_set_arrays():
    models, params, seeds = model_set_arrays(SPECS)
    assert models.dtype == np.int32 and params.dtype == np.float64 and seeds.dtype == np.uint64
    assert models.tolist() == [m for m, _, _ in SPECS] and seeds.tolist() == [s for _, _, s in SPECS]
    assert model_set_arrays([(_lib.MR_STOCH, 0.5, -1)])[2][0] == 2**64 - 1       # seeds are taken modulo 2^64, as in getTopK
    assert len(model_set_arrays([(_lib.MR_UBM, 0.5, 0)] * 16)[0]) == 16          # duplicates are allowed
    for bad in ([], [(_lib.MR_UBM, 0.5, 0)] * 17):
        with pytest.raises(ValueError, match="1..16 entries"):
            model_set_arrays(bad)
    with pytest.raises(ValueError, match="entry 1: expected"):
        model_set_arrays([(_lib.MR_UBM, 0.5, 0), (_lib.MR_LC, 0.5)])
    with pytest.raises(ValueError, match="entry 2: unknown model selector"):
        model_set_arrays([(_lib.MR_UBM, 0.5, 0), (_lib.MR_IBM, 0.5, 0), (7, 0.5, 0)])
