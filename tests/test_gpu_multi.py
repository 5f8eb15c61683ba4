"""GPU tests (-m gpu) of model sets (mr_topk_multi*, mr_eval_range_multi / mr_eval_counts_multi, DESIGN.md §4.6): every entry's outputs
have the bits of the single-model call, the shard is scored once per batch whatever the set's size, and partitions still sum up."""
import ctypes as C
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import synth, synth_config
from musicrecommendation_b200.distributed import pair_index_bases, shard_range, song_window
from musicrecommendation_b200.recommender import MusicRecommender, ParameterRange, _p, eval_finish, model_set_arrays

ROOT = Path(__file__).resolve().parent.parent
ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
SET = [(_lib.MR_UBM, 0.5, 0), (_lib.MR_IBM, 0.5, 0), (_lib.MR_LC, 0.3, 0), (_lib.MR_AGG, 0.5, 0), (_lib.MR_STOCH, 0.5, 42),
       (_lib.MR_LC, 0.0, 0), (_lib.MR_LC, 1.0, 0), (_lib.MR_STOCH, 0.5, 7)]
SMALL = dict(T=300, U=40, S=2000, seed=3)
ITEMDS = dict(T=800, U=300, S=3001, seed=5)


def bits(x) -> str:
    return float(x).hex()


def dense_set(oracle, ds, specs):
    ubm, ibm = oracle.canon_scores(ds, oracle.UBM), oracle.canon_scores(ds, oracle.IBM)
    kinds = {_lib.MR_LC: oracle.LC, _lib.MR_AGG: oracle.AGG, _lib.MR_STOCH: oracle.STOCH}
    return [ubm if m == _lib.MR_UBM else ibm if m == _lib.MR_IBM else oracle.blend_dense(kinds[m], p, ubm, ibm, seed=s) for m, p, s in specs]


def check_set(mr, ds, specs, oracle=None, k=50, n_thr=10):
    """Every output of the set calls against the single-model calls, entry by entry (and against the oracle's dense models)."""
    multi_top = mr.getTopKMulti(specs, k)
    for (m, p, s), got in zip(specs, multi_top):
        want = mr.getTopK(m, k, p, s)
        np.testing.assert_array_equal(got[2], want[2])
        np.testing.assert_array_equal(got[0], want[0])
        np.testing.assert_array_equal(got[1].view(np.int64), want[1].view(np.int64))
    mn, mx = mr.eval_range_multi(specs)
    new = np.unique(ds.lab_col)
    pred, tp, nlab = mr.eval_counts_multi(specs, mn, mx, new, n_thr)
    maps = mr.evaluateAllOnDevice(specs, n_thr)
    models = dense_set(oracle, ds, specs) if oracle is not None else None
    for i, (m, p, s) in enumerate(specs):
        a, b = mr.eval_range(m, p, s)
        assert (bits(mn[i]), bits(mx[i])) == (bits(a), bits(b)), i
        c = mr.eval_counts(m, a, b, new, p, s, n_thr)
        np.testing.assert_array_equal(pred[i], c[0])
        np.testing.assert_array_equal(tp[i], c[1])
        np.testing.assert_array_equal(nlab, c[2])
        single = mr.evaluateOnDevice(m, p, s, n_thr)
        assert bits(maps[i]) == bits(single) == bits(eval_finish(pred[i], tp[i], nlab, n_thr)), i
        if models is not None:
            assert bits(single) == bits(oracle.evaluate(models[i], ds, n_thr)), i


@pytest.mark.parametrize("cfg", ["tensor_user", "sparse_user", "item_one_batch", "item_batches", "item_batches_serial", "head_exceptions", "c3"])
def test_set_equals_single_calls(mrlib, oracle_lib, monkeypatch, cfg):
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
    with MusicRecommender(ds, **kw) as mr:
        if cfg.startswith("item_batches"):
            assert mr.info()["batch_rows"] == 128
        check_set(mr, ds, SET, oracle_lib, n_thr=11 if cfg == "c3" else 10)
        if cfg == "head_exceptions":
            assert mr.info()["head_exceptions"] > 0


@pytest.mark.parametrize("cfg", ["user", "item_batches", "item_one_batch"])
def test_one_scoring_per_batch(mrlib, cfg):
    ds = synth(**ITEMDS)
    kw = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER) if cfg == "user" else dict(ITEM, item_batch=128 if cfg == "item_batches" else 0)
    new = np.unique(ds.lab_col)
    with MusicRecommender(ds, **kw) as mr:
        rows = 128 if cfg != "item_one_batch" else mr.info()["batch_rows"]
        n_batches = -(-ds.U // rows)
        assert n_batches == (1 if cfg == "item_one_batch" else 3)
        for specs in (SET[:1], SET[:5], SET, SET * 2):
            p0 = mr.info()["scoring_passes"]
            mr.getTopKMulti(specs, 20)
            assert mr.info()["scoring_passes"] - p0 == n_batches
            mn, mx = mr.eval_range_multi(specs)
            assert mr.info()["scoring_passes"] - p0 == 2 * n_batches
            mr.eval_counts_multi(specs, mn, mx, new)
            # a single-batch item-space shard keeps its panels from the range pass: one scoring for both
            assert mr.info()["scoring_passes"] - p0 == (2 if cfg == "item_one_batch" else 3) * n_batches
        p0 = mr.info()["scoring_passes"]
        mn, mx = mr.eval_range_multi(SET)
        mr.eval_counts_multi(SET[::-1], mn[::-1], mx[::-1], new)         # another set: scored again
        assert mr.info()["scoring_passes"] - p0 == 2 * n_batches


def test_partition_invariance(mrlib, oracle_lib):
    """3 song windows x 2 user shards: per entry the summed counts and the combined min / max are the whole model's; the song partitions'
    top-k lists from mr_topk_multi_ptrs joined by mr_topk_merge equal the whole-model lists."""
    import torch
    ds = synth(T=800, U=61, S=3001, seed=5)
    specs, k, n_win = SET, 40, 3
    models = dense_set(oracle_lib, ds, specs)
    new = np.unique(ds.lab_col)
    starts, n_total = pair_index_bases(ds, 2)
    shards = [ds.shard_test_users(*shard_range(ds.U, r, 2)) for r in range(2)]
    with MusicRecommender(ds, **ITEM) as whole:
        want_top = whole.getTopKMulti(specs, k)
    rngs, tot, parts = [], None, [[] for _ in specs]
    for sweep in ("range", "counts"):
        if sweep == "counts":
            mn = np.min([a for a, _ in rngs], axis=0)
            mx = np.max([b for _, b in rngs], axis=0)
        for w in range(n_win):
            with MusicRecommender(ds, song_window=song_window(ds.S, w, n_win), **ITEM) as mr:
                if sweep == "range":
                    mr.topk_multi_device(specs, k)
                    mr.sync()
                    for i in range(len(specs)):
                        parts[i].append([t.clone() for t in mr.topk_multi_device_tensors(i, k)])
                for r, sh in enumerate(shards):
                    mr.set_test_users(sh, int(starts[r]), n_total)
                    if sweep == "range":
                        rngs.append(mr.eval_range_multi(specs))
                    else:
                        c = mr.eval_counts_multi(specs, mn, mx, new)
                        tot = list(c) if tot is None else [a + b for a, b in zip(tot, c)]
    for i, sc in enumerate(models):
        assert (mn[i], mx[i]) == (np.nanmin(sc), np.nanmax(sc)), i
        assert bits(eval_finish(tot[0][i], tot[1][i], tot[2], 10)) == bits(oracle_lib.evaluate(sc, ds, 10)), i
    with MusicRecommender(ds, **ITEM) as merger:
        for i in range(len(specs)):
            ps = torch.stack([p[0] for p in parts[i]]); pv = torch.stack([p[1] for p in parts[i]]); pl = torch.stack([p[2] for p in parts[i]])
            out = (torch.empty_like(ps[0]), torch.empty_like(pv[0]), torch.empty_like(pl[0]))
            merger.mergeTopK(ps, pv, pl, *out)
            merger.sync()
            np.testing.assert_array_equal(out[2].cpu().numpy(), want_top[i][2])
            np.testing.assert_array_equal(out[0].cpu().numpy(), want_top[i][0])
            np.testing.assert_array_equal(out[1].cpu().numpy().view(np.int64), want_top[i][1].view(np.int64))


def test_state_separation(mrlib):
    """A device-resident single-model top-k, its device pointers and mapAtK(top=None) survive the set calls."""
    import torch
    ds = synth(**ITEMDS)
    with MusicRecommender(ds, **ITEM) as mr:
        mr._check(mr._lib.mr_topk_device(mr._h, _lib.MR_AGG, 0.5, C.c_uint64(0), 50))
        before = mr.mapAtK(50, top=None)
        song, score, ln = [t.clone() for t in mr.topk_device_tensors(50)]
        mr.getTopKMulti(SET, 50)
        mr.topk_multi_device(SET, 30)
        mr.evaluateAllOnDevice(SET)
        assert mr.mapAtK(50, top=None) == before
        s2, v2, l2 = mr.topk_device_tensors(50)
        assert torch.equal(s2, song) and torch.equal(v2.view(torch.int64), score.view(torch.int64)) and torch.equal(l2, ln)
        host = np.empty((ds.U, 50), np.int32), np.empty((ds.U, 50), np.float64), np.empty(ds.U, np.int32)
        mr._check(mr._lib.mr_topk_fetch(mr._h, 50, _p(host[0]), _p(host[1]), _p(host[2])))
        np.testing.assert_array_equal(host[0], song.cpu().numpy())
        with pytest.raises(_lib.MrError) as e:                           # the set result is at k = 30
            mr.topk_multi_device_tensors(0, 50)
        assert e.value.code == _lib.MR_ERR_STATE
        with pytest.raises(_lib.MrError) as e:
            mr.topk_multi_device_tensors(len(SET), 30)
        assert e.value.code == _lib.MR_ERR_BAD_ARG


def test_guards(mrlib):
    ds = synth(**SMALL)
    new = np.unique(ds.lab_col)
    lib = mrlib
    with MusicRecommender(ds, **ITEM) as mr:
        h = mr._h
        for bad in ((_lib.MR_LC, 1.5, 0), (_lib.MR_LC, float("nan"), 0), (_lib.MR_LC, -0.5, 0), (_lib.MR_AGG, 1.5, 0), (_lib.MR_STOCH, -0.1, 0)):
            specs = [SET[0], SET[3], bad, (bad[0], 2.0, 0)]
            for call in (lambda: mr.getTopKMulti(specs, 10), lambda: mr.eval_range_multi(specs),
                         lambda: mr.eval_counts_multi(specs, [0.0] * 4, [1.0] * 4, new)):
                p0 = mr.info()["scoring_passes"]
                with pytest.raises(ParameterRange, match="^entry 2: "):
                    call()
                assert mr.info()["scoring_passes"] == p0
        m, p, s = model_set_arrays(SET)
        mn, mx = np.zeros(len(SET)), np.ones(len(SET))
        out = np.zeros(len(SET) * len(new) * 11, np.int64)

        def code(rc):
            assert rc == _lib.MR_ERR_BAD_ARG, rc
            return lib.mr_last_error(h).decode()
        for n in (0, 17):
            assert "n_models" in code(lib.mr_topk_multi_device(h, n, _p(m), _p(p), _p(s), 10))
            assert "n_models" in code(lib.mr_eval_range_multi(h, n, _p(m), _p(p), _p(s), _p(mn), _p(mx)))
            assert "n_models" in code(lib.mr_eval_counts_multi(h, n, _p(m), _p(p), _p(s), _p(mn), _p(mx), 10, _p(ds.lab_ptr), _p(ds.lab_col),
                                                               _p(new), len(new), _p(out), _p(out), _p(out)))
        code(lib.mr_topk_multi_device(h, len(SET), None, _p(p), _p(s), 10))
        code(lib.mr_eval_range_multi(h, len(SET), _p(m), None, _p(s), _p(mn), _p(mx)))
        for k in (0, 1025):
            assert "k must be" in code(lib.mr_topk_multi_device(h, len(SET), _p(m), _p(p), _p(s), k))
        for nth in (9, 12):
            assert "n_thresholds" in code(lib.mr_eval_counts_multi(h, len(SET), _p(m), _p(p), _p(s), _p(mn), _p(mx), nth, _p(ds.lab_ptr),
                                                                   _p(ds.lab_col), _p(new), len(new), _p(out), _p(out), _p(out)))
        bad_m = m.copy(); bad_m[5] = 9
        assert code(lib.mr_eval_range_multi(h, len(SET), _p(bad_m), _p(p), _p(s), _p(mn), _p(mx))).startswith("entry 5: unknown model")
        neg = mn.copy(); neg[3] = -1.0
        assert code(lib.mr_eval_counts_multi(h, len(SET), _p(m), _p(p), _p(s), _p(neg), _p(mx), 10, _p(ds.lab_ptr), _p(ds.lab_col), _p(new),
                                             len(new), _p(out), _p(out), _p(out))).startswith("entry 3: mn must be")
        missing = int(new[len(new) // 2])
        with pytest.raises(_lib.MrError, match=f"lacks label song {missing}") as e:
            mr.eval_counts_multi(SET, mn, mx, new[new != missing])
        assert e.value.code == _lib.MR_ERR_BAD_ARG
        null = (C.c_void_p * 2)(None, None)
        assert "null output" in code(lib.mr_topk_multi(h, 2, _p(m), _p(p), _p(s), 10, null, null, null))
        starts, n_total = pair_index_bases(ds, 2)
        mr.set_test_users(ds.shard_test_users(*shard_range(ds.U, 1, 2)), int(starts[1]), n_total)
        with pytest.raises(ValueError):                                  # a shard's own mAP is not the model's
            mr.evaluateAllOnDevice(SET)
    with MusicRecommender(ds, song_window=(0, 1000), **ITEM) as mr:
        with pytest.raises(ValueError):
            mr.evaluateAllOnDevice(SET)


def test_result_blocks_beyond_the_reserve(mrlib):
    """The set's top-k blocks must fit in the caller's 6 GB reserve: 16 x 40 000 users x k = 1024 x 12 B = 7.9 GB is MR_ERR_OOM stating the
    bytes, and leaves the handle usable; 8 entries (3.9 GB) run."""
    ds = synth(T=300, U=40000, S=1100, seed=8)
    specs = [(_lib.MR_LC, i / 15, 0) for i in range(16)]
    with MusicRecommender(ds, **ITEM) as mr:
        with pytest.raises(_lib.MrError, match=f"need {16 * 40000 * 1024 * 12 + 16 * 160000} bytes") as e:
            mr.topk_multi_device(specs, 1024)
        assert e.value.code == _lib.MR_ERR_OOM
        mr.topk_multi_device(specs[:8], 1024)
        mr.sync()
        song, score, ln = mr.topk_multi_device_tensors(7, 1024)
        want = mr.getTopK(_lib.MR_LC, 1024, 7 / 15, 0)
        np.testing.assert_array_equal(song.cpu().numpy(), want[0])
        np.testing.assert_array_equal(ln.cpu().numpy(), want[2])


def test_msd_shape(mrlib):
    """configs[3] (MSD) shape, a 2 560-user shard, default engine: one batch and 640-user batches, the set results equal the per-model calls."""
    ds = synth_config("c4").shard_test_users(0, 2560)
    specs = SET[:5] + [(_lib.MR_LC, a, 0) for a in (0.1, 0.9)]
    res = None
    for kw in ({}, dict(item_batch=640)):
        with MusicRecommender(ds, **kw) as mr:
            if kw:
                assert mr.info()["batch_rows"] == 640
            check_set(mr, ds, specs, None, k=100)
            maps = mr.evaluateAllOnDevice(specs)
            if res is None:
                res = maps
            assert [bits(x) for x in maps] == [bits(x) for x in res]


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_reference_map_multi_two_ranks_under_torchrun(mrlib):
    """distributed.evaluate_reference_map_multi over two song partitions on two GPUs (NCCL) equals the single-process set mAPs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port",
           str(_free_port()), str(ROOT / "tools" / "multi_bench.py"), "--mode", "dist", "--config", "c3", "--reps", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, OMP_NUM_THREADS="4"))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["check_equal_single_process"] is True
