"""GPU tests (-m gpu) of the streamed evaluateModel (mr_eval_range / mr_eval_counts / mr_eval_finish, DESIGN.md §4.5): the reference's
threshold-sweep mAP without a materialised model has the same bits as mr_evaluate_dense on the materialised one and as the oracle, on
every engine, space, batch plan, user sharding and song partitioning."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import Dataset, from_triplets, synth, synth_config
from musicrecommendation_b200.distributed import pair_index_bases, shard_range, song_window
from musicrecommendation_b200.recommender import Model, MusicRecommender, ParameterRange, eval_counts_host, eval_finish

ROOT = Path(__file__).resolve().parent.parent
ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
KINDS = ((_lib.MR_UBM, "ubm", 0.5, 0), (_lib.MR_IBM, "ibm", 0.5, 0), (_lib.MR_LC, "lc", 0.3, 0), (_lib.MR_AGG, "agg", 0.5, 0),
         (_lib.MR_STOCH, "stoch", 0.5, 42))


def dense_models(oracle_lib, ds):
    ubm, ibm = oracle_lib.canon_scores(ds, oracle_lib.UBM), oracle_lib.canon_scores(ds, oracle_lib.IBM)
    return {"ubm": ubm, "ibm": ibm, "lc": oracle_lib.blend_dense(oracle_lib.LC, 0.3, ubm, ibm),
            "agg": oracle_lib.blend_dense(oracle_lib.AGG, 0.5, ubm, ibm), "stoch": oracle_lib.blend_dense(oracle_lib.STOCH, 0.5, ubm, ibm, seed=42)}


def bits(x: float) -> str:
    return float(x).hex()


def check_models(mr, oracle_lib, ds, models, n_thrs=(10, 11)):
    for kind, name, param, seed in KINDS:
        for n in n_thrs:
            got = mr.evaluateOnDevice(kind, param, seed, n)
            dense = mr.evaluateModel(Model(models[name]), n_thresholds=n)           # mr_evaluate_dense on the materialised model
            assert bits(got) == bits(dense) == bits(oracle_lib.evaluate(models[name], ds, n)), (name, n)


SMALL = dict(T=300, U=40, S=2000, seed=3)
ITEMDS = dict(T=800, U=300, S=3001, seed=5)


@pytest.mark.parametrize("cfg", ["tensor_user", "sparse_user", "item_one_batch", "item_batches", "item_batches_serial", "head_exceptions", "c3"])
def test_on_device_equals_materialised(mrlib, oracle_lib, monkeypatch, cfg):
    kw, ds = {}, None
    if cfg == "tensor_user":
        ds, kw = synth(**SMALL), dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER)
    elif cfg == "sparse_user":
        ds, kw = synth(**SMALL), dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER)
    elif cfg == "item_one_batch":
        ds, kw = synth(**ITEMDS), ITEM
    elif cfg in ("item_batches", "item_batches_serial"):
        if cfg.endswith("serial"):
            monkeypatch.setenv("MRSCORE_NO_PIPELINE", "1")
        ds, kw = synth(**ITEMDS), dict(ITEM, item_batch=128)
    elif cfg == "head_exceptions":
        ds, kw = synth(T=12000, U=1040, S=30000, seed=6), dict(ITEM, head_min_deg=8)
    else:
        ds = synth_config("c3")
    models = dense_models(oracle_lib, ds)
    with MusicRecommender(ds, **kw) as mr:
        if cfg.startswith("item_batches"):
            assert mr.info()["batch_rows"] == 128 and mr.info()["space"] == _lib.MR_SPACE_ITEM
        check_models(mr, oracle_lib, ds, models)
        if cfg == "head_exceptions":
            assert mr.info()["head_exceptions"] > 0


def test_per_song_ap_equals_oracle(mrlib, oracle_lib):
    """out_ap of mr_eval_finish: the AP of each label song equals the oracle's mAP over that song alone (same global min / max)."""
    ds = synth(**ITEMDS)
    ibm = oracle_lib.canon_scores(ds, oracle_lib.IBM)
    with MusicRecommender(ds, **ITEM) as mr:
        mn, mx = mr.eval_range(_lib.MR_IBM)
        new = np.unique(ds.lab_col)
        m, ap = eval_finish(*mr.eval_counts(_lib.MR_IBM, mn, mx, new), 10, per_song=True)
    assert bits(m) == bits(oracle_lib.evaluate(ibm, ds, 10))
    rows = np.repeat(np.arange(ds.U), np.diff(ds.lab_ptr))
    for j in np.linspace(0, len(new) - 1, 40).astype(int):
        keep = ds.lab_col == new[j]
        one = Dataset(ds.T, ds.U, ds.S, ds.tr_ptr, ds.tr_col, ds.te_ptr, ds.te_col,
                      np.concatenate([[0], np.cumsum(np.bincount(rows[keep], minlength=ds.U))]).astype(np.int64), ds.lab_col[keep],
                      ds.deg_tr, ds.deg_te, ds.deg_song)
        assert bits(ap[j]) == bits(oracle_lib.evaluate(ibm, one, 10)), j


def partitioned(oracle_lib, ds, models, n_win, n_shard, kinds=KINDS, n_thr=10, handle_kw=ITEM):
    """n_win song windows x n_shard user shards on one GPU: ranges combined by min / max, counts by a numpy sum.  One handle at a time
    (a window handle of the MSD shape sizes its panels and head rows to the HBM it finds): a first sweep takes the ranges, a second the counts."""
    starts, n_total = pair_index_bases(ds, n_shard)
    new = np.unique(ds.lab_col)
    shards = [ds.shard_test_users(*shard_range(ds.U, r, n_shard)) for r in range(n_shard)]
    rng = {name: [] for _, name, _, _ in kinds}
    tot = {name: None for _, name, _, _ in kinds}
    for sweep in ("range", "counts"):
        if sweep == "counts":
            glob = {name: (min(a for a, _ in r), max(b for _, b in r)) for name, r in rng.items()}
        for w in range(n_win):
            with MusicRecommender(ds, song_window=song_window(ds.S, w, n_win), **handle_kw) as mr:
                for r, sh in enumerate(shards):
                    mr.set_test_users(sh, int(starts[r]), n_total)
                    for kind, name, param, seed in kinds:
                        if sweep == "range":
                            rng[name].append(mr.eval_range(kind, param, seed))
                        else:
                            c = mr.eval_counts(kind, *glob[name], new, param, seed, n_thr)
                            tot[name] = list(c) if tot[name] is None else [a + b for a, b in zip(tot[name], c)]
    return {name: (*glob[name], tot[name], eval_finish(*tot[name], n_thr), rng[name]) for name in rng}


def test_partition_invariance(mrlib, oracle_lib):
    ds = synth(T=800, U=61, S=3001, seed=5)
    models = dense_models(oracle_lib, ds)
    new = np.unique(ds.lab_col)
    for name, (mn, mx, tot, m, _) in partitioned(oracle_lib, ds, models, 3, 2).items():
        sc = models[name]
        assert (mn, mx) == (np.nanmin(sc), np.nanmax(sc))
        for a, b in zip(tot, eval_counts_host(sc, ds, 0, mn, mx, 10, new)):
            np.testing.assert_array_equal(a, b, err_msg=name)
        assert bits(m) == bits(oracle_lib.evaluate(sc, ds, 10)), name


def edge_dataset():
    """Labels the user also listened to, label-only songs (ids >= S), users without labels; songs 0..3 listened by every test user."""
    rng = np.random.default_rng(3)
    T, U, S = 30, 6, 60
    tr = [(v, s) for v in range(T) for s in rng.choice(np.arange(4, S), 8, replace=False)] + [(v, s) for v in range(5) for s in range(4)]
    te = [(u, s) for u in range(U) for s in range(4)] + [(u, s) for u in range(U) for s in rng.choice(np.arange(4, S), 3, replace=False)]
    te_set = set(te)
    lab = [(0, 4 + i) for i in range(5)] + [(1, S + 2), (1, S + 7), (1, 10)] + [(2, s) for u, s in te if u == 2][:3] + [(2, 50)] + [(4, 5), (4, 6)]
    assert any(p in te_set for p in lab)
    tr, te, lab = (np.array(x).T for x in (tr, te, lab))
    return from_triplets(tr, te, lab, T, U, S)


def test_edge_data(mrlib, oracle_lib):
    ds = edge_dataset()
    assert np.diff(ds.lab_ptr)[3] == 0 and ds.lab_col.max() >= ds.S
    models = dense_models(oracle_lib, ds)
    with MusicRecommender(ds, **ITEM) as mr:
        check_models(mr, oracle_lib, ds, models)
    # a window in which every pair is listened emits nothing; combined with the rest, still exact
    out = partitioned(oracle_lib, ds, models, 1, 1, kinds=KINDS[:1])   # sanity: one part
    assert bits(out["ubm"][3]) == bits(oracle_lib.evaluate(models["ubm"], ds, 10))
    new = np.unique(ds.lab_col)
    parts = [MusicRecommender(ds, song_window=w, **ITEM) for w in ((0, 4), (4, ds.S))]
    try:
        rng = [mr.eval_range(_lib.MR_UBM) for mr in parts]
        assert rng[0] == (np.inf, -np.inf)
        mn, mx = min(a for a, _ in rng), max(b for _, b in rng)
        c = [mr.eval_counts(_lib.MR_UBM, mn, mx, new) for mr in parts]
        assert bits(eval_finish(*[a + b for a, b in zip(*c)], 10)) == bits(oracle_lib.evaluate(models["ubm"], ds, 10))
    finally:
        for mr in parts:
            mr.close()
    # all-zero model: no test user shares a song with a train user -> max == min -> 0.0
    z = from_triplets((np.arange(10), np.arange(10)), (np.repeat(np.arange(3), 2), np.arange(20, 26)), (np.array([0, 1]), np.array([12, 30])),
                      10, 3, 40)
    zm = dense_models(oracle_lib, z)
    assert np.nanmax(zm["ubm"]) == np.nanmin(zm["ubm"]) == 0.0
    with MusicRecommender(z, **ITEM) as mr:
        for kind, name, param, seed in KINDS:
            assert mr.evaluateOnDevice(kind, param, seed) == 0.0 == oracle_lib.evaluate(zm[name], z, 10)


def test_resident_reuse(mrlib, oracle_lib):
    """Single-batch item-space shard under MR_PROFILE: range then counts scores once (head_rowsum time does not grow); a top-k call in
    between forces a second scoring; results identical; a device-resident top-k survives an evaluation."""
    ds = synth(**ITEMDS)
    new = np.unique(ds.lab_col)
    with MusicRecommender(ds, profile=True, **ITEM) as mr:
        assert mr.info()["batch_rows"] >= ds.U
        for kind, name, param, seed in KINDS:
            mr.timing(reset=True)
            mn, mx = mr.eval_range(kind, param, seed)
            h1 = mr.timing()["head_rowsum"]
            assert h1 > 0
            a = mr.eval_counts(kind, mn, mx, new, param, seed)
            assert mr.timing()["head_rowsum"] == h1
            mr.eval_range(kind, param, seed)
            mr.getTopK(kind, k=20, param=param, seed=seed)
            h2 = mr.timing()["head_rowsum"]
            b = mr.eval_counts(kind, mn, mx, new, param, seed)
            assert mr.timing()["head_rowsum"] > h2
            for x, y in zip(a, b):
                np.testing.assert_array_equal(x, y)
        mr.getTopK(_lib.MR_UBM, k=50)
        before = mr.mapAtK(50, top=None)
        mr.evaluateOnDevice(_lib.MR_IBM)
        assert mr.mapAtK(50, top=None) == before


def test_guards(mrlib):
    ds = synth(**SMALL)
    new = np.unique(ds.lab_col)
    with MusicRecommender(ds, **ITEM) as mr:
        for kind, p in ((_lib.MR_LC, 1.5), (_lib.MR_LC, float("nan")), (_lib.MR_AGG, 1.5), (_lib.MR_STOCH, -0.1)):
            with pytest.raises(ParameterRange):
                mr.eval_range(kind, p)
            with pytest.raises(ParameterRange):
                mr.eval_counts(kind, 0.0, 1.0, new, p)
        with pytest.raises(_lib.MrError) as e:
            mr.eval_counts(_lib.MR_UBM, 0.0, 1.0, new, n_thresholds=9)
        assert e.value.code == _lib.MR_ERR_BAD_ARG
        bad = ds.shard_test_users(0, ds.U)
        r = int(np.flatnonzero(np.diff(bad.lab_ptr) >= 2)[0])
        bad.lab_col = bad.lab_col.copy()
        i = int(bad.lab_ptr[r])
        bad.lab_col[i], bad.lab_col[i + 1] = bad.lab_col[i + 1], bad.lab_col[i]
        with pytest.raises(_lib.MrError, match=f"label row {r} not ascending") as e:
            mr.eval_counts(_lib.MR_UBM, 0.0, 1.0, new, labels=bad)
        assert e.value.code == _lib.MR_ERR_BAD_ARG
        with pytest.raises(ValueError):                                  # label rows of another shard
            mr.eval_counts(_lib.MR_UBM, 0.0, 1.0, new, labels=ds.shard_test_users(0, ds.U - 1))
        starts, n_total = pair_index_bases(ds, 2)
        mr.set_test_users(ds.shard_test_users(*shard_range(ds.U, 1, 2)), int(starts[1]), n_total)
        with pytest.raises(ValueError):                                  # a shard's own mAP is not the model's
            mr.evaluateOnDevice(_lib.MR_UBM)
        mr.set_test_users(ds)
        missing = int(new[len(new) // 2])
        with pytest.raises(_lib.MrError, match=f"lacks label song {missing}") as e:
            mr.eval_counts(_lib.MR_UBM, 0.0, 1.0, new[new != missing])
        assert e.value.code == _lib.MR_ERR_BAD_ARG


def test_msd_shape(mrlib):
    """configs[3] (MSD) shape, a 2 560-user shard, default engine: the mAP bits agree across one batch, 640-user batches and 4 song windows x
    2 user shards; the counts of 200 label songs equal the numpy mirror over exact dense columns (getRanks2), and min / max equal those of
    getRanks1 rows taken in chunks."""
    ds = synth_config("c4").shard_test_users(0, 2560)
    new = np.unique(ds.lab_col)
    res = {}
    with MusicRecommender(ds) as mr:
        for kind in (_lib.MR_UBM, _lib.MR_IBM):
            mn, mx = mr.eval_range(kind)
            cnt = mr.eval_counts(kind, mn, mx, new)
            res[kind] = (mn, mx, eval_finish(*cnt, 10))
            lo, hi = np.inf, -np.inf
            for u in range(0, ds.U, 512):
                r = mr.getRanks1(kind, np.arange(u, min(u + 512, ds.U)))
                lo, hi = min(lo, np.nanmin(r)), max(hi, np.nanmax(r))
            assert (mn, mx) == (lo, hi)
            pick = np.random.default_rng(1).choice(np.flatnonzero(new < ds.S), 200, replace=False)
            cols = mr.getRanks2(kind, new[pick])
            for j, c in zip(pick, cols):
                want = eval_counts_host(c[:, None], ds, int(new[j]), mn, mx, 10, new[j:j + 1])
                for a, b in zip(cnt, want):
                    np.testing.assert_array_equal(a[j], b[0])
    with MusicRecommender(ds, item_batch=640) as mr:
        assert mr.info()["batch_rows"] == 640
        for kind in (_lib.MR_UBM, _lib.MR_IBM):
            assert bits(mr.evaluateOnDevice(kind)) == bits(res[kind][2])
    part = partitioned(None, ds, None, 4, 2, kinds=((_lib.MR_UBM, "ubm", 0.5, 0), (_lib.MR_IBM, "ibm", 0.5, 0)), handle_kw={})
    for kind, name in ((_lib.MR_UBM, "ubm"), (_lib.MR_IBM, "ibm")):
        assert (part[name][0], part[name][1]) == res[kind][:2]
        assert bits(part[name][3]) == bits(res[kind][2])


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_reference_map_two_ranks_under_torchrun(mrlib):
    """distributed.evaluate_reference_map over two song partitions on two GPUs (NCCL) equals the single-process mAP."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           str(ROOT / "tools" / "eval_bench.py"), "--mode", "dist", "--config", "c3", "--check", "--reps", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, OMP_NUM_THREADS="4"))
    assert out.returncode == 0, out.stderr[-2000:]
    import json
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["check_equal_single_process"] is True
