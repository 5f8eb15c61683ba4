"""GPU tests (-m gpu) of the handle's device memory: repeated calls hold device_bytes steady (per-call temporaries are released), the Gram
workspace frees what it outgrows, and malformed label rows are refused before any of them is read on the host or the device."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import synth
from musicrecommendation_b200.recommender import MusicRecommender, _p

CONFIGS = {"tensor_user": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER),
           "sparse_user": dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER),
           "tensor_item": dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_ITEM),
           "sparse_item": dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)}
DS = dict(T=1500, U=200, S=4200, seed=11)      # S >= 4096: room for a 4096-row Gram workspace


def device_bytes(mr):
    return mr.info()["device_bytes"]


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_device_bytes_steady(mrlib, cfg):
    ds = synth(**DS)
    users, songs = np.arange(0, ds.U, 7), np.arange(0, ds.S, 97)
    with MusicRecommender(ds, **CONFIGS[cfg]) as mr:
        tensor = mr.info()["engine"] == _lib.MR_ENGINE_TENSOR
        ubm, ibm = mr.getUserBasedModel(), mr.getItemBasedModel()

        def one_round():
            top = mr.getTopK(_lib.MR_UBM, k=20)
            mr.mapAtK(20, top=(top[0], top[2]))
            mr.mapAtK(20, top=None)
            mr.evaluateModel(ubm)
            mr.getRanks1(_lib.MR_UBM, users)
            mr.getRanks2(_lib.MR_IBM, songs)
            mr.counts_ibm(0, 1500)
            mr.similarity_ibm(0, 1500)
            mr.getLinearCombinationModel(ubm, ibm, 0.5)
            if tensor:
                mr.invalidate_prepared()
                mr.prepare()
            return device_bytes(mr)

        one_round()                                  # warm-up: the grow-only slots reach their sizes
        assert one_round() == one_round()


@pytest.mark.parametrize("engine", [_lib.MR_ENGINE_TENSOR, _lib.MR_ENGINE_SPARSE], ids=["tensor", "sparse"])
def test_gram_workspace_does_not_leak(mrlib, engine):
    ds = synth(**DS)
    with MusicRecommender(ds, engine=engine, space=_lib.MR_SPACE_USER) as mr:
        assert mr.info()["engine"] == engine
        ptr, ld = C.c_void_p(), C.c_int64()

        def rows(n):
            mr._check(mr._lib.mr_gram_rows_device(mr._h, 0, n, C.byref(ptr), C.byref(ld)))
            return device_bytes(mr)

        b0 = rows(1024)
        b1 = rows(4096)
        grown = 4096 - 1024
        want = grown * ld.value * 4
        if engine == _lib.MR_ENGINE_TENSOR:
            want += grown * (-(-ds.T // 128) * 128)      # the 0/1 operand rows, T rounded up to 128 bytes
        ids = lambda n: 4 * n + (4 * n) // 4 + 256       # noqa: E731  the row id list, a grow-only slot with a quarter of headroom
        want += ids(4096) - ids(1024)
        assert b1 - b0 == want
        mr.counts_ibm(0, 2000)                           # 1024-row chunks: the workspace is large enough, the temporaries go
        assert device_bytes(mr) == b1


def test_malformed_label_rows_refused(mrlib):
    ds = synth(T=300, U=40, S=900, seed=4)
    lp = np.ascontiguousarray(ds.lab_ptr, np.int64)
    lc = np.ascontiguousarray(ds.lab_col, np.int32)
    r = int(np.flatnonzero(np.diff(lp) >= 2)[0])
    i = int(lp[r])
    start = lp.copy(); start[0] = 1
    falling = lp.copy(); falling[r + 1] = lp[r] - 1
    descending = lc.copy(); descending[i], descending[i + 1] = lc[i + 1], lc[i]
    negative = lc.copy(); negative[i] = -1
    cases = [(start, lc, r"label: rowptr\[0\] != 0"),
             (falling, lc, f"label: rowptr not monotone at row {r}\\b"),
             (lp, descending, f"label row {r} not ascending/unique"),
             (lp, negative, f"label: column id -1 out of range at row {r}\\b")]
    k = 10
    top_song, top_len = np.zeros((ds.U, k), np.int32), np.zeros(ds.U, np.int32)
    scores = np.zeros((ds.U, ds.S), np.float64)
    new = np.unique(lc)
    pred, tp = np.zeros((len(new), 10), np.int64), np.zeros((len(new), 10), np.int64)
    nlab = np.zeros(len(new), np.int64)
    with MusicRecommender(ds, engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER) as mr:
        lib, h, out = mr._lib, mr._h, C.c_double()
        calls = {"mr_map_at_k": lambda p, c: lib.mr_map_at_k(h, k, _p(top_song), _p(top_len), ds.U, _p(p), _p(c), C.byref(out), None),
                 "mr_evaluate_dense": lambda p, c: lib.mr_evaluate_dense(h, _p(scores), ds.U, ds.S, _p(p), _p(c), 10, C.byref(out)),
                 "mr_eval_counts": lambda p, c: lib.mr_eval_counts(h, _lib.MR_UBM, 0.5, C.c_uint64(0), 0.0, 1.0, 10, _p(p), _p(c), _p(new),
                                                                    len(new), _p(pred), _p(tp), _p(nlab))}
        for name, call in calls.items():
            for p, c, msg in cases:
                with pytest.raises(_lib.MrError, match=msg) as e:
                    mr._check(call(p, c))
                assert e.value.code == _lib.MR_ERR_BAD_ARG, name
            mr._check(call(lp, lc))                      # the well-formed rows pass
