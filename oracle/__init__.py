"""CPU oracle for the MusicRecommendation scoring hot path — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / ``--impl reference`` legs may
import this package.  The product path (musicrecommendation_b200/ and libmrscore.so) never does;
it fails loudly when its CUDA library is missing instead of falling back to anything in here.

Parity status: **parity unpinned** — the Scala reference has no tests, fixtures or datasets and
there is no JVM in this image (SURVEY.md §4, §8c); see the header of mr_oracle.c for what pins the
restatement instead.

The arithmetic lives in mr_oracle.c (plain C, compiled by ``build()`` with gcc); this module is the
ctypes binding.  Every function takes a dataset object exposing the int-id CSR fields produced by
``musicrecommendation_b200.dataset.Dataset``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SRC = _HERE / "mr_oracle.c"
_BUILD = _HERE / "_build"
_SO = _BUILD / "libmroracle.so"
_lib = None

LC, AGG, STOCH = 0, 1, 2
UBM, IBM = 0, 1


def build(force: bool = False) -> Path:
    """Compile mr_oracle.c → oracle/_build/libmroracle.so (gcc, OpenMP, no FMA contraction).  A tree that cannot be written (a
    read-only checkout running bench.py) gets the library in a temporary directory instead."""
    global _SO
    if force or not _SO.exists() or _SO.stat().st_mtime < _SRC.stat().st_mtime:
        if os.access(_BUILD if _BUILD.exists() else _HERE, os.W_OK):
            _BUILD.mkdir(exist_ok=True)
        else:
            _SO = Path(tempfile.mkdtemp(prefix="mroracle-")) / _SO.name
        cmd = ["gcc", "-O2", "-std=c11", "-fopenmp", "-ffp-contract=off", "-fvisibility=hidden", "-shared", "-fPIC",
               str(_SRC), "-o", str(_SO), "-lm"]
        subprocess.run(cmd, check=True)
    return _SO


class _Data(C.Structure):
    _fields_ = [("T", C.c_int32), ("U", C.c_int32), ("S", C.c_int32),
                ("tr_ptr", C.c_void_p), ("tr_col", C.c_void_p),
                ("te_ptr", C.c_void_p), ("te_col", C.c_void_p),
                ("deg_tr", C.c_void_p), ("deg_te", C.c_void_p), ("deg_song", C.c_void_p)]


def lib():
    global _lib
    if _lib is None:
        if not _SO.exists():
            build()
        _lib = C.CDLL(str(_SO))
        _lib.mro_q.restype = C.c_int64
        _lib.mro_q.argtypes = [C.c_int32, C.c_int]
        _lib.mro_rs.restype = C.c_double
        _lib.mro_rs.argtypes = [C.c_int32, C.c_int]
        _lib.mro_num_threads.restype = C.c_int
        _lib.mro_naive_sample.restype = C.c_int64
        _lib.mro_evaluate.restype = C.c_double
        _lib.mro_round_at.restype = C.c_double
        _lib.mro_round_at.argtypes = [C.c_int, C.c_double]
        _lib.mro_blend.restype = C.c_int
        _lib.mro_map_at_k.restype = C.c_double
    return _lib


def _p(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def _data(ds) -> tuple[_Data, list]:
    keep = [np.ascontiguousarray(ds.tr_ptr, np.int64), np.ascontiguousarray(ds.tr_col, np.int32),
            np.ascontiguousarray(ds.te_ptr, np.int64), np.ascontiguousarray(ds.te_col, np.int32),
            np.ascontiguousarray(ds.deg_tr, np.int32), np.ascontiguousarray(ds.deg_te, np.int32),
            np.ascontiguousarray(ds.deg_song, np.int32)]
    d = _Data(ds.T, ds.U, ds.S, *[a.ctypes.data for a in keep])
    return d, keep


def num_threads() -> int:
    return int(lib().mro_num_threads())


def set_threads(n: int) -> None:
    os.environ["OMP_NUM_THREADS"] = str(n)


def set_num_threads(n: int) -> None:
    """omp_set_num_threads: overrides an inherited OMP_NUM_THREADS (torchrun exports 1) for every later call."""
    lib().mro_set_num_threads(C.c_int(int(n)))


def q(deg: int, model: int = UBM) -> int:
    return int(lib().mro_q(int(deg), int(model)))


def naive_scores(ds, model: int, par: bool = False) -> np.ndarray:
    """MusicRecommender.scala as written (MR:105-307); dense [U,S] fp64, NaN at listened pairs."""
    d, keep = _data(ds)
    out = np.empty((ds.U, ds.S), np.float64)
    fn = lib().mro_naive_ubm if model == UBM else lib().mro_naive_ibm
    fn(C.byref(d), _p(out), C.c_int(int(par)))
    return out


def naive_sample(ds, model: int, u0: int, u1: int, stride: int, phase: int = 0, par: bool = False):
    """Timed-baseline helper: the as-written loops on every `stride`-th song; returns (pairs, checksum)."""
    d, keep = _data(ds)
    cs = C.c_double(0.0)
    n = lib().mro_naive_sample(C.byref(d), C.c_int(model), C.c_int32(u0), C.c_int32(u1), C.c_int32(stride),
                               C.c_int32(phase), C.c_int(int(par)), C.byref(cs))
    return int(n), float(cs.value)


def counts_ubm(ds) -> np.ndarray:
    d, keep = _data(ds)
    out = np.empty((ds.U, ds.T), np.int32)
    lib().mro_counts_ubm(C.byref(d), _p(out))
    return out


def gram_rows(ds, rows) -> np.ndarray:
    d, keep = _data(ds)
    rows = np.ascontiguousarray(rows, np.int32)
    out = np.empty((len(rows), ds.S), np.int32)
    lib().mro_gram_rows(C.byref(d), _p(rows), C.c_int32(len(rows)), _p(out))
    return out


def canon_sint(ds, model: int, u0: int = 0, u1: int | None = None) -> np.ndarray:
    d, keep = _data(ds)
    u1 = ds.U if u1 is None else u1
    out = np.empty((u1 - u0, ds.S), np.int64)
    lib().mro_canon_sint(C.byref(d), C.c_int(model), C.c_int32(u0), C.c_int32(u1), _p(out))
    return out


def canon_scores(ds, model: int, u0: int = 0, u1: int | None = None) -> np.ndarray:
    """Canonical exact-arithmetic scores; dense [u1-u0, S] fp64, NaN at listened pairs."""
    d, keep = _data(ds)
    u1 = ds.U if u1 is None else u1
    out = np.empty((u1 - u0, ds.S), np.float64)
    lib().mro_canon_scores(C.byref(d), C.c_int(model), C.c_int32(u0), C.c_int32(u1), _p(out))
    return out


def fp64_scores(ds, model: int, u0: int = 0, u1: int | None = None) -> np.ndarray:
    """The reference's fp64 terms c/(sqrt(a)*sqrt(b)) summed in ascending-id order through the inverted index (no fixed point):
    the third restatement, used by the ranking differential test.  Dense [u1-u0, S], NaN at listened pairs."""
    d, keep = _data(ds)
    u1 = ds.U if u1 is None else u1
    out = np.empty((u1 - u0, ds.S), np.float64)
    lib().mro_fp64_scores(C.byref(d), C.c_int(model), C.c_int32(u0), C.c_int32(u1), _p(out))
    return out


def map_at_k(top_song: np.ndarray, top_len: np.ndarray, ds, per_user: bool = False):
    """MSD-challenge mAP@k of ranked lists [U,k] against the label CSR of ds (definition in mr_oracle.c)."""
    top_song = np.ascontiguousarray(top_song, np.int32)
    top_len = np.ascontiguousarray(top_len, np.int32)
    U, k = top_song.shape
    lab_ptr = np.ascontiguousarray(ds.lab_ptr, np.int64)
    lab_col = np.ascontiguousarray(ds.lab_col, np.int32)
    ap = np.zeros(U, np.float64)
    m = float(lib().mro_map_at_k(_p(top_song), _p(top_len), C.c_int32(U), C.c_int32(k), _p(lab_ptr), _p(lab_col), _p(ap)))
    return (m, ap) if per_user else m


def blend(kind: int, param: float, ubm: np.ndarray, ibm: np.ndarray, seed: int = 0, first_index: int = 0,
          n_total: int | None = None) -> np.ndarray:
    """MR:317-481 on compact (user, song)-sorted arrays.  Raises ValueError where the reference exits(-1)."""
    ubm = np.ascontiguousarray(ubm, np.float64)
    ibm = np.ascontiguousarray(ibm, np.float64)
    n = min(len(ubm), len(ibm))  # zip truncates to the shorter input (MR:322)
    out = np.empty(n, np.float64)
    rc = lib().mro_blend(C.c_int(kind), C.c_double(param), C.c_uint64(seed & (2**64 - 1)), _p(ubm), _p(ibm), _p(out),
                         C.c_int64(n), C.c_int64(first_index), C.c_int64(len(ubm) if n_total is None else n_total))
    if rc == -1:
        raise ValueError("Percentage must be between 0 and 1" if kind == AGG else "Probability must be between 0 and 1")
    if rc != 0:
        raise ValueError(f"bad blend kind {kind}")
    return out


def blend_dense(kind: int, param: float, ubm: np.ndarray, ibm: np.ndarray, seed: int = 0) -> np.ndarray:
    """Blend two dense [U,S] models (NaN at listened pairs): compacts to MAIN:57-59 order, blends, re-expands."""
    mask = ~np.isnan(ubm)
    out = np.full(ubm.shape, np.nan)
    out[mask] = blend(kind, param, ubm[mask], ibm[mask], seed)
    return out


def topk(scores: np.ndarray, k: int):
    scores = np.ascontiguousarray(scores, np.float64)
    U, S = scores.shape
    song = np.empty((U, k), np.int32)
    val = np.empty((U, k), np.float64)
    ln = np.empty(U, np.int32)
    lib().mro_topk(_p(scores), C.c_int32(U), C.c_int32(S), C.c_int32(k), _p(song), _p(val), _p(ln))
    return song, val, ln


def evaluate(scores: np.ndarray, ds, n_thresholds: int = 10) -> float:
    """The reference's threshold-sweep mAP (MR:521-639; n_thresholds=11 for DIST:395)."""
    scores = np.ascontiguousarray(scores, np.float64)
    U, S = scores.shape
    lab_ptr = np.ascontiguousarray(ds.lab_ptr, np.int64)
    lab_col = np.ascontiguousarray(ds.lab_col, np.int32)
    new = np.unique(lab_col).astype(np.int32)
    return float(lib().mro_evaluate(_p(scores), C.c_int32(U), C.c_int32(S), _p(lab_ptr), _p(lab_col), _p(new),
                                    C.c_int32(len(new)), C.c_int32(n_thresholds)))


def round_at(p: int, x: float) -> float:
    return float(lib().mro_round_at(p, x))


def java_random_floats(seed: int, n: int) -> np.ndarray:
    """java.util.Random(seed).nextFloat() stream in pure Python (SURVEY A.4) — independent check of the C LCG."""
    mask = (1 << 48) - 1
    s = (seed ^ 0x5DEECE66D) & mask
    out = np.empty(n, np.float32)
    for i in range(n):
        s = (s * 0x5DEECE66D + 0xB) & mask
        out[i] = np.float32(s >> 24) / np.float32(1 << 24)
    return out
