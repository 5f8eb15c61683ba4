"""Similar songs (mr_similar_songs, DESIGN.md §4.7) on the MSD shape, one GPU.  Prints one JSON line and writes it to --out.

synth_config("c4"), the train replica with a 2 560-user test shard (the call does not read the test shard), default engine.  For every
k in --ks: all S songs as the query list, wall time of the call (it returns with its work complete; the clock ends after mr_sync) as the
median of --reps after one warm-up; the rows each path answered (mr_get_info 21 / 22); then a separate MR_PROFILE pass for the CUDA-event
phases (count rows: expand + count, long-row select: topk, short rows and the E_i count: other).  Also timed: 1 000 random songs and the
1 000 most popular songs (by train listeners).
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200.dataset import synth_config  # noqa: E402
from musicrecommendation_b200.recommender import MusicRecommender  # noqa: E402

sys.path.insert(0, str(ROOT / "tools"))
from eval_bench import gpu_info  # noqa: E402


def timed_median(mr, songs, k, reps):
    mr.getSimilarSongs(songs, k)                     # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        mr.getSimilarSongs(songs, k)
        mr.sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 1) for t in ts]


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config", default="c4")
    ap.add_argument("--ks", default="100,500")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_similar_1gpu.json"))
    a = ap.parse_args()
    ds = synth_config(a.config)
    ds = ds.shard_test_users(0, min(ds.U, 2560))
    deg_tr = np.bincount(ds.tr_col, minlength=ds.S)
    deg = np.diff(ds.tr_ptr)
    ev = np.bincount(ds.tr_col, weights=deg[np.repeat(np.arange(ds.T), deg)], minlength=ds.S).astype(np.int64)
    res = dict(config=a.config, T=ds.T, S=ds.S, nnz_train=int(ds.nnz_tr), events_total=int(ev.sum()), events_max=int(ev.max()),
               gpu=gpu_info(), runs={})
    rng = np.random.default_rng(0)
    batches = {"random_1000": rng.choice(ds.S, 1000, replace=False).astype(np.int32),
               "popular_1000": np.argsort(-deg_tr, kind="stable")[:1000].astype(np.int32)}
    with MusicRecommender(ds) as mr:
        res["engine"] = mr.info()["engine"]
        for k in (int(x) for x in a.ks.split(",")):
            r = {}
            i0 = mr.info()
            r["all_ms"], r["all_ms_runs"] = timed_median(mr, None, k, a.reps)
            i1 = mr.info()
            calls = a.reps + 1
            r["short_rows"] = (i1["similar_short_rows"] - i0["similar_short_rows"]) // calls
            r["long_rows"] = (i1["similar_long_rows"] - i0["similar_long_rows"]) // calls
            for name, songs in batches.items():
                r[name + "_ms"], r[name + "_ms_runs"] = timed_median(mr, songs, k, a.reps)
            mr._lib.mr_set_profile(mr._h, 1)
            mr.timing(reset=True)
            t0 = time.perf_counter()
            mr.getSimilarSongs(None, k)
            r["profiled_all_ms"] = (time.perf_counter() - t0) * 1e3
            r["phases_ms"] = {n: round(v, 2) for n, v in mr.timing(reset=True).items() if v}
            mr._lib.mr_set_profile(mr._h, 0)
            res["runs"][f"k{k}"] = r
            Path(a.out).parent.mkdir(parents=True, exist_ok=True)
            Path(a.out).write_text(json.dumps(res) + "\n")      # after every k, so that a cut-short run keeps what it measured
    print(json.dumps(res))


if __name__ == "__main__":
    main()
