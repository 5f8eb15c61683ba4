"""Explanations (mr_explain, DESIGN.md §4.9) on the MSD shape, one GPU.  Prints one JSON line and writes it to --out.

synth_config("c4"), all 110 000 test users, default engine and space.  Cases, each for UBM and IBM:
  one_pair        one (test user, song) pair: the first song of test user 0's top-10, m = 10;
  top10_1000      the top-10 of 1 000 random test users (10 000 pairs), m = 5;
  top500_100      the top-500 of 100 random test users (50 000 pairs), m = 10.
The pairs come from getTopK of the same handle (k = 10 and k = 500, computed before the timed calls).  Per case: wall time of the call (it
returns with its work complete; the clock ends after mr_sync) as the median of --reps after one warm-up, the count rows built per call
(mr_get_info 25), the distinct keys, and the CUDA-event phases of a separate MR_PROFILE pass (count rows: expand + count, the explain
kernel: topk).
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

from musicrecommendation_b200 import _lib  # noqa: E402
from musicrecommendation_b200.dataset import synth_config  # noqa: E402
from musicrecommendation_b200.recommender import MusicRecommender  # noqa: E402

sys.path.insert(0, str(ROOT / "tools"))
from eval_bench import gpu_info  # noqa: E402


def timed_median(mr, model, u, s, m, reps):
    mr.explain(model, u, s, m)                        # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        mr.explain(model, u, s, m)
        mr.sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 2) for t in ts]


def top_pairs(top, users):
    song, _, ln = top
    u = np.repeat(users, ln[users]).astype(np.int32)
    s = np.concatenate([song[i, :ln[i]] for i in users]).astype(np.int32)
    return u, s


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config", default="c4")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r11_explain_1gpu.json"))
    a = ap.parse_args()
    ds = synth_config(a.config)
    res = dict(config=a.config, T=ds.T, U=ds.U, S=ds.S, nnz_test=int(ds.te_ptr[-1]), gpu=gpu_info(), runs={})
    out = Path(a.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(0)
    u1000 = np.sort(rng.choice(ds.U, 1000, replace=False))
    u100 = np.sort(rng.choice(ds.U, 100, replace=False))
    with MusicRecommender(ds) as mr:
        res["engine"] = mr.info()["engine"]
        res["space"] = mr.info()["space"]
        for model, name in ((_lib.MR_UBM, "ubm"), (_lib.MR_IBM, "ibm")):
            top10 = mr.getTopK(model, 10)
            top500 = mr.getTopK(model, 500)
            u0, s0 = top_pairs(top10, np.array([0]))
            cases = {"one_pair": (u0[:1], s0[:1], 10), "top10_1000": (*top_pairs(top10, u1000), 5),
                     "top500_100": (*top_pairs(top500, u100), 10)}
            for case, (u, s, m) in cases.items():
                r = dict(pairs=len(u), m=m, keys=int(len(np.unique(u if model == _lib.MR_UBM else s))))
                i0 = mr.info()["explain_rows"]
                r["ms"], r["ms_runs"] = timed_median(mr, model, u, s, m, a.reps)
                r["rows_per_call"] = (mr.info()["explain_rows"] - i0) // (a.reps + 1)
                mr._lib.mr_set_profile(mr._h, 1)
                mr.timing(reset=True)
                t0 = time.perf_counter()
                e = mr.explain(model, u, s, m)
                r["profiled_ms"] = (time.perf_counter() - t0) * 1e3
                r["phases_ms"] = {n: round(v, 3) for n, v in mr.timing(reset=True).items() if v}
                mr._lib.mr_set_profile(mr._h, 0)
                r["contributors_mean"] = float(e.count.mean())
                r["contributors_max"] = int(e.count.max())
                res["runs"][f"{name}_{case}"] = r
                out.write_text(json.dumps(res) + "\n")   # after every case, so that a cut-short run keeps what it measured
        res["device_bytes"] = mr.info()["device_bytes"]
    out.write_text(json.dumps(res) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
