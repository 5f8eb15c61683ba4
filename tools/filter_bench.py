"""Filtered top-k (mr_topk_filtered, DESIGN.md §4.11) on the MSD shape, one GPU.  Prints one JSON line and writes it to --out.

synth_config("c4"), all 110 000 test users, default engine and space, k = 500.  Per model (UBM, IBM, AGG 0.5):
  topk                   getTopK(500), the reference point;
  nofilter               a filter with empty exclusion rows and every song allowed: the filtered call's own path without any mask;
  page2                  page 2 of 500: page 1 (55 M entries) excluded.  page2 - nofilter is the exclusion mask's time; set_ms is the
                         host-side mr_set_topk_filter (validation and upload of the rows);
  allow_<set>_<path>     allowed sets of 1 000 songs and of 1, 5, 10, 25, 50 and 90 % of the catalogue, random and most popular, each on
                         both paths (MRSCORE_FILTER_PATH=full / candidate), so that the crossover is measured; lists_equal: both paths
                         gave the same ids and score bits.
Wall time of each call (it returns with its lists on the host; the clock ends after mr_sync): median of --reps after one warm-up.
page2_equal: UBM's page 2 equals entries [500, 1000) of getTopK(1000).  Phases: one MR_PROFILE pass of page2 and of the 1 % random set per
path (topk = listened and exclusion masks + select).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200 import _lib  # noqa: E402
from musicrecommendation_b200.dataset import synth_config  # noqa: E402
from musicrecommendation_b200.recommender import MusicRecommender, exclusions_from_topk  # noqa: E402

sys.path.insert(0, str(ROOT / "tools"))
from eval_bench import gpu_info  # noqa: E402

K = 500


def timed_median(mr, fn, reps):
    out = fn()                                        # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        mr.sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 2) for t in ts], out


def same(a, b):
    return bool(np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.int64), b[1].view(np.int64)) and np.array_equal(a[2], b[2]))


def profiled(mr, fn):
    mr._lib.mr_set_profile(mr._h, 1)
    mr.timing(reset=True)
    t0 = time.perf_counter()
    fn()
    ms = (time.perf_counter() - t0) * 1e3
    phases = {n: round(v, 3) for n, v in mr.timing(reset=True).items() if v}
    mr._lib.mr_set_profile(mr._h, 0)
    return dict(profiled_ms=round(ms, 2), phases_ms=phases)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config", default="c4")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--models", default="ubm,ibm,agg")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r14_filter_1gpu.json"))
    a = ap.parse_args()
    ds = synth_config(a.config)
    res = dict(config=a.config, T=ds.T, U=ds.U, S=ds.S, k=K, gpu=gpu_info(), runs={})
    out = Path(a.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(0)
    pop = np.argsort(-np.asarray(ds.deg_song), kind="stable").astype(np.int32)
    sets = {"1000": 1000}
    sets.update({f"{p}pct": ds.S * p // 100 for p in (1, 5, 10, 25, 50, 90)})
    allowed = {}
    for name, n in sets.items():
        allowed[f"rand{name}"] = rng.choice(ds.S, n, replace=False).astype(np.int32)
        allowed[f"pop{name}"] = pop[:n]
    empty = (np.zeros(ds.U + 1, np.int64), np.empty(0, np.int32))
    models = {"ubm": (_lib.MR_UBM, 0.5), "ibm": (_lib.MR_IBM, 0.5), "agg": (_lib.MR_AGG, 0.5)}
    with MusicRecommender(ds) as mr:
        info = mr.info()
        res.update(engine=info["engine"], space=info["space"], batch_rows=info["batch_rows"])
        for name in a.models.split(","):
            model, param = models[name]
            run = lambda: mr.getTopKFiltered(model, K, param)  # noqa: E731
            r = res["runs"]
            ms, runs, top = timed_median(mr, lambda: mr.getTopK(model, K, param), a.reps)
            r[f"{name}_topk"] = dict(ms=ms, ms_runs=runs)
            mr.setTopKFilter(None, empty)
            ms, runs, _ = timed_median(mr, run, a.reps)
            r[f"{name}_nofilter"] = dict(ms=ms, ms_runs=runs)
            ex = exclusions_from_topk(top[0], top[2])
            t0 = time.perf_counter()
            mr.setTopKFilter(None, ex)
            set_ms = (time.perf_counter() - t0) * 1e3
            ms, runs, page2 = timed_median(mr, run, a.reps)
            r[f"{name}_page2"] = dict(ms=ms, ms_runs=runs, set_ms=round(set_ms, 2), exclusions=int(ex[0][-1]),
                                      mask_ms=round(ms - r[f"{name}_nofilter"]["ms"], 2), profile=profiled(mr, run))
            if name == "ubm":
                song, score, ln = mr.getTopK(model, 2 * K, param)
                res["page2_equal"] = same(page2, (song[:, K:], score[:, K:], np.maximum(ln - K, 0).astype(np.int32)))
            out.write_text(json.dumps(res) + "\n")
            for aname, ids in allowed.items():
                mr.setTopKFilter(ids, None)
                lists = {}
                for path in ("full", "candidate"):
                    os.environ["MRSCORE_FILTER_PATH"] = path
                    ms, runs, lists[path] = timed_median(mr, run, a.reps)
                    case = dict(ms=ms, ms_runs=runs, allowed=len(ids))
                    if aname == "rand1pct":
                        case["profile"] = profiled(mr, run)
                    r[f"{name}_allow_{aname}_{path}"] = case
                del os.environ["MRSCORE_FILTER_PATH"]
                i0 = mr.info()
                run()
                i1 = mr.info()
                auto = "candidate" if i1["filter_candidate_rows"] > i0["filter_candidate_rows"] else "full"
                r[f"{name}_allow_{aname}_full"].update(lists_equal=same(lists["full"], lists["candidate"]), auto_path=auto)
                out.write_text(json.dumps(res) + "\n")   # after every case, so that a cut-short run keeps what it measured
            mr.clearTopKFilter()
        res["device_bytes"] = mr.info()["device_bytes"]
    out.write_text(json.dumps(res) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
