"""Similar users (mr_similar_users, DESIGN.md §4.8) on the MSD shape, one GPU.  Prints one JSON line and writes it to --out.

synth_config("c4"), all 110 000 test users, default engine.  First, on the fresh handle: one item-space top-k call (UBM, k = 500), whose
batch plan leaves only the 6 GB caller reserve free, then all test users at k = 100 (time and whether it completed).  Then for every k in
--ks: all test users as the query list, wall time of the call (it returns with its work complete; the clock ends after mr_sync) as the
median of --reps after one warm-up; the rows each path answered (mr_get_info 23 / 24); 1 000 random test users and the 1 000 heaviest by
E_u (sum over the visible songs of their train listeners); then a separate MR_PROFILE pass for the CUDA-event phases (count rows: expand +
count, long-row select: topk, short rows and the E_u count: other).
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200 import _lib  # noqa: E402
from musicrecommendation_b200.dataset import synth_config  # noqa: E402
from musicrecommendation_b200.recommender import MusicRecommender  # noqa: E402

sys.path.insert(0, str(ROOT / "tools"))
from eval_bench import gpu_info  # noqa: E402


def timed_median(mr, users, k, reps):
    mr.getSimilarUsers(users, k)                     # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        mr.getSimilarUsers(users, k)
        mr.sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 1) for t in ts]


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config", default="c4")
    ap.add_argument("--ks", default="100,500")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r08_similar_users_1gpu.json"))
    a = ap.parse_args()
    ds = synth_config(a.config)
    deg_tr = np.bincount(ds.tr_col, minlength=ds.S)
    owner = np.repeat(np.arange(ds.U), np.diff(ds.te_ptr))
    ev = np.bincount(owner, weights=deg_tr[ds.te_col], minlength=ds.U).astype(np.int64)
    res = dict(config=a.config, T=ds.T, U=ds.U, S=ds.S, nnz_test=int(ds.te_ptr[-1]), events_total=int(ev.sum()), events_max=int(ev.max()),
               events_median=int(np.median(ev)), gpu=gpu_info(), runs={})
    # bytes of the dense count rows of all test users (T padded to 32, int32): what one pass of the long-row select reads
    res["count_row_bytes_all"] = int(ds.U) * ((ds.T + 31) // 32 * 32) * 4
    res["events_long"] = int(ev[ev > 8192].sum())      # E_u of the rows above kSimShortMax: the work of the long-row counts
    rng = np.random.default_rng(0)
    batches = {"random_1000": rng.choice(ds.U, 1000, replace=False).astype(np.int32),
               "heaviest_1000": np.argsort(-ev, kind="stable")[:1000].astype(np.int32)}
    out = Path(a.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    with MusicRecommender(ds) as mr:
        res["engine"] = mr.info()["engine"]
        res["space"] = mr.info()["space"]
        mr.getTopK(_lib.MR_UBM, 500)
        free_b, _ = torch.cuda.mem_get_info()
        r = dict(free_bytes_before=int(free_b))
        t0 = time.perf_counter()
        try:
            mr.getSimilarUsers(None, 100)
            mr.sync()
            r["ms"], r["completed"] = (time.perf_counter() - t0) * 1e3, True
        except _lib.MrError as e:
            r["completed"], r["error"] = False, str(e)
        res["after_item_topk_k100"] = r
        out.write_text(json.dumps(res) + "\n")
        for k in (int(x) for x in a.ks.split(",")):
            r = {}
            i0 = mr.info()
            r["all_ms"], r["all_ms_runs"] = timed_median(mr, None, k, a.reps)
            i1 = mr.info()
            calls = a.reps + 1
            r["short_rows"] = (i1["similar_user_short_rows"] - i0["similar_user_short_rows"]) // calls
            r["long_rows"] = (i1["similar_user_long_rows"] - i0["similar_user_long_rows"]) // calls
            for name, users in batches.items():
                r[name + "_ms"], r[name + "_ms_runs"] = timed_median(mr, users, k, a.reps)
            mr._lib.mr_set_profile(mr._h, 1)
            mr.timing(reset=True)
            t0 = time.perf_counter()
            mr.getSimilarUsers(None, k)
            r["profiled_all_ms"] = (time.perf_counter() - t0) * 1e3
            r["phases_ms"] = {n: round(v, 2) for n, v in mr.timing(reset=True).items() if v}
            mr._lib.mr_set_profile(mr._h, 0)
            if r["phases_ms"].get("count"):
                r["long_count_events_per_s"] = res["events_long"] / (r["phases_ms"]["count"] * 1e-3)
            res["runs"][f"k{k}"] = r
            out.write_text(json.dumps(res) + "\n")      # after every k, so that a cut-short run keeps what it measured
        res["device_bytes"] = mr.info()["device_bytes"]
    out.write_text(json.dumps(res) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
