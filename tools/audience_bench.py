"""Song audiences (mr_song_audience, DESIGN.md §4.10) on the MSD shape, one GPU.  Prints one JSON line and writes it to --out.

synth_config("c4"), all 110 000 test users, default engine and space.  Per model (UBM, IBM, AGG 0.5):
  all_k100 / all_k500   every song (384 546 query rows) at k = 100 and k = 500;
  rand1000_k100         1 000 random songs at k = 100;
  topk_k100             getTopK of the same model at k = 100, for context.
The cases run in that order, rand1000 first.  Wall time of each call (it returns with its work complete; the clock ends after mr_sync): median of --reps after one warm-up.  Phases from
a separate MR_PROFILE pass of the k = 100 all-songs call: head pass (head_rowsum), tail scatter, and topk = listened mask + select-plane
build + column select.  The column select must read every panel entry once per batch: 8 B per pair and panel, so U x S x 8 B = 338 GB per
pure model over the shard (two panels for a blend); bytes_per_s relates that to the topk phase.  A sample of 16 songs is checked against
the ranked getRanks2 columns (UBM and IBM) inside the run.  Per case the column selects that took the radix select (mr_get_info 27);
per model the kernel times of one all-songs call from torch.profiler.
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
from musicrecommendation_b200.recommender import MusicRecommender, song_audience_host  # noqa: E402

sys.path.insert(0, str(ROOT / "tools"))
from eval_bench import gpu_info  # noqa: E402


def timed_median(mr, fn, reps):
    fn()                                              # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        mr.sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 2) for t in ts]


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config", default="c4")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r13_audience_1gpu.json"))
    a = ap.parse_args()
    ds = synth_config(a.config)
    res = dict(config=a.config, T=ds.T, U=ds.U, S=ds.S, nnz_test=int(ds.te_ptr[-1]), gpu=gpu_info(), runs={})
    out = Path(a.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(0)
    rand1000 = rng.choice(ds.S, 1000, replace=False).astype(np.int32)
    sample = rng.choice(ds.S, 16, replace=False).astype(np.int32)
    with MusicRecommender(ds) as mr:
        info = mr.info()
        res.update(engine=info["engine"], space=info["space"], batch_rows=info["batch_rows"], batches=-(-ds.U // info["batch_rows"]))
        for model, name, param in ((_lib.MR_UBM, "ubm", 0.5), (_lib.MR_IBM, "ibm", 0.5), (_lib.MR_AGG, "agg", 0.5)):
            if model != _lib.MR_AGG:   # the bits check: the sample's lists against its ranked getRanks2 columns
                got = mr.getSongAudience(model, sample, 100, param)
                want = song_audience_host(mr.getRanks2(model, sample).T, np.arange(len(sample)), 100)
                res[f"{name}_sample16_equal"] = bool(all(np.array_equal(g.view(np.int64) if g.dtype == np.float64 else g,
                                                                        w.view(np.int64) if w.dtype == np.float64 else w) for g, w in zip(got, want)))
            cases = {"rand1000_k100": (rand1000, 100), "all_k100": (None, 100), "all_k500": (None, 500)}
            for case, (songs, k) in cases.items():
                r = dict(rows=ds.S if songs is None else len(songs), k=k)
                i0 = mr.info()
                r["ms"], r["ms_runs"] = timed_median(mr, lambda: mr.getSongAudience(model, songs, k, param), a.reps)
                i1 = mr.info()
                r["passes_per_call"] = (i1["scoring_passes"] - i0["scoring_passes"]) // (a.reps + 1)
                r["radix_selects_per_call"] = (i1["audience_radix_selects"] - i0["audience_radix_selects"]) // (a.reps + 1)
                res["runs"][f"{name}_{case}"] = r
                out.write_text(json.dumps(res) + "\n")   # after every case, so that a cut-short run keeps what it measured
            r = dict(k=100)
            r["ms"], r["ms_runs"] = timed_median(mr, lambda: mr.getTopK(model, 100, param), a.reps)
            res["runs"][f"{name}_topk_k100"] = r
            mr._lib.mr_set_profile(mr._h, 1)
            mr.timing(reset=True)
            r0 = mr.info()["audience_radix_selects"]
            t0 = time.perf_counter()
            mr.getSongAudience(model, None, 100, param)
            prof = dict(profiled_ms=(time.perf_counter() - t0) * 1e3, phases_ms={n: round(v, 3) for n, v in mr.timing(reset=True).items() if v},
                        radix_selects=mr.info()["audience_radix_selects"] - r0)
            mr._lib.mr_set_profile(mr._h, 0)
            panels = 1 if model in (_lib.MR_UBM, _lib.MR_IBM) else 2
            prof["panel_bytes"] = ds.U * ds.S * 8 * panels
            if prof["phases_ms"].get("topk"):
                prof["bytes_per_s"] = prof["panel_bytes"] / (prof["phases_ms"]["topk"] * 1e-3)
            res["runs"][f"{name}_all_k100"]["profile"] = prof
            # kernel times of the same call from torch.profiler (CUPTI), summed per kernel name
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as tp:
                mr.getSongAudience(model, None, 100, param)
                mr.sync()
            kern = {}
            for e in tp.key_averages():
                t = getattr(e, "self_device_time_total", None)
                if t is None:
                    t = getattr(e, "self_cuda_time_total", 0)
                if t:
                    kern[e.key[:60]] = dict(ms=round(t / 1e3, 3), calls=e.count)
            res["runs"][f"{name}_all_k100"]["kernels"] = dict(sorted(kern.items(), key=lambda kv: -kv[1]["ms"])[:8])
            out.write_text(json.dumps(res) + "\n")
        res["device_bytes"] = mr.info()["device_bytes"]
    out.write_text(json.dumps(res) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
