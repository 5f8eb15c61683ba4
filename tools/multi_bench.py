"""Model sets (DESIGN.md §4.6) against one call per model, in the same process.  Prints one JSON line and writes it to --out.

  --mode 1gpu   synth_config("c4"), all 110 000 test users on one GPU, head rows built once, the five models of main.scala (UBM, IBM,
                LC 0.5, AGG 0.5, STOCH 0.5 seed 42):
                (a) five evaluateOnDevice calls against one evaluateAllOnDevice (mAP bits compared);
                (b) five mr_topk_device calls against one mr_topk_multi_device, top-500 (ids and score bits compared on the device);
                (c) an 11-point LC alpha sweep: one evaluateAllOnDevice against 11 evaluateOnDevice calls.
                Wall times end in a device synchronise; single and set calls alternate over --reps.  A separate MR_PROFILE pass gives the
                CUDA-event phases of the set calls, MRSCORE_DEBUG_TIMING the host stages of one count call (single and set), and a
                16-entry top-500 set is tried, which does not fit next to the batch plan (MR_ERR_OOM with the bytes).
  --mode parts  the same data as --parts song partitions scored one after the other on this GPU (the per-GPU work of a song-partitioned
                job): per partition the five models' range + counts as a set against one model at a time.
  --mode dist   under torch.distributed.run, one song partition per rank through distributed.evaluate_reference_map_multi (NCCL);
                rank 0 checks the mAPs against a single-process evaluateAllOnDevice.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import sys
import tempfile
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

MAIN = [(_lib.MR_UBM, 0.5, 0), (_lib.MR_IBM, 0.5, 0), (_lib.MR_LC, 0.5, 0), (_lib.MR_AGG, 0.5, 0), (_lib.MR_STOCH, 0.5, 42)]
SWEEP = [(_lib.MR_LC, a / 10, 0) for a in range(11)]


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t0) * 1e3


def alternate(single, multi, reps):
    """single / multi alternated reps times after one warm-up each: (last results, median ms, all ms)."""
    rs, rm = single(), multi()
    ts, tm = [], []
    for _ in range(reps):
        rs, t = timed(single); ts.append(t)
        rm, t = timed(multi); tm.append(t)
    return rs, rm, float(np.median(ts)), float(np.median(tm)), [round(t, 1) for t in ts], [round(t, 1) for t in tm]


def host_stages(mr, call) -> str:
    """The MRSCORE_DEBUG_TIMING line a count call writes to stderr (fd 2 captured into a temporary file)."""
    os.environ["MRSCORE_DEBUG_TIMING"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as f:
        os.dup2(f.fileno(), 2)
        try:
            call()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["MRSCORE_DEBUG_TIMING"]
        f.seek(0)
        lines = [ln for ln in f.read().decode(errors="replace").splitlines() if "eval_counts host stages" in ln]
    return lines[-1] if lines else ""


def parse_stages(line: str) -> dict:
    return {k: float(v) for k, v in re.findall(r"(\w+)=([0-9.]+)", line)}


def one_gpu(args, ds):
    res = {}
    new = np.unique(ds.lab_col)
    with MusicRecommender(ds) as mr:
        mr.prepare()
        lib, h = mr._lib, mr._h

        # (a) five models evaluated
        single = lambda specs: (lambda: [mr.evaluateOnDevice(m, p, s) for m, p, s in specs])   # noqa: E731
        multi = lambda specs: (lambda: mr.evaluateAllOnDevice(specs))                             # noqa: E731
        rs, rm, ts, tm, all_s, all_m = alternate(single(MAIN), multi(MAIN), args.reps)
        res["evaluate_five"] = dict(single_calls_ms=ts, set_call_ms=tm, single_all_ms=all_s, set_all_ms=all_m, speedup=ts / tm,
                                    map_hex=[float(x).hex() for x in rm], equal_bits=[float(a).hex() for a in rs] == [float(b).hex() for b in rm])

        # (b) five top-500 lists kept on the device
        k = 500

        def topk_single():
            for m, p, s in MAIN:
                mr._check(lib.mr_topk_device(h, m, p, C.c_uint64(s), k))
            mr.sync()

        def topk_multi():
            mr.topk_multi_device(MAIN, k)
            mr.sync()
        _, _, ts, tm, all_s, all_m = alternate(topk_single, topk_multi, args.reps)
        import torch
        eq = []
        for i, (m, p, s) in enumerate(MAIN):
            mr._check(lib.mr_topk_device(h, m, p, C.c_uint64(s), k))
            mr.sync()
            a, b = mr.topk_device_tensors(k), mr.topk_multi_device_tensors(i, k)
            eq.append(bool(torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int64), b[1].view(torch.int64)) and torch.equal(a[2], b[2])))
        res["topk500_five"] = dict(single_calls_ms=ts, set_call_ms=tm, single_all_ms=all_s, set_all_ms=all_m, speedup=ts / tm, equal_bits=eq,
                                   all_equal=all(eq))

        # (c) 11-point LC alpha sweep, evaluated
        rs, rm, ts, tm, all_s, all_m = alternate(single(SWEEP), multi(SWEEP), max(1, args.reps - 1))
        res["lc_sweep_11"] = dict(single_calls_ms=ts, set_call_ms=tm, single_all_ms=all_s, set_all_ms=all_m, speedup=ts / tm,
                                  map_hex=[float(x).hex() for x in rm], equal_bits=[float(a).hex() for a in rs] == [float(b).hex() for b in rm])

        # wall time of the parts of one set evaluation, and of a single count call (its fixed cost outside the GPU phases)
        (mn, mx), t_range = timed(lambda: mr.eval_range_multi(MAIN))
        _, t_counts = timed(lambda: mr.eval_counts_multi(MAIN, mn, mx, new))
        (a, b), t_range1 = timed(lambda: mr.eval_range(*MAIN[0]))
        _, t_counts1 = timed(lambda: mr.eval_counts(MAIN[0][0], a, b, new))
        res["wall_ms"] = dict(range_multi=t_range, counts_multi=t_counts, range_ubm=t_range1, counts_ubm=t_counts1)
        res["count_call_host_stages_ms"] = dict(
            ubm=parse_stages(host_stages(mr, lambda: mr.eval_counts(MAIN[0][0], a, b, new))),
            set5=parse_stages(host_stages(mr, lambda: mr.eval_counts_multi(MAIN, mn, mx, new))))

        # MR_PROFILE pass: CUDA-event phases of the set calls (serial order, no overlap)
        lib.mr_set_profile(h, 1)
        mr.timing(reset=True)
        mn, mx = mr.eval_range_multi(MAIN)
        ev_range = mr.timing(reset=True)
        mr.eval_counts_multi(MAIN, mn, mx, new)
        ev_counts = mr.timing(reset=True)
        mr.topk_multi_device(MAIN, k); mr.sync()
        ev_topk = mr.timing(reset=True)
        mr.evaluateOnDevice(*MAIN[3])
        ev_agg_single = mr.timing(reset=True)
        lib.mr_set_profile(h, 0)
        res["profiled_events_ms"] = dict(range_multi=ev_range, counts_multi=ev_counts, topk500_multi=ev_topk, evaluate_agg_single=ev_agg_single)

        # sixteen top-500 lists of 110 000 users (10.6 GB) do not fit next to the batch plan
        try:
            mr.topk_multi_device([(_lib.MR_LC, i / 15, 0) for i in range(16)], k)
            res["sixteen_topk500"] = dict(code=0)
        except _lib.MrError as e:
            res["sixteen_topk500"] = dict(code=e.code, oom=e.code == _lib.MR_ERR_OOM, msg=e.msg)
        res["info"] = mr.info()
    return res


def parts(args, ds):
    from musicrecommendation_b200.distributed import song_window
    new = np.unique(ds.lab_col)
    per = []
    for r in range(args.parts):
        with MusicRecommender(ds, song_window=song_window(ds.S, r, args.parts)) as mr:
            mr.prepare()

            def single():
                out = []
                for m, p, s in MAIN:
                    a, b = mr.eval_range(m, p, s)
                    out.append(mr.eval_counts(m, a, b, new, p, s))
                return out

            def multi():
                mn, mx = mr.eval_range_multi(MAIN)
                return mr.eval_counts_multi(MAIN, mn, mx, new)
            rs, rm, ts, tm, _, _ = alternate(single, multi, args.reps)
            eq = all(np.array_equal(rs[i][0], rm[0][i]) and np.array_equal(rs[i][1], rm[1][i]) for i in range(len(MAIN)))
            per.append(dict(single_calls_ms=ts, set_call_ms=tm, equal_counts=eq))
    return dict(partitions=per, max_single_ms=max(p["single_calls_ms"] for p in per), max_set_ms=max(p["set_call_ms"] for p in per),
                all_equal=all(p["equal_counts"] for p in per))


def dist_mode(args, ds):
    import torch
    import torch.distributed as dist
    from musicrecommendation_b200.distributed import evaluate_reference_map_multi, song_window
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl")
    new = np.unique(ds.lab_col)
    with MusicRecommender(ds, device=torch.cuda.current_device(), song_window=song_window(ds.S, rank, world)) as mr:
        mr.prepare()
        evaluate_reference_map_multi(mr, MAIN, 10, new)
        dist.barrier()
        maps, t = timed(lambda: evaluate_reference_map_multi(mr, MAIN, 10, new))
    res = dict(world=world, map_hex=[float(x).hex() for x in maps], evaluate_reference_map_multi_ms=t)
    ok = True
    if rank == 0:
        with MusicRecommender(ds, device=torch.cuda.current_device()) as mr:
            ok = [float(x).hex() for x in mr.evaluateAllOnDevice(MAIN)] == res["map_hex"]
    res["check_equal_single_process"] = ok
    dist.barrier()
    dist.destroy_process_group()
    return res if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["1gpu", "parts", "dist"], required=True)
    ap.add_argument("--config", default="c4")
    ap.add_argument("--parts", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    t0 = time.perf_counter()
    ds = synth_config(args.config)
    t_data = time.perf_counter() - t0
    info = gpu_info()
    res = {"1gpu": one_gpu, "parts": parts, "dist": dist_mode}[args.mode](args, ds)
    if res is None:
        return
    line = dict(mode=args.mode, config=args.config, users=ds.U, songs=ds.S, reps=args.reps, synth_s=round(t_data, 1), **info, **res)
    if args.mode == "parts":
        line["parts"] = args.parts
    s = json.dumps(line, default=lambda o: o.item() if hasattr(o, "item") else str(o))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")
    print(s)


if __name__ == "__main__":
    main()
