"""Timing of the streamed evaluateModel (mr_eval_range / mr_eval_counts / mr_eval_finish; DESIGN.md §4.5).  Prints one JSON line and
writes it to --out.

  --mode 1gpu   synth_config("c4"), all 110 000 test users on one GPU, head rows built once: per model the wall time of evaluateOnDevice
                (it ends in a device synchronise), of its range and count passes (host work included: label checks, uploads, copy-back),
                and of a device top-500 (mr_topk_device) of the same model, which scores the same panels once.  Then, in a separate
                MR_PROFILE pass, the CUDA-event time of every phase of the three calls: count_kernels_bytes_per_s = bytes_count_pass over
                the count pass's "other" phase (mask + select bits + count kernels), select_bytes_per_s = the same bytes over the top-k
                call's "topk" phase (mask + select bits + select) on the same slices.  bytes_count_pass = what the count pass must move:
                8 B per pair for a pure model, 16 B plus one select bit for a blend, plus the label entries.
  --mode parts  the same data as --parts song partitions scored one after the other on this GPU: the per-GPU work of an N-GPU song-
                partitioned job (each partition is one batch, so the count pass reuses the range pass's panels); counts summed on the host,
                the all-reduce of a real job is not in these numbers.  --check: the mAP equals the one-GPU result.
  --mode dist   under torch.distributed.run, one song partition per rank through distributed.evaluate_reference_map (NCCL).
  --mode c3     synth_config("c3"): evaluateOnDevice against the materialised path (mr_score_dense [+ mr_blend_dense] + mr_evaluate_dense).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from musicrecommendation_b200 import _lib  # noqa: E402
from musicrecommendation_b200.dataset import synth_config  # noqa: E402
from musicrecommendation_b200.recommender import Model, MusicRecommender, eval_finish  # noqa: E402

MODELS = {"ubm": (_lib.MR_UBM, 0.5, 0), "ibm": (_lib.MR_IBM, 0.5, 0), "lc": (_lib.MR_LC, 0.5, 0), "agg": (_lib.MR_AGG, 0.5, 0),
          "stoch": (_lib.MR_STOCH, 0.5, 42)}


def gpu_info() -> dict:
    import torch
    out = {"gpu": torch.cuda.get_device_name(0), "gpus_visible": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        out["power_limit"], out["sm_clock"], out["sm_clock_max"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # noqa: BLE001
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def wall(fn, reps: int):
    ts, r = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return r, float(np.median(ts)), [round(t, 2) for t in ts]


def count_bytes(ds, name: str) -> int:
    pairs = ds.n_pairs
    per = 8 if name in ("ubm", "ibm") else 16
    return pairs * per + (ds.U * ds.S // 8 if name in ("agg", "stoch") else 0) + int(ds.lab_ptr[-1]) * 12


def on_device(mr, name, n_thr=10):
    kind, p, seed = MODELS[name]
    return mr.evaluateOnDevice(kind, p, seed, n_thr)


def one_gpu(args, ds):
    res = {}
    new = np.unique(ds.lab_col)
    with MusicRecommender(ds) as mr:
        mr.prepare()
        for name in args.models:
            kind, p, seed = MODELS[name]
            on_device(mr, name)                                     # warm-up of every kernel and buffer
            m, t_all, ts = wall(lambda: on_device(mr, name), args.reps)
            (mn, mx), t_range, _ = wall(lambda: mr.eval_range(kind, p, seed), args.reps)
            cnt, t_count, _ = wall(lambda: mr.eval_counts(kind, mn, mx, new, p, seed), args.reps)
            lib, h = mr._lib, mr._h
            import ctypes as C
            lib.mr_topk_device(h, kind, p, C.c_uint64(seed), 500)
            _, t_topk, _ = wall(lambda: mr._check(lib.mr_topk_device(h, kind, p, C.c_uint64(seed), 500)) or mr.sync(), args.reps)
            # separate profiled pass (MR_PROFILE: CUDA events around every phase, serial order): where the passes spend their GPU time.
            # "other" of an eval call = mask + select bits + eval kernels of every slice; "topk" of a top-k call = mask + select bits + select.
            lib.mr_set_profile(h, 1)
            mr.timing(reset=True)
            mr.eval_range(kind, p, seed)
            ev_range = mr.timing(reset=True)
            mr.eval_counts(kind, mn, mx, new, p, seed)
            ev_count = mr.timing(reset=True)
            mr._check(lib.mr_topk_device(h, kind, p, C.c_uint64(seed), 500))
            ev_topk = mr.timing(reset=True)
            lib.mr_set_profile(h, 0)
            b = count_bytes(ds, name)
            res[name] = dict(map=m, map_hex=float(m).hex(), evaluate_on_device_ms=t_all, evaluate_on_device_all_ms=ts,
                             range_pass_wall_ms=t_range, count_pass_wall_ms=t_count, topk500_device_wall_ms=t_topk, bytes_count_pass=b,
                             profiled_events_ms=dict(range_pass=ev_range, count_pass=ev_count, topk500=ev_topk),
                             count_kernels_bytes_per_s=b / (ev_count["other"] * 1e-3), select_bytes_per_s=b / (ev_topk["topk"] * 1e-3),
                             mn=mn, mx=mx)
        res["info"] = mr.info()
    return res


def parts(args, ds):
    """One handle at a time (each sizes its panels to the HBM it finds, as on its own GPU): a first sweep takes every partition's range,
    the second times, per partition, what its GPU does in a job — range pass, then the count pass under the global (mn, mx), which reuses
    the range pass's panels (one batch per partition)."""
    from musicrecommendation_b200.distributed import song_window
    res, new = {}, np.unique(ds.lab_col)
    wins = [song_window(ds.S, r, args.parts) for r in range(args.parts)]
    rngs = {name: [] for name in args.models}
    for w in wins:
        with MusicRecommender(ds, song_window=w) as mr:
            for name in args.models:
                kind, p, seed = MODELS[name]
                rngs[name].append(mr.eval_range(kind, p, seed))
    glob = {name: (min(a for a, _ in r), max(b for _, b in r)) for name, r in rngs.items()}
    per = {name: [] for name in args.models}
    tot = {name: None for name in args.models}
    for w in wins:
        with MusicRecommender(ds, song_window=w) as mr:
            mr.prepare()
            for name in args.models:
                kind, p, seed = MODELS[name]

                def step():
                    mr.eval_range(kind, p, seed)
                    return mr.eval_counts(kind, *glob[name], new, p, seed)
                step()                                              # warm-up
                c, t, _ = wall(step, args.reps)
                per[name].append(round(t, 2))
                tot[name] = list(c) if tot[name] is None else [a + b for a, b in zip(tot[name], c)]
            res.setdefault("info_partition0", mr.info())
    for name in args.models:
        m = eval_finish(*tot[name], 10)
        res[name] = dict(map=m, map_hex=float(m).hex(), per_partition_range_plus_counts_ms=per[name], max_partition_ms=max(per[name]),
                         allreduce_bytes=len(new) * 21 * 8)
    if args.check:
        with MusicRecommender(ds) as mr:
            for name in args.models:
                res[name]["equals_one_gpu"] = float(on_device(mr, name)).hex() == res[name]["map_hex"]
    return res


def dist_mode(args, ds):
    import torch
    import torch.distributed as dist
    from musicrecommendation_b200.distributed import evaluate_reference_map, song_window
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl")
    res = {"world": world}
    new = np.unique(ds.lab_col)
    with MusicRecommender(ds, device=torch.cuda.current_device(), song_window=song_window(ds.S, rank, world)) as mr:
        mr.prepare()
        for name in args.models:
            kind, p, seed = MODELS[name]
            evaluate_reference_map(mr, kind, p, seed, 10, new)
            dist.barrier()
            m, t, ts = wall(lambda: evaluate_reference_map(mr, kind, p, seed, 10, new), args.reps)
            res[name] = dict(map=m, map_hex=float(m).hex(), evaluate_reference_map_ms=t, all_ms=ts)
    ok = True
    if args.check and rank == 0:
        with MusicRecommender(ds, device=torch.cuda.current_device()) as mr:
            ok = all(float(on_device(mr, n)).hex() == res[n]["map_hex"] for n in args.models)
    res["check_equal_single_process"] = ok
    dist.barrier()
    dist.destroy_process_group()
    return res if rank == 0 else None


def c3(args, ds):
    res = {}
    with MusicRecommender(ds) as mr:
        def materialised(name):
            kind, p, seed = MODELS[name]
            u = mr.getUserBasedModel() if name != "ibm" else None
            i = mr.getItemBasedModel() if name != "ubm" else None
            model = {"ubm": lambda: u, "ibm": lambda: i, "lc": lambda: mr.getLinearCombinationModel(u, i, p),
                     "agg": lambda: mr.getAggregationModel(u, i, p), "stoch": lambda: mr.getStochasticCombinationModel(u, i, p, seed)}[name]()
            return mr.evaluateModel(Model(model.scores))
        for name in args.models:
            on_device(mr, name); materialised(name)
            m1, t1, _ = wall(lambda: on_device(mr, name), args.reps)
            m2, t2, _ = wall(lambda: materialised(name), args.reps)
            res[name] = dict(map_hex=float(m1).hex(), equal_bits=float(m1).hex() == float(m2).hex(), evaluate_on_device_ms=t1,
                             materialised_score_dense_plus_evaluate_dense_ms=t2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["1gpu", "parts", "dist", "c3"], required=True)
    ap.add_argument("--config", default=None)
    ap.add_argument("--models", default="ubm,ibm,agg")
    ap.add_argument("--parts", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="MRSCORE_NO_PIPELINE=1: every pass in the serial order on one stream")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.no_pipeline:
        os.environ["MRSCORE_NO_PIPELINE"] = "1"
    args.models = args.models.split(",")
    cfg = args.config or ("c3" if args.mode == "c3" else "c4")
    t0 = time.perf_counter()
    ds = synth_config(cfg)
    t_data = time.perf_counter() - t0
    info = gpu_info()
    res = {"1gpu": one_gpu, "parts": parts, "dist": dist_mode, "c3": c3}[args.mode](args, ds)
    if res is None:
        return
    line = dict(mode=args.mode, config=cfg, no_pipeline=args.no_pipeline, users=ds.U, songs=ds.S, label_songs=int(len(np.unique(ds.lab_col))), reps=args.reps,
                synth_s=round(t_data, 1), **info, **res)
    if args.mode in ("parts", "dist"):
        line["parts"] = args.parts if args.mode == "parts" else res.get("world")
    s = json.dumps(line, default=lambda o: o.item() if hasattr(o, "item") else str(o))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")
    print(s)


if __name__ == "__main__":
    main()
