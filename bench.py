#!/usr/bin/env python
"""bench.py — scored (test-user, song) pairs / second for UBM + IBM scoring with top-500 ranking (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--workload msd|c1|c2|c3|ksplit] [--impl reference]

Workload `msd` (default) is BASELINE.json configs[3], the whole job: the MSD-shaped synthetic data set (909 318 train users, 384 546
songs, ~42 M train triplets) and ALL 110 000 test users on N GPUs.  STRONG scaling: the work is fixed, N GPUs split it — by default
(N > 1) by SONG: every GPU scores all test users against its 1/N of the songs (the reference's second partitioning,
distributed.scala:459-461), the ranked lists are exchanged with one NCCL all-to-all per array and joined exactly (mr_topk_merge), so the
head-row precompute is divided by N instead of replicated; `--partition users` shards the test users instead (distributed.scala:450-452).  One step = what getUserBasedModel + getItemBasedModel
(+ the new top-500) do for the whole test set, with nothing amortised across steps:

    head-row precompute (the only place the item-item intersection counts |U_i ∩ U_j| are computed at this scale; the reference's
    model builders have no reusable half, MR:132-170, 222-261)  ->  per batch of test users: head pass, tail scatter, top-500 select,
    for UBM and for IBM            = 2 * (110 000 * S - nnz_test) scored pairs per step.

One JSON line on rank 0:
  value         whole-job pairs/s, test CSR already resident in HBM, CUDA events on the library stream, max over ranks
  e2e           the same through the host-buffer C-ABI: mr_prepare_async + mr_set_test_users (pinned host -> device) + scoring + the lists
                of this rank's users copied device -> host and, for N > 1, the NCCL gather of the packed top-k blocks to rank 0 (the
                reference's `.collect`, DIST:451, 461)
  steady_state  the per-step figure WITHOUT the precompute (a service that keeps the train set's head rows): secondary
  roofline      dominant kernel (by CUDA-event share): algorithmic bytes per launch / average launch time vs the measured HBM peak
  cpu_baseline  the oracle's canonical CPU port (OpenMP, all host threads) on a bounded sample of the same test users
`--impl reference` times that CPU port alone (the Scala reference cannot run here: no JVM; its loops as written are infeasible beyond
configs[0]/[1] — SURVEY.md §8d) on rank 0 with every host thread the process may use and prints the same line with "impl": "reference".
`--workload c1|c2` add the as-written sequential and `.par` CPU legs; `--workload ksplit` is BASELINE configs[4] (K-split item-item sweep).
`--dump-outputs DIR` writes the UBM and IBM top-500 lists that the last timed step computed for a fixed, seeded sample of rank 0's test
users to DIR/*.npy (float64), so that two builds can be compared output for output on identical inputs.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

K_TOP = 500
N_TEST_USERS = 110000          # BASELINE configs[3]
METRIC = "scored (test-user, song) pairs/sec, UBM+IBM with top-500"
DUMP_USERS = 2048              # --dump-outputs: 2 models x (song, score) x 2048 x 500 float64 = 33 MB, under the 64 MB a dump may take
DUMP_SEED = 0


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." to fd 1), so fd 1 is pointed at
# stderr for the whole run and the JSON line goes to a private duplicate of the original stdout.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)
sys.stdout = sys.stderr


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def host_threads() -> int:
    """Threads this process may run on (torchrun exports OMP_NUM_THREADS=1; the CPU legs set their thread count explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def make_workload(name: str, rank: int, world: int, users_total: int = 0, partition: str = "users"):
    from musicrecommendation_b200.dataset import synth_config
    from musicrecommendation_b200.distributed import shard_range
    t0 = time.time()
    if name == "msd":
        full = synth_config("c4")
        n_users = min(users_total or N_TEST_USERS, full.U)
        u0, u1 = (0, n_users) if partition == "songs" else shard_range(n_users, rank, world)
        ds = full.shard_test_users(u0, u1)
        how = (f"songs partitioned over {world} GPU(s) (distributed.scala:459-461), every GPU scores all test users against its songs, all-to-all + join of the ranked lists"
               if partition == "songs" else f"sharded by test user over {world} GPU(s)")
        desc = (f"BASELINE configs[3]: MSD-shaped synthetic, T={full.T} train users, S={full.S} songs, nnz_train={full.nnz_tr}, all {n_users} test users, "
                f"{how}, train replica per GPU; head-row precompute inside every step")
        total_pairs = 2 * (n_users * full.S - int(full.te_ptr[n_users]))
    else:
        full = synth_config(name)
        ds = full            # the small shapes do not shard (U = 10..100): every rank scores the same users (replicas)
        desc = f"BASELINE {name}: T={full.T}, U={full.U}, S={full.S}" + (f" (replicated on {world} GPUs)" if world > 1 else "")
        total_pairs = 2 * ds.n_pairs * world
    log(f"[rank {rank}] workload {name} generated in {time.time() - t0:.1f}s: T={ds.T} U={ds.U} S={ds.S} nnz_tr={ds.nnz_tr} nnz_te={ds.nnz_te}")
    return ds, desc, total_pairs


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason samples during the timed region (via NVML)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.sm = []
        self.reasons = set()
        self.sm_max = None
        self.err = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop_flag.is_set():
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(h))
                for bit, nm in names.items():
                    if mask & bit:
                        self.reasons.add(nm)
                time.sleep(0.1)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm), **({"error": self.err} if self.err else {})}


def pinned(a: np.ndarray):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


# ------------------------------------------------------------------------------------------------------------------ CPU legs
def cpu_port_sample(ds, n_users: int):
    """The oracle's canonical CPU port (CSR + inverted index, exact integer accumulation, fp64 finalisation, full-sort top-k) on the
    first n_users test users of the shard, UBM + IBM, on every host thread; returns (pairs, seconds, threads, top-k lists)."""
    import oracle
    oracle.build()
    oracle.set_num_threads(host_threads())
    n_users = min(n_users, ds.U)
    sub = ds.shard_test_users(0, n_users)
    t0 = time.perf_counter()
    pairs = 0
    tops = []
    for m in (oracle.UBM, oracle.IBM):
        sc = oracle.canon_scores(sub, m)
        tops.append(oracle.topk(sc, K_TOP))
        pairs += sub.n_pairs
    return pairs, time.perf_counter() - t0, oracle.num_threads(), tops


def as_written_sample(ds, n_songs_ubm: int = 48, n_songs_ibm: int = 48):
    """The reference's loops AS WRITTEN (oracle.naive_sample: MusicRecommender.scala:105-307, linear `contains` scans, cosine
    recomputed per neighbour) with OpenMP over the pair loop (= `.par`, MR:119-125) on a handful of pairs of test user 0."""
    import oracle
    oracle.set_num_threads(host_threads())
    out = {}
    for name, model, n_songs in (("ubm", oracle.UBM, n_songs_ubm), ("ibm", oracle.IBM, n_songs_ibm)):
        stride = max(1, ds.S // n_songs)
        t0 = time.perf_counter()
        pairs, _ = oracle.naive_sample(ds, model, 0, 1, stride, phase=stride // 2, par=True)
        dt = time.perf_counter() - t0
        out[name] = {"pairs": pairs, "seconds": dt, "pairs_per_s": pairs / dt if dt > 0 else None}
    out["cores"] = oracle.num_threads()
    out["sample"] = f"test user 0 x every {max(1, ds.S // n_songs_ubm)}-th song, loops as written, OpenMP over pairs"
    return out


def naive_legs(ds, name: str):
    """BASELINE.md §2: the reference's sequential (MR:132-170, 222-261) and `.par` (MR:177-215, 268-307) model builders as written,
    timed on this box's host cores.  c1 in full; c2 in full for `.par` and on every 4th song for the sequential leg (say so)."""
    import oracle
    oracle.build()
    oracle.set_num_threads(host_threads())
    out = {"cores": host_threads(), "published_i5_8250U_ms": {"c1": {"ubm_seq": 42857, "ubm_par": 15507, "ibm_seq": 70839, "ibm_par": 25829},
                                                             "c2": {"ubm_seq": 1090257, "ubm_par": 425118, "ibm_seq": 823119, "ibm_par": 330385}}.get(name)}
    for mname, model in (("ubm", oracle.UBM), ("ibm", oracle.IBM)):
        for leg, par in (("seq", False), ("par", True)):
            stride = 1 if (name == "c1" or par) else 4
            t0 = time.perf_counter()
            pairs, _ = oracle.naive_sample(ds, model, 0, ds.U, stride, phase=0, par=par)
            dt = time.perf_counter() - t0
            out[f"{mname}_{leg}"] = {"pairs": pairs, "seconds": round(dt, 3), "pairs_per_s": pairs / dt, "threads": host_threads() if par else 1,
                                     "sample": "whole model" if stride == 1 else f"every {stride}-th song of every test user"}
    return out


def k1_probe(device: int):
    """Kernel K1 (tcgen05 int8 count GEMM) where it dominates: item-space head rows of a dense-friendly shape (65 536 train users x
    16 384 songs) computed as 1 count GEMM + 3 byte-plane GEMMs; dense-equivalent int8 TOP/s from CUDA events around the GEMM launches,
    against the int8 peak measured in the same process."""
    from musicrecommendation_b200 import _lib
    from musicrecommendation_b200.dataset import synth
    from musicrecommendation_b200.recommender import MusicRecommender
    from musicrecommendation_b200.ksplit import int8_peak
    peak = None
    try:
        peak = int8_peak(device)
    except Exception as e:  # noqa: BLE001
        log("int8 peak probe failed:", repr(e))
    ds = synth(T=65536, U=256, S=16384, seed=20230005)
    with MusicRecommender(ds, device=device, engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_ITEM, profile=True) as m:
        m._lib.mr_reset_timing(m._h)
        m.prepare()
        t = m.timing()
        H = m.info()["n_head"]
    q_max = int(round(2 ** 24 / np.sqrt(max(1, int(ds.deg_tr.min())))))
    gemms = 1 + max(1, (q_max.bit_length() + 7) // 8)
    ops = 2.0 * H * ds.S * ((ds.T + 127) // 128 * 128) * gemms
    tops = ops / (t["count"] * 1e-3) / 1e12
    return {"kernel": "count_gemm_kernel<256> (tcgen05.mma.cta_group::1.kind::i8 M128 N256 K32, TMA 128B swizzle, TMEM double buffer)",
            "M": H, "N": ds.S, "K": ds.T, "gemms": gemms, "gemm_ms": t["count"], "dense_int8_tops": tops,
            "int8_peak_tops_measured": peak, "frac_of_measured_int8_peak": (tops / peak) if peak else None,
            "peak_how": "torch._int_mm (cuBLASLt) int8 8192^3, best of 10, same process", "ncu": "profiles/r01_gemm_summary.md"}


def run_reference(args, rank, world):
    """The reference arm: the CPU port on rank 0's host cores (all of them, set explicitly — torchrun exports OMP_NUM_THREADS=1),
    each step a bounded sample of the workload."""
    if rank != 0:
        return
    if args.workload == "ksplit":
        emit({"impl": "reference", "unavailable": "the K-split sweep has no separate CPU arm; its rows are checked against the oracle inside the job"})
        return
    ds, desc, _ = make_workload(args.workload, 0, 1, args.users)
    n_users = args.ref_users
    times = []
    pairs = 0
    thr = 0
    for i in range(args.warmup + args.steps):
        p, dt, thr, _ = cpu_port_sample(ds, n_users)
        log(f"[reference] step {i}: {p} pairs in {dt:.2f}s on {thr} threads")
        if i >= args.warmup:
            times.append(dt)
            pairs = p
    ms = 1e3 * float(np.mean(times))
    val = pairs / (ms / 1e3)
    sample = f"first {min(n_users, ds.U)} test users per step, UBM+IBM canonical CPU port + top-{K_TOP}, OpenMP on {thr} threads"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if args.workload == "msd" else "weak", "vs_baseline": None, "dtype": "int64 accumulate / f64 scores", "data": "synthetic",
            "config": {"workload": desc, "k": K_TOP},
            "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": thr, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="msd", choices=["msd", "c1", "c2", "c3", "ksplit"])
    ap.add_argument("--engine", default="auto", choices=["auto", "tensor", "sparse"])
    ap.add_argument("--space", default="auto", choices=["auto", "user", "item"])
    ap.add_argument("--ref-users", type=int, default=96, help="test users per step of the CPU port sample (reference arm / cpu_baseline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-as-written", action="store_true", help="skip the as-written (naive) CPU samples")
    ap.add_argument("--no-k1-probe", action="store_true", help="skip the tensor-core count-GEMM probe")
    ap.add_argument("--users", type=int, default=0, help="profiling aid: total test users of the job instead of 110 000 (not a bench line)")
    ap.add_argument("--head-min-deg", type=int, default=-1, help="MR_OPT_HEAD_MIN_DEG (-1: picked from the batches per GPU, 0: library default)")
    ap.add_argument("--partition", default="auto", choices=["auto", "users", "songs"],
                    help="msd on N > 1 GPUs: shard the test users (DIST:450-452) or partition the songs (DIST:459-461; auto = songs: the head-row "
                         "precompute is divided by N instead of replicated)")
    ap.add_argument("--emulate-song-partition", default="", metavar="R/N",
                    help="profiling aid on ONE GPU (not a bench line): score all test users against song partition R of N, i.e. what one GPU of an "
                         "N-GPU song-partitioned job computes, without the exchange")
    ap.add_argument("--batch-users", type=int, default=0, help="MR_OPT_ITEM_BATCH: cap on test users per batch (0: as many as fit in HBM)")
    ap.add_argument("--ksplit-songs", type=int, nargs="+", default=[20000])
    ap.add_argument("--ksplit-mode", default="auto", choices=["auto", "fused", "nccl"])
    ap.add_argument("--ksplit-panel", type=int, default=4096)
    ap.add_argument("--ksplit-verify", action="store_true", help="check every row of every panel against the oracle (small S only)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help=f"write the top-{K_TOP} lists of UBM and IBM (song, score, len) that the last timed step computed for {DUMP_USERS} test users "
                         f"of rank 0 (seeded sample, ids in users.npy) as DIR/<model>_<array>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "ksplit"):
        ap.error("--dump-outputs covers the GPU scoring path (--impl ours, workloads msd and c1-c3)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the scoring path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.workload == "ksplit":
        from musicrecommendation_b200.ksplit import run_ksplit_bench
        checker = None
        if args.ksplit_verify:       # the CPU oracle as the checker of every Gram row (small S only)
            import oracle
            oracle.build()
            oracle.set_num_threads(max(1, host_threads() // world))
            checker = lambda d, r0, n: oracle.gram_rows(d, np.arange(r0, r0 + n))  # noqa: E731
        line = run_ksplit_bench(args, rank, world, local_rank, log, checker)
        if rank == 0:
            emit(line)
        if world > 1:
            dist.destroy_process_group()
        return

    from musicrecommendation_b200 import _lib
    from musicrecommendation_b200.recommender import MusicRecommender
    from musicrecommendation_b200.distributed import gather_topk_packed, shard_range, song_window, exchange_song_partitions

    msd = args.workload == "msd"
    n_job_users = min(args.users or N_TEST_USERS, N_TEST_USERS)
    by_songs = msd and world > 1 and args.partition in ("auto", "songs") and n_job_users % world == 0    # equal user ranges: one gather of equal blocks
    ds, desc, total_pairs = make_workload(args.workload, rank, world, args.users, "songs" if by_songs else "users")
    window = song_window(ds.S, rank, world) if by_songs else None
    if args.emulate_song_partition and world == 1:
        r_emu, n_emu = (int(x) for x in args.emulate_song_partition.split("/"))
        window = song_window(ds.S, r_emu, n_emu)
        desc += f" [EMULATION: song partition {r_emu} of {n_emu} only, no exchange — not a bench line]"
    my_u0, my_u1 = shard_range(ds.U, rank, world) if by_songs else (0, ds.U)     # the users whose joined lists this rank ends up with
    engine = {"auto": _lib.MR_ENGINE_AUTO, "tensor": _lib.MR_ENGINE_TENSOR, "sparse": _lib.MR_ENGINE_SPARSE}[args.engine]
    space = {"auto": _lib.MR_SPACE_AUTO, "user": _lib.MR_SPACE_USER, "item": _lib.MR_SPACE_ITEM}[args.space]
    # head size: a dense head row pays off when several batches of test users reuse it; a GPU that scores a single batch builds fewer
    head_min_deg = args.head_min_deg
    if head_min_deg < 0:
        # measured on one B200 (gpurun_out/r02_bench_u13750_md*.json): per 13 750-user batch the step costs 88.7 / 89.7 / 100.3 / 129.7 ms and the
        # precompute 130 / 113 / 57 / 35 ms at min_deg 64 / 150 / 400 / 1000 — few batches per GPU favour a small head
        batches = -(-ds.U // 13750)
        # song partitions (gpurun_out/ps_*.json, one GPU emulating 1 of N partitions): 125-150 beats the default 64 by 3-7 % at N = 2, 4, 8
        head_min_deg = 125 if (by_songs or window) else ((400 if batches <= 5 else 150) if msd else 0)
    t_load0 = time.perf_counter()
    mr = MusicRecommender(ds, device=local_rank, engine=engine, space=space, head_min_deg=head_min_deg, item_batch=args.batch_users, song_window=window)
    lib, h = mr._lib, mr._h
    load_ms = 1e3 * (time.perf_counter() - t_load0)
    log(f"[rank {rank}] mr_load done in {load_ms / 1e3:.1f}s, info={mr.info()}")
    stream = torch.cuda.ExternalStream(int(lib.mr_stream(h)), device=local_rank)
    U, S, k = ds.U, ds.S, K_TOP
    item_space = mr.info()["space"] == _lib.MR_SPACE_ITEM

    def check(rc):
        mr._check(rc)

    t0 = time.perf_counter()
    mr.prepare()                                   # cold: includes the cudaMalloc of the head rows
    cold_precompute_ms = 1e3 * (time.perf_counter() - t0)

    # song partitioning: per model one joined block (song | score | len of this rank's users) that the partitions' lists are merged into
    n_mine = my_u1 - my_u0
    joined = {}
    if by_songs:
        song_b, score_b = -(-n_mine * k * 4 // 16) * 16, n_mine * k * 8
        for model in (_lib.MR_UBM, _lib.MR_IBM):
            block = torch.empty(song_b + score_b + -(-n_mine * 4 // 16) * 16, dtype=torch.uint8, device="cuda")
            joined[model] = (block, block[:n_mine * k * 4].view(torch.int32).view(n_mine, k), block[song_b:song_b + score_b].view(torch.float64).view(n_mine, k),
                             block[song_b + score_b:song_b + score_b + n_mine * 4].view(torch.int32))

    # --dump-outputs: the sampled rows of rank 0's lists are copied aside right after each model, on the library stream, because the next
    # model's mr_topk_device reuses the result block
    dump_rows = None
    if args.dump_outputs and rank == 0:
        pick = np.random.default_rng(DUMP_SEED).choice(n_mine, min(n_mine, DUMP_USERS), replace=False)
        dump_rows = torch.from_numpy(np.sort(pick)).cuda()
    dumped = {}

    def score_model(model, keep=None):
        """One model for this rank's part of the job, result left on the device; `keep` receives the dump rows of its lists."""
        check(lib.mr_topk_device(h, model, 0.0, 0, k))
        if by_songs:      # exchange step of the song partitioning: all-to-all of the ranked lists, then the join (mr_topk_merge), in stream order
            with torch.cuda.stream(stream):
                parts = exchange_song_partitions(*mr.topk_device_tensors(k), ds.U, world, rank)
            mr.mergeTopK(*parts, *joined[model][1:])
        if keep is not None:
            with torch.cuda.stream(stream):
                keep[model] = [t.index_select(0, dump_rows) for t in (joined[model][1:] if by_songs else mr.topk_device_tensors(k))]

    def step_device(rebuild=True, keep=None):
        if rebuild and item_space:
            check(lib.mr_invalidate_prepared(h))
            check(lib.mr_prepare(h))
        score_model(_lib.MR_UBM, keep)
        score_model(_lib.MR_IBM, keep)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, last=None):
        """n steps between two events on the library stream; the n-th step is `last` where one is given."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        for i in range(n):
            (last if last is not None and i == n - 1 else fn)()
        ev1.record(stream)
        ev1.synchronize()
        barrier()
        return ev0.elapsed_time(ev1)

    # ---------------- device-resident timing (value): the whole job, precompute included
    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = mr.info()["launches"]
    dev_ms = timed(step_device, args.steps, last=(lambda: step_device(keep=dumped)) if dump_rows is not None else None)
    launches = mr.info()["launches"] - l0
    if dump_rows is not None:       # timed() ends in a device synchronise
        dump_dir = Path(args.dump_outputs)
        dump_dir.mkdir(parents=True, exist_ok=True)
        arrays = {"users": my_u0 + dump_rows.cpu().numpy()}
        for model, name in ((_lib.MR_UBM, "ubm"), (_lib.MR_IBM, "ibm")):
            arrays.update({f"{name}_{part}": t.cpu().numpy() for part, t in zip(("song", "score", "len"), dumped[model])})
        for name, a in arrays.items():
            np.save(dump_dir / f"{name}.npy", a.astype(np.float64))
        log(f"[rank {rank}] top-{k} lists of {len(arrays['users'])} sampled users written to {dump_dir}")
    # secondary: steady state of a service that keeps the head rows of its train set (no precompute in the step)
    steady_ms = timed(lambda: step_device(rebuild=False), args.steps)

    # ---------------- end-to-end through the host-buffer C-ABI (pinned host -> device, device -> host every step)
    keep = [pinned(ds.te_ptr.astype(np.int64)), pinned(ds.te_col.astype(np.int32)), pinned(ds.deg_te.astype(np.int32))]
    out = [pinned(np.empty((n_mine, k), np.int32)), pinned(np.empty((n_mine, k), np.float64)), pinned(np.empty(n_mine, np.int32))]
    h2d = sum(a.nbytes for _, a in keep)
    d2h = 2 * sum(a.nbytes for _, a in out)
    gather_recv = {}
    if by_songs and rank == 0:
        gather_recv = {m: [torch.empty_like(joined[m][0]) for _ in range(world)] for m in joined}
    comm_stream = torch.cuda.Stream(device=local_rank) if world > 1 else None

    def p(a):
        return C.c_void_p(a.ctypes.data)

    e2e_parts = {"precompute": 0.0, "mr_set_test_users": 0.0, "mr_topk_ubm": 0.0, "mr_topk_ibm": 0.0, "gather_join": 0.0}

    def step_e2e(verbose=False):
        t = [time.perf_counter()]
        if item_space:      # the build is started on its own stream: the host work of mr_set_test_users below overlaps it, the first mr_topk completes it
            check(lib.mr_invalidate_prepared(h))
            check(lib.mr_prepare_async(h))
        t.append(time.perf_counter())
        check(lib.mr_set_test_users(h, U, p(keep[0][1]), p(keep[1][1]), p(keep[2][1]), 0, 0))
        t.append(time.perf_counter())
        for model in (_lib.MR_UBM, _lib.MR_IBM):
            if by_songs:
                score_model(model)
                # this rank's joined lists go to the host, and — the reference's `.collect` (DIST:461) — to rank 0, both on the comm stream
                comm_stream.wait_stream(stream)
                with torch.cuda.stream(comm_stream):
                    for (dst, _), src in zip(out, joined[model][1:]):
                        dst.copy_(src, non_blocking=True)
                    dist.gather(joined[model][0], gather_list=gather_recv.get(model), dst=0)
            else:
                check(lib.mr_topk(h, model, 0.0, 0, k, p(out[0][1]), p(out[1][1]), p(out[2][1])))
                if world > 1:   # the reference's `.collect` (DIST:451-478): ONE gather of the packed (song | score | len) block to rank 0,
                                # on its own stream so that the UBM block travels while the IBM model is computed
                    gather_topk_packed(mr, k, world, rank, stream, comm_stream)
            t.append(time.perf_counter())
        if comm_stream is not None:
            comm_stream.synchronize()
        t.append(time.perf_counter())
        for name, a, b in zip(e2e_parts, t[:-1], t[1:]):
            e2e_parts[name] += 1e3 * (b - a)
        if verbose:
            log(f"[rank {rank}] e2e step: " + ", ".join(f"{n} {1e3 * (b - a):.1f} ms" for n, a, b in zip(e2e_parts, t[:-1], t[1:])))

    step_e2e(verbose=True)
    for name in e2e_parts:
        e2e_parts[name] = 0.0
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_parts = {n: v / args.steps for n, v in e2e_parts.items()}
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    checksum = int(out[0][1][:, 0].astype(np.int64).sum())

    # ---------------- per-phase CUDA-event profile of one extra step (for the roofline of the dominant kernel)
    lib.mr_set_profile(h, 1)
    lib.mr_reset_timing(h)
    step_device()
    torch.cuda.synchronize()
    phases = mr.timing()
    lib.mr_set_profile(h, 0)
    info = mr.info()
    batch = int(info["batch_rows"]) if item_space else 128    # test users per batch (mr_get_info) / kUserBatch
    n_batches = (U + batch - 1) // batch

    # max over ranks
    t = torch.tensor([dev_ms, e2e_s * 1e3, steady_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max, steady_ms_max = (float(x) for x in t.tolist())

    line = None
    if rank == 0:
        peaks = {}
        pk = ROOT / "MEASURED_PEAKS.json"
        if pk.exists():
            peaks = json.loads(pk.read_text())
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy figure)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        # dominant phase and its algorithmic bytes per launch (DESIGN.md §5): every operand crosses HBM once per launch
        T, nnz = ds.T, ds.nnz_tr
        sparse = info["engine"] == _lib.MR_ENGINE_SPARSE
        Sc = int(info["n_cols"])                      # scored columns of this GPU (its song partition; S without one)
        Sp = (Sc + 31) // 32 * 32
        # distinct head songs per batch (head = the n_head songs with most train listeners, ties by id — as mr_load selects them)
        deg_train = np.bincount(ds.tr_col, minlength=S)
        is_head = np.zeros(S, bool)
        is_head[np.argsort(-deg_train, kind="stable")[:info["n_head"]]] = True
        distinct_head_rows = 0
        for b0 in range(0, U, batch):
            cols = ds.te_col[int(ds.te_ptr[b0]):int(ds.te_ptr[min(U, b0 + batch)])]
            distinct_head_rows += int(np.count_nonzero(is_head[np.unique(cols)]))
        n_launch = {"agg_ubm": n_batches, "agg_ibm": n_batches, "topk": 2 * n_batches, "count": 2 * n_batches, "expand": n_batches,
                    "head_rowsum": 2 * n_batches, "tail_scatter": 2 * n_batches, "precompute": 1}
        # algorithmic bytes PER STEP of each phase (DESIGN.md §4/§5): every operand crosses HBM once
        alg = {
            # user space: count panel + inverted index + q table + Sint panel written, per 128-user batch
            "agg_ubm": n_batches * (2 * 128 * T + 4 * nnz + 8 * (S + 1) + 4 * T + 8 * 128 * S),
            "agg_ibm": n_batches * (4 * 128 * T + 4 * nnz + 8 * (S + 1) + 8 * 128 * S) if sparse else None,
            # item space: every DISTINCT head row a batch needs crosses HBM once per pass (4 B/song of packed Gq in the UBM pass, 2 B/song of
            # packed G in the IBM pass; users of the batch that share a song reuse its tiles out of L2), plus the Sint rows written
            # (8 B per (user, song) and model)
            "head_rowsum": distinct_head_rows * Sp * 6 + 2 * U * Sp * 8,
            # top-k: 1.125 (UBM) / 1.25 (IBM, + 4 B fp32 bound per song) streaming passes over the Sint rows, k results written
            "topk": 1.125 * U * Sc * 8 + 1.25 * U * Sc * 8 + U * Sc * 4 + 2 * 12 * U * k,
            # precompute: the packed head rows written once (6 B per entry) + the train CSR / CSC read
            "precompute": info["n_head"] * Sp * 6 + 8 * nnz,
        }
        names = {"agg_ubm": "aggregate_panel_kernel<true>", "agg_ibm": "aggregate_panel_kernel<false>" if sparse else "aggregate_ibm_kernel",
                 "topk": "topk_kernel", "count": "sparse_count / count_gemm", "expand": "expand_rows_kernel",
                 "head_rowsum": "head_rowsum_kernel", "tail_scatter": "tail_scatter_kernel",
                 "precompute": "gram_head_direct_kernel + gram_head_scatter_kernel"}
        dom = max(n_launch, key=lambda n: phases.get(n, 0.0))
        dom_ms = phases[dom] / n_launch[dom]
        roof = {"bound": "hbm", "kernel": names[dom], "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": None,
                "peak_source": peak_src, "ms_per_launch": dom_ms, "launches_per_step": n_launch[dom], "phase_ms_per_step": phases,
                "phase_note": "phases and ms_per_launch come from a separate MR_PROFILE pass of the same step (CUDA events around every phase, which "
                              "serialises the stream, and builds the head rows on one stream); the timed step runs the batches as a two-stream pipeline and the "
                              "head-row build on four streams (113 -> 73 ms, profiles/r02_summary.md §10), so it is shorter than their sum"}
        if alg.get(dom):
            roof["achieved"] = alg[dom] / (phases[dom] * 1e-3) / 1e9
            roof["frac"] = roof["achieved"] / hbm_peak
            roof["algorithmic_bytes_per_launch"] = alg[dom] / n_launch[dom]
            if dom == "head_rowsum":
                gathered = info["head_entries"] * Sp * 6 + 2 * U * Sp * 8
                roof["gathered_bytes_per_launch"] = gathered / n_launch[dom]
                roof["gathered_gbs"] = gathered / (phases[dom] * 1e-3) / 1e9
                roof["note"] = ("algorithmic = each distinct head row of a batch once per pass + what the pass writes (what must cross HBM); gathered = one "
                                "row read per (user, head song) entry = what crosses the L2 -> SM fabric.  With one wave of balanced CTAs per song tile the "
                                "DRAM traffic equals the algorithmic bytes (ncu, profiles/), so the pass is bound by the L2 -> SM fabric: it runs at "
                                "gathered_gbs against the ~12.4 TB/s LTS cap of B300_MICROARCH (6300 B/clk)")
        traffic_file = ROOT / "profiles" / "traffic.json"      # dram bytes per launch from the committed ncu --set full capture
        if traffic_file.exists() and window is None:     # captured on the whole-row configuration of one GPU (profiles/r02_traffic.md)
            roof["traffic"] = json.loads(traffic_file.read_text()).get(names[dom])
        line = {
            "metric": METRIC, "value": total_pairs * args.steps / (dev_ms_max * 1e-3),
            "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong" if msd else "weak", "vs_baseline": None, "dtype": "int64 accumulate / f64 scores", "data": "synthetic",
            "config": {"workload": desc, "k": K_TOP, "engine": ["auto", "tensor", "sparse"][info["engine"]],
                       "space": {8: "user", 16: "item"}.get(info["space"]), "head_songs": info["n_head"], "users_per_gpu": U, "users_per_batch": batch,
                       "batches_per_gpu": n_batches, "partition": "songs" if by_songs else "test users", "songs_per_gpu": Sc,
                       "l2": "inputs (head rows >= 10 GB rebuilt every step, train CSR/CSC 0.7 GB, the Sint panel of a batch: 8 B per (user, song)) exceed the 126 MB L2; no explicit flush",
                       "pairs_per_step": total_pairs},
            "e2e": {"value": total_pairs * args.steps / (e2e_ms_max * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms_max / args.steps, "host_wall_ms_per_call_rank0": e2e_parts},
            "gpu_launches": int(launches), "clocks": sampler.summary(), "roofline": roof, "checksum": checksum,
            "topk_select_rows_since_load": {"fast_path_handed_back": info["topk_fast_rejects"], "short_rows_exact_path": info["topk_short_rows"],
                                            "degenerate_radix": info["topk_degenerate_rows"]},
            "steady_state": {"value": total_pairs * args.steps / (steady_ms_max * 1e-3), "unit": "pairs/s", "ms_per_step": steady_ms_max / args.steps,
                             "what": "the same step without the head-row precompute (head rows of the train set kept across steps)"},
            "precompute_ms_per_step": phases.get("precompute", 0.0) + phases.get("count", 0.0) + phases.get("expand", 0.0) if item_space else 0.0,
            "cold_start_ms": {"mr_load": load_ms, "first_precompute_incl_cudaMalloc": cold_precompute_ms},
        }
        # mAP@500 of this rank's users from the device-resident lists (north_star's second parity target)
        map500 = {}
        mine = ds.shard_test_users(my_u0, my_u1) if by_songs else ds
        final = {}
        for name, model in (("ubm", _lib.MR_UBM), ("ibm", _lib.MR_IBM)):
            if by_songs:        # rank 0's users: the joined lists of the last step
                torch.cuda.synchronize()
                final[name] = tuple(t.cpu().numpy() for t in joined[model][1:])
                map500[name] = mr.mapAtK(k, top=(final[name][0], final[name][2]), labels=mine)
            else:
                check(lib.mr_topk_device(h, model, 0.0, 0, k))
                map500[name] = mr.mapAtK(k)
        line["map_at_500"] = dict(map500, users=mine.U, what="MSD-challenge mAP@500 of rank 0's test users against their hidden halves (mr_map_at_k)")
        if not args.no_cpu_baseline:
            import oracle
            pairs_c, sec_c, thr, tops = cpu_port_sample(mine, args.ref_users)
            # full-size parity: the same users' top-500 from the CUDA path must equal the oracle's bit for bit, and so must mAP@500
            n_chk = min(args.ref_users, mine.U)
            sub = mine.shard_test_users(0, n_chk)
            equal = {}
            map_equal = {}
            for name, model, (ws, wv, wl) in (("ubm", _lib.MR_UBM, tops[0]), ("ibm", _lib.MR_IBM, tops[1])):
                gs, gv, gl = final[name] if by_songs else mr.getTopK(model, k=k)
                equal[name] = bool(np.array_equal(gs[:n_chk], ws) and np.array_equal(gv[:n_chk].view(np.int64), wv.view(np.int64))
                                   and np.array_equal(gl[:n_chk], wl))
                map_equal[name] = bool(oracle.map_at_k(gs, gl, mine) == map500[name] and oracle.map_at_k(gs[:n_chk], gl[:n_chk], sub) == oracle.map_at_k(ws, wl, sub))
            line["parity"] = {"users_checked": n_chk, "top500_ids_and_scores_bit_equal": equal, "map_at_500_identical": map_equal}
            line["cpu_baseline_as_written"] = as_written_sample(mine) if not args.no_as_written else None
            if args.workload in ("c1", "c2") and not args.no_as_written:
                line["cpu_baseline_naive_seq_par"] = naive_legs(ds, args.workload)
            line["cpu_baseline"] = {"value": pairs_c / sec_c, "unit": "pairs/s", "cores": thr, "kind": "port",
                                    "sample": f"first {n_chk} test users of rank 0's shard, UBM+IBM canonical CPU port + top-{K_TOP}, {sec_c:.1f}s"}
    mr.close()
    if rank == 0:
        if not args.no_k1_probe:   # after the scorer released its HBM (it sizes its batches to fill the GPU)
            try:
                line["k1_count_gemm_probe"] = k1_probe(local_rank)
            except Exception as e:  # noqa: BLE001
                line["k1_count_gemm_probe"] = {"error": repr(e)}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
