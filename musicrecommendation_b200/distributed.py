"""Multi-GPU plumbing: one process per GPU; test users sharded with no data-path collective, or songs partitioned with one all-to-all.

The reference distributes the same way (distributed.scala:450-452: `ctx.parallelize(testUsers, slices).map(getRanks1).collect`):
every worker holds the whole train set (there: the task closure; here: a train replica in each GPU's HBM) and scores a
contiguous range of test users.  Scored pairs are independent, so the only exchange is the `collect` — here an all-gather of the
fixed-size top-k blocks (k * 12 bytes per test user) over NCCL.  The index-dependent blends (Aggregation MR:372-382, Stochastic
MR:447) need each shard's position in the global (user, song)-sorted pair list; `pair_index_bases` computes it from the CSR alone.

Works with any torch.distributed backend: `nccl` with CUDA tensors on the GPU box, `gloo` with CPU tensors in the tests.
"""
from __future__ import annotations

import numpy as np

from .dataset import Dataset


def shard_range(n_users: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous, balanced test-user range of `rank` (first n_users % world ranks get one extra user)."""
    base, rem = divmod(n_users, world)
    u0 = rank * base + min(rank, rem)
    return u0, u0 + base + (1 if rank < rem else 0)


def pair_index_bases(ds: Dataset, world: int) -> tuple[np.ndarray, int]:
    """(index of each rank's first scored pair in the global MAIN:57-59 order, total number of scored pairs)."""
    per_user = ds.S - np.diff(ds.te_ptr)                       # unlistened songs per test user (MR:109)
    prefix = np.concatenate([[0], np.cumsum(per_user)])
    starts = np.array([prefix[shard_range(ds.U, r, world)[0]] for r in range(world)], np.int64)
    return starts, int(prefix[-1])


_GATHER_BUFFERS: dict = {}


def gather_topk(song, score, length, n_users_total: int, world: int, rank: int, group=None, reuse_buffers: bool = False):
    """All-gather the per-shard top-k blocks into the full [U, k] result (the reference's `.collect`).  Accepts numpy arrays or
    torch tensors (CPU for gloo, CUDA for nccl); returns torch tensors on the same device.  Equal shards (the usual case) are gathered
    by one `all_gather_into_tensor` per array straight into the result; with reuse_buffers=True that result lives in a per-shape
    buffer that the next call overwrites (a steady-state scoring loop then allocates nothing)."""
    import torch
    import torch.distributed as dist
    song = torch.as_tensor(song)
    score = torch.as_tensor(score)
    length = torch.as_tensor(length)
    if world == 1:
        return song, score, length
    sizes = [shard_range(n_users_total, r, world) for r in range(world)]
    max_n = max(b - a for a, b in sizes)
    equal = all(b - a == max_n for a, b in sizes)

    def pad(t, fill):
        if t.shape[0] == max_n:
            return t.contiguous()
        extra = torch.full((max_n - t.shape[0],) + tuple(t.shape[1:]), fill, dtype=t.dtype, device=t.device)
        return torch.cat([t, extra]).contiguous()

    outs = []
    for t, fill in ((song, -1), (score, 0.0), (length, 0)):
        p = pad(t, fill)
        shape = (world * max_n,) + tuple(p.shape[1:])
        key = (str(p.device), p.dtype, shape)
        full = _GATHER_BUFFERS.get(key) if reuse_buffers else None
        if full is None:
            full = torch.empty(shape, dtype=p.dtype, device=p.device)
            if reuse_buffers:
                _GATHER_BUFFERS[key] = full
        dist.all_gather_into_tensor(full, p, group=group)
        if equal:
            outs.append(full)
        else:
            outs.append(torch.cat([full[r * max_n: r * max_n + (hi - lo)] for r, (lo, hi) in enumerate(sizes)]))
    return tuple(outs)


_PACKED: dict = {}


def gather_topk_packed(mr, k: int, world: int, rank: int, lib_stream, comm_stream, dst: int = 0):
    """The reference's `.collect` (distributed.scala:451-452: results go to the driver only) as ONE NCCL gather of the packed
    (song | score | len) block of every rank's shard to rank `dst`, issued on `comm_stream` so that it overlaps whatever the handle
    computes next.  The block is first copied device-to-device into a staging tensor (the library reuses its result block for the
    next model); the library stream waits for that copy, nothing waits for the gather until the caller joins comm_stream.
    Returns the list of per-rank uint8 blocks on rank dst (None elsewhere); equal shard sizes are required (pad the shards otherwise)."""
    import torch
    import torch.distributed as dist
    block, _, _ = mr.topk_packed_tensor(k)
    key = (block.numel(), world, rank)
    st = _PACKED.get(key)
    if st is None:
        recv = [[torch.empty(block.numel(), dtype=torch.uint8, device=block.device) for _ in range(world)] for _ in range(2)] if rank == dst else None
        st = _PACKED[key] = {"stage": torch.empty_like(block), "recv": recv, "turn": 0, "copied": torch.cuda.Event()}
    comm_stream.wait_stream(lib_stream)
    with torch.cuda.stream(comm_stream):
        st["stage"].copy_(block, non_blocking=True)
        st["copied"].record(comm_stream)
        bufs = None
        if rank == dst:
            bufs = st["recv"][st["turn"]]
            st["turn"] ^= 1
        dist.gather(st["stage"], gather_list=bufs, dst=dst)
    lib_stream.wait_event(st["copied"])
    return bufs


def song_window(n_songs: int, rank: int, world: int) -> tuple[int, int]:
    """Song partition of `rank` (the reference's second partitioning, distributed.scala:459-461: `ctx.parallelize(songs, n)`): a contiguous,
    balanced range of song ids.  A handle created with this window scores ALL test users against its songs only."""
    return shard_range(n_songs, rank, world)


_EXCHANGE: dict = {}


def exchange_song_partitions(song, score, length, n_users_total: int, world: int, rank: int, group=None):
    """Song partitioning's exchange step: every rank holds, for ALL test users, the ranked list of its own song window; afterwards rank r
    holds all `world` lists of the users of ITS test-user range (shard_range): one all-to-all per array (row blocks of unequal size
    allowed).  Returns (parts_song [world, n_r, k], parts_score [world, n_r, k], parts_len [world, n_r]); the receive buffers are reused
    by the next call with the same shapes.  Tensors live where the backend needs them (CUDA for nccl, CPU for gloo)."""
    import torch
    import torch.distributed as dist
    song, score, length = torch.as_tensor(song), torch.as_tensor(score), torch.as_tensor(length)
    ranges = [shard_range(n_users_total, r, world) for r in range(world)]
    n_mine = ranges[rank][1] - ranges[rank][0]
    send_rows = [b - a for a, b in ranges]
    outs = []
    for t in (song, score, length):
        shape = (world, n_mine) + tuple(t.shape[1:])
        key = (str(t.device), t.dtype, shape)
        recv = _EXCHANGE.get(key)
        if recv is None:
            recv = _EXCHANGE[key] = torch.empty(shape, dtype=t.dtype, device=t.device)
        if world == 1:
            recv[0].copy_(t)
        else:
            dist.all_to_all_single(recv.view((world * n_mine,) + tuple(t.shape[1:])), t.contiguous(), [n_mine] * world, send_rows, group=group)
        outs.append(recv)
    return tuple(outs)


def audience_shard_parts(user, score, length, u0: int, world: int, rank: int, group=None):
    """The host part of song_audience under test-user sharding: every rank holds, for ALL query songs, the audience lists of its shard
    (user indices into the shard, -1 past the length).  The ids are made global by adding the shard's first user u0, then
    exchange_song_partitions hands rank r every rank's lists of ITS rows of the query list (shard_range over the queries): the exchange is
    row-generic, the rows here are query songs.  Returns (parts_user [world, n_r, k], parts_score, parts_len [world, n_r]); the parts hold
    disjoint user sets, each ordered by (score descending, user ascending), so their join (mr_topk_merge) is exact."""
    import torch
    user = torch.as_tensor(user)
    user = torch.where(user >= 0, user + int(u0), user)
    return exchange_song_partitions(user, score, length, user.shape[0], world, rank, group)


def song_audience(mr, model: int, k: int, param: float = 0.5, seed: int = 0, songs=None, group=None):
    """getSongAudience of a job whose ranks each hold one part of the model (DESIGN.md §4.10).  Every rank passes the same query list
    (default: every song).
      song partitioning (the handle has a song window, and sees every test user): each rank answers the queries inside its window, and
        rank 0 gathers them in window order.  Returns (songs, user, score, len) on rank 0, None elsewhere.
      test-user sharding (mr.ds is the shard [u0, u1) of shard_test_users): each rank ranks its shard for every query, the ids are made
        global, audience_shard_parts moves the lists by query rows and mr_topk_merge joins them on the GPU.  Returns (songs, user, score,
        len) of this rank's rows shard_range(n, rank, world) of the query list; user ids index the whole test set."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    lo, hi = mr.song_window
    ids = np.arange(mr.ds.S, dtype=np.int32) if songs is None else np.ascontiguousarray(songs, np.int32).reshape(-1)
    if (lo, hi) != (0, mr.ds.S):
        mine = ids[(ids >= lo) & (ids < hi)]
        part = (mine,) + tuple(mr.getSongAudience(model, mine, k, param, seed))
        parts = [None] * world if rank == 0 else None
        dist.gather_object(part, parts, dst=0, group=group)
        if rank != 0:
            return None
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(4))
    user, score, ln = mr.getSongAudience(model, ids, k, param, seed)
    dev = _collective_device(group)
    u0 = mr.ds.meta.get("shard", (0, mr.ds.U))[0]
    ps, pv, pl = audience_shard_parts(torch.from_numpy(user).to(dev), torch.from_numpy(score).to(dev), torch.from_numpy(ln).to(dev), u0,
                                      world, rank, group)
    r0, r1 = shard_range(len(ids), rank, world)
    ps, pv, pl = ps.cuda(), pv.cuda(), pl.cuda()
    out = (torch.empty_like(ps[0]), torch.empty_like(pv[0]), torch.empty_like(pl[0]))
    torch.cuda.synchronize()          # the parts are written on torch's streams, the join runs on the library stream
    mr.mergeTopK(ps, pv, pl, *out)
    mr.sync()
    return (ids[r0:r1],) + tuple(t.cpu().numpy() for t in out)


def shard_exclusions(ex_ptr, ex_col, u0: int, u1: int):
    """Rows [u0, u1) of an exclusion CSR over the whole test set, as the CSR of that test-user shard (rowptr from 0)."""
    ex_ptr = np.asarray(ex_ptr, np.int64)
    return ex_ptr[u0:u1 + 1] - ex_ptr[u0], np.asarray(ex_col, np.int32)[ex_ptr[u0]:ex_ptr[u1]]


def topk_filtered(mr, specs, k: int, allowed=None, exclude=None, group=None):
    """getTopKMultiFiltered of a job whose ranks each hold one part of the model (DESIGN.md §4.11).  Every rank passes the same global
    filter: `allowed` song ids (None = every song) and `exclude`, a CSR (rowptr, col) over ALL test users (None = no exclusions).
      song partitioning (the handle has a song window, and sees every test user): each rank ranks its window under the filter (the handle
        keeps the in-window part), exchange_song_partitions hands rank r every window's lists of ITS users shard_range(U, rank, world), and
        mr_topk_merge joins them on the GPU: exact, the windows are disjoint.
      test-user sharding (mr.ds is the shard [u0, u1) of shard_test_users, set with its pair base): each rank filters with its rows of
        `exclude` and ranks its shard.
    Either way returns, per entry, (song, score, len) as numpy arrays of this rank's users, rows shard_range(U, rank, world)."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    lo, hi = mr.song_window
    windowed = (lo, hi) != (0, mr.ds.S)
    if exclude is not None and not windowed:
        u0, u1 = mr.ds.meta.get("shard", (0, mr.ds.U))
        exclude = shard_exclusions(exclude[0], exclude[1], u0, u1)
    mr.setTopKFilter(allowed, exclude)
    lists = mr.getTopKMultiFiltered(specs, k)
    if not windowed:
        return lists
    dev = _collective_device(group)
    out = []
    for song, score, ln in lists:
        ps, pv, pl = exchange_song_partitions(torch.from_numpy(song).to(dev), torch.from_numpy(score).to(dev), torch.from_numpy(ln).to(dev),
                                              mr.ds.U, world, rank, group)
        ps, pv, pl = ps.cuda(), pv.cuda(), pl.cuda()
        res = (torch.empty_like(ps[0]), torch.empty_like(pv[0]), torch.empty_like(pl[0]))
        torch.cuda.synchronize()      # the parts are written on torch's streams, the join runs on the library stream
        mr.mergeTopK(ps, pv, pl, *res)
        mr.sync()
        out.append(tuple(t.cpu().numpy() for t in res))
    return out


def _collective_device(group):
    import torch
    import torch.distributed as dist
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")


def global_label_songs(lab_col, group=None) -> np.ndarray:
    """newSongs of the whole test set (MR:72, 79) when each rank holds only its own users' labels: all-gather of the ranks' distinct
    label songs, ascending int32."""
    import torch
    import torch.distributed as dist
    dev = _collective_device(group)
    mine = torch.from_numpy(np.unique(np.asarray(lab_col, np.int64))).to(dev)
    world = dist.get_world_size(group)
    n = torch.tensor([mine.numel()], dtype=torch.int64, device=dev)
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n, group=group)
    sizes = [int(x.item()) for x in sizes]
    pad = torch.full((max(sizes),), -1, dtype=torch.int64, device=dev)
    pad[:mine.numel()] = mine
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    allv = torch.cat([p[:k] for p, k in zip(parts, sizes)]).cpu().numpy()
    return np.unique(allv).astype(np.int32)


def evaluate_reference_map(mr, model: int, param: float = 0.5, seed: int = 0, n_thresholds: int = 10, new_songs=None, group=None,
                           labels: Dataset | None = None) -> float:
    """evaluateModel (MR:521-639) of a model whose parts are scored by the ranks of a job (user shards, song windows, or both), with
    the same bits as on the materialised whole model: every rank's handle gives the min / max of its part, one all-reduce makes them
    global, every rank counts its part's label pairs under the global normalisation, one all-reduce sums the integer counts, and every
    rank finishes the mAP.  new_songs: the distinct label songs of ALL test users (default: global_label_songs of this rank's labels).
    CUDA tensors under NCCL, CPU tensors under gloo."""
    import torch
    import torch.distributed as dist
    from .recommender import eval_finish
    dev = _collective_device(group)
    lab = labels if labels is not None else mr.ds
    if new_songs is None:
        new_songs = global_label_songs(lab.lab_col, group)
    mn, mx = mr.eval_range(model, param, seed)
    r = torch.tensor([mn, -mx], dtype=torch.float64, device=dev)      # min of (mn, -mx): the global min and max in one collective
    dist.all_reduce(r, op=dist.ReduceOp.MIN, group=group)
    mn, mx = float(r[0].item()), -float(r[1].item())
    pred, tp, nlab = mr.eval_counts(model, mn, mx, new_songs, param, seed, n_thresholds, lab)
    c = torch.from_numpy(np.concatenate([pred.ravel(), tp.ravel(), nlab])).to(dev)
    dist.all_reduce(c, group=group)
    c = c.cpu().numpy()
    n, k = len(nlab), n_thresholds
    return eval_finish(c[:n * k].reshape(n, k), c[n * k:2 * n * k].reshape(n, k), c[2 * n * k:], n_thresholds)


def evaluate_reference_map_multi(mr, specs, n_thresholds: int = 10, new_songs=None, group=None, labels: Dataset | None = None) -> list[float]:
    """evaluate_reference_map for every entry (model, param, seed) of a model set, from one scoring per batch on every rank: one MIN
    all-reduce of the 2 M values (mn, -mx), one sum all-reduce of the M count blocks and nlab, and a finish per entry.  One mAP per entry,
    each with the bits of evaluate_reference_map for that entry."""
    import torch
    import torch.distributed as dist
    from .recommender import eval_finish
    dev = _collective_device(group)
    lab = labels if labels is not None else mr.ds
    if new_songs is None:
        new_songs = global_label_songs(lab.lab_col, group)
    mn, mx = mr.eval_range_multi(specs)
    m = len(mn)
    r = torch.from_numpy(np.concatenate([np.asarray(mn, np.float64), -np.asarray(mx, np.float64)])).to(dev)
    dist.all_reduce(r, op=dist.ReduceOp.MIN, group=group)
    r = r.cpu().numpy()
    mn, mx = r[:m].copy(), -r[m:]
    pred, tp, nlab = mr.eval_counts_multi(specs, mn, mx, new_songs, n_thresholds, lab)
    c = torch.from_numpy(np.concatenate([np.asarray(pred).reshape(m, -1), np.asarray(tp).reshape(m, -1)], axis=1).ravel())
    c = torch.cat([c, torch.from_numpy(np.asarray(nlab, np.int64))]).to(dev)
    dist.all_reduce(c, group=group)
    c = c.cpu().numpy()
    n, k = len(nlab), n_thresholds
    blocks, nl = c[:2 * m * n * k].reshape(m, 2, n, k), c[2 * m * n * k:]
    return [eval_finish(blocks[i, 0], blocks[i, 1], nl, n_thresholds) for i in range(m)]


def split_train_users(ds: Dataset, rank: int, world: int) -> Dataset:
    """K-split of the item-item Gram (BASELINE configs[4]): rank r keeps the train users of its contiguous range, every song.
    deg_song stays global — the cosine denominators count all listeners (MR:237)."""
    v0, v1 = shard_range(ds.T, rank, world)
    a, b = int(ds.tr_ptr[v0]), int(ds.tr_ptr[v1])
    return Dataset(v1 - v0, ds.U, ds.S, (ds.tr_ptr[v0:v1 + 1] - a).astype(np.int64), ds.tr_col[a:b], ds.te_ptr, ds.te_col, ds.lab_ptr,
                   ds.lab_col, ds.deg_tr[v0:v1], ds.deg_te, ds.deg_song, None, ds.test_users, ds.songs, dict(ds.meta, train_shard=(v0, v1)))


def reduce_scatter_rows(partial, world: int, rank: int, group=None):
    """Sum the ranks' partial int32 panels [n, ld] and leave rows [rank*n/world, (rank+1)*n/world) on each rank: one NCCL
    reduce-scatter (integer sums: bit-exact in any reduction order).  n must be a multiple of world.  gloo (CPU tests) has no
    reduce-scatter, so it all-reduces and slices."""
    import torch
    import torch.distributed as dist
    n = partial.shape[0]
    assert n % world == 0
    if world == 1:
        return partial
    if dist.get_backend(group) == "gloo":
        full = partial.clone()
        dist.all_reduce(full, group=group)
        return full[rank * (n // world):(rank + 1) * (n // world)]
    out = torch.empty((n // world, partial.shape[1]), dtype=partial.dtype, device=partial.device)
    dist.reduce_scatter_tensor(out, partial.contiguous(), group=group)
    return out
