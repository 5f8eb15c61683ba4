"""The paths of the top-k select (topk_kernel, csrc/k3_topk.cu) on rows built to force each one, against the oracle's ranking.

Long rows (more than 16 384 scored columns) take a sampled fast path: a cut from every 8th chunk of 2 048 songs, then one collect pass.
It hands a row to the exact path when too few sampled keys are positive (cut < 2) or when it collects fewer than
need = min(k, unlistened songs) keys or more than 2 048.  The exact path bins the row with a scale taken from the sampled maximum
(scores above it share the top bin), and a bin of more than 2 048 keys goes to the 8-bit radix select over the 96-bit key.  Short rows
take the exact path from the start.  Each test user range holds one row kind; the CPU tests check on the oracle's scores that every
kind has the property that sends it down its path, and the GPU tests rank every kind and read the library's select counters
(mr_get_info: topk_fast_rejects, topk_short_rows, topk_degenerate_rows) to show that it took that path.

  A control        ordinary rows: accepted by the fast path, no radix
  B zero           the user's songs have no train listener, every score is 0: hand-back, then radix over the whole row
  D few            1 to 60 positive scores: hand-back (cut < 2), then radix (the zeros fill the k-th bin)
  E sampled-only   600 positive scores, all in sampled chunks, 300 of them far above the others: the cut keeps only those 300 < need,
                   hand-back, exact path without radix
  F crowded tie    2 500 songs tied above every sampled key, in unsampled chunks: the collect pass finds more than 2 048 keys, hand-back,
                   the tie lands in the clamped top bin, radix; the list is the k smallest tie ids
  G boundary tie   300 distinct top scores, then 600 songs tied at rank 500: accepted, and the trim before the sort meets a bin too
                   crowded to compact
  H near-full      the user listened to all but 200 songs: need = 200, the list ends after 200 entries
"""
import numpy as np
import pytest

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import from_triplets
from musicrecommendation_b200.distributed import song_window
from musicrecommendation_b200.recommender import MusicRecommender

# topk_kernel reads 4 * kTopkThreads songs per chunk and, on long rows, samples every stride = 8th chunk: column c of a row (c counted
# from the first column of the song window) is sampled iff (c // CHUNK) % STRIDE == 0
CHUNK = 4 * 512
STRIDE = 8
LONG_ROW = 16384            # rows of more scored columns take the sampled fast path
CAP = 2048                  # candidate buffer of the select (kTopkCap)
K = 500

N_USERS = dict(A=3, B=3, D=3, E=2, F=2, G=2, H=2)
COLD = (0, 3, 4, 10, 63, 257, 498, 1023)    # window columns nobody in train listens to (the B users' songs)
D_SIZES = (1, 7, 60)                         # positive scores of the D users
N_TIE, N_W_SAMPLED, N_W_LOW = 2500, 700, 2048
N_TOP, N_TOP_SAMPLED, N_TIE_G, N_TIE_G_SAMPLED = 300, 40, 600, 100
N_NEAR_FULL = 200

ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
MODELS = ((_lib.MR_UBM, "ubm", 0.0, 0), (_lib.MR_IBM, "ibm", 0.0, 0), (_lib.MR_LC, "lc", 0.5, 0), (_lib.MR_AGG, "agg", 0.5, 0),
          (_lib.MR_STOCH, "stoch", 0.5, 42))


def sampled(c):
    """Whether window column c lies in a chunk the fast path samples."""
    return (np.asarray(c) // CHUNK) % STRIDE == 0


def want_sampled(k):
    """Sampled keys the cut aims to keep at or above it: (k + 46 k / 100 + stride - 1) / stride in topk_fast_path."""
    return (k + (46 * k) // 100 + STRIDE - 1) // STRIDE


def paths_dataset(n_cols, n_parts=1, kinds="ABDEFGH", seed=0):
    """S = n_cols songs, split into n_parts song windows (distributed.song_window); every row kind is built inside each window from that
    window's own columns.  Test users come in one contiguous range per kind; ds.meta["kinds"][kind] = (u0, u1) and
    ds.meta["windows"][r] holds the columns each kind was given in window r."""
    rng = np.random.default_rng(seed)
    train = []                                                   # song lists of the train users
    listens = {kind: [[] for _ in range(N_USERS[kind])] for kind in kinds}
    windows = []
    for r in range(n_parts):
        lo, hi = song_window(n_cols, r, n_parts)
        samp = sampled(np.arange(hi - lo))
        free = np.ones(hi - lo, bool)

        def take(n, where=None, lowest=False):
            """n free window columns (global ids): sampled ones (where=True), unsampled ones (False) or any (None)."""
            cand = np.flatnonzero(free & (samp if where is True else ~samp if where is False else True))
            pick = cand[:n] if lowest else np.sort(rng.choice(cand, n, replace=False))
            free[pick] = False
            return pick + lo

        w = dict(lo=lo, hi=hi, cold=np.array(COLD) + lo)
        free[list(COLD)] = False
        free[-1] = "A" not in kinds                             # the last column goes to the A pool (and is open for H)
        for i, user in enumerate(listens.get("B", [])):
            user += list(w["cold"][i::3])
        if "F" in kinds:   # v* = {a, b} + tie, w = {a} + W: 2 / sqrt(|v*|) > 1 / sqrt(|w|), so for {a, b} the tie is above W
            a, b = take(2, False)
            w["w_low"] = take(N_W_LOW, False, lowest=True)    # keys a select keeping the first 2 048 met in column order would take
            w["w_sampled"] = take(N_W_SAMPLED, True)
            w["tie"] = take(N_TIE, False)
            train += [[a, b, *w["tie"]], [a, *w["w_low"], *w["w_sampled"]]]
            for user in listens["F"]:
                user += [a, b]
        if "E" in kinds:   # hi songs in two train users, lo songs in one: hi >= sqrt(2) * lo for both models
            w["hi_songs"], w["lo_songs"] = take(300, True), take(300, True)
            for user in listens["E"]:
                (e,) = take(1, False)
                train += [[e, *w["hi_songs"]], [e, *w["hi_songs"], *w["lo_songs"]]]
                user.append(e)
        if "G" in kinds:   # nested train users {g} + top[:j + 1] give the top songs 300 distinct scores, one more user the tie below them
            (g,) = take(1, False)
            top = rng.permutation(np.concatenate([take(N_TOP_SAMPLED, True), take(N_TOP - N_TOP_SAMPLED, False)]))
            w["top"], w["tie_g"] = top, np.concatenate([take(N_TIE_G_SAMPLED, True), take(N_TIE_G - N_TIE_G_SAMPLED, False)])
            train += [[g, *top[:j + 1]] for j in range(N_TOP)] + [[g, *top], [g, *w["tie_g"]]]
            for user in listens["G"]:
                user.append(g)
        if "D" in kinds:
            w["few"] = []
            for i, user in enumerate(listens["D"]):
                (d,) = take(1, False)
                p = take(D_SIZES[i], False if D_SIZES[i] == 1 else None)
                train += [[d, *p], [d, *p[::2]]]
                user.append(d)
                w["few"].append(p)
        if "A" in kinds:   # 60 train users, each with one of 12 anchors and ~30 % of a 3 200-song pool; anchors of distinct popularity
            anchors = take(12, False)
            w["pool"] = np.concatenate([[hi - 1], take(400 - samp[-1], True), take(2800 - (not samp[-1]), False)])
            for m in range(60):
                train.append([anchors[m % 12], *w["pool"][rng.random(len(w["pool"])) < 0.3]])
            train += [[anchors[j]] for j in range(12) for _ in range(j)]
            for i, user in enumerate(listens["A"]):
                user += [anchors[j] for j in range(12) if j % 3 != i % 3]
        if "H" in kinds:
            pool = np.sort(w["pool"])
            w["near_full_open"] = np.sort(np.concatenate([pool[np.linspace(0, len(pool) - 1, N_NEAR_FULL - len(COLD)).astype(int)], w["cold"]]))
            rest = np.setdiff1d(np.arange(lo, hi), w["near_full_open"])
            for user in listens["H"]:
                user += list(rest)
        windows.append(w)
    tests = [user for kind in kinds for user in listens[kind]]
    tr = (np.repeat(np.arange(len(train)), [len(t) for t in train]), np.concatenate([np.asarray(t, np.int64) for t in train]))
    te = (np.repeat(np.arange(len(tests)), [len(t) for t in tests]), np.concatenate([np.asarray(t, np.int64) for t in tests]))
    lab = (np.arange(len(tests)), np.full(len(tests), n_cols))             # one label-only song per user
    ds = from_triplets(tr, te, lab, len(train), len(tests), n_cols)
    bounds = np.cumsum([0] + [N_USERS[kind] for kind in kinds])
    ds.meta.update(kinds={kind: (int(bounds[i]), int(bounds[i + 1])) for i, kind in enumerate(kinds)}, windows=windows)
    return ds


def reference_models(oracle_lib, ds):
    ubm, ibm = oracle_lib.canon_scores(ds, oracle_lib.UBM), oracle_lib.canon_scores(ds, oracle_lib.IBM)
    return dict(ubm=ubm, ibm=ibm, lc=oracle_lib.blend_dense(oracle_lib.LC, 0.5, ubm, ibm), agg=oracle_lib.blend_dense(oracle_lib.AGG, 0.5, ubm, ibm),
                stoch=oracle_lib.blend_dense(oracle_lib.STOCH, 0.5, ubm, ibm, 42))


def window_topk(oracle_lib, model, lo, hi, k):
    """The oracle's ranking of the columns [lo, hi) of a dense model, with global song ids."""
    song, score, ln = oracle_lib.topk(np.ascontiguousarray(model[:, lo:hi]), k)
    return np.where(song >= 0, song + lo, song).astype(np.int32), score, ln


def hand_lists(ds, kind, k, lo=0, hi=None):
    """(song [n, k], len [n]) derived by hand inside window [lo, hi): for B the first k unlistened ids, for F the k smallest tie ids,
    for H (k >= 200) its 200 open songs in ascending order, then -1.  None for the other kinds."""
    hi = ds.S if hi is None else hi
    w = next(w for w in ds.meta["windows"] if w["lo"] == lo)
    u0, u1 = ds.meta["kinds"][kind]
    if kind not in "BFH" or (kind == "H" and k < N_NEAR_FULL):
        return None
    rows = []
    for u in range(u0, u1):
        heard = set(ds.te_col[ds.te_ptr[u]:ds.te_ptr[u + 1]].tolist())
        rows.append([s for s in range(lo, hi) if s not in heard][:k] if kind == "B" else list(w["tie" if kind == "F" else "near_full_open"][:k]))
    song = np.full((u1 - u0, k), -1, np.int32)
    for i, r in enumerate(rows):
        song[i, :len(r)] = r
    return song, np.array([len(r) for r in rows], np.int32)


def assert_hand_list(got, hand, kind, ctx=""):
    """A ranked list (song, score, len) against hand_lists: the same ids (H: the same set of open songs), all-zero scores for B, one
    tie score for F, -1 / 0.0 past the length."""
    song, score, ln = got
    np.testing.assert_array_equal(ln, hand[1], err_msg=ctx)
    if kind == "H":
        song = np.concatenate([np.sort(song[:, :N_NEAR_FULL], axis=1), song[:, N_NEAR_FULL:]], axis=1)
    np.testing.assert_array_equal(song, hand[0], err_msg=ctx)
    assert np.all(score[hand[0] == -1] == 0.0), ctx
    if kind == "B":
        assert np.all(score == 0.0), ctx
    if kind == "F":
        assert np.all(score == score[:, :1]) and np.all(score > 0), ctx


SHAPES = [(16384, 1, "ABDEFGH"), (16385, 1, "ABDEFGH"), (40000, 1, "ABDEFGH"), (50000, 3, "BDFG")]


@pytest.fixture(scope="module")
def built(oracle_lib):
    cache = {}

    def get(n_cols, n_parts, kinds):
        if (n_cols, n_parts) not in cache:
            ds = paths_dataset(n_cols, n_parts, kinds)
            cache[n_cols, n_parts] = ds, reference_models(oracle_lib, ds)
        return cache[n_cols, n_parts]
    return get


# ------------------------------------------------------------------------------------------------ CPU: the constructions hold
@pytest.mark.parametrize("n_cols,n_parts,kinds", SHAPES)
def test_row_kinds_have_their_properties(built, n_cols, n_parts, kinds):
    """Each kind's property, per song window, on the oracle's UBM, IBM and LC 0.5 scores."""
    ds, models = built(n_cols, n_parts, kinds)
    listened = ds.listened_mask()
    for w in ds.meta["windows"]:
        lo, hi = w["lo"], w["hi"]
        assert hi - lo >= LONG_ROW
        samp = sampled(np.arange(hi - lo))
        for name in ("ubm", "ibm", "lc"):
            rows = models[name][:, lo:hi]
            for kind, (u0, u1) in ds.meta["kinds"].items():
                for i, u in enumerate(range(u0, u1)):
                    row = rows[u]
                    pos = np.flatnonzero(row > 0)            # NaN (listened) compares false
                    vals = np.sort(row[pos])[::-1]
                    n_samp = int(samp[pos].sum())
                    ctx = f"{name} kind {kind} user {u} window {lo}"
                    if kind == "A":
                        assert len(pos) >= 1024 and n_samp >= want_sampled(1024), ctx
                    elif kind == "B":
                        assert len(pos) == 0 and np.all(row[~np.isnan(row)] == 0), ctx
                        assert set(np.flatnonzero(listened[u, lo:hi]) + lo) <= set(w["cold"].tolist()), ctx
                    elif kind == "D":
                        assert 1 <= len(pos) <= 60 and np.array_equal(pos + lo, w["few"][i]), ctx
                        assert n_samp < want_sampled(K), ctx                            # cut < 2
                    elif kind == "E":
                        assert len(pos) == 600 and n_samp == 600, ctx
                        # a log bin spans at most a factor 65/64 (6 mantissa bits), so the cut bin of the 92nd best sampled key starts
                        # at or above v92 * 64/65 and the collect pass keeps no more keys than lie there
                        v = vals[want_sampled(K) - 1]
                        assert np.count_nonzero(vals >= v * 64 / 65) < K, ctx
                    elif kind == "F":
                        top = vals[0]
                        tie = np.flatnonzero(row == top) + lo
                        assert np.array_equal(tie, w["tie"]) and not samp[tie - lo].any(), ctx
                        below = row[samp & (row > 0)]
                        assert len(below) >= 100 and below.max() < top, ctx          # every sampled key is below the tie
                        assert np.count_nonzero(pos + lo < tie[0]) >= CAP, ctx         # the first 2 048 keys met in column order miss it
                    elif kind == "G":
                        assert len(pos) == N_TOP + N_TIE_G, ctx
                        assert len(np.unique(vals[:N_TOP])) == N_TOP and vals[N_TOP - 1] > vals[N_TOP], ctx
                        assert np.all(vals[N_TOP:] == vals[K - 1]), ctx                # the tie holds rank 500
                        # fewer sampled keys than the cut wants above the tie, enough with it: the cut is the tie's bin, 900 collected
                        n_top_samp = int(samp[w["top"] - lo].sum())
                        assert n_top_samp < want_sampled(K) <= n_samp, ctx
                    elif kind == "H":
                        assert np.array_equal(np.flatnonzero(~listened[u, lo:hi]) + lo, w["near_full_open"]), ctx
                        assert n_samp < want_sampled(K), ctx


@pytest.mark.parametrize("n_cols,n_parts,kinds", SHAPES)
def test_oracle_gives_the_hand_derived_lists(built, oracle_lib, n_cols, n_parts, kinds):
    """The oracle's top-500 of kinds B, F and H (UBM, IBM, LC) is the list derived by hand, in every window."""
    ds, models = built(n_cols, n_parts, kinds)
    for w in ds.meta["windows"]:
        lo, hi = w["lo"], w["hi"]
        for name in ("ubm", "ibm", "lc"):
            for kind in "BFH":
                if kind not in ds.meta["kinds"]:
                    continue
                u0, u1 = ds.meta["kinds"][kind]
                assert_hand_list(window_topk(oracle_lib, models[name][u0:u1], lo, hi, K), hand_lists(ds, kind, K, lo, hi), kind,
                                 f"{name} kind {kind} window {lo}")


# ------------------------------------------------------------------------------------------------ GPU: each kind takes its path
def expected_counters(kind, n_cols, n):
    """(topk_fast_rejects, topk_short_rows, topk_degenerate_rows) of one top-500 call on n rows of the kind (UBM, IBM, LC)."""
    radix = n if kind in "BDF" else 0
    if n_cols <= LONG_ROW:
        return 0, n, radix
    return (n if kind in "BDEFH" else 0), 0, radix


def counters(mr):
    i = mr.info()
    return np.array([i["topk_fast_rejects"], i["topk_short_rows"], i["topk_degenerate_rows"]])


def assert_bits_equal(a, b):
    a = np.ascontiguousarray(a, np.float64)
    b = np.ascontiguousarray(b, np.float64)
    np.testing.assert_array_equal(a.view(np.int64), b.view(np.int64))


def assert_topk_equal(got, want, ctx):
    np.testing.assert_array_equal(got[2], want[2], err_msg=ctx)
    np.testing.assert_array_equal(got[0], want[0], err_msg=ctx)
    assert_bits_equal(got[1], want[1])


@pytest.mark.gpu
@pytest.mark.parametrize("n_cols", [16384, 16385, 40000])
def test_each_row_kind_takes_its_select_path(mrlib, oracle_lib, built, n_cols):
    """Per row kind (its user range as the shard, with its global pair index base): the lists of UBM, IBM, LC, AGG and STOCH equal
    the oracle's, the hand-derived lists too for B, F and H, and the select counters show the path of the kind at k = 500."""
    ds, models = built(n_cols, 1, "ABDEFGH")
    ks = (K, 1, 1024) if n_cols == 40000 else (K,)
    want = {(name, k): oracle_lib.topk(models[name], k) for _, name, _, _ in MODELS for k in ks}
    base = np.concatenate([[0], np.cumsum(ds.S - np.diff(ds.te_ptr))])
    with MusicRecommender(ds, **ITEM) as mr:
        for kind, (u0, u1) in ds.meta["kinds"].items():
            mr.set_test_users(ds.shard_test_users(u0, u1), int(base[u0]), ds.n_pairs)
            for k in ks:
                hand = hand_lists(ds, kind, k)
                for model, name, param, seed in MODELS:
                    ctx = f"kind {kind} model {name} k {k}"
                    before = counters(mr)
                    got = mr.getTopK(model, k=k, param=param, seed=seed)
                    delta = counters(mr) - before
                    assert_topk_equal(got, tuple(a[u0:u1] for a in want[name, k]), ctx)
                    if hand is not None and name in ("ubm", "ibm", "lc"):
                        assert_hand_list(got, hand, kind, ctx)
                    if k == K and name in ("ubm", "ibm", "lc"):
                        assert tuple(delta) == expected_counters(kind, n_cols, u1 - u0), ctx


@pytest.mark.gpu
def test_song_windows_take_the_long_row_paths_and_join(mrlib, oracle_lib, built):
    """S = 50 000 in three song windows of more than 16 384 columns, kinds B, D, F and G built in each window's own columns: every
    window's lists equal the oracle's ranking of its columns, and the device join of the three equals the oracle's global top-500
    (for the all-zero and tied rows the joined order comes from song ids across windows alone)."""
    ds, models = built(50000, 3, "BDFG")
    parts = {name: [] for _, name, _, _ in MODELS}
    for w in ds.meta["windows"]:
        lo, hi = w["lo"], w["hi"]
        with MusicRecommender(ds, song_window=(lo, hi), **ITEM) as mr:
            assert mr.info()["n_cols"] == hi - lo
            for model, name, param, seed in MODELS:
                got = mr.getTopK(model, k=K, param=param, seed=seed)
                assert_topk_equal(got, window_topk(oracle_lib, models[name], lo, hi, K), f"window {lo} model {name}")
                parts[name].append(got)
            if hi == ds.S:
                for _, name, _, _ in MODELS:
                    assert_topk_equal(merge_on_device(mr, parts[name], K), oracle_lib.topk(models[name], K), f"join model {name}")


def merge_on_device(mr, parts, k):
    import torch
    ps, pv, pl = (torch.from_numpy(np.stack([p[i] for p in parts])).cuda() for i in range(3))
    n = ps.shape[1]
    out = (torch.empty((n, k), dtype=torch.int32, device="cuda"), torch.empty((n, k), dtype=torch.float64, device="cuda"),
           torch.empty(n, dtype=torch.int32, device="cuda"))
    mr.mergeTopK(ps, pv, pl, *out)
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in out)
