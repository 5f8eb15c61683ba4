"""The narrow counters of the exact scoring (DESIGN.md §3), crossed on purpose: constructed data sets put chosen entries just below and
just at or above each counter's width, the CPU tests show from the oracle that they sit there, and the GPU tests show that the scores
and lists stay bit-exact and read the library's counters (mr_get_info) to show that each data set took its path.

  carry       sparse user-space IBM panel Wi, u32: one train user shares n songs of visible degree 2 with each of five test users (batch
              rows 0, 1, 127 of the first batch, 1 and 127 of the second), so Wi = n q_26(2); n just below the first wrap, at it, at the
              second.  Every wrap is a carry event that carry_fixup_kernel pays back with 2^32.
  overflow    the same under a carry list of one entry (MRSCORE_CARRY_CAP): the call fails, and a shard without carries then scores
  u16 panel   user-space UBM count panel Ct, u16 pairs in one 32-bit word: two test users (rows 0 and 1) with 65 535 songs, all shared
              with one train user; a user with 65 536 songs is refused
  split       item-space head rows: a head song whose listeners all have two songs is built in place while its weighted listener sum is
              below 2^32 and staged, with exception entries, from there on
  u16 rows    two staged head songs with 65 535 and 65 536 common listeners (the 16-bit count row)
  packed      the staged rows' 64-bit accumulator, packed (count in bits 44..63) only while every train degree is < 2^20 and every
              weighted listener sum < 2^44: about 2^20 one-song train users on one song, on each side of both conditions
  planes      the tensor engine's byte-plane GEMMs of the weights q_24(|I_v|): a one-song train user has q_24 = 2^24, a fourth byte
  int select  the UBM top-k may rank the integers when every user's numerator is < 2^52: a cheap bound (longest row x largest weighted
              listener sum) fails, the exact per-user sums decide; MRSCORE_UBM_FP64_SELECT forces the fp64 select, with the same lists
"""
import numpy as np
import pytest

from musicrecommendation_b200 import _lib
from musicrecommendation_b200.dataset import from_triplets
from musicrecommendation_b200.recommender import MusicRecommender

K = 100
SPARSE_USER = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_USER)
SPARSE_ITEM = dict(engine=_lib.MR_ENGINE_SPARSE, space=_lib.MR_SPACE_ITEM)
TENSOR_USER = dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_USER)
TENSOR_ITEM = dict(engine=_lib.MR_ENGINE_TENSOR, space=_lib.MR_SPACE_ITEM)
POOL = 300                  # background songs of the item-space constructions


# ------------------------------------------------------------------------------------------------ constructions
def lists_to_pairs(lists, base=0):
    rows = np.repeat(np.arange(base, base + len(lists)), [len(t) for t in lists])
    cols = np.concatenate([np.asarray(t, np.int64) for t in lists]) if lists else np.zeros(0, np.int64)
    return rows.astype(np.int64), cols


def dataset(train, tests, S, T=None):
    """train / tests: lists of song lists, or (rows, cols) pair arrays for train; one label-only song per test user."""
    tr = train if isinstance(train, tuple) else lists_to_pairs(train)
    T = int(tr[0].max()) + 1 if T is None else T
    te = lists_to_pairs(tests)
    lab = (np.arange(len(tests)), np.full(len(tests), S))
    return from_triplets(tr, te, lab, T, len(tests), S)


def train_weights(oracle_lib, ds):
    """q_24(|I_v|) per train user, exact (oracle.q)."""
    degs, inv = np.unique(ds.deg_tr, return_inverse=True)
    return np.array([oracle_lib.q(int(d), oracle_lib.UBM) for d in degs], np.int64)[inv]


def train_users_of_entries(ds):
    return np.repeat(np.arange(ds.T), np.diff(ds.tr_ptr))


def weighted_rows(oracle_lib, ds, rows):
    """Gq[r][s] = sum of q_24(|I_v|) over the train users v who listened to rows[r] and to s: the UBM head rows, exact."""
    qv, user = train_weights(oracle_lib, ds), train_users_of_entries(ds)
    out = np.zeros((len(rows), ds.S), np.int64)
    for i, r in enumerate(rows):
        sel = np.isin(user, user[ds.tr_col == r])
        np.add.at(out[i], ds.tr_col[sel], qv[user[sel]])
    return out


def song_qsum(oracle_lib, ds):
    """Per song: the sum of q_24(|I_v|) over its train listeners (the bound of every weighted head-row entry of the song)."""
    out = np.zeros(ds.S, np.int64)
    np.add.at(out, ds.tr_col, train_weights(oracle_lib, ds)[train_users_of_entries(ds)])
    return out


def exceptions(oracle_lib, ds, rows):
    """Entries of the staged rows that leave the 6-byte form: count >= 2^16 or weighted sum >= 2^32."""
    g, gq = oracle_lib.gram_rows(ds, rows), weighted_rows(oracle_lib, ds, rows)
    return int(np.count_nonzero((g >= 1 << 16) | (gq >= 1 << 32)))


def with_pool(tests, head_songs, n_pool_users=40, seed=0):
    """Adds POOL background songs after the head_songs construction songs: 40 train users with 30 of them each, and 5 of them to every
    listed test user (plus two test users of pool songs only).  No pool song reaches 41 listeners."""
    rng = np.random.default_rng(seed)
    pool = np.arange(head_songs, head_songs + POOL)
    bg = [np.sort(rng.choice(pool, 30, replace=False)) for _ in range(n_pool_users)]
    tests = [sorted(t) + sorted(rng.choice(pool, 5, replace=False).tolist()) for t in tests] + \
            [sorted(rng.choice(pool, 8, replace=False).tolist()) for _ in range(2)]
    return bg, tests, head_songs + POOL


# carry: five wrapping test users and 255 users of two private songs each; rows 256..259 are the clean shard of the recovery test
CARRY_ROWS = (0, 1, 127, 129, 255)
CARRY_U, CLEAN = 260, (256, 260)
N_X, N_Y = 64, 32


def carry_cases(oracle_lib):
    """n just below the first wrap of n q_26(2), at it, at the second."""
    q = oracle_lib.q(2, oracle_lib.IBM)
    first, second = -(-(1 << 32) // q), -(-(1 << 33) // q)
    return first - 1, first, second


def carry_dataset(n):
    """v0 listens to every wrapping user's block of n songs and to X; v1 to the fillers' songs and Y; v2 to one more song z_b of each
    wrapping user, X[:32] and Y[:16].  Every block song and z_b has visible degree 2."""
    blocks = {u: list(range(i * n, (i + 1) * n)) for i, u in enumerate(CARRY_ROWS)}
    nxt = len(CARRY_ROWS) * n
    X = list(range(nxt, nxt + N_X)); nxt += N_X
    Z = {u: nxt + i for i, u in enumerate(CARRY_ROWS)}; nxt += len(CARRY_ROWS)
    tests, F = [], []
    for u in range(CARRY_U):
        if u in blocks:
            tests.append(blocks[u] + [Z[u]])
        else:
            tests.append([nxt, nxt + 1]); F += [nxt, nxt + 1]; nxt += 2
    Y = list(range(nxt, nxt + N_Y)); nxt += N_Y
    train = [sum(blocks.values(), []) + X, F + Y, list(Z.values()) + X[:32] + Y[:16]]
    ds = dataset(train, tests, nxt)
    ds.meta.update(n=n, X=np.array(X))
    return ds


# u16 count panel: two test users with 65 535 songs, all listened to by train user v0
U16 = (1 << 16) - 1


def u16_dataset():
    S = U16 + 200
    E0, E1 = list(range(U16, U16 + 100)), list(range(U16 + 100, U16 + 200))
    train = [list(range(U16)) + E0, list(range(50)) + E1]
    tests = [list(range(U16)), list(range(U16)), list(range(10)) + E1[:5]]
    return dataset(train, tests, S)


def split_cases(oracle_lib):
    """Listeners of the boundary head song (two songs each): the most with a weighted sum < 2^32, and one more."""
    n = ((1 << 32) - 1) // oracle_lib.q(2, oracle_lib.UBM)
    return n, n + 1


def pair_song_dataset(n_pair, n_single=0, seed=0, pool_users=40):
    """Songs 0 and 1: n_pair train users listen to both, n_single more to song 0 only; then the pool.  Test users: two with song 0,
    two with song 1, one with both, two with pool songs only."""
    bg, tests, S = with_pool([[0], [0], [1], [1], [0, 1]], 2, pool_users, seed)
    T0 = n_pair + n_single
    rows = np.concatenate([np.repeat(np.arange(n_pair), 2), np.arange(n_pair, T0), *[np.full(len(b), T0 + i) for i, b in enumerate(bg)]])
    cols = np.concatenate([np.tile([0, 1], n_pair), np.zeros(n_single, np.int64), *bg])
    return dataset((rows.astype(np.int64), cols.astype(np.int64)), tests, S, T0 + len(bg))


PACKED_PAIRS = 70000         # two-song users on songs 0 and 1: G[0][1] >= 2^16 and Gq[0][1] >= 2^32 in every case


def packed_cases(oracle_lib):
    """One-song users on song 0 next to PACKED_PAIRS two-song users: train degree of song 0 = 2^20 - 1 (packed), = 2^20 (only the degree
    rule fails), the largest weighted sum < 2^44 (degree > 2^20), the smallest >= 2^44."""
    q1, q2 = oracle_lib.q(1, oracle_lib.UBM), oracle_lib.q(2, oracle_lib.UBM)
    below = ((1 << 44) - 1 - PACKED_PAIRS * q2) // q1
    return dict(deg_below=(1 << 20) - 1 - PACKED_PAIRS, deg_at=(1 << 20) - PACKED_PAIRS, qsum_below=below, qsum_at=below + 1)


def planes_dataset(one_song_users, seed=1):
    rng = np.random.default_rng(seed)
    S = 400
    train = [np.sort(rng.choice(S, 30, replace=False)).tolist() for _ in range(60)] + [[s] for s in range(one_song_users)]
    tests = [np.sort(rng.choice(S, 6, replace=False)).tolist() for _ in range(8)]
    return dataset(train, tests, S)


# int select: a long test row of L songs next to a song p of n one-song train users, with n q_24(1) L >= 2^52
INT_L = 1 << 14


def int_select_dataset(oracle_lib):
    n = -(-(1 << 52) // (oracle_lib.q(1, oracle_lib.UBM) * INT_L))
    p, E = INT_L, list(range(INT_L + 1, INT_L + 65))
    chunk = INT_L // 32
    train = [list(range(c * chunk, (c + 1) * chunk)) + [E[c], E[c + 32]] for c in range(32)] + [[p]] * n
    tests = [list(range(INT_L)), [p] + E[:3], list(range(0, INT_L, INT_L // 20))]
    ds = dataset(train, tests, INT_L + 65)
    ds.meta.update(p=p, n_single=n)
    return ds


# ------------------------------------------------------------------------------------------------ references
@pytest.fixture(scope="module")
def built(oracle_lib):
    cache = {}

    def get(name, arg=None):
        if (name, arg) not in cache:
            ds = dict(carry=lambda: carry_dataset(arg), u16=u16_dataset, pair=lambda: pair_song_dataset(*arg),
                      planes=lambda: planes_dataset(arg), int_select=lambda: int_select_dataset(oracle_lib))[name]()
            cache[name, arg] = ds
        return cache[name, arg]
    return get


def reference(oracle_lib, ds, u0=0, u1=None):
    ubm, ibm = oracle_lib.canon_scores(ds, oracle_lib.UBM, u0, u1), oracle_lib.canon_scores(ds, oracle_lib.IBM, u0, u1)
    return dict(ubm=ubm, ibm=ibm, lc=oracle_lib.blend_dense(oracle_lib.LC, 0.5, ubm, ibm))


def assert_bits_equal(got, want, ctx):
    got, want = np.ascontiguousarray(got, np.float64), np.ascontiguousarray(want, np.float64)
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want), err_msg=ctx)
    np.testing.assert_array_equal(np.nan_to_num(got).view(np.int64), np.nan_to_num(want).view(np.int64), err_msg=ctx)


def assert_models(mr, oracle_lib, ref, ctx=""):
    """Dense UBM, IBM and LC 0.5, then the top-K of UBM, LC and IBM (IBM last: the carry counter reads that call), bit for bit."""
    ubm, ibm = mr.getUserBasedModel(), mr.getItemBasedModel()
    assert_bits_equal(ubm.scores, ref["ubm"], f"{ctx} dense ubm")
    assert_bits_equal(ibm.scores, ref["ibm"], f"{ctx} dense ibm")
    assert_bits_equal(mr.getLinearCombinationModel(ubm, ibm, 0.5).scores, ref["lc"], f"{ctx} dense lc")
    for model, name in ((_lib.MR_UBM, "ubm"), (_lib.MR_LC, "lc"), (_lib.MR_IBM, "ibm")):
        song, score, ln = mr.getTopK(model, k=K, param=0.5)
        ws, wv, wl = oracle_lib.topk(ref[name], K)
        np.testing.assert_array_equal(ln, wl, err_msg=f"{ctx} top-k {name}")
        np.testing.assert_array_equal(song, ws, err_msg=f"{ctx} top-k {name}")
        assert_bits_equal(score, wv, f"{ctx} top-k {name}")


# ------------------------------------------------------------------------------------------------ CPU: the constructions hold
def test_carry_cases_sit_on_both_sides_of_each_wrap(oracle_lib, built):
    """Wi[v0][b] = n q_26(2) for every wrapping user, seen in the oracle's IBM numerators at the songs of X that only v0 shares with
    them: below 2^32, then wrapping once, then twice; the fillers and clean users never reach 2^32."""
    q = oracle_lib.q(2, oracle_lib.IBM)
    for wraps, n in enumerate(carry_cases(oracle_lib)):
        ds = built("carry", n)
        assert np.all(ds.deg_song[:len(CARRY_ROWS) * n] == 2)
        sint = oracle_lib.canon_sint(ds, oracle_lib.IBM)
        X = ds.meta["X"]
        for u in CARRY_ROWS:
            assert np.all(sint[u, X[32:]] == n * q) and np.all(sint[u, X[:32]] == (n + 1) * q)
        assert (n * q) >> 32 == wraps and ((n + 1) * q >> 32 == 1 if wraps == 0 else (n - 1) * q >> 32 == wraps - 1)
        assert sint[[u for u in range(CARRY_U) if u not in CARRY_ROWS]].max() < 1 << 32


def test_u16_panel_rows_hold_the_largest_count(oracle_lib, built):
    ds = built("u16")
    c = oracle_lib.counts_ubm(ds)
    assert c[0, 0] == c[1, 0] == U16 == (1 << 16) - 1 and c.max() == U16
    assert np.diff(ds.te_ptr).max() == U16


def test_split_boundary_song(oracle_lib, built):
    """The boundary song's weighted listener sum, which is its row's largest entry (at the other pair song), is below 2^32 with n
    listeners and not with n + 1; its listeners all have two songs, and no pool song reaches the head-degree cut."""
    for n, staged in zip(split_cases(oracle_lib), (False, True)):
        ds = built("pair", (n, 0))
        qsum = song_qsum(oracle_lib, ds)
        gq = weighted_rows(oracle_lib, ds, [0, 1])
        assert gq[0, 1] == gq.max() == qsum[0] == qsum[1] == n * oracle_lib.q(2, oracle_lib.UBM)
        assert (qsum[0] >= 1 << 32) == staged and np.all(ds.deg_tr[:n] == 2)
        assert np.bincount(ds.tr_col, minlength=ds.S)[2:].max() < split_cases(oracle_lib)[0]
        # the user of song 0 alone: its UBM numerator at song 1 is that entry
        assert oracle_lib.canon_sint(ds, oracle_lib.UBM, 0, 1)[0, 1] == gq[0, 1]
        assert exceptions(oracle_lib, ds, [0, 1]) == (4 if staged else 0)


@pytest.mark.parametrize("m", [U16, U16 + 1])
def test_u16_row_counts(oracle_lib, built, m):
    ds = built("pair", (m, 0))
    g = oracle_lib.gram_rows(ds, [0, 1])
    assert g[0, 1] == g[1, 0] == m and ((g[0, 1] >> 16) == (m > U16))
    assert song_qsum(oracle_lib, ds)[1] >= 1 << 32                    # both rows are staged
    assert exceptions(oracle_lib, ds, [0, 1]) == 4


def test_packed_cases(oracle_lib):
    """Train degree and weighted listener sum of song 0 on the intended side of 2^20 and 2^44 (no other song comes close)."""
    want = dict(deg_below=(True, True), deg_at=(False, True), qsum_below=(False, True), qsum_at=(False, False))
    for case, n_single in packed_cases(oracle_lib).items():
        ds = pair_song_dataset(PACKED_PAIRS, n_single)
        deg = np.bincount(ds.tr_col, minlength=ds.S)
        qsum = song_qsum(oracle_lib, ds)
        assert deg.argmax() == qsum.argmax() == 0
        assert (deg[0] < 1 << 20, qsum[0] < 1 << 44) == want[case], case
        q1 = oracle_lib.q(1, oracle_lib.UBM)
        if case in ("deg_below", "deg_at"):
            assert deg[0] == (1 << 20) - (case == "deg_below")
        elif case == "qsum_below":
            assert qsum[0] < 1 << 44 <= qsum[0] + q1                 # one more one-song listener crosses
        else:
            assert qsum[0] - q1 < 1 << 44 <= qsum[0]


@pytest.mark.parametrize("one_song", [0, 6])
def test_plane_weights(oracle_lib, built, one_song):
    ds = built("planes", one_song)
    qmax = int(train_weights(oracle_lib, ds).max())
    assert (qmax >> 24 != 0) == (one_song > 0) and qmax >> 16 != 0


def test_int_select_cheap_bound_fails_exact_sums_hold(oracle_lib, built):
    ds = built("int_select")
    qsum = song_qsum(oracle_lib, ds)
    longest = int(np.diff(ds.te_ptr).max())
    assert int(qsum.max()) * longest >= 1 << 52
    per_user = [int(qsum[ds.te_col[ds.te_ptr[u]:ds.te_ptr[u + 1]]].sum()) for u in range(ds.U)]
    assert max(per_user) < 1 << 52
    assert np.all(oracle_lib.canon_sint(ds, oracle_lib.UBM).max(axis=1) <= per_user)


# ------------------------------------------------------------------------------------------------ GPU: exact, and on the path
@pytest.mark.gpu
@pytest.mark.parametrize("case", [0, 1, 2])
def test_carry_events_are_paid_back(mrlib, oracle_lib, built, case):
    """Sparse user-space IBM with 0, 1 and 2 wraps of Wi per wrapping user: scores and lists bit-exact (listened pairs NaN / never
    ranked), carry_events = wraps x wrapping users for every IBM call and 0 for a UBM call."""
    n = carry_cases(oracle_lib)[case]
    ds = built("carry", n)
    ref = reference(oracle_lib, ds)
    events = len(CARRY_ROWS) * ((n * oracle_lib.q(2, oracle_lib.IBM)) >> 32)
    assert events == len(CARRY_ROWS) * case
    with MusicRecommender(ds, **SPARSE_USER) as mr:
        assert_models(mr, oracle_lib, ref, f"n {n}")
        assert mr.info()["carry_events"] == events
        mr.getItemBasedModel()
        assert mr.info()["carry_events"] == events
        mr.getTopK(_lib.MR_UBM, k=K)
        assert mr.info()["carry_events"] == 0


@pytest.mark.gpu
def test_carry_overflow_fails_the_call_and_the_next_shard_scores(mrlib, oracle_lib, built, monkeypatch):
    """A carry list of one entry: the IBM call over the wrapping users returns MR_ERR_OOM; then, on the same handle, a shard without
    carries scores and ranks bit-exactly (the overflow belongs to the call that met it)."""
    ds = built("carry", carry_cases(oracle_lib)[2])
    monkeypatch.setenv("MRSCORE_CARRY_CAP", "1")
    with MusicRecommender(ds, **SPARSE_USER) as mr:
        for call in (lambda: mr.getTopK(_lib.MR_IBM, k=K), mr.getItemBasedModel):
            with pytest.raises(_lib.MrError) as err:
                call()
            assert err.value.code == _lib.MR_ERR_OOM and "carry list overflowed" in err.value.msg
        u0, u1 = CLEAN
        mr.set_test_users(ds.shard_test_users(u0, u1))
        assert_models(mr, oracle_lib, reference(oracle_lib, ds, u0, u1), "clean shard")
        assert mr.info()["carry_events"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("engine", [SPARSE_USER, TENSOR_USER], ids=["sparse", "tensor"])
def test_u16_count_panel_at_its_largest_count(mrlib, oracle_lib, built, engine):
    ds = built("u16")
    with MusicRecommender(ds, **engine) as mr:
        assert mr.info()["space"] == _lib.MR_SPACE_USER
        np.testing.assert_array_equal(mr.counts_ubm(), oracle_lib.counts_ubm(ds))
        assert_models(mr, oracle_lib, reference(oracle_lib, ds), "u16 panel")


@pytest.mark.gpu
def test_user_with_65536_songs_is_refused(mrlib, built):
    ds = built("u16")
    bad = dataset([list(range(U16)), list(range(50))], [list(range(10)), list(range(U16 + 1))], ds.S)
    with MusicRecommender(ds, **SPARSE_USER) as mr:
        with pytest.raises(_lib.MrError) as err:
            mr.set_test_users(bad)
        assert err.value.code == _lib.MR_ERR_BAD_ARG and "test user 1 has more than 65535" in err.value.msg


@pytest.mark.gpu
@pytest.mark.parametrize("staged", [False, True])
def test_direct_and_staged_split_at_2_32(mrlib, oracle_lib, built, staged):
    """Head rows = the two pair songs (MR_OPT_HEAD_MIN_DEG): in place with n listeners, staged with 4 exception entries with n + 1."""
    n = split_cases(oracle_lib)[staged]
    ds = built("pair", (n, 0))
    with MusicRecommender(ds, head_min_deg=split_cases(oracle_lib)[0], **SPARSE_ITEM) as mr:
        assert_models(mr, oracle_lib, reference(oracle_lib, ds), f"split n {n}")
        i = mr.info()
        assert (i["n_head"], i["head_staged_rows"], i["head_exceptions"]) == (2, 2 * staged, exceptions(oracle_lib, ds, [0, 1]))


@pytest.mark.gpu
@pytest.mark.parametrize("m", [U16, U16 + 1])
def test_u16_head_row_exceptions(mrlib, oracle_lib, built, m):
    ds = built("pair", (m, 0))
    with MusicRecommender(ds, **SPARSE_ITEM) as mr:
        assert_models(mr, oracle_lib, reference(oracle_lib, ds), f"u16 rows m {m}")
        i = mr.info()
        assert (i["head_staged_rows"], i["head_exceptions"], i["head_packed"]) == (2, 4, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["deg_below", "deg_at", "qsum_below", "qsum_at"])
def test_packed_accumulator_chosen_from_data(mrlib, oracle_lib, case, monkeypatch):
    monkeypatch.delenv("MRSCORE_PRECOMPUTE_UNPACKED", raising=False)
    ds = pair_song_dataset(PACKED_PAIRS, packed_cases(oracle_lib)[case])
    with MusicRecommender(ds, **SPARSE_ITEM) as mr:
        assert_models(mr, oracle_lib, reference(oracle_lib, ds), case)
        i = mr.info()
        assert (i["head_packed"], i["head_staged_rows"], i["head_exceptions"]) == (case == "deg_below", 2, exceptions(oracle_lib, ds, [0, 1]))


@pytest.mark.gpu
@pytest.mark.parametrize("one_song", [0, 6])
def test_tensor_head_rows_take_a_fourth_byte_plane(mrlib, oracle_lib, built, one_song):
    ds = built("planes", one_song)
    with MusicRecommender(ds, **TENSOR_ITEM) as mr:
        assert_models(mr, oracle_lib, reference(oracle_lib, ds), f"planes one_song {one_song}")
        assert mr.info()["head_planes"] == (4 if one_song else 3)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", [SPARSE_USER, SPARSE_ITEM], ids=["user", "item"])
def test_ubm_int_select_from_exact_sums_and_fp64_select(mrlib, oracle_lib, built, engine, monkeypatch):
    """The exact per-user sums keep the integer select (flag 1); MRSCORE_UBM_FP64_SELECT gives the fp64 select (flag 0) the same lists."""
    ds = built("int_select")
    ref = reference(oracle_lib, ds)
    lists = {}
    for forced in (False, True):
        if forced:
            monkeypatch.setenv("MRSCORE_UBM_FP64_SELECT", "1")
        with MusicRecommender(ds, **engine) as mr:
            assert mr.info()["ubm_int_ok"] == (0 if forced else 1)
            assert_models(mr, oracle_lib, ref, f"forced {forced}")
            lists[forced] = [mr.getTopK(m, k=K, param=0.5) for m in (_lib.MR_UBM, _lib.MR_LC)]
    for a, b in zip(lists[False], lists[True]):
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)
