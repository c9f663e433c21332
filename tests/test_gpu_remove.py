"""muse_group_remove: series leave a resident store in place.  The removed rows below the new size m take, in ascending order,
the kept rows at or above m.  After any sequence of appends, rolls and removals the store must be indistinguishable from a
fresh store that appended the resulting rows and label ids in their resulting order: the rows, every kind of run, bit for
bit, and the pairs the call returns must be that pairing.  GPU tests need a B200; the argument checks and the facade's host
paths at the end run without one."""
import contextlib
import ctypes as C
import gc

import numpy as np
import pytest

import muse_b200 as mb

gpu = pytest.mark.gpu
MODES = (mb.MODE_EXACT, mb.MODE_SCREEN, mb.MODE_AUTO)
PTR64 = C.POINTER(C.c_int64)


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _rows(rng, S, N):
    Y = rng.normal(size=(S, N)) * rng.uniform(0.1, 10.0, size=(S, 1)) + rng.uniform(-50, 50, size=(S, 1))
    for i in range(0, S, 3):
        m, w = int(rng.integers(0, N)), int(rng.integers(1, max(2, N // 20)))
        Y[i, m:m + w] += rng.uniform(5, 60)
    return Y


def _ref(rng, N):
    r = 0.1 * rng.random(N)
    r[N // 2 - max(1, N // 100): N // 2 + max(1, N // 100)] += 1.5
    return r


def _ids(S, offset=0):
    i = np.arange(offset, offset + S)
    return np.stack([i % 7, (i // 3) % 5], axis=1).astype(np.int32)


def _store(ctx, rows, ids, offset=0):
    st = mb.DeviceStore(ctx, rows.shape[1], 2, max(rows.shape[0], 1))
    if offset:
        st.set_global_offset(offset)
    st.append(rows, ids)
    return st


def _model(R, I, rows):
    """The documented pairing on the host: (rows and ids left, moved_from, moved_to).  Holes: the removed rows below
    m = S - len(rows); fillers: the kept rows at or above m; the j-th hole takes the j-th filler."""
    S = len(R)
    gone = set(int(r) for r in rows)
    m = S - len(gone)
    holes = sorted(r for r in gone if r < m)
    fillers = [r for r in range(m, S) if r not in gone]
    assert len(holes) == len(fillers)
    R2, I2 = R.copy(), I.copy()
    R2[holes], I2[holes] = R[fillers], I[fillers]
    return R2[:m], I2[:m], np.array(fillers, dtype=np.int64), np.array(holes, dtype=np.int64)


def _remove(st, R, I, rows):
    """Remove `rows` from the store and from the host model; checks the returned pairs against the model."""
    rows = np.sort(np.asarray(rows, dtype=np.int64))
    got_from, got_to = st.remove(rows)
    R, I, want_from, want_to = _model(R, I, rows)
    assert np.array_equal(got_from, want_from) and np.array_equal(got_to, want_to)
    return R, I


def _same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True), (x, y)


def _same_partials(a, b):
    a, b = np.sort(a, order=["group_key", "series_idx"]), np.sort(b, order=["group_key", "series_idx"])
    for f in mb.PARTIAL_DTYPE.names:
        assert np.array_equal(a[f], b[f], equal_nan=True), f


def _check_equivalent(ctx, got, R, I, ref, offset=0, old_batches=(), modes=MODES):
    """`got` (after appends, rolls and removals) against a fresh store of rows R with label ids I: rows, runs in every mode
    grouped by two keys and ungrouped with unsigned and signed scores and the path they took, filtered runs, grouped partials,
    score_all and the refined screening bounds -- all bit for bit."""
    S, N = R.shape
    assert got.size() == S
    if S:
        assert np.array_equal(got.read_rows(0, S), R, equal_nan=True)
    want = _store(ctx, R, I, offset)
    bw = mb.DeviceBatch(ctx, want, ref)
    max_lag = max(1, N // 4)
    for b in [mb.DeviceBatch(ctx, got, ref)] + list(old_batches):
        if S == 0:          # an empty store: no records, on the paths that do not screen
            for mode in (mb.MODE_EXACT, mb.MODE_AUTO):
                for keys in ([], [0, 1]):
                    assert len(b.run(keys, max_lag, 25, 0.0, mode=mode)[0]) == 0
                    assert len(bw.run(keys, max_lag, 25, 0.0, mode=mode)[0]) == 0
            continue
        for mode in modes:
            for keys in ([], [0, 1]):
                for signed in (False, True):
                    _same(b.run(keys, max_lag, 25, 0.1, mode=mode, signed_scores=signed),
                          bw.run(keys, max_lag, 25, 0.1, mode=mode, signed_scores=signed))
                    assert b.timing().mode == bw.timing().mode
                _same_partials(b.run_partial(keys, max_lag, 25, 0.1, mode=mode), bw.run_partial(keys, max_lag, 25, 0.1, mode=mode))
            for cols, vals in (([0], [int(I[0, 0])]), ([0, 1], [int(I[S // 2, 0]), int(I[S // 2, 1])])):
                for keys in ([], [1]):
                    _same(b.run_where(cols, vals, keys, max_lag, 25, 0.1, mode=mode),
                          bw.run_where(cols, vals, keys, max_lag, 25, 0.1, mode=mode))
                    assert b.timing().mode == bw.timing().mode
        _same(b.score_all(), bw.score_all())
        _same(b.score_all(signed_scores=True), bw.score_all(signed_scores=True))
        try:
            wb = bw.screen_bounds(refine=True, max_lag=max_lag)
        except mb.MuseError as e:          # the shape has no screening kernel: the same answer on both
            assert e.code == mb.MUSE_ERR_UNSUPPORTED
            with pytest.raises(mb.MuseError):
                b.screen_bounds(refine=True, max_lag=max_lag)
        else:
            _same(b.screen_bounds(refine=True, max_lag=max_lag), wb)
    want.close()


# N = 50: fp64 only; 100, 480: sub-warp; 1440: warp; 1441: odd (pad column); 3000, 10080: n = 4096 / 16384; 20000: long
SHAPES = [(50, 600), (100, 600), (480, 600), (1440, 600), (1441, 600), (3000, 300), (10080, 160), (20000, 48)]


def _pattern(name, S, rng):
    return {"first": [0], "middle": [S // 2], "last": [S - 1],
            "scattered": np.sort(rng.choice(S, S // 10, replace=False)),
            "block": np.arange(S // 3, S // 3 + S // 5),
            "tail": np.arange(S - S // 4, S),                       # exactly the tail: nothing moves
            "all_but_one": np.delete(np.arange(S), S // 3),
            "all": np.arange(S),
            "none": []}[name]


@gpu
@pytest.mark.parametrize("N,S", SHAPES)
@pytest.mark.parametrize("pattern", ["first", "middle", "last", "scattered", "block", "tail", "all_but_one", "all", "none"])
def test_removal_equals_fresh_store(ctx, N, S, pattern):
    rng = np.random.default_rng(N * 10 + len(pattern))
    R, I = _rows(rng, S, N), _ids(S)
    ref = _ref(rng, N)
    st = _store(ctx, R, I)
    before = mb.DeviceBatch(ctx, st, ref)          # a batch made before the removal sees the remaining rows
    rows = _pattern(pattern, S, rng)
    R2, I2 = _remove(st, R, I, rows)
    if pattern == "tail":
        assert np.array_equal(R2, R[:S - S // 4])
    _check_equivalent(ctx, st, R2, I2, ref, old_batches=[before])


@gpu
def test_larger_store_crosses_the_screening_rule(ctx):
    """20 000 rows down to 15 000 at N = 1440: AUTO screens before (>= 16384 rows) and scores exactly after, as a fresh store
    of the remaining rows does."""
    N, S = 1440, 20000
    rng = np.random.default_rng(11)
    R, I = _rows(rng, S, N), _ids(S)
    ref = _ref(rng, N)
    st = _store(ctx, R, I)
    b = mb.DeviceBatch(ctx, st, ref)
    b.run([], 60, 20, 0.3)
    assert b.timing().mode == mb.MODE_SCREEN
    R, I = _remove(st, R, I, np.sort(rng.choice(S, 5000, replace=False)))
    b.run([], 60, 20, 0.3)
    assert b.timing().mode == mb.MODE_EXACT
    _check_equivalent(ctx, st, R, I, ref, old_batches=[b], modes=(mb.MODE_AUTO, mb.MODE_SCREEN))


@gpu
def test_multi_run_on_tensor_cores_after_removal(ctx):
    """muse_multi_run on the tensor-core path (n = 2048, >= 16384 series, several queries) after a removal that keeps the store
    at or above 16384 rows equals it on a fresh store, and each query equals a batch made before the removal."""
    N, S = 1440, 20000
    st = mb.DeviceStore(ctx, N, 2, S)
    st.append_synthetic(S, 20261018, 0)
    i = np.arange(S)
    R, I = st.read_rows(0, S), np.stack([i // 1000, i % 1000], axis=1).astype(np.int32)
    rng = np.random.default_rng(9)
    refs = np.stack([mb.synth_reference(20261018, N), _ref(rng, N), mb.synth_row(20261018, 3, N)])
    before = [mb.DeviceBatch(ctx, st, r) for r in refs]
    R, I = _remove(st, R, I, np.sort(rng.choice(S, 3000, replace=False)))
    assert st.size() == 17000
    fresh = _store(ctx, R, I)
    got = mb.multi_run(st, refs, [], 60, 20, 0.3, mode=mb.MODE_SCREEN)
    n_refined, _ = mb.multi_last_stats(ctx)
    assert n_refined > 0                            # the tensor-core path ran
    want = mb.multi_run(fresh, refs, [], 60, 20, 0.3, mode=mb.MODE_SCREEN)
    for q in range(len(refs)):
        _same(got[q], want[q])
        _same(before[q].run([], 60, 20, 0.3, mode=mb.MODE_SCREEN), want[q])
    fresh.close()


@gpu
def test_more_pairs_than_one_chunk(ctx):
    """More than 2^20 rows move: the pairs reach the device in several chunks."""
    N, S = 50, 2_200_000
    st = mb.DeviceStore(ctx, N, 2, S)
    st.append_synthetic(S, 5, 0)
    i = np.arange(S)
    R, I = st.read_rows(0, S), np.stack([i // 1000, i % 1000], axis=1).astype(np.int32)
    rows = np.concatenate([np.arange(0, 1_099_990), np.arange(S - 10, S)])      # m = 1 100 000: 1 099 990 holes below m
    R, I = _remove(st, R, I, rows)
    assert np.array_equal(st.read_rows(0, len(R)), R)
    fresh = _store(ctx, R, I)
    ref = _ref(np.random.default_rng(1), N)
    b, bw = mb.DeviceBatch(ctx, st, ref), mb.DeviceBatch(ctx, fresh, ref)
    for keys in ([], [0, 1]):
        _same(b.run(keys, 10, 30, 0.2), bw.run(keys, 10, 30, 0.2))
    _same(b.score_all(), bw.score_all())
    fresh.close()
    st.close()


@gpu
@pytest.mark.parametrize("N", [480, 1441])
def test_sequences_of_appends_rolls_and_removals(ctx, N):
    S = 400
    rng = np.random.default_rng(N + 3)
    R, I = _rows(rng, S, N), _ids(S)
    ref = _ref(rng, N)
    st = _store(ctx, R, I)
    before = mb.DeviceBatch(ctx, st, ref)
    R, I = _remove(st, R, I, np.sort(rng.choice(S, 60, replace=False)))
    A, IA = _rows(rng, 50, N), _ids(50, 1000)      # append after removal: written at index m
    st.append(A, IA)
    R, I = np.concatenate([R, A]), np.concatenate([I, IA])
    _check_equivalent(ctx, st, R, I, ref, old_batches=[before], modes=(mb.MODE_SCREEN,))
    X = _rows(rng, len(R), 7)                       # roll after removal
    st.roll(X)
    R = np.concatenate([R[:, 7:], X], axis=1)
    R, I = _remove(st, R, I, [0, 5, len(R) - 3])    # removal after a roll
    for _ in range(3):                              # a chain of removals
        R, I = _remove(st, R, I, np.sort(rng.choice(len(R), int(rng.integers(1, 40)), replace=False)))
    _check_equivalent(ctx, st, R, I, ref, old_batches=[before])


@gpu
def test_nan_and_constant_rows_and_a_global_offset(ctx):
    """NaN and std-zero rows among the removed and among the moved rows, on a shard whose rows have global indices
    1000 + local; N odd, so the pad column moves with its row."""
    N, S, off = 1441, 600, 1000
    rng = np.random.default_rng(12)
    R, I = _rows(rng, S, N), _ids(S, off)
    ref = _ref(rng, N)
    R[11] = R[11] * 0.01 + 2.0 * ref + 3.0          # the top result, removed
    R[594] = R[594] * 0.01 + 2.0 * ref + 3.0        # the top result once 11 is gone, moved
    for r in (5, 590):
        R[r, 100] = np.nan
    for r in (7, 595):
        R[r] = 4.25
    st = _store(ctx, R, I, off)
    b = mb.DeviceBatch(ctx, st, ref)
    assert sorted(b.run([], N // 2, 2, 0.0)[2]) == [off + 11, off + 594]
    # m = 562; holes 5, 7, 11, 12, 13, 560, 561 take fillers 590, 593, 594, 595, 596, 597, 598
    rows = [5, 7, 11, 12, 13] + list(range(560, 590)) + [591, 592, 599]
    R, I = _remove(st, R, I, rows)
    assert np.isnan(R).any(axis=1).sum() == 1 and np.isnan(R[5]).any()      # the moved NaN row; the removed one is gone
    assert np.all(R[12] == 4.25) and (R == 4.25).all(axis=1).sum() == 1      # the moved constant row
    assert b.run([], N // 2, 1, 0.0)[2][0] == off + 11                       # 594 now sits at local 11
    _check_equivalent(ctx, st, R, I, ref, offset=off, old_batches=[b])


@gpu
def test_label_id_range_follows_the_remaining_rows(ctx):
    """Group-key widths come from the largest label id of each column: after the rows with large ids leave, grouped runs and
    the partials' group keys are a fresh store's, and a grouping that needed more than 64 key bits works again."""
    N, S = 100, 300
    rng = np.random.default_rng(13)
    R = _rows(rng, S, N)
    I = np.stack([np.arange(S) % 5, np.arange(S) % 3, np.arange(S) % 4], axis=1).astype(np.int32)
    I[40, 0] = 1 << 22                              # 23 bits: over the 21 of three fixed-width columns
    I[250] = (1 << 22) + 1                          # three 23-bit columns: 69 bits
    ref = _ref(rng, N)
    st = mb.DeviceStore(ctx, N, 3, S)
    st.append(R, I)
    b = mb.DeviceBatch(ctx, st, ref)
    with pytest.raises(mb.MuseError) as e:
        b.run([0, 1, 2], 20, 10, 0.1)
    assert e.value.code == mb.MUSE_ERR_UNSUPPORTED
    def partials(batch, keys):      # shards need fixed-width keys: MUSE_ERR_UNSUPPORTED while a column needs more
        try:
            return batch.run_partial(keys, 20, 10, 0.1)
        except mb.MuseError as e:
            return e.code

    for rows, fixed in (([250], False), ([40], True)):      # packed widths first, then fixed widths
        R, I = _remove(st, R, I, rows)
        fresh = mb.DeviceStore(ctx, N, 3, S)
        fresh.append(R, I)
        bf = mb.DeviceBatch(ctx, fresh, ref)
        for keys in ([0, 1, 2], [0, 2]):
            _same(b.run(keys, 20, 10, 0.1), bf.run(keys, 20, 10, 0.1))
            got, want = partials(b, keys), partials(bf, keys)
            if keys == [0, 1, 2] and not fixed:
                assert got == want == mb.MUSE_ERR_UNSUPPORTED
            else:
                _same_partials(got, want)
        bf.close()
        fresh.close()


@gpu
def test_held_bytes_do_not_grow_with_removals():
    @contextlib.contextmanager
    def held_unchanged():
        before = _held()
        yield
        assert _held() == before

    gc.collect()
    start = _held()
    N, S = 1440, 5000
    c = mb.Context(0)
    st = mb.DeviceStore(c, N, 2, S)
    rng = np.random.default_rng(2)
    st.append(rng.random((S, N)), np.zeros((S, 2), dtype=np.int32))      # pageable: the context's pinned staging ring
    st.remove(np.arange(0, 200, 2))                 # the first removal that moves rows: the context's pair buffer
    with held_unchanged():
        st.remove(np.sort(rng.choice(st.size(), 1500, replace=False)))
        st.remove(np.arange(st.size() - 10, st.size()))
        st.remove(np.arange(100, 1100))
        st.remove([])
        st.append(rng.random((2000, N)), np.zeros((2000, 2), dtype=np.int32))
    st.close()
    c.close()
    assert _held() == start


def _held():
    dev, pinned = C.c_int64(-1), C.c_int64(-1)
    mb._check(mb.lib().muse_held_bytes(C.byref(dev), C.byref(pinned)))
    return dev.value, pinned.value


def _p(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int64).ctypes.data_as(PTR64)


@gpu
def test_argument_errors_leave_the_store_untouched(ctx):
    N, S = 480, 100
    rng = np.random.default_rng(4)
    R, I = _rows(rng, S, N), _ids(S)
    st = _store(ctx, R, I)
    L = mb.lib()
    out = np.zeros(S + 2, dtype=np.int64)
    n = C.c_int64(99)
    bad = [(np.array([1, 2]), 2, out, out, None),        # n_moved NULL
           (None, 1, out, out, C.byref(n)),              # rows NULL
           (np.array([1]), -1, out, out, C.byref(n)),
           (np.arange(S + 1), S + 1, out, out, C.byref(n)),
           (np.array([-1, 3]), 2, out, out, C.byref(n)),
           (np.array([3, S]), 2, out, out, C.byref(n)),
           (np.array([3, 3]), 2, out, out, C.byref(n)),  # repeated
           (np.array([5, 3]), 2, out, out, C.byref(n)),  # out of order
           (np.array([3, 5]), 2, None, out, C.byref(n)),
           (np.array([3, 5]), 2, out, None, C.byref(n))]
    for rows, k, mf, mt, pn in bad:
        assert L.muse_group_remove(st.h, _p(rows), k, _p(mf), _p(mt), pn) == mb.MUSE_ERR_INVALID_ARG
        assert st.size() == S
    assert L.muse_group_remove(None, _p([1]), 1, _p(out), _p(out), C.byref(n)) == mb.MUSE_ERR_INVALID_ARG
    n.value = 99
    assert L.muse_group_remove(st.h, None, 0, None, None, C.byref(n)) == mb.MUSE_OK and n.value == 0      # nothing to do
    assert L.muse_group_remove(st.h, _p([S - 1]), 1, None, None, C.byref(n)) == mb.MUSE_OK and n.value == 0   # no pairs asked
    R, I = R[:S - 1], I[:S - 1]
    _check_equivalent(ctx, st, R, I, _ref(rng, N), modes=(mb.MODE_SCREEN,))


# ---- the Python facade ------------------------------------------------------------------------------------------------
def _series(rows, first=0, tag="h"):
    return [mb.NewSeries(rows[i], mb.NewLabels({"graph": "g%d" % ((first + i) % 9), tag: "%s%d" % (tag, first + i)}))
            for i in range(len(rows))]


@gpu
def test_group_remove_facade(ctx):
    N, S = 480, 300
    rng = np.random.default_rng(8)
    R = _rows(rng, S, N)
    ref = mb.NewSeries(_ref(rng, N))
    where = mb.NewLabels({"graph": "g4"})

    def run(group):
        b = mb.NewBatch(ref, group, mb.NewResults(100, 20, 0.1, mb.SignFilter_ANY), 1)
        b.Run(["graph"])
        got, _ = b.Results.Fetch()
        b.RunWhere(where)
        got2, _ = b.Results.Fetch()
        return [(s.Labels.ID(), s.Lag, s.PercentScore) for s in got + got2]

    def same_as_fresh(g):
        fresh = mb.NewGroup("fresh")
        fresh.Add(*[mb.NewSeries(s.Values(), s.Labels()) for s in g.series])
        assert g.Length() == fresh.Length() and len(g.registry) == len(g.series)
        assert [s.UID() for s in g.FilterByLabelValues(where)] == [s.UID() for s in fresh.FilterByLabelValues(where)]
        assert run(g) == run(fresh)

    g = mb.NewGroup("remove")
    members = _series(R[:250])
    g.Add(*members)
    b = mb.NewBatch(ref, g, mb.NewResults(100, 20, 0.1, mb.SignFilter_ANY), 1)
    store = g._store
    pending = _series(R[250:], 250)
    g.Add(*pending)                                 # not uploaded yet: Remove uploads them first
    order = members + pending
    gone = [order[i] for i in (0, 17, 18, 140, 260, 299)]
    g.Remove(*gone)
    _, _, moved_from, moved_to = _model(np.arange(S)[:, None], np.zeros((S, 1)), [0, 17, 18, 140, 260, 299])
    for f, t in zip(moved_from, moved_to):
        order[t] = order[f]
    order = order[:S - len(gone)]
    assert g.series == order and g._store is store       # the pairs applied on the host; the store kept
    assert all(g.registry[s.UID()] == i for i, s in enumerate(g.series))
    same_as_fresh(g)
    b.Run(None)                                     # the batch made before the removal still runs
    # the only series with the key "colo" leaves: the key keeps its column, the store is not rebuilt
    extra = mb.NewSeries(_rows(rng, 1, N)[0], mb.NewLabels({"graph": "g4", "colo": "c1"}))
    g.Add(extra)
    same_as_fresh(g)
    store = g._store
    g.Remove(extra)
    assert g._store is store
    same_as_fresh(g)
    # remove then add of the same UID replaces a series
    s = g.series[3]
    g.Remove(s)
    g.Add(mb.NewSeries(R[0] * 2.0 + 1.0, s.Labels()))
    same_as_fresh(g)
    g.Remove(s)                                     # by UID: the new member
    with pytest.raises(mb.MuseError):
        g.Remove(s)
    same_as_fresh(g)


# ---- without a device ----------------------------------------------------------------------------------------------------
def test_remove_abi_rejects_a_null_group_without_a_device():
    mb.build()
    L = mb.lib()
    n = C.c_int64(0)
    assert L.muse_group_remove(None, _p([0]), 1, None, None, C.byref(n)) == mb.MUSE_ERR_INVALID_ARG
    assert L.muse_group_remove(None, None, 0, None, None, None) == mb.MUSE_ERR_INVALID_ARG


def test_group_remove_before_any_upload_keeps_add_order(monkeypatch):
    g = mb.NewGroup("cpu")

    def no_device():
        raise AssertionError("a removal without a store needs no device")

    monkeypatch.setattr(g, "_sync_device", no_device)
    S = _series(np.arange(60.0).reshape(6, 10))
    g.Add(*S)
    with pytest.raises(mb.MuseError) as e:         # a stranger: nothing is removed
        g.Remove(S[1], mb.NewSeries(np.zeros(10), mb.NewLabels({"graph": "g1", "h": "nobody"})))
    assert e.value.code == mb.MUSE_ERR_INVALID_ARG and g.series == S
    g.Remove(S[1], S[4], S[1])
    assert g.series == [S[0], S[2], S[3], S[5]] and g.registry == {s.UID(): i for i, s in enumerate(g.series)}
    g.Add(mb.NewSeries(np.ones(10), S[4].Labels()))        # remove then add of a UID
    assert g.series[-1].UID() == S[4].UID() and g.registry[S[4].UID()] == 4
    g.Remove(*g.series)                            # empty again: the length is free, as in a new Group
    assert g.Length() == 0 and g.series == [] and g.registry == {}
    g.Add(mb.NewSeries(np.ones(7), mb.NewLabels({"a": "b"})))
    assert g.Length() == 7
