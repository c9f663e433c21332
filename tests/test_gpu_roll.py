"""muse_group_roll: every series of a resident store slides forward by k new samples, in place on the device.  After any
sequence of appends and rolls the store must be indistinguishable from a fresh store that appended the resulting rows with
the same labels: the rows, every kind of run, bit for bit.  GPU tests need a B200; the argument checks at the end run
without one."""
import ctypes as C

import numpy as np
import pytest

import muse_b200 as mb

gpu = pytest.mark.gpu
MODES = (mb.MODE_EXACT, mb.MODE_SCREEN, mb.MODE_AUTO)


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


def _store(ctx, rows, offset=0):
    st = mb.DeviceStore(ctx, rows.shape[1], 2, rows.shape[0])
    if offset:
        st.set_global_offset(offset)
    st.append(rows, _ids(rows.shape[0], offset))
    return st


def _rolled(R, X, first=0):
    """What a roll of rows [first, first + len(X)) by k = X.shape[1] leaves in R (host model)."""
    R = R.copy()
    k = X.shape[1]
    if len(X) and k:
        R[first:first + len(X)] = np.concatenate([R[first:first + len(X), k:], X], axis=1)
    return R


def _same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True), (x, y)


def _check_equivalent(ctx, got, R, ref, offset=0, old_batches=(), modes=MODES):
    """`got` (after appends and rolls) against a fresh store of rows R: rows, runs in every mode grouped and ungrouped with
    unsigned and signed scores, score_all and the refined screening bounds -- all bit for bit."""
    S, N = R.shape
    assert got.size() == S
    assert np.array_equal(got.read_rows(0, S), R, equal_nan=True)
    want = _store(ctx, R, offset)
    bw = mb.DeviceBatch(ctx, want, ref)
    max_lag = max(1, N // 4)
    for b in [mb.DeviceBatch(ctx, got, ref)] + list(old_batches):
        for mode in modes:
            for keys in ([], [0, 1]):
                for signed in (False, True):
                    _same(b.run(keys, max_lag, 25, 0.1, mode=mode, signed_scores=signed),
                          bw.run(keys, max_lag, 25, 0.1, mode=mode, signed_scores=signed))
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


@gpu
@pytest.mark.parametrize("N,S", SHAPES)
@pytest.mark.parametrize("kk", ["1", "7", "N-1", "N"])
def test_roll_whole_store_equals_fresh_store(ctx, N, S, kk):
    k = {"1": 1, "7": 7, "N-1": N - 1, "N": N}[kk]
    rng = np.random.default_rng(N * 10 + k)
    R = _rows(rng, S, N)
    ref = _ref(rng, N)
    st = _store(ctx, R)
    before = mb.DeviceBatch(ctx, st, ref)          # a batch made before the roll sees the new rows
    X = _rows(rng, S, k)
    st.roll(X)
    _check_equivalent(ctx, st, _rolled(R, X), ref, old_batches=[before])


@gpu
@pytest.mark.parametrize("N", [480, 1441, 10080])
def test_chain_of_rolls_over_ranges(ctx, N):
    """Three rolls with different k over a sub-range, one row, an empty range and the whole store."""
    S = 200
    rng = np.random.default_rng(N)
    R = _rows(rng, S, N)
    ref = _ref(rng, N)
    st = _store(ctx, R)
    for first, n, k in ((37, 101, 3), (150, 1, N - 1), (5, 0, 9), (0, S, 60)):
        X = _rows(rng, n, k)
        st.roll(X, first)
        R = _rolled(R, X, first)
        assert np.array_equal(st.read_rows(0, S), R)
    _check_equivalent(ctx, st, R, ref)


@gpu
def test_nan_sample_until_pushed_out_and_constant_window(ctx):
    N, S = 1440, 3000
    rng = np.random.default_rng(5)
    R = _rows(rng, S, N)
    ref = _ref(rng, N)
    R[11] = R[11] * 0.01 + 2.0 * ref + 3.0         # a series that would be the top result
    st = _store(ctx, R)
    b = mb.DeviceBatch(ctx, st, ref)
    everyone = lambda: b.run([], N // 2, S, 0.0)[2]      # every series whose score is not NaN
    assert 11 in everyone()
    X = _rows(rng, S, 7)
    X[11, 0] = np.nan                              # lands at N - 7
    st.roll(X)
    st.roll(np.full((1, N), 4.25), 12)             # k == N on one row: a constant window
    R = _rolled(_rolled(R, X), np.full((1, N), 4.25), 12)
    assert 11 not in everyone()                    # never passes, as at ingest
    assert np.isnan(b.score_all()[0][11])
    _check_equivalent(ctx, st, R, ref, modes=(mb.MODE_SCREEN,))
    X = _rows(rng, S, N - 100)
    X[11] = 0.01 * X[11] + 2.0 * ref[100:] + 3.0
    X[12] = 4.25
    st.roll(X)
    R = _rolled(R, X)                              # the NaN now at position 93, row 12 constant
    assert np.isnan(R[11]).any() and np.all(R[12] == 4.25)
    assert 11 not in everyone()
    _check_equivalent(ctx, st, R, ref, modes=(mb.MODE_SCREEN,))
    X = _rows(rng, S, 200)
    X[11] = 0.01 * X[11] + 2.0 * ref[N - 200:] + 3.0
    st.roll(X)
    R = _rolled(R, X)                              # the NaN is pushed out: the series is back
    assert not np.isnan(R[11]).any()
    assert 11 in everyone() and b.score_all()[0][11] > 0.5
    _check_equivalent(ctx, st, R, ref, modes=(mb.MODE_SCREEN,))


@gpu
def test_multi_run_on_tensor_cores_after_roll(ctx):
    """muse_multi_run on the tensor-core path (n = 2048, >= 16384 series, several queries) after a roll equals it on a fresh
    store, and each query equals a batch made before the roll."""
    N, S = 1440, 20000
    st = mb.DeviceStore(ctx, N, 2, S)
    st.append_synthetic(S, 20261018, 0)
    rng = np.random.default_rng(9)
    refs = np.stack([mb.synth_reference(20261018, N), _ref(rng, N), mb.synth_row(20261018, 3, N)])
    before = [mb.DeviceBatch(ctx, st, r) for r in refs]
    X = _rows(rng, S, 60)
    st.roll(X)
    R = st.read_rows(0, S)
    fresh = mb.DeviceStore(ctx, N, 2, S)
    fresh.append(R, _ids(S))
    got = mb.multi_run(st, refs, [], 60, 20, 0.3, mode=mb.MODE_SCREEN)
    n_refined, _ = mb.multi_last_stats(ctx)
    assert n_refined > 0                            # the tensor-core path ran
    want = mb.multi_run(fresh, refs, [], 60, 20, 0.3, mode=mb.MODE_SCREEN)
    for q in range(len(refs)):
        _same(got[q], want[q])
        _same(before[q].run([], 60, 20, 0.3, mode=mb.MODE_SCREEN), want[q])


@gpu
def test_rows_rolled_from_the_previous_synthetic_rows(ctx):
    """The rolled rows are the old rows shifted: read back before and after (synthetic store, odd length)."""
    N, S, k = 1441, 5000, 33
    st = mb.DeviceStore(ctx, N, 2, S)
    st.append_synthetic(S, 7, 0)
    R = st.read_rows(0, S)
    X = _rows(np.random.default_rng(2), S, k)
    st.roll(X)
    assert np.array_equal(st.read_rows(0, S), _rolled(R, X))


@gpu
def test_staging_paths(ctx):
    import torch
    N = 1440
    rng = np.random.default_rng(3)
    # pageable samples larger than one 64 MB staging chunk (60 000 x 1440 x 8 = 691 MB at k = N)
    S = 60000
    st = mb.DeviceStore(ctx, N, 2, S)
    st.append_synthetic(S, 11, 0)
    X = rng.normal(size=(S, N))
    st.roll(X)
    assert np.array_equal(st.read_rows(0, S), X)
    ref = _ref(rng, N)
    fresh = _store(ctx, X)
    fresh_b, b = mb.DeviceBatch(ctx, fresh, ref), mb.DeviceBatch(ctx, st, ref)
    _same(b.run([], 100, 30, 0.1, mode=mb.MODE_SCREEN), fresh_b.run([], 100, 30, 0.1, mode=mb.MODE_SCREEN))
    _same(b.score_all(), fresh_b.score_all())
    fresh.close()
    st.close()
    # page-locked samples (muse_host_alloc)
    S, k = 3000, 90
    R = _rows(rng, S, N)
    st = _store(ctx, R)
    p = C.c_void_p()
    mb._check(mb.lib().muse_host_alloc(C.byref(p), S * k * 8))
    try:
        X = np.ctypeslib.as_array((C.c_double * (S * k)).from_address(p.value)).reshape(S, k)
        X[:] = _rows(rng, S, k)
        st.roll(X)
        R = _rolled(R, X)
    finally:
        mb.lib().muse_host_free(p)
    _check_equivalent(ctx, st, R, ref, modes=(mb.MODE_SCREEN,))
    # device samples: a torch tensor on the context's device
    Xd = torch.from_numpy(_rows(rng, 500, k)).cuda()
    torch.cuda.synchronize()
    st.roll_device(Xd.data_ptr(), 1000, 500, k)
    R = _rolled(R, Xd.cpu().numpy(), 1000)
    _check_equivalent(ctx, st, R, ref, modes=(mb.MODE_SCREEN,))


@gpu
def test_argument_errors_leave_the_store_untouched(ctx):
    N, S = 480, 100
    rng = np.random.default_rng(4)
    R = _rows(rng, S, N)
    st = _store(ctx, R)
    L = mb.lib()
    X = np.ones((S, N + 1))
    Xp = X.ctypes.data_as(C.c_void_p)
    for first, n, k, p in ((0, S, N + 1, Xp), (0, S, -1, Xp), (-1, 2, 1, Xp), (S - 1, 2, 1, Xp), (0, S, 1, None),
                           (S + 1, 0, 1, Xp)):
        assert L.muse_group_roll(st.h, first, n, p, k) == mb.MUSE_ERR_INVALID_ARG
        assert L.muse_group_roll_device(st.h, first, n, p, k) == mb.MUSE_ERR_INVALID_ARG
    assert L.muse_group_roll(None, 0, 1, Xp, 1) == mb.MUSE_ERR_INVALID_ARG
    assert L.muse_group_roll(st.h, 0, 0, None, 5) == mb.MUSE_OK      # nothing to do
    assert L.muse_group_roll(st.h, 0, S, None, 0) == mb.MUSE_OK
    _check_equivalent(ctx, st, R, _ref(rng, N), modes=(mb.MODE_SCREEN,))


@gpu
def test_sharded_rolls_merge_to_one_rolled_store(ctx):
    N, S, k = 1440, 4000, 25
    rng = np.random.default_rng(6)
    R = _rows(rng, S, N)
    ref = _ref(rng, N)
    X = _rows(rng, S, k)
    whole = _store(ctx, R)
    whole.roll(X)
    h = S // 2
    shards = [_store(ctx, R[:h], 0), _store(ctx, R[h:], h)]
    shards[0].roll(X[:h])
    shards[1].roll(X[h:])
    _check_equivalent(ctx, shards[1], _rolled(R, X)[h:], ref, offset=h, modes=(mb.MODE_SCREEN,))
    bw = mb.DeviceBatch(ctx, whole, ref)
    for keys in ([], [0, 1]):
        parts = np.concatenate([mb.DeviceBatch(ctx, s, ref).run_partial(keys, 100, 20, 0.1, mode=mb.MODE_SCREEN) for s in shards])
        got = mb.merge_partials(parts, 100, 20, 0.1)
        _same(got, bw.run(keys, 100, 20, 0.1, mode=mb.MODE_SCREEN))
    assert np.all(mb.DeviceBatch(ctx, shards[1], ref).run([], 100, 20, 0.1)[2] >= h)     # global indices kept


@gpu
def test_group_roll_facade(ctx):
    N, S, k = 480, 300, 12
    rng = np.random.default_rng(8)
    R = _rows(rng, S, N)
    ref = mb.NewSeries(_ref(rng, N))

    def series(rows, tag="h"):
        return [mb.NewSeries(rows[i], mb.NewLabels({"graph": "g%d" % (i % 9), tag: "%s%d" % (tag, i)})) for i in range(len(rows))]

    def run(group):
        b = mb.NewBatch(ref, group, mb.NewResults(100, 20, 0.1, mb.SignFilter_ANY), 1)
        b.Run(["graph"])
        got, _ = b.Results.Fetch()
        return [(s.Labels.ID(), s.Lag, s.PercentScore) for s in got]

    g = mb.NewGroup("roll")
    g.Add(*series(R[:200]))
    b = mb.NewBatch(ref, g, mb.NewResults(100, 20, 0.1, mb.SignFilter_ANY), 1)
    g.Add(*[mb.NewSeries(R[i], mb.NewLabels({"graph": "g%d" % (i % 9), "h": "h%d" % i})) for i in range(200, S)])   # pending
    X = _rows(rng, S, k)
    g.Roll(X)
    R2 = _rolled(R, X)
    for i, s in enumerate(g.series):
        assert np.array_equal(s.Values(), R2[i])
    fresh = mb.NewGroup("fresh")
    fresh.Add(*series(R2))
    assert run(g) == run(fresh)
    b.Run(None)                                     # the batch made before the roll still runs
    # a series with a new label key rebuilds the store from the host values
    extra = _rows(rng, 1, N)[0]
    g.Add(mb.NewSeries(extra, mb.NewLabels({"graph": "g0", "colo": "c1"})))
    fresh.Add(mb.NewSeries(extra, mb.NewLabels({"graph": "g0", "colo": "c1"})))
    assert run(g) == run(fresh)
    X = _rows(rng, S + 1, N)
    g.Roll(X)
    fresh2 = mb.NewGroup("fresh2")
    fresh2.Add(*series(X[:S]), mb.NewSeries(X[S], mb.NewLabels({"graph": "g0", "colo": "c1"})))
    assert run(g) == run(fresh2)


# ---- argument checks without a device ----------------------------------------------------------------------------------
class _NoDevice:
    def __getattr__(self, name):
        raise AssertionError("device call %s before the arguments were checked" % name)


def test_device_store_roll_checks_before_any_call(monkeypatch):
    st = object.__new__(mb.DeviceStore)
    st.h, st.series_len, st.n_label_keys = C.c_void_p(), 100, 0
    monkeypatch.setattr(mb, "_lib", _NoDevice())
    for bad, first in ((np.zeros(5), 0), (np.zeros((2, 2, 2)), 0), (np.zeros((3, 101)), 0), (np.zeros((3, 4)), -1)):
        with pytest.raises(mb.MuseError) as e:
            st.roll(bad, first)
        assert e.value.code == mb.MUSE_ERR_INVALID_ARG


def test_group_roll_checks_before_any_call(monkeypatch):
    g = mb.NewGroup("cpu")
    vals = [np.arange(10.0) + i for i in range(3)]
    g.Add(*[mb.NewSeries(v, mb.NewLabels({"h": str(i)})) for i, v in enumerate(vals)])

    def no_device():
        raise AssertionError("device call before the arguments were checked")

    monkeypatch.setattr(g, "_sync_device", no_device)
    for bad in ([[1.0]] * 2, [[1.0], [2.0, 3.0], [4.0]], [[1.0] * 11] * 3, np.zeros((3, 2, 2))):
        with pytest.raises(mb.MuseError) as e:
            g.Roll(bad)
        assert e.value.code == mb.MUSE_ERR_INVALID_ARG
    g.Roll(np.zeros((3, 0)))                       # k == 0: nothing to do, no device call
    for s, v in zip(g.series, vals):
        assert np.array_equal(s.Values(), v)


def test_roll_abi_rejects_a_null_group_without_a_device():
    mb.build()
    L = mb.lib()
    x = np.zeros(4)
    assert L.muse_group_roll(None, 0, 1, x.ctypes.data_as(C.c_void_p), 4) == mb.MUSE_ERR_INVALID_ARG
    assert L.muse_group_roll_device(None, 0, 1, None, 0) == mb.MUSE_ERR_INVALID_ARG
