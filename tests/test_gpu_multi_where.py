"""muse_multi_run_where: many references against the series of a resident store whose label ids match.  Row q of the
outputs must be what muse_multi_run writes for reference q on a fresh store that holds only the matching rows, in the same
order: scores bit for bit, lags and order identical, indices mapped through the selection.  GPU tests need a B200; the
argument checks of the facade at the end run without one."""
import ctypes as C

import numpy as np
import pytest

import muse_b200 as mb

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _rows(rng, S, N):
    Y = 0.1 * (rng.random((S, N)) - 0.5)
    for i in range(0, S, 3):
        m, w = int(rng.integers(0, N - 20)), int(rng.integers(3, 20))
        Y[i, m:m + w] += rng.uniform(0.5, 40)
    Y[::17] = 3.5                   # std == 0 on both sides of every selection
    Y[5::19, N // 3] = np.nan       # NaN samples, likewise
    return Y


def _refs(rng, Q, N):
    refs = 0.1 * (rng.random((Q, N)) - 0.5)
    for q in range(Q):
        mid, w = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8)), int(rng.integers(3, 21))
        refs[q, mid - w // 2: mid - w // 2 + w] += 1.5
    if Q > 3:
        refs[3] = 2.0               # std == 0: n_out = -1 for this reference alone
    return refs


def _ids(S, offset=0):
    """col 0: 1 for i % 3 == 0 (id 0 selects two thirds); col 1: i % 7; col 2: i % 2, absent (-1) for i % 13 == 0."""
    i = np.arange(offset, offset + S)
    return np.stack([(i % 3 == 0), i % 7, np.where(i % 13 == 0, -1, i % 2)], axis=1).astype(np.int32)


def _store(ctx, rows, ids, offset=0):
    st = mb.DeviceStore(ctx, rows.shape[1], ids.shape[1], max(1, rows.shape[0]))
    if offset:
        st.set_global_offset(offset)
    if rows.shape[0]:
        st.append(rows, ids)
    return st


def _mask(ids, cols, vals):
    m = np.ones(ids.shape[0], dtype=bool)
    for c, v in zip(cols, vals):
        m &= ids[:, c] == v
    return m


def _same(got, want, sel, offset=0):
    """raw outputs (scores, lags, series_idx, n_out) of a filtered call against those of a fresh store of the selection"""
    gsc, glg, gix, gn = got
    wsc, wlg, wix, wn = want
    assert np.array_equal(gn, wn), (gn[:8], wn[:8])
    for q in range(len(gn)):
        k = max(int(gn[q]), 0)
        assert np.array_equal(gsc[q, :k], wsc[q, :k]), q
        assert np.array_equal(glg[q, :k], wlg[q, :k]), q
        assert np.array_equal(gix[q, :k], offset + sel[wix[q, :k]]), q


def _check(ctx, st, R, ids, refs, cols, vals, keys, max_lag, top_n, thr, sign=0, mode=mb.MODE_AUTO, offset=0, per_query=(),
           tc=None):
    """multi_run_where against multi_run on a fresh store of the selection and, for the references in per_query, against
    DeviceBatch.run_where; tc: whether the tensor-core path must (True) or must not (False) have run."""
    sel = np.flatnonzero(_mask(ids, cols, vals))
    got = mb.multi_run_where(st, refs, cols, vals, keys, max_lag, top_n, thr, sign, mode, raw=True)
    stats = mb.multi_last_stats(ctx)
    if tc is not None:
        assert (stats[0] > 0) == tc, stats
    fresh = _store(ctx, R[sel], ids[sel])
    want = mb.multi_run(fresh, refs, keys, max_lag, top_n, thr, sign, mode, raw=True)
    fresh.close()
    _same(got, want, sel, offset)
    for q in per_query:
        if got[3][q] < 0:           # std == 0: no batch
            continue
        b = mb.DeviceBatch(ctx, st, refs[q])
        sc, lg, ix = b.run_where(cols, vals, keys, max_lag, top_n, thr, sign, mode=mode)
        b.close()
        k = int(got[3][q])
        assert np.array_equal(sc, got[0][q, :k]) and np.array_equal(lg, got[1][q, :k]) and np.array_equal(ix, got[2][q, :k]), q
    return got, sel


@gpu
@pytest.mark.parametrize("N", [1440, 1283])
def test_tensor_core_path_equals_fresh_store(ctx, N):
    """FFT length 2048, a 40 k store with 26.7 k rows selected (AUTO takes the tensor-core path); 33 and 257 references (two
    launch groups, the second of one query)."""
    rng = np.random.default_rng(N)
    S = 40000
    R = _rows(rng, S, N)
    ids = _ids(S)
    st = _store(ctx, R, ids)
    for Q in (33, 257):
        refs = _refs(rng, Q, N)
        got, sel = _check(ctx, st, R, ids, refs, [0], [0], [], 60, 100, 0.0, per_query=(0, 3, Q - 1), tc=True)
        assert len(sel) >= 16384 and got[3][3] == -1 and np.all(got[3][np.arange(Q) != 3] > 0)
    _check(ctx, st, R, ids, _refs(rng, 9, N), [0, 2], [0, 1], [], N, 50, 0.0, mb.SignFilter_POS, tc=False)   # 12 k rows: separate
    st.close()


@gpu
def test_screen_mode_below_the_auto_size_takes_the_tensor_core_path(ctx):
    rng = np.random.default_rng(2)
    S, N = 9000, 1440
    R = _rows(rng, S, N)
    ids = _ids(S)
    st = _store(ctx, R, ids)
    refs = _refs(rng, 6, N)
    _check(ctx, st, R, ids, refs, [0], [0], [], 60, 100, 0.5, mode=mb.MODE_SCREEN, per_query=(1,), tc=True)
    _check(ctx, st, R, ids, refs, [1], [4], [], 60, 100, 0.5, mode=mb.MODE_SCREEN, tc=True)
    st.close()


@gpu
@pytest.mark.parametrize("N", [480, 1440, 5000])
def test_separate_path_equals_fresh_store(ctx, N):
    """AUTO below 16384 selected rows, grouped runs (one and two key columns), SIGN_NEG, MODE_EXACT, one reference."""
    rng = np.random.default_rng(N + 1)
    S = 3000
    R = _rows(rng, S, N)
    ids = _ids(S)
    st = _store(ctx, R, ids)
    refs = _refs(rng, 5, N)
    for cols, vals in (([0], [0]), ([2, 1], [1, 3])):
        _check(ctx, st, R, ids, refs, cols, vals, [], 60, 100, 0.5, per_query=(0,), tc=False)
        _check(ctx, st, R, ids, refs, cols, vals, [1], 60, 100, 0.0, per_query=(1,), tc=False)
        _check(ctx, st, R, ids, refs, cols, vals, [1, 2], N, 30, 0.3, tc=False)
        _check(ctx, st, R, ids, refs, cols, vals, [], 60, 100, 0.2, mb.SignFilter_NEG, tc=False)
        _check(ctx, st, R, ids, refs, cols, vals, [], 60, 100, 0.5, mode=mb.MODE_EXACT, tc=False)
        _check(ctx, st, R, ids, refs[:1], cols, vals, [], 60, 100, 0.5, mode=mb.MODE_SCREEN, per_query=(0,), tc=False)
    st.close()


@gpu
def test_unselected_rows_that_would_win_never_appear(ctx):
    rng = np.random.default_rng(4)
    S, N = 24000, 1440
    R = _rows(rng, S, N)
    ids = _ids(S)
    refs = _refs(rng, 4, N)
    out = np.flatnonzero(ids[:, 0] != 0)
    R[out] = refs[0] * 2.0 + 1.0 + 1e-3 * rng.random((len(out), N))     # score ~1 at lag 0 against reference 0
    st = _store(ctx, R, ids)
    for mode, tc in ((mb.MODE_AUTO, False), (mb.MODE_SCREEN, True)):
        got, sel = _check(ctx, st, R, ids, refs, [0], [0], [], N, 200, 0.0, mode=mode, tc=tc)
        for q in range(4):
            ix = got[2][q, :max(int(got[3][q]), 0)]
            assert np.all(ids[ix, 0] == 0)
        assert got[3][0] > 0
    st.close()


@gpu
def test_edges(ctx):
    rng = np.random.default_rng(5)
    S, N = 20000, 1440
    R = _rows(rng, S, N)
    ids = _ids(S)
    ids[:, 1] = 6                   # every series: col 1 == 6
    st = _store(ctx, R, ids)
    refs = _refs(rng, 5, N)
    whole = mb.multi_run(st, refs, [], 60, 100, 0.5, raw=True)
    for got in (mb.multi_run_where(st, refs, [], [], [], 60, 100, 0.5, raw=True),
                mb.multi_run_where(st, refs, [1], [6], [], 60, 100, 0.5, raw=True)):
        _same(got, whole, np.arange(S))
    for cols, vals in (([1], [2]), ([2, 0], [5, 0])):      # nothing matches
        for keys in ([], [1]):
            sc, lg, ix, n = mb.multi_run_where(st, refs, cols, vals, keys, 60, 100, 0.5, raw=True)
            assert n.tolist() == [0, 0, 0, -1, 0]
    _check(ctx, st, R, ids, refs, [0], [0], [], 60, len(np.flatnonzero(ids[:, 0] == 0)) + 7, 0.0, tc=False)   # top_n > selection
    _check(ctx, st, R, ids, refs, [0], [0], [], 60, 3300, 0.0, mode=mb.MODE_SCREEN, tc=True)      # top_n * 4 <= rows
    _check(ctx, st, R, ids, refs, [0], [0], [], 60, 0, 0.5, tc=None)
    st.close()
    empty = mb.DeviceStore(ctx, N, 3, 1)
    _same(mb.multi_run_where(empty, refs, [0], [0], [], 60, 100, 0.5, raw=True), mb.multi_run(empty, refs, [], 60, 100, 0.5, raw=True),
          np.arange(0))
    empty.close()


@gpu
def test_global_offset_roll_and_remove(ctx):
    rng = np.random.default_rng(6)
    S, N, off = 30000, 1440, 777777
    R = _rows(rng, S, N)
    ids = _ids(S, off)
    st = _store(ctx, R, ids, off)
    refs = _refs(rng, 6, N)
    _check(ctx, st, R, ids, refs, [0], [0], [], 60, 100, 0.5, offset=off, tc=True)
    X = _rows(rng, S, 41)
    st.roll(X)
    R = np.concatenate([R[:, 41:], X], axis=1)
    _check(ctx, st, R, ids, refs, [0], [0], [], 60, 100, 0.5, offset=off, tc=True)
    gone = np.arange(0, S, 5)
    moved_from, moved_to = st.remove(gone)
    keep = np.ones(S, dtype=bool)
    keep[gone] = False
    order = np.flatnonzero(keep)
    pos = np.arange(S)
    pos[moved_to] = moved_from          # row r of the store after the removal holds old row pos[r]
    new = pos[:S - len(gone)]
    assert set(new.tolist()) == set(order.tolist())
    R, ids = R[new], ids[new]
    _check(ctx, st, R, ids, refs, [0], [0], [], 60, 100, 0.5, mode=mb.MODE_SCREEN, offset=off, per_query=(0,), tc=True)
    st.close()


@gpu
def test_top_n_beyond_the_device_side_select_and_the_list_fallback(ctx):
    """Contiguous selections of synthetic stores (a fresh store of the selection is the same synthetic rows): top_n above the
    device-side select (33000), and the adversarial rect store whose exact list exceeds the launch bound -- both reach a
    query's fallback (flags == 2), which finishes as a filtered run of that query."""
    N = 1026
    for S, variant, top_n, max_lag in ((280000, 0, 33000, N), (80000, 1, 10000, N)):
        half = S // 2
        st = mb.DeviceStore(ctx, N, 2, S)
        st.append_synthetic(S, 20261018, 0, variant)
        st.set_synthetic_labels([half, 1], [2, 5])
        refs = _refs(np.random.default_rng(S), 3, N)
        got = mb.multi_run_where(st, refs, [0], [1], [], max_lag, top_n, 0.0, raw=True)
        rescored = mb.multi_last_stats(ctx)[1]
        assert rescored > 32768, rescored
        fresh = mb.DeviceStore(ctx, N, 0, half)
        fresh.append_synthetic(half, 20261018, half, variant)
        want = mb.multi_run(fresh, refs, [], max_lag, top_n, 0.0, raw=True)
        _same(got, want, np.arange(half, S))
        assert np.all(got[3] == top_n)
        fresh.close()
        st.close()


@gpu
def test_argument_errors_leave_the_store_usable_and_memory_is_not_held(ctx):
    rng = np.random.default_rng(7)
    S, N = 18000, 1440
    R = _rows(rng, S, N)
    ids = _ids(S)
    st = _store(ctx, R, ids)
    refs = _refs(rng, 4, N)
    want = mb.multi_run_where(st, refs, [0], [0], [], 60, 20, 0.5, raw=True)
    L = mb.lib()
    Q, k = 4, 20
    sc, lg, ix, n = np.zeros((Q, k)), np.zeros((Q, k), dtype=np.int64), np.zeros((Q, k), dtype=np.int64), np.zeros(Q, dtype=np.int64)
    P = lambda a: a.ctypes.data_as(mb._ip32)
    c17, v17 = np.zeros(17, dtype=np.int32), np.zeros(17, dtype=np.int32)

    def call(cols, vals, nw, keys=None, nk=0, top_n=k, out=True, refs_p=mb._d(refs), nq=Q):
        return L.muse_multi_run_where(ctx.h, st.h, refs_p, nq, N, cols, vals, nw, keys, nk, 60, top_n, 0.5, 0, 0,
                                      mb._d(sc) if out else None, lg.ctypes.data_as(mb._ip64), ix.ctypes.data_as(mb._ip64),
                                      n.ctypes.data_as(mb._ip64))

    one = np.zeros(1, dtype=np.int32)
    for rc in (call(P(c17), P(v17), -1), call(P(c17), P(v17), 17), call(None, P(v17), 1), call(P(c17), None, 1),
               call(P(np.array([3], dtype=np.int32)), P(one), 1), call(P(np.array([-1], dtype=np.int32)), P(one), 1),
               call(P(one), P(np.array([-1], dtype=np.int32)), 1), call(P(one), P(one), 1, None, 1), call(P(one), P(one), 1, top_n=-1),
               call(P(one), P(one), 1, out=False), call(P(one), P(one), 1, refs_p=None), call(P(one), P(one), 1, nq=-1)):
        assert rc == mb.MUSE_ERR_INVALID_ARG
    assert L.muse_multi_run_where(None, st.h, mb._d(refs), Q, N, P(one), P(one), 1, None, 0, 60, k, 0.5, 0, 0, mb._d(sc),
                                  lg.ctypes.data_as(mb._ip64), ix.ctypes.data_as(mb._ip64), n.ctypes.data_as(mb._ip64)) == mb.MUSE_ERR_INVALID_ARG
    assert call(P(c17), P(v17), 16) == mb.MUSE_OK          # sixteen equalities are allowed
    _same(mb.multi_run_where(st, refs, [0], [0], [], 60, 20, 0.5, raw=True), want, np.arange(S))
    held = []
    for _ in range(5):
        mb.multi_run_where(st, refs, [0], [0], [], 60, 20, 0.5)
        mb.multi_run_where(st, refs, [2], [1], [1], 60, 20, 0.5)
        d, p = C.c_int64(0), C.c_int64(0)
        mb._check(L.muse_held_bytes(C.byref(d), C.byref(p)))
        held.append((d.value, p.value))
    assert held[2:] == held[1:-1], held          # the first round may size buffers that later rounds reuse
    st.close()


# ---- facade --------------------------------------------------------------------------------------------------------
def _facade_group(rng, S, N):
    Y = _rows(rng, S, N)
    g = mb.NewGroup("many")
    series = []
    for i in range(S):
        lab = {"uid": "s%d" % i, "svc": "svc%d" % (i % 4), "colo": "c%d" % (i // 7 % 3)}
        if i % 5:
            lab["host"] = "h%d" % (i % 9)
        series.append(mb.NewSeries(Y[i], mb.NewLabels(lab)))
    g.Add(*series)
    return g


def _fetch(r):
    got, _ = r.Fetch()
    return [(s.PercentScore, s.Lag, s.Labels) for s in got]


@gpu
@pytest.mark.parametrize("N", [480, 1440])
def test_facade_run_many_and_run_many_where_equal_loops_of_batches(ctx, N):
    rng = np.random.default_rng(N + 11)
    g = _facade_group(rng, 1300, N)
    refs = [mb.NewSeries(r) for r in _refs(rng, 5, N)]
    for labels, group_by in ((None, None), (None, ["colo"]), ({"svc": "svc1"}, None), ({"svc": "svc2", "host": "h4"}, ["colo"]),
                             ({"host": "h3"}, ["host", "colo"])):
        L = mb.NewLabels(labels) if labels else None
        res = [mb.NewResults(N, 10, 0.1, mb.SignFilter_ANY) for _ in refs]
        errs, err = mb.RunManyWhere(refs, g, res, L, group_by) if L else mb.RunMany(refs, g, res, group_by)
        assert err is None
        for q, ref in enumerate(refs):
            want = mb.NewResults(N, 10, 0.1, mb.SignFilter_ANY)
            if q == 3:                                        # constant reference: NewBatch fails, Results untouched
                assert errs[q] is not None and errs[q].code == mb.MUSE_ERR_STDDEV_ZERO and res[q]._heap == []
                continue
            assert errs[q] is None
            b = mb.NewBatch(ref, g, want, 1)
            b.RunWhere(L, group_by) if L else b.Run(group_by)
            got, exp = _fetch(res[q]), _fetch(want)
            assert len(got) == len(exp) > 0
            for (gs, gl, glab), (ws, wl, wlab) in zip(got, exp):
                assert gs == ws and gl == wl and glab is wlab


@gpu
def test_facade_run_many_where_unknown_label_leaves_results_untouched(ctx):
    rng = np.random.default_rng(3)
    g = _facade_group(rng, 300, 480)
    refs = [mb.NewSeries(r) for r in _refs(rng, 4, 480)]
    for labels in ({"svc": "nope"}, {"nokey": "svc1"}, {}, {"svc": "svc1", "host": "nope"}):
        res = [mb.NewResults(60, 10, 0.0, mb.SignFilter_ANY) for _ in refs]
        mb.RunMany(refs, g, res, None)
        before = [[(s, -q, x.PercentScore, x.Lag, x.Labels) for s, q, x in r._heap] for r in res]
        errs, err = mb.RunManyWhere(refs, g, res, mb.NewLabels(labels), ["colo"])
        assert err is None and errs == [None] * 4
        assert [[(s, -q, x.PercentScore, x.Lag, x.Labels) for s, q, x in r._heap] for r in res] == before


# ---- checks that need no device -------------------------------------------------------------------------------------
class _NoDevice:
    def __getattr__(self, name):
        raise AssertionError("device call %s" % name)


def _cpu_group():
    g = mb.NewGroup("cpu")
    g.Add(*[mb.NewSeries(np.arange(10.0) + i, mb.NewLabels({"h": str(i % 2), "uid": str(i)})) for i in range(4)])
    g._cols = ["h", "uid"]
    g._dict = {"h": {"0": 0, "1": 1}, "uid": {str(i): i for i in range(4)}}
    return g


def test_facade_run_many_checks_without_a_device(monkeypatch):
    g = _cpu_group()
    monkeypatch.setattr(mb, "_lib", _NoDevice())
    monkeypatch.setattr(g, "_sync_device", lambda: None)
    ref, short = mb.NewSeries(np.arange(10.0) * 2), mb.NewSeries(np.arange(9.0))
    r = lambda top=5, lag=5: mb.NewResults(lag, top, 0.0, 0)
    for fn, extra in ((mb.RunMany, ()), (mb.RunManyWhere, (mb.NewLabels({"h": "1"}),))):
        errs, err = fn([ref, ref], g, [r()], *extra)                   # one Results per reference
        assert errs is None and err.code == mb.MUSE_ERR_INVALID_ARG
        errs, err = fn([ref, short], g, [r(), r()], *extra)            # every reference has the group's length
        assert errs is None and err is not None
        errs, err = fn([ref, ref], g, [r(), r(lag=6)], *extra)         # the same filter on every Results
        assert errs is None and err is not None
        assert fn([], g, [], *extra) == ([], None)
        assert fn([ref], mb.NewGroup("empty"), [r()], *extra) == ([None], None)
        assert fn([ref, ref], g, [r(0), r(0)], *extra) == ([None, None], None)     # TopN 0: nothing to keep
    for labels in ({"h": "7"}, {"x": "0"}, {"h": "0", "uid": "9"}, {}):
        res = [r(), r()]
        assert mb.RunManyWhere([ref, ref], g, res, mb.NewLabels(labels)) == ([None, None], None)
        assert all(x._heap == [] for x in res)
    assert mb.RunManyWhere([ref], g, [r()], None) == ([None], None)


def test_multi_run_where_checks_lengths_before_any_call(monkeypatch):
    monkeypatch.setattr(mb, "_lib", _NoDevice())
    st = object.__new__(mb.DeviceStore)
    with pytest.raises(mb.MuseError) as e:
        mb.multi_run_where(st, np.zeros((2, 8)), [0, 1], [2], [], 60, 10, 0.5)
    assert e.value.code == mb.MUSE_ERR_INVALID_ARG


def test_multi_run_where_abi_rejects_null_arguments_without_a_device():
    mb.build()
    L = mb.lib()
    n = np.zeros(1, dtype=np.int64)
    assert L.muse_multi_run_where(None, None, None, 0, 8, None, None, 0, None, 0, 60, 10, 0.5, 0, 0, None, None, None,
                                  n.ctypes.data_as(mb._ip64)) == mb.MUSE_ERR_INVALID_ARG
