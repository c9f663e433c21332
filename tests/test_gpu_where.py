"""muse_batch_run_where: Batch.Run over the series of a resident store whose label ids match.  A filtered run must return
what muse_batch_run_ex returns on a fresh store that holds only the matching rows, in the same order: scores bit for bit,
lags and order identical, indices mapped through the selection, and the same scoring path (timing.mode).  GPU tests need a
B200; the argument checks of the facade at the end run without one."""
import ctypes as C

import numpy as np
import pytest

import muse_b200 as mb

gpu = pytest.mark.gpu
MODES = (mb.MODE_AUTO, mb.MODE_EXACT, mb.MODE_SCREEN)
NKEYS = 4


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _rows(rng, S, N):
    Y = rng.normal(size=(S, N)) * rng.uniform(0.1, 10.0, size=(S, 1)) + rng.uniform(-50, 50, size=(S, 1))
    for i in range(0, S, 3):
        m, w = int(rng.integers(0, N)), int(rng.integers(1, max(2, N // 20)))
        Y[i, m:m + w] += rng.uniform(5, 60)
    Y[::17] = 3.5                   # std == 0 on both sides of every selection
    Y[5::19, N // 3] = np.nan       # NaN samples, likewise
    return Y


def _ref(rng, N):
    r = 0.1 * rng.random(N)
    r[N // 2 - max(1, N // 100): N // 2 + max(1, N // 100)] += 1.5
    return r


def _ids(S, offset=0):
    """col 0: i % 11, col 1: (i // 5) % 4 (group keys that straddle every selection); col 2: i % 3, absent (-1) for
    i % 13 == 0 (such a series never matches); col 3: (i // 50) % 4, contiguous blocks."""
    i = np.arange(offset, offset + S)
    c2 = np.where(i % 13 == 0, -1, i % 3)
    return np.stack([i % 11, (i // 5) % 4, c2, (i // 50) % 4], axis=1).astype(np.int32)


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


def _same_as_fresh(got, want, sel, offset, t_got, t_want, S=None, same_path=True):
    """got, t_got: the records and timing of a run over the rows sel of a store of S rows; want, t_want: those of the run it
    must equal.  S = None: both runs made the same selection (or none).  same_path: both runs ranked their records on the
    same side (device or host), so they re-scored as many series and launched the same work.  n_refined is not compared: it
    counts the second stages, which depend on how far the running cut-off had risen when each series was screened, and the
    work counter hands the series out in a different order on every run, even of one store."""
    gsc, glg, gix = got
    wsc, wlg, wix = want
    assert np.array_equal(gsc, wsc), (gsc[:8], wsc[:8])
    assert np.array_equal(glg, wlg)
    assert np.array_equal(gix, offset + sel[wix]), (gix[:8], (offset + sel[wix])[:8])
    assert t_got.mode == t_want.mode
    if not same_path:
        return
    assert t_got.n_rescored == t_want.n_rescored
    # the selection's count, scan and write, and the neutral fill of the rows outside a selection that is not the store
    extra = 0 if S is None else 3 + (0 < len(sel) < S)
    assert t_got.n_launches == t_want.n_launches + extra, (t_got.n_launches, t_want.n_launches, extra)


# (key columns, max_lag, top_n (None: more than the selection), threshold, sign filter, signed scores)
RUNS = [
    ([], 60, 100, 0.5, mb.SignFilter_ANY, False),
    ([], 0, 1, 0.0, mb.SignFilter_ANY, False),
    ([], 60, None, 0.0, mb.SignFilter_POS, False),
    ([], 60, 100, 0.5, mb.SignFilter_NEG, False),
    ([], 60, 100, 0.0, mb.SignFilter_ANY, True),
    ([], 60, 100, 0.5, mb.SignFilter_POS, True),
    ([0], 60, 100, 0.5, mb.SignFilter_ANY, False),
    ([0, 1], 60, None, 0.0, mb.SignFilter_ANY, False),
    ([0], 0, 1, 0.0, mb.SignFilter_POS, True),
    ([1, 0], 60, 100, 0.5, mb.SignFilter_NEG, False),
]
PREDICATES = [([2], [1]), ([2, 3], [0, 2]), ([3], [1])]


def _check_runs(ctx, st, R, ids, ref, offset=0, runs=RUNS, predicates=PREDICATES, modes=MODES, batch=None):
    b = batch or mb.DeviceBatch(ctx, st, ref)
    for cols, vals in predicates:
        sel = np.flatnonzero(_mask(ids, cols, vals))
        fresh = _store(ctx, R[sel], ids[sel])
        bf = mb.DeviceBatch(ctx, fresh, ref)
        for keys, max_lag, top_n, thr, sign, signed in runs:
            top_n = len(sel) + 7 if top_n is None else top_n
            for mode in modes:
                got = b.run_where(cols, vals, keys, max_lag, top_n, thr, sign, mode=mode, signed_scores=signed)
                tg = b.timing()
                want = bf.run(keys, max_lag, top_n, thr, sign, mode=mode, signed_scores=signed)
                # a filtered run ranks ungrouped records on the device when they fit a store of the selection's size (4 sort
                # entries per record, at least 1024 entries); the fresh batch may reuse a larger scratch set from the
                # context's pool, in which they fit where they do not fit the selection
                same_path = bool(keys) or 4 * top_n <= max(len(sel), 1024)
                _same_as_fresh(got, want, sel, offset, tg, bf.timing(), len(ids), same_path)
        bf.close()
        fresh.close()
    return b


# N = 120, 480, 1000: sub-warp; 1440: warp; 1441: odd (pad column); 2500, 10080: n = 4096 / 16384; 20000: long
SHAPES = [(120, 1500), (480, 1500), (1000, 1200), (1440, 1500), (1441, 1200), (2500, 600), (10080, 300), (20000, 90)]


@gpu
@pytest.mark.parametrize("N,S", SHAPES)
def test_where_equals_fresh_store_of_the_selection(ctx, N, S):
    rng = np.random.default_rng(N)
    R = _rows(rng, S, N)
    ids = _ids(S)
    ref = _ref(rng, N)
    st = _store(ctx, R, ids)
    _check_runs(ctx, st, R, ids, ref)


def _synthetic(ctx, S, N, div, mod, variant=0, seed=7):
    st = mb.DeviceStore(ctx, N, len(div), S)
    st.append_synthetic(S, seed, 0, variant)
    st.set_synthetic_labels(div, mod)
    i = np.arange(S)
    ids = np.stack([(i // d) % m for d, m in zip(div, mod)], axis=1).astype(np.int32)
    return st, ids


@gpu
def test_where_above_and_below_the_screening_size(ctx):
    """A 40 k store: a selection of 20 k rows screens under AUTO, one of 10 k does not (the rule follows the selection's
    size, not the store's); every mode, grouped and ungrouped, against fresh stores of the selections."""
    S, N = 40000, 1440
    st, ids = _synthetic(ctx, S, N, [1, 5, 1, 50], [11, 4, 2, 4])
    R = st.read_rows(0, S)
    ref = mb.synth_reference(7, N)
    above, below = ([2], [0]), ([1], [0])
    assert _mask(ids, *above).sum() == 20000 and _mask(ids, *below).sum() == 10000
    runs = [r for r in RUNS if r[2] is not None] + [([], 60, 20000, 0.5, mb.SignFilter_ANY, False)]
    b = _check_runs(ctx, st, R, ids, ref, runs=runs, predicates=[above, below, ([2, 1], [1, 3])])
    b.run_where(*above, [], 60, 100, 0.5, mode=mb.MODE_AUTO)
    assert b.timing().mode == mb.MODE_SCREEN
    b.run_where(*below, [], 60, 100, 0.5, mode=mb.MODE_AUTO)
    assert b.timing().mode == mb.MODE_EXACT


@gpu
def test_where_empty_and_whole_selection(ctx):
    N, S = 1440, 2000
    rng = np.random.default_rng(1)
    R = _rows(rng, S, N)
    ids = _ids(S)
    ids[:, 3] = 2                           # every series has col 3 == 2
    ref = _ref(rng, N)
    st = _store(ctx, R, ids)
    b = mb.DeviceBatch(ctx, st, ref)
    for mode in MODES:
        for keys in ([], [0]):
            sc, lg, ix = b.run_where([2], [7], keys, 60, 100, 0.0, mode=mode)      # no series has id 7
            assert len(sc) == len(lg) == len(ix) == 0
            sc, lg, ix = b.run_where([3, 2], [2, 5], keys, 60, 100, 0.0, mode=mode)
            assert len(sc) == 0
            got = b.run_where([3], [2], keys, 60, 100, 0.5, mode=mode)
            tg = b.timing()
            want = b.run(keys, 60, 100, 0.5, mode=mode)
            tw = b.timing()
            _same_as_fresh(got, want, np.arange(S), 0, tg, tw, S)
            # no where columns: the whole store
            got = b.run_where([], [], keys, 60, 100, 0.5, mode=mode)
            _same_as_fresh(got, want, np.arange(S), 0, b.timing(), tw)


@gpu
@pytest.mark.parametrize("N", [480, 1440, 10080])
def test_unselected_rows_that_outscore_the_selection_never_appear(ctx, N):
    S = 1200
    rng = np.random.default_rng(N + 3)
    R = _rows(rng, S, N)
    ids = _ids(S)
    ref = _ref(rng, N)
    out = np.flatnonzero(ids[:, 2] != 1)
    R[out] = ref * 2.0 + 1.0 + 1e-3 * rng.random((len(out), N))     # score ~1 at lag 0
    st = _store(ctx, R, ids)
    b = _check_runs(ctx, st, R, ids, ref, predicates=[([2], [1])])
    for mode in MODES:
        for keys in ([], [0], [0, 1]):
            sc, lg, ix = b.run_where([2], [1], keys, N, S, 0.0, mode=mode)      # every lag passes
            assert len(ix) > 0 and np.all(ids[ix, 2] == 1)


@gpu
def test_where_adversarial_rect_store(ctx):
    """variant 1: every series a rect of the reference's width, nearly every score within the slack of the cut-off; 20 k of
    60 k rows selected (below the fused path's exact launch bound of 32768, so the exact list always fits the launch)."""
    S, N = 60000, 1440
    st, ids = _synthetic(ctx, S, N, [1, 5, 1, 50], [11, 4, 3, 4], variant=1, seed=11)
    assert _mask(ids, [2], [1]).sum() == 20000
    R = st.read_rows(0, S)
    ref = mb.synth_reference(11, N)
    runs = [([], 60, 100, 0.5, mb.SignFilter_ANY, False), ([], 60, 5000, 0.0, mb.SignFilter_ANY, False),
            ([0, 1], 60, 100, 0.5, mb.SignFilter_ANY, False)]
    _check_runs(ctx, st, R, ids, ref, runs=runs, predicates=[([2], [1])])


@gpu
def test_where_exact_list_longer_than_the_launch_bound(ctx):
    """40 k of 80 k rect rows selected with top_n above the selection and every lag allowed: the cut-off never rises, every
    selected series reaches the exact list, and the list is longer than the fused path's launch bound (32768) -- the overflow
    fallback scores the rest of the list, the selected rows only."""
    S, N = 80000, 1440
    st, ids = _synthetic(ctx, S, N, [1, 1], [2, 3], variant=1, seed=13)
    sel = ([0], [1])
    assert _mask(ids, *sel).sum() == 40000
    R = st.read_rows(0, S)
    ref = mb.synth_reference(13, N)
    runs = [([], N, None, 0.0, mb.SignFilter_ANY, False), ([], 60, 100, 0.5, mb.SignFilter_ANY, False),
            ([1], 60, 100, 0.0, mb.SignFilter_ANY, False)]
    b = _check_runs(ctx, st, R, ids, ref, runs=runs, predicates=[sel])
    b.run_where(*sel, [], N, 40007, 0.0, mode=mb.MODE_SCREEN)
    t = b.timing()
    assert t.mode == mb.MODE_SCREEN and t.n_rescored > 32768


@gpu
@pytest.mark.parametrize("N", [480, 1441, 10080])
def test_where_after_roll_and_with_global_offset(ctx, N):
    S, off = 900, 123456
    rng = np.random.default_rng(N + 5)
    R = _rows(rng, S, N)
    ids = _ids(S, off)
    ref = _ref(rng, N)
    st = _store(ctx, R, ids, off)
    b = mb.DeviceBatch(ctx, st, ref)
    X = _rows(rng, S, 37)
    st.roll(X)
    R = np.concatenate([R[:, 37:], X], axis=1)
    runs = [RUNS[0], RUNS[4], RUNS[7]]
    _check_runs(ctx, st, R, ids, ref, offset=off, runs=runs, batch=b)


@gpu
@pytest.mark.parametrize("N", [480, 1440, 10080])
def test_alternating_runs_leak_no_state(ctx, N):
    S = 1500
    rng = np.random.default_rng(N + 9)
    R = _rows(rng, S, N)
    ids = _ids(S)
    ref = _ref(rng, N)
    st = _store(ctx, R, ids)
    b = mb.DeviceBatch(ctx, st, ref)
    whole = _store(ctx, R, ids)
    bw = mb.DeviceBatch(ctx, whole, ref)
    preds = [([2], [1]), None, ([3, 2], [1, 0]), None, ([0], [4]), ([2], [2])]
    for keys in ([], [0]):
        for mode in MODES:
            for p in preds:
                if p is None:
                    got = b.run(keys, 60, 50, 0.3, mode=mode)
                    tg = b.timing()
                    want = bw.run(keys, 60, 50, 0.3, mode=mode)
                    _same_as_fresh(got, want, np.arange(S), 0, tg, bw.timing())
                    continue
                sel = np.flatnonzero(_mask(ids, *p))
                fresh = _store(ctx, R[sel], ids[sel])
                bf = mb.DeviceBatch(ctx, fresh, ref)
                got = b.run_where(p[0], p[1], keys, 60, 50, 0.3, mode=mode)
                tg = b.timing()
                want = bf.run(keys, 60, 50, 0.3, mode=mode)
                _same_as_fresh(got, want, sel, 0, tg, bf.timing(), S)
                bf.close()
                fresh.close()


@gpu
def test_where_argument_errors_leave_the_batch_usable(ctx):
    N, S = 480, 600
    rng = np.random.default_rng(2)
    R = _rows(rng, S, N)
    ids = _ids(S)
    ref = _ref(rng, N)
    st = _store(ctx, R, ids)
    b = mb.DeviceBatch(ctx, st, ref)
    want = b.run_where([2], [1], [0], 60, 20, 0.3)
    tw = b.timing()
    L = mb.lib()
    sc, lg, ix, n = np.zeros(20), np.zeros(20, dtype=np.int64), np.zeros(20, dtype=np.int64), C.c_int64(0)
    c = np.array([2] * 17, dtype=np.int32)
    v = np.array([1] * 17, dtype=np.int32)
    P = lambda a: a.ctypes.data_as(mb._ip32)

    def call(cols, vals, nw):
        return L.muse_batch_run_where(b.h, cols, vals, nw, None, 0, 60, 20, 0.3, 0, 0, 0, mb._d(sc),
                                      lg.ctypes.data_as(mb._ip64), ix.ctypes.data_as(mb._ip64), C.byref(n))

    bad_col = np.array([NKEYS], dtype=np.int32)
    neg_col = np.array([-1], dtype=np.int32)
    neg_id = np.array([-1], dtype=np.int32)
    for rc in (call(P(c), P(v), -1), call(P(c), P(v), 17), call(None, P(v), 1), call(P(c), None, 1),
               call(P(bad_col), P(v), 1), call(P(neg_col), P(v), 1), call(P(c), P(neg_id), 1)):
        assert rc == mb.MUSE_ERR_INVALID_ARG
    assert call(P(c), P(v), 16) == mb.MUSE_OK          # sixteen equalities are allowed
    _same_as_fresh(b.run_where([2], [1], [0], 60, 20, 0.3), want, np.arange(S), 0, b.timing(), tw)


# ---- facade --------------------------------------------------------------------------------------------------------
def _facade_group(rng, S, N):
    Y = _rows(rng, S, N)
    g = mb.NewGroup("where")
    series = []
    for i in range(S):
        lab = {"uid": "s%d" % i, "svc": "svc%d" % (i % 4), "colo": "c%d" % (i // 7 % 3)}
        if i % 5:                                            # every fifth series lacks "host"
            lab["host"] = "h%d" % (i % 9)
        series.append(mb.NewSeries(Y[i], mb.NewLabels(lab)))
    g.Add(*series)
    return g


def _fetch(r):
    got, _ = r.Fetch()
    return [(s.PercentScore, s.Lag, s.Labels) for s in got]


@gpu
@pytest.mark.parametrize("N", [480, 1440])
def test_facade_run_where_equals_run_on_a_filtered_group(ctx, N):
    rng = np.random.default_rng(N + 11)
    S = 1300
    g = _facade_group(rng, S, N)
    ref = mb.NewSeries(_ref(rng, N))
    for labels in ({"svc": "svc1"}, {"svc": "svc2", "host": "h4"}, {"host": "h3"}, {"colo": "c0", "svc": "svc3"}):
        L = mb.NewLabels(labels)
        G = mb.NewGroup("filtered")
        G.Add(*g.FilterByLabelValues(L))
        assert G.Length() == N and len(G.series) > 0
        for group_by in (None, ["colo"], ["host", "colo"], ["nokey"]):
            for max_lag, top_n, thr, sign in ((N, 10, 0.1, mb.SignFilter_ANY), (N, len(G.series) + 3, 0.0, mb.SignFilter_POS),
                                              (60, 10, 0.0, mb.SignFilter_ANY)):
                b = mb.NewBatch(ref, g, mb.NewResults(max_lag, top_n, thr, sign), 2)
                b.RunWhere(L, group_by)
                w = mb.NewBatch(ref, G, mb.NewResults(max_lag, top_n, thr, sign), 2)
                w.Run(group_by)
                got, want = _fetch(b.Results), _fetch(w.Results)
                assert len(got) == len(want) and (len(got) > 0 or max_lag < N)
                for (gs, gl, glab), (ws, wl, wlab) in zip(got, want):
                    assert gs == ws and gl == wl and glab is wlab


@gpu
def test_facade_run_where_nothing_matches(ctx):
    rng = np.random.default_rng(3)
    g = _facade_group(rng, 300, 480)
    ref = mb.NewSeries(_ref(rng, 480))
    for labels in ({"svc": "nope"}, {"nokey": "svc1"}, {}, {"svc": "svc1", "host": "nope"}):
        r = mb.NewResults(60, 10, 0.0, mb.SignFilter_ANY)
        b = mb.NewBatch(ref, g, r, 1)
        b.Run(None)                                          # Results hold one run's records ...
        before = [(s, -q, x.PercentScore, x.Lag, x.Labels) for s, q, x in r._heap]
        assert before
        b.RunWhere(mb.NewLabels(labels), ["colo"])           # ... which a run that matches nothing leaves as they are
        assert [(s, -q, x.PercentScore, x.Lag, x.Labels) for s, q, x in r._heap] == before
        assert g.FilterByLabelValues(mb.NewLabels(labels)) == []


# ---- checks that need no device -------------------------------------------------------------------------------------
class _NoDevice:
    def __getattr__(self, name):
        raise AssertionError("device call %s where nothing can match" % name)


def _cpu_batch():
    g = mb.NewGroup("cpu")
    g.Add(*[mb.NewSeries(np.arange(10.0) + i, mb.NewLabels({"h": str(i % 2), "uid": str(i)})) for i in range(4)])
    g._cols = ["h", "uid"]                                   # what _sync_device leaves: columns and value ids
    g._dict = {"h": {"0": 0, "1": 1}, "uid": {str(i): i for i in range(4)}}
    b = object.__new__(mb.Batch)
    b.Comparison, b.Results, b.mode, b._batch = g, mb.NewResults(5, 5, 0.0, 0), mb.MODE_AUTO, None
    return g, b


def test_group_where_maps_labels_to_columns_and_ids():
    g, _ = _cpu_batch()
    assert g._where(mb.NewLabels({"h": "1"})) == ([0], [1])
    assert g._where(mb.NewLabels({"uid": "3", "h": "1"})) == ([0, 1], [1, 3])
    assert g._where(mb.NewLabels({"h": "7"})) is None
    assert g._where(mb.NewLabels({"x": "1"})) is None
    assert g._where(mb.NewLabels({})) is None


def test_run_where_without_a_match_makes_no_device_call(monkeypatch):
    g, b = _cpu_batch()
    monkeypatch.setattr(mb, "_lib", _NoDevice())
    monkeypatch.setattr(g, "_sync_device", lambda: None)
    for labels in ({"h": "7"}, {"x": "0"}, {"h": "0", "uid": "9"}):
        assert b.RunWhere(mb.NewLabels(labels), ["h"]) is None
        assert b.Results._heap == []

    def no_sync():
        raise AssertionError("empty labels: not even the store is synchronised")

    monkeypatch.setattr(g, "_sync_device", no_sync)
    assert b.RunWhere(mb.NewLabels({}), None) is None


def test_device_batch_run_where_checks_lengths_before_any_call(monkeypatch):
    b = object.__new__(mb.DeviceBatch)
    b.h = C.c_void_p()
    monkeypatch.setattr(mb, "_lib", _NoDevice())
    with pytest.raises(mb.MuseError) as e:
        b.run_where([0, 1], [2], [], 60, 10, 0.5)
    assert e.value.code == mb.MUSE_ERR_INVALID_ARG


def test_run_where_abi_rejects_a_null_batch_without_a_device():
    mb.build()
    L = mb.lib()
    n = C.c_int64(0)
    assert L.muse_batch_run_where(None, None, None, 0, None, 0, 60, 10, 0.5, 0, 0, 0, None, None, None,
                                  C.byref(n)) == mb.MUSE_ERR_INVALID_ARG
