"""Parity of the CUDA path (through the C ABI) with the oracle.  Needs a B200."""
import os

import numpy as np
import pytest

import muse_b200 as mb
from oracle import c_oracle as co
from oracle import muse_oracle as mo

pytestmark = pytest.mark.gpu

SCORE_TOL = 1e-9   # north_star: scores within 1e-9 absolute in fp64


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _mk(entries):
    return [mb.NewSeries(e["y"], mb.NewLabels(e["labels"])) for e in entries]


def _compare_scores(scores, expected, tol):
    # muse_test.go:11-39 compareScores (+ the F4 tie-lag allowance)
    assert len(scores) == len(expected)
    for got, want in zip(scores, expected):
        assert got.Lag in want.get("tie_lags", [want["lag"]])
        assert abs(got.PercentScore - want["score"]) <= tol
        assert got.Labels.labels == want["labels"]


@pytest.mark.parametrize("name", ["batch_run_simple", "batch_run_multi_dimensional"])
def test_reference_batch_kats(kats, name):
    # muse_batch_test.go:9-82 through NewSeries/NewGroup/NewBatch/Run/Fetch
    k = kats[name]
    ref = mb.NewSeries(k["ref"]["y"], mb.NewLabels(k["ref"]["labels"]))
    g = mb.NewGroup("targets")
    assert g.Add(*_mk(k["comp"])) is None
    r = k["results"]
    b = mb.NewBatch(ref, g, mb.NewResults(r["max_lag"], r["top_n"], r["threshold"], r["sign_filter"]), k["concurrency"])
    assert b.Run(list(k["group_by"])) is None
    scores, _ = b.Results.Fetch()
    _compare_scores(scores, k["expected"], k["score_tol"])


def test_reference_batch_errors(kats):
    # muse_batch_test.go:83-102 and muse_batch.go:38-41
    k = kats["batch_run_with_larger_group"]
    g = mb.NewGroup("targets")
    g.Add(*_mk(k["comp"]))
    with pytest.raises(mb.MuseError) as e:
        mb.NewBatch(mb.NewSeries(k["ref"]["y"], mb.NewLabels(k["ref"]["labels"])), g, mb.NewResults(10, 20, 0, 0), 1)
    assert e.value.code == mb.MUSE_ERR_LENGTH_MISMATCH
    g = mb.NewGroup("t")
    g.Add(mb.NewSeries([1.0, 2.0, 3.0, 4.0], mb.NewLabels({"a": "b"})))
    with pytest.raises(mb.MuseError) as e:
        mb.NewBatch(mb.NewSeries([2.0, 2.0, 2.0, 2.0]), g, mb.NewResults(1, 1, 0, 0), 1)
    assert e.value.code == mb.MUSE_ERR_STDDEV_ZERO and "Invalid input query" in str(e.value)


def test_reference_muse_run_kats(kats):
    # muse_test.go:41-142: the signed Muse.Run path with all three sign filters, one series per Run
    k = kats["muse_run_simple"]
    for key, sf in (("expected_any", mb.SignFilter_ANY), ("expected_pos", mb.SignFilter_POS),
                    ("expected_neg", mb.SignFilter_NEG)):
        ref = mb.NewSeries(k["ref"]["y"], mb.NewLabels(k["ref"]["labels"]))
        m = mb.New(ref, mb.NewResults(k["results"]["max_lag"], k["results"]["top_n"], k["results"]["threshold"], sf))
        for s in _mk(k["comp"]):
            assert m.Run([s]) is None
        scores, _ = m.Results.Fetch()
        _compare_scores(scores, k[key], k["score_tol"])
    # one Run over the whole list keeps only the member with the largest |score| (muse.go:86)
    ref = mb.NewSeries(k["ref"]["y"], mb.NewLabels(k["ref"]["labels"]))
    m = mb.New(ref, mb.NewResults(k["results"]["max_lag"], k["results"]["top_n"], k["results"]["threshold"], mb.SignFilter_ANY))
    assert m.Run(_mk(k["comp"])) is None
    scores, _ = m.Results.Fetch()
    om = mo.Muse(mo.Series(k["ref"]["y"], mo.Labels(k["ref"]["labels"])),
                 mo.Results(k["results"]["max_lag"], k["results"]["top_n"], k["results"]["threshold"], mo.SIGN_FILTER_ANY))
    om.Run([mo.Series(e["y"], mo.Labels(e["labels"])) for e in k["comp"]])
    want, _ = om.Results.Fetch()
    assert len(scores) == len(want)
    for g, w in zip(scores, want):
        assert abs(g.PercentScore - w.PercentScore) <= 1e-9 and g.Lag == w.Lag and g.Labels.labels == w.Labels.labels
    # TestRunNoInput (muse_test.go) and the length check (muse.go:70-72)
    m = mb.New(ref, mb.NewResults(10, 20, 0, 0))
    assert m.Run([]) is None
    scores, mean = m.Results.Fetch()
    assert scores == [] and mean != mean
    err = m.Run([mb.NewSeries([1.0, 2.0, 3.0], mb.NewLabels({"a": "b"}))])
    assert isinstance(err, mb.MuseError) and "differing length" in str(err)
    with pytest.raises(mb.MuseError) as e:
        mb.New(mb.NewSeries([3.0, 3.0, 3.0, 3.0]), mb.NewResults(1, 1, 0, 0))
    assert e.value.code == mb.MUSE_ERR_STDDEV_ZERO


def test_example_structure(kats):
    # example_test.go:9-94 shape (C1): Run(nil) / ["graph"] / ["host"] on one Batch, Results reused
    rng = np.random.default_rng(5)
    N = 480

    def rect(amp, mid, width):
        y = np.zeros(N)
        y[mid - width // 2: mid - width // 2 + width] = amp
        return y

    noise = lambda: 0.1 * (rng.random(N) - 0.5)
    ref = mb.NewSeries(rect(1.5, 240, 10) + noise(), mb.NewLabels({"graph": "CallTime99Pct", "host": "host1"}))
    comp = mb.NewGroup("comparison")
    comp.Add(ref,
             mb.NewSeries(rect(1.5, 242, 7) + noise(), mb.NewLabels({"graph": "CallTime99Pct", "host": "host2"})),
             mb.NewSeries(rect(43, 240, 10) + noise(), mb.NewLabels({"graph": "ErrorRate", "host": "host1"})),
             mb.NewSeries(np.full(N, 0.1) + noise(), mb.NewLabels({"graph": "ErrorRate", "host": "host2"})),
             mb.NewSeries(np.full(N, 0.1), mb.NewLabels({"graph": "ErrorRate", "host": "host3"})))
    Y = np.stack([s.Values() for s in comp.series])
    m = mb.NewBatch(ref, comp, mb.NewResults(15, 4, 0.0, mb.SignFilter_ANY), 2)
    graph_ids = np.array([0, 0, 1, 1, 1])
    host_ids = np.array([0, 1, 0, 1, 2])
    for group_by, gids in ((None, None), (["graph"], graph_ids), (["host"], host_ids)):
        m.Run(group_by)
        res, _ = m.Results.Fetch()
        sc, lg, ix = mo.batch_run_arrays(ref.Values(), Y, gids, 15, 4, 0.0)
        assert [comp.series[int(i)].UID() for i in ix] == [s.Labels.ID(list(s.Labels.Keys())) for s in res]
        for s, a, l in zip(res, sc, lg):
            assert abs(s.PercentScore - a) <= SCORE_TOL and s.Lag == l
    # structure pinned by the Example: the constant series scores 0.000 at lag 0
    m.Run(None)
    res, _ = m.Results.Fetch()
    assert res[0].PercentScore == pytest.approx(1.0, abs=1e-12) and res[0].Lag == 0
    ids = [s.Labels.ID(list(s.Labels.Keys())) for s in res]
    assert "graph:ErrorRate,host:host3" in ids
    z = res[ids.index("graph:ErrorRate,host:host3")]
    assert z.PercentScore == 0.0 and z.Lag == 0


def _siggen(rng, S, N, pulse_every=3):
    ref = np.zeros(N)
    ref[N // 2 - min(5, N // 4): N // 2 + max(1, min(5, N // 4))] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    Y = 0.1 * (rng.random((S, N)) - 0.5)
    for i in range(0, S, pulse_every):
        w = int(rng.integers(1, max(2, min(20, N // 2))))
        m = int(rng.integers(0, max(1, N - w)))
        Y[i, m:m + w] += rng.uniform(0.5, 40)
    for i in range(1, S, pulse_every):
        Y[i] += rng.uniform(-0.01, 0.01) * np.arange(N) + rng.uniform(0, 100)
    return ref, Y


def _check_scores(ref, Y, sc, lg, tol=SCORE_TOL):
    want_s, want_l, ties = mo.score_series_batch(ref, Y, want_ties=True)
    assert np.max(np.abs(sc - want_s)) <= tol
    for i in range(Y.shape[0]):
        assert lg[i] == want_l[i] or lg[i] in ties[i], (i, lg[i], want_l[i])


@pytest.mark.parametrize("N", [2, 3, 4, 5, 8, 12, 31, 33, 100, 255, 480, 1000, 1440, 2500, 5000, 10080])
def test_score_all_matches_oracle(ctx, N):
    # every FFT size the kernels are instantiated for, odd and even lengths
    rng = np.random.default_rng(N)
    S = 257 if N <= 2500 else 37
    ref, Y = _siggen(rng, S, N)
    if N >= 8:
        Y[3] = 7.25                      # constant -> score 0, lag 0 (xcorr.go:165-168)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    b = mb.DeviceBatch(ctx, store, ref)
    assert b.fft_len() == mo.next_pow_of2(float(N))
    sc, lg = b.score_all()
    _check_scores(ref, Y, sc, lg)
    if N >= 8:
        assert sc[3] == 0.0 and lg[3] == 0
    # signed scores (muse.go:72-76)
    ssc, slg = b.score_all(signed_scores=True)
    want_s, want_l = mo.score_series_batch(ref, Y, signed=True)
    assert np.max(np.abs(ssc - want_s)) <= SCORE_TOL
    np.testing.assert_array_equal(np.abs(ssc), sc)


def test_xcorr_vector_kats(ctx, kats):
    # TestXCorrWithX inputs (xcorr_test.go:204-286) through the Batch path: N=5 -> n=8
    # (NewBatch always pads to a power of two); full cc vector against the oracle, plus the
    # lag/sign expectations that do not depend on n.
    k = kats["x_corr_with_x"]
    for c in k["cases"]:
        x, y = np.array(c["x"], dtype=float), np.array(c["y"], dtype=float)
        store = mb.DeviceStore(ctx, 5, 0, 1)
        store.append(y)
        b = mb.DeviceBatch(ctx, store, x)
        cc, std_zero = b.xcorr(0)
        X, n = mo.ref_spectrum(x)
        want_cc, want_lag, want_mv = mo.x_corr_with_x(X, y, n)
        if c["cc"] is None:
            assert std_zero and cc is None and want_cc is None
            continue
        assert np.max(np.abs(cc - want_cc)) <= 1e-12
        sc, lg = b.score_all(signed_scores=True)
        assert lg[0] == c["lag"] and np.sign(sc[0]) == c["sign"]
        assert abs(sc[0] - max(-1.0, min(1.0, want_mv))) <= 1e-12 and lg[0] == want_lag


def test_generic_xcorr_kats(ctx, kats):
    # TestXCorr (xcorr_test.go:86-202): n = 5, normalised and not, a constant input -> (nil, 0, 0)
    k = kats["x_corr"]
    for c in k["cases"]:
        cc, lag, mv = mb.xCorr(c["x"], c["y"], len(c["x"]), c["normalize"], ctx)
        if c["cc"] is None:
            assert cc is None and lag == 0 and mv == 0.0
            continue
        assert np.max(np.abs(cc - np.array(c["cc"], dtype=float))) <= k["tol"]
        assert lag == c["lag"] and np.sign(mv) == c["sign"]
        want_cc, want_lag, want_mv = mo.x_corr(c["x"], c["y"], len(c["x"]), c["normalize"])
        assert np.max(np.abs(cc - want_cc)) <= 1e-12 and lag == want_lag and abs(mv - want_mv) <= 1e-12


@pytest.mark.parametrize("lx,ly,n", [(5, 5, 5), (7, 5, 0), (5, 9, 12), (480, 480, 512), (1000, 1000, 1000),
                                     (1441, 1440, 2048), (3001, 2999, 3001), (16385, 16385, 32768)])
@pytest.mark.parametrize("normalize", [False, True])
def test_generic_xcorr_matches_oracle(ctx, lx, ly, n, normalize):
    # any n (not only powers of two), inputs of different lengths, n below / at / above the lengths;
    # the last shape is BenchmarkXCorr's (xcorr_test.go:310-326)
    rng = np.random.default_rng(lx * 31 + ly * 7 + n)
    x, y = rng.random(lx), rng.random(ly)
    y[ly // 3] += 25.0
    x[lx // 2] += 25.0
    cc, lag, mv = mb.xCorr(x, y, n, normalize, ctx)
    want_cc, want_lag, want_mv = mo.x_corr(x, y, n, normalize)
    assert cc.shape == want_cc.shape
    scale = max(1.0, float(np.max(np.abs(want_cc))))
    assert np.max(np.abs(cc - want_cc)) <= SCORE_TOL * scale
    assert lag == want_lag and abs(mv - want_mv) <= SCORE_TOL * scale


def test_generic_xcorr_edge_cases(ctx):
    # a constant input is only an error when normalising (xcorr.go:108-127)
    cc, lag, mv = mb.xCorr([3, 3, 3, 3], [0, 1, 0, 0], 4, False, ctx)
    np.testing.assert_allclose(cc, [3, 3, 3, 3])
    assert (lag, mv) == (0, 3.0)                     # first index wins the tie (xcorr.go:39-50)
    assert mb.xCorr([3, 3, 3, 3], [0, 1, 0, 0], 4, True, ctx) == (None, 0, 0.0)
    assert mb.xCorr([0, 1, 0, 0], [2, 2, 2, 2], 4, True, ctx) == (None, 0, 0.0)
    # all-zero correlation: index 0, value 0
    cc, lag, mv = mb.xCorr([0, 0, 0], [1, 2, 3], 3, False, ctx)
    assert not cc.any() and (lag, mv) == (0, 0.0)
    # NaN samples never win the arg-max (math.Abs(NaN) > x is false)
    cc, lag, mv = mb.xCorr([1, 0, 0, 0], [float("nan"), 0, 0, 0], 4, False, ctx)
    want_cc, want_lag, want_mv = mo.x_corr([1, 0, 0, 0], [float("nan"), 0, 0, 0], 4, False)
    assert lag == want_lag
    with pytest.raises(mb.MuseError):
        mb.xCorr([], [1.0], 4, False, ctx)


def test_run_matches_oracle_ungrouped_and_grouped(ctx):
    rng = np.random.default_rng(11)
    S, N = 6000, 480
    ref, Y = _siggen(rng, S, N)
    graph = (np.arange(S) // 50).astype(np.int32)
    host = (np.arange(S) % 50).astype(np.int32)
    colo = rng.integers(0, 3, S).astype(np.int32)
    ids = np.stack([graph, host, colo], axis=1)
    store = mb.DeviceStore(ctx, N, 3, S)
    store.append(Y, ids)
    b = mb.DeviceBatch(ctx, store, ref)
    sl = mo.score_series_batch(ref, Y)

    def dense(*cols):
        _, inv = np.unique(np.stack(cols, axis=1), axis=0, return_inverse=True)
        # first-appearance order
        first = {}
        out = np.zeros(S, dtype=np.int64)
        for i, g in enumerate(inv.ravel()):
            out[i] = first.setdefault(int(g), len(first))
        return out

    cases = [([], None), ([0], dense(graph)), ([1], dense(host)), ([0, 2], dense(graph, colo)),
             ([0, 1, 2], dense(graph, host, colo))]
    for cols, gids in cases:
        for max_lag, top_n, thr in ((10, 20, 0.0), (60, 100, 0.5), (240, 5, 0.2), (3, 7000, 0.0)):
            sc, lg, ix = b.run(cols, max_lag, top_n, thr, mode=mb.MODE_EXACT)
            wsc, wlg, wix = mo.batch_run_arrays(ref, Y, gids, max_lag, top_n, thr, scores_lags=sl)
            assert len(sc) == len(wsc), (cols, max_lag, top_n, thr)
            assert np.max(np.abs(sc - wsc), initial=0.0) <= SCORE_TOL
            np.testing.assert_array_equal(ix, wix)
            np.testing.assert_array_equal(lg, wlg)
    t = b.timing()
    assert t.n_launches >= 2 and t.total_ms > 0


def test_top_n_device_select_with_ties(ctx):
    # heavy ties: many exact duplicates of a few rows, so the top-N must cut by (score desc, index asc).  Every series
    # passes the filter: a store of 20000 takes the device-side rank-by-counting top-N; one of 300000 has more candidates
    # than that ranks (32768) and than run_select leaves to the host (262144), so it takes the device radix select, whose
    # last digits are the ~index ones
    rng = np.random.default_rng(2)
    N = 64
    ref, base = _siggen(rng, 8, N, pulse_every=1)
    for S in (20000, 300000):
        Y = base[rng.integers(0, 8, S)]
        store = mb.DeviceStore(ctx, N, 0, S)
        store.append(Y)
        b = mb.DeviceBatch(ctx, store, ref)
        sl = mo.score_series_batch(ref, Y)
        for top_n in (1, 100, 4500, 12345):
            sc, lg, ix = b.run([], N, top_n, 0.0, mode=mb.MODE_EXACT)
            wsc, wlg, wix = mo.batch_run_arrays(ref, Y, None, N, top_n, 0.0, scores_lags=sl)
            assert len(sc) == len(wsc), (S, top_n)
            np.testing.assert_array_equal(ix, wix, err_msg="S = %d, top_n = %d" % (S, top_n))
            assert np.max(np.abs(sc - wsc), initial=0.0) <= SCORE_TOL, (S, top_n)


def test_hash_group_table(ctx):
    # label cardinalities whose product exceeds the dense table -> open-addressing path
    rng = np.random.default_rng(3)
    S, N = 3000, 100
    ref, Y = _siggen(rng, S, N)
    a = rng.integers(0, 2_000_000, S).astype(np.int32)
    a[::7] = a[0]                      # some real groups
    c = rng.integers(0, 1_000_000, S).astype(np.int32)
    c[::7] = c[0]
    a[5], c[5] = -1, -1                # absent labels share the "" group (labels.go:61-65)
    a[6], c[6] = -1, -1
    store = mb.DeviceStore(ctx, N, 2, S)
    store.append(Y, np.stack([a, c], axis=1))
    b = mb.DeviceBatch(ctx, store, ref)
    key = {}
    gids = np.array([key.setdefault((int(x), int(y)), len(key)) for x, y in zip(a, c)])
    sc, lg, ix = b.run([0, 1], 100, 50, 0.0, mode=mb.MODE_EXACT)
    wsc, wlg, wix = mo.batch_run_arrays(ref, Y, gids, 100, 50, 0.0)
    np.testing.assert_array_equal(ix, wix)
    assert np.max(np.abs(sc - wsc)) <= SCORE_TOL


def test_group_by_six_keys(ctx):
    # labels.go:54-73 takes any number of keys: six group-by columns (10 key bits each when packed evenly; one column
    # of cardinality 5000 forces the per-column widths), against the oracle; 9 wide columns do not fit 64 bits -> an error
    rng = np.random.default_rng(17)
    S, N = 4000, 100
    ref, Y = _siggen(rng, S, N)
    cards = [7, 3, 5000, 2, 11, 4, 200000, 200000, 200000, 200000, 200000, 200000, 200000, 200000, 200000]
    ids = np.stack([rng.integers(0, c, S) for c in cards], axis=1).astype(np.int32)
    ids[::5, 2] = 17                       # real groups
    ids[::5, :2] = 1
    ids[3, 4] = -1                         # an absent label is a value of its own (labels.go:61-65)
    store = mb.DeviceStore(ctx, N, len(cards), S)
    store.append(Y, ids)
    b = mb.DeviceBatch(ctx, store, ref)
    for cols in ([0, 1, 2, 3, 4, 5], [0, 1, 3, 4, 5], [5, 4, 3, 2, 1, 0]):
        key = {}
        gids = np.array([key.setdefault(tuple(int(v) for v in row), len(key)) for row in ids[:, sorted(cols)]])
        sc, lg, ix = b.run(cols, 100, 60, 0.0, mode=mb.MODE_EXACT)
        wsc, wlg, wix = mo.batch_run_arrays(ref, Y, gids, 100, 60, 0.0)
        np.testing.assert_array_equal(ix, wix)
        np.testing.assert_array_equal(lg, wlg)
        assert np.max(np.abs(sc - wsc)) <= SCORE_TOL
    with pytest.raises(mb.MuseError) as ei:
        b.run(list(range(6, 15)), 100, 60, 0.0, mode=mb.MODE_EXACT)
    assert ei.value.code == mb.MUSE_ERR_UNSUPPORTED


def test_synthetic_rows_identical_on_host_and_device(ctx):
    N, S, seed, first = 1440, 64, 20261018, 999_990
    store = mb.DeviceStore(ctx, N, 2, S)
    store.append_synthetic(S, seed, first)
    for i in (0, 1, 2, 9, 10, 63):
        np.testing.assert_array_equal(store.read_row(i), mb.synth_row(seed, first + i, N))
    kinds = [np.ptp(mb.synth_row(seed, first + i, N)) for i in range(3)]
    assert max(kinds) > 0.4                      # a rect pulse is in there
    ref = mb.synth_reference(seed, N)
    assert ref[N // 2] > 1.4 and abs(ref[10]) <= 0.05


def test_sharded_partials_merge_equals_single_store(ctx):
    # two shards with global offsets -> partials -> merge == one store (F2: group max before filter)
    rng = np.random.default_rng(17)
    S, N = 4000, 256
    ref, Y = _siggen(rng, S, N)
    graph = rng.integers(0, 40, S).astype(np.int32)      # groups straddle the shard boundary
    ids = graph[:, None]
    whole = mb.DeviceStore(ctx, N, 1, S)
    whole.append(Y, ids)
    bw = mb.DeviceBatch(ctx, whole, ref)
    cut = 1700
    shards = []
    for lo, hi in ((0, cut), (cut, S)):
        st = mb.DeviceStore(ctx, N, 1, hi - lo)
        st.append(Y[lo:hi], ids[lo:hi])
        st.set_global_offset(lo)
        shards.append(mb.DeviceBatch(ctx, st, ref))
    for cols in ([], [0]):
        for max_lag, top_n, thr in ((20, 10, 0.0), (128, 100, 0.3)):
            parts = np.concatenate([s.run_partial(cols, max_lag, top_n, thr, mode=mb.MODE_EXACT) for s in shards])
            sc, lg, ix = mb.merge_partials(parts, max_lag, top_n, thr)
            wsc, wlg, wix = bw.run(cols, max_lag, top_n, thr, mode=mb.MODE_EXACT)
            np.testing.assert_array_equal(ix, wix)
            np.testing.assert_array_equal(lg, wlg)
            np.testing.assert_array_equal(sc, wsc)


def test_device_side_partials_equal_host_partials(ctx):
    # muse_batch_run_partial_device: the shard's filtered top_n written to device memory == run_partial's records
    import torch
    rng = np.random.default_rng(29)
    for S, N in ((3000, 256), (40_000, 1440)):
        ref, Y = _siggen(rng, S, N)
        Y[5] = Y[4]                                  # an exact tie: lowest index first
        st = mb.DeviceStore(ctx, N, 0, S)
        st.append(Y)
        st.set_global_offset(1_000_000)
        b = mb.DeviceBatch(ctx, st, ref)
        for max_lag, top_n, thr in ((20, 10, 0.0), (128, 100, 0.3), (N, 500, 0.0)):
            want = b.run_partial([], max_lag, top_n, thr)
            t = torch.zeros(top_n * 32, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            b.run_partial_device(max_lag, top_n, thr, 0, mb.MODE_AUTO, t.data_ptr(), top_n)
            ctx.synchronize()
            got = t.cpu().numpy().view(mb.PARTIAL_DTYPE)
            if np.any(got["flags"] == 2):            # more than 32768 passing candidates: the documented overflow signal
                assert thr == 0.0 and max_lag == N
                continue
            k = len(want)
            np.testing.assert_array_equal(got[:k], want)
            assert np.all(got["flags"][k:] == 1)
            tm = b.timing()
            assert tm.total_ms > 0 and tm.n_launches >= 2
        b.close()


def test_c_oracle_agrees_at_larger_size(ctx):
    # the fast C oracle as checker at a size the numpy form would take long on
    rng = np.random.default_rng(23)
    S, N = 20000, 1440
    ref, Y = _siggen(rng, S, N)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    b = mb.DeviceBatch(ctx, store, ref)
    sc, lg = b.score_all()
    wsc, wlg = co.score_all(ref, Y)
    assert np.max(np.abs(sc - wsc)) <= SCORE_TOL
    bad = np.nonzero(lg != wlg)[0]
    for i in bad[:50]:      # any lag mismatch must be a tie within tolerance
        _, _, ties = mo.score_series_batch(ref, Y[i:i + 1], want_ties=True)
        assert lg[i] in ties[0]
    assert bad.size <= 50


def test_pageable_rows_are_staged_through_the_pinned_ring(ctx):
    """muse_group_append from PAGEABLE host memory (a numpy array, a Go slice): chunks go through the context's ring of pinned
    buffers, filled by several host threads while the previous chunk is on the wire.  Rows must arrive intact (also at a
    pitch that needs a 2-D copy), and the rate must be that of a staged copy, not of a single-threaded bounce buffer."""
    import time
    rng = np.random.default_rng(8)
    S, N = 150_000, 1440
    Y = rng.standard_normal((S, N))                      # 1.7 GB, pageable
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y[:1000])                               # warm: ring allocation, thread start-up
    store.clear()
    t0 = time.perf_counter()
    store.append(Y)
    dt = time.perf_counter() - t0
    gbs = Y.nbytes / dt / 1e9
    print("pageable append: %.1f GB/s (%d threads available)" % (gbs, os.cpu_count()))
    for i in (0, 1, 4095, 4096, 77_777, S - 1):
        np.testing.assert_array_equal(store.read_row(i), Y[i])
    assert gbs >= 10.0
    store.close()
    N2 = 1001                                            # odd length: pitched rows, pad column
    Z = rng.standard_normal((70_000, N2))
    st2 = mb.DeviceStore(ctx, N2, 0, 70_000)
    st2.append(Z)
    for i in (0, 8190, 69_999):
        np.testing.assert_array_equal(st2.read_row(i), Z[i])
    st2.close()


def test_peer_memory_exchange_single_rank(ctx):
    # muse_batch_run_exchange with world_size 1: the selection kernel pushes into its own receive buffer, waits
    # on its own flag, merges -> must be the plain Run; repeated calls alternate the two buffer parities
    rng = np.random.default_rng(5)
    S, N = 20000, 480
    ref, Y = _siggen(rng, S, N)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    b = mb.DeviceBatch(ctx, store, ref)
    ex = mb.Exchange(ctx, 64)
    for max_lag, top_n, thr in ((15, 50, 0.3), (15, 64, 0.0), (3, 1, 0.9), (15, 50, 0.3), (0, 7, 0.0)):
        want = b.run([], max_lag, top_n, thr)
        got = ex.run(b, max_lag, top_n, thr)
        assert got is not None
        for g, w in zip(got, want):
            np.testing.assert_array_equal(g, w)
    with pytest.raises(mb.MuseError):
        ex.run(b, 15, 65, 0.3)                      # above the exchange's capacity
    ex.close()


def test_peer_memory_exchange_grouped_single_rank(ctx):
    # grouped runs through the exchange: every group representative of the shard is pushed (unfiltered, SURVEY F2), the
    # group max across shards, the filter and the top-N run on the device -> with one shard it must be the plain grouped Run
    rng = np.random.default_rng(6)
    S, N = 12000, 480
    ref, Y = _siggen(rng, S, N)
    ids = np.stack([np.arange(S) // 40, np.arange(S) % 40, rng.integers(0, 3, S)], axis=1).astype(np.int32)
    store = mb.DeviceStore(ctx, N, 3, S)
    store.append(Y, ids)
    b = mb.DeviceBatch(ctx, store, ref)
    ex = mb.Exchange(ctx, 1024)
    for cols in ([0], [1], [0, 2]):
        for max_lag, top_n, thr in ((15, 50, 0.3), (15, 1000, 0.0), (3, 1, 0.9)):
            want = b.run(cols, max_lag, top_n, thr)
            got = ex.run(b, max_lag, top_n, thr, key_cols=cols)
            assert got is not None
            for g, w in zip(got, want):
                np.testing.assert_array_equal(g, w)
    assert ex.run(b, 15, 50, 0.3, key_cols=[0, 1]) is None      # 12000 groups do not fit 1024 records: the host path is asked for
    ex.close()


def test_peer_memory_exchange_two_gpus():
    # two ranks, one per GPU (skipped on a one-GPU box): tools/exchange_check.py compares the peer-memory push
    # with the NCCL all-gather path and the host path for several argument sets
    import os, subprocess, sys, torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CHECK_SERIES="200000")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(root, "tools", "exchange_check.py")],
                       env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL IDENTICAL" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_multi_reference_run_equals_separate_batches(ctx):
    # muse_multi_run: Q references against one resident store == Q x (NewBatch + Run); a constant reference
    # fails for itself only (muse_batch.go:38-41)
    rng = np.random.default_rng(17)
    S, N, Q = 3000, 480, 5
    _, Y = _siggen(rng, S, N)
    refs = np.zeros((Q, N))
    for q in range(Q):
        m = int(rng.integers(100, 380))
        refs[q, m:m + 4 + 2 * q] = 1.0 + q
        refs[q] += 0.1 * (rng.random(N) - 0.5)
    refs[3] = 7.0
    ids = np.stack([np.arange(S) // 30, np.arange(S) % 30], axis=1).astype(np.int32)
    store = mb.DeviceStore(ctx, N, 2, S)
    store.append(Y, ids)
    for cols in ([], [0]):
        got = mb.multi_run(store, refs, cols, 20, 15, 0.2)
        assert got[3] is None
        for q in (0, 1, 2, 4):
            b = mb.DeviceBatch(ctx, store, refs[q])
            want = b.run(cols, 20, 15, 0.2)
            for g, w in zip(got[q], want):
                np.testing.assert_array_equal(g, w)
            wsc, wlg, wix = co.batch_run(refs[q], Y, (ids[:, 0] if cols else None), 20, 15, 0.2)
            assert np.max(np.abs(got[q][0] - wsc), initial=0) <= SCORE_TOL
            np.testing.assert_array_equal(got[q][1], wlg)
            np.testing.assert_array_equal(got[q][2], wix)
            b.close()


def test_incremental_store_growth(ctx):
    # SURVEY 8f rank 4: Group.Add after the first upload and after a Batch exists.  The store grows (slab
    # reallocation, row statistics extended for the new rows only), the existing batch sees the new series.
    rng = np.random.default_rng(23)
    S, N = 24000, 1440
    ref, Y = _siggen(rng, S, N)
    store = mb.DeviceStore(ctx, N, 0, 16)                 # tiny reservation: forces several reallocations
    b = None
    done = 0
    for chunk in (5000, 1, 12999, 6000):
        store.append(Y[done:done + chunk])
        done += chunk
        if b is None:
            b = mb.DeviceBatch(ctx, store, ref)
        for mode in (mb.MODE_SCREEN, mb.MODE_EXACT):
            sc, lg, ix = b.run([], 60, 50, 0.3, mode=mode)
            wsc, wlg, wix = co.batch_run(ref, Y[:done], None, 60, 50, 0.3)
            assert np.max(np.abs(sc - wsc), initial=0) <= SCORE_TOL
            np.testing.assert_array_equal(lg, wlg)
            np.testing.assert_array_equal(ix, wix)
    assert store.size() == S
    # the same through the facade: Add between two Runs of one Batch (Results is not reset between Runs, results.go:55-72)
    g = mb.NewGroup("grow")
    mk = lambda i: mb.NewSeries(Y[i, :480].copy(), mb.NewLabels({"host": "h%d" % i}))
    g.Add(*[mk(i) for i in range(0, 300)])
    batch = mb.NewBatch(mb.NewSeries(ref[480:960].copy()), g, mb.NewResults(20, 400, 0.0, mb.SignFilter_ANY), 1)
    batch.Run(None)
    first, _ = batch.Results.Fetch()
    g.Add(*[mk(i) for i in range(300, 700)])
    with pytest.raises(mb.MuseError):
        g.Add(mk(5))                                       # duplicate UID (group.go:39-41)
    with pytest.raises(mb.MuseError):
        g.Add(mb.NewSeries(Y[0, :100].copy(), mb.NewLabels({"host": "short"})))   # length (group.go:45-51)
    batch.Run(None)
    second, _ = batch.Results.Fetch()
    sl = mo.score_series_batch(ref[480:960], Y[:700, :480])
    want = sorted([(min(abs(float(s)), 1.0), i) for i, (s, l) in enumerate(zip(*sl)) if abs(l) <= 20], key=lambda x: (-x[0], x[1]))[:400]
    assert len(first) <= 300 and len(second) == len(want)
    for got, (ws, wi) in zip(second, want):
        assert abs(got.PercentScore - ws) <= SCORE_TOL and got.Labels is g.series[wi].Labels()
