"""The fp32 screening pass: its bound must dominate the exact score on every input, and a
screened Batch.Run must return exactly what the all-exact run returns.  Needs a B200."""
import numpy as np
import pytest

import muse_b200 as mb
from oracle import c_oracle as co
from oracle import muse_oracle as mo

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _adversarial(rng, S, N):
    """siggen-style rows plus the inputs that stress an fp32 pass."""
    Y = 0.1 * (rng.random((S, N)) - 0.5)
    t = np.arange(N)
    for i in range(S):
        k = i % 12
        if k == 0:      # rect pulse near the reference's
            m = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8))
            Y[i, m:m + int(rng.integers(3, 20))] += rng.uniform(0.5, 40)
        elif k == 1:    # huge offset, unit noise
            Y[i] = 1e9 + rng.standard_normal(N)
        elif k == 2:    # tiny amplitude
            Y[i] *= 1e-12
        elif k == 3:    # huge amplitude
            Y[i] = 1e12 * rng.standard_normal(N)
        elif k == 4:    # one spike
            Y[i, int(rng.integers(0, N))] += 1e6
        elif k == 5:    # trend
            Y[i] += 3.0 * t + 1e5
        elif k == 6:    # exact copy of a shifted reference-like pulse (score ~ 1)
            Y[i] = 0.0
            Y[i, N // 2 - 5:N // 2 + 5] = 2.0
        elif k == 7:    # constant
            Y[i] = 0.1
        elif k == 8:    # almost constant: one ulp-level wiggle
            Y[i] = 5.0
            Y[i, 7] = np.nextafter(5.0, 6.0)
        elif k == 9:    # first sample is an outlier (the fp32 pivot)
            Y[i, 0] = 1e8
        elif k == 10:   # sinusoid
            Y[i] = np.sin(2 * np.pi * t / rng.uniform(5, 200)) + 100.0
        # k == 11: plain noise
    return Y


@pytest.mark.parametrize("N", [1440, 1030, 2048, 480, 300, 700, 1000, 1024, 2500, 4096, 6000, 10080,
                               1441, 1027, 2047, 481, 999, 2049, 4097, 10081, 16383, 66, 100, 127, 128, 130, 200, 255, 256, 257, 259, 513])
def test_screened_run_equals_exact_run(ctx, N):
    rng = np.random.default_rng(N)
    S = 30000 if N <= 2048 else 6000
    Y = _adversarial(rng, S, N)
    ref = np.zeros(N)
    ref[N // 2 - 5:N // 2 + 5] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    b = mb.DeviceBatch(ctx, store, ref)
    for max_lag, top_n, thr in ((60, 100, 0.5), (15, 10, 0.0), (N, 2000, 0.9), (5, 50000, 0.2), (60, 0, 0.0)):
        e = b.run([], max_lag, top_n, thr, mode=mb.MODE_EXACT)
        assert b.timing().mode == mb.MODE_EXACT
        s = b.run([], max_lag, top_n, thr, mode=mb.MODE_SCREEN)
        t = b.timing()
        assert t.mode == mb.MODE_SCREEN
        for x, y in zip(e, s):
            np.testing.assert_array_equal(x, y)      # bit-identical scores, lags and indices
    # the oracle agrees with both
    sc, lg, ix = b.run([], 60, 100, 0.5, mode=mb.MODE_SCREEN)
    wsc, wlg, wix = co.batch_run(ref, Y, None, 60, 100, 0.5)
    assert np.max(np.abs(sc - wsc), initial=0) <= 1e-9
    same = ix == wix
    assert same.mean() > 0.9    # identical rows (k == 6) tie exactly; order among ties may differ from the oracle's
    assert set(ix[~same]) == set(wix[~same])


@pytest.mark.parametrize("N", [10080, 16384, 8195])
def test_n16384_screened_runs_equal_exact_runs(ctx, N):
    """The n = 16384 screening kernel on short, full and odd rows: ungrouped and grouped screened runs must be the
    all-exact run, bit for bit, and the refined bounds must dominate the exact scores."""
    rng = np.random.default_rng(13 * N)
    S = 5000
    Y = _adversarial(rng, S, N)
    ref = np.zeros(N)
    ref[N // 2 - 5:N // 2 + 5] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    store = mb.DeviceStore(ctx, N, 1, S)
    store.append(Y, (np.arange(S) // 25).astype(np.int32)[:, None])
    b = mb.DeviceBatch(ctx, store, ref)
    for cols in ([], [0]):
        for max_lag, top_n, thr in ((240, 100, 0.5), (N, 300, 0.0)):
            e = b.run(cols, max_lag, top_n, thr, mode=mb.MODE_EXACT)
            s = b.run(cols, max_lag, top_n, thr, mode=mb.MODE_SCREEN)
            assert b.timing().mode == mb.MODE_SCREEN
            for x, y in zip(e, s):
                np.testing.assert_array_equal(x, y)
    up, lo = b.screen_bounds(refine=True, max_lag=240)
    sc, lg = b.score_all()
    dec = up >= 0
    assert np.all(up[dec].astype(np.float64) >= sc[dec] + 0.5e-4)


@pytest.mark.parametrize("N", [1440, 1441, 480, 10080])
def test_signed_screened_run_equals_exact_run(ctx, N):
    """Signed scores (Muse.Run, muse.go:72-76: the sign is kept, clamp to [-1, 1], ranking by |score|) through the
    screening: the bounds hold for |score|, the survivors are re-scored signed -> the all-exact signed run, bit for bit."""
    rng = np.random.default_rng(7 * N)
    S = 30000 if N <= 2048 else 6000
    Y = _adversarial(rng, S, N)
    Y[::2] *= -1.0                                   # half of the pulses point down: negative peaks
    ref = np.zeros(N)
    ref[N // 2 - 5:N // 2 + 5] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    store = mb.DeviceStore(ctx, N, 1, S)
    store.append(Y, (np.arange(S) // 25).astype(np.int32)[:, None])
    b = mb.DeviceBatch(ctx, store, ref)
    for cols in ([], [0]):
        for max_lag, top_n, thr in ((60, 100, 0.5), (N, 500, 0.0)):
            e = b.run(cols, max_lag, top_n, thr, mode=mb.MODE_EXACT, signed_scores=True)
            s = b.run(cols, max_lag, top_n, thr, mode=mb.MODE_SCREEN, signed_scores=True)
            assert b.timing().mode == mb.MODE_SCREEN
            for x, y in zip(e, s):
                np.testing.assert_array_equal(x, y)
            assert (e[0] < 0).any()
    # a sign filter on signed scores cannot be screened (no bound knows the sign): the exact path serves it
    s = b.run([], 60, 100, 0.5, sign_filter=mb.SignFilter_NEG, mode=mb.MODE_AUTO, signed_scores=True)
    assert b.timing().mode == mb.MODE_EXACT and len(s[0]) > 0 and np.all(s[0] < 0)


@pytest.mark.parametrize("N", [1440, 1026, 1030, 1088, 1090, 1500, 1984, 2046, 2048, 480, 300, 258, 512, 514, 720, 1000, 1024,
                               2050, 3000, 4096, 4098, 7000, 8192, 8194, 10080, 16384, 66, 101, 128, 130, 199, 256])
def test_bound_dominates_exact_score(ctx, N):
    """U >= exact fp64 score for every series, on the adversarial inputs and on siggen-style rows;
    the margin U - score is reported (it must never be negative)."""
    rng = np.random.default_rng(7 * N)
    S = 6000 if N <= 2048 else 1200
    Y = _adversarial(rng, S, N)
    ref = np.zeros(N)
    ref[N // 2 - 5:N // 2 + 5] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    b = mb.DeviceBatch(ctx, store, ref)
    u = b.screen_bounds().astype(np.float64)
    sc, _ = b.score_all()
    assert np.all(np.isfinite(u))
    margin = u - sc
    # at least half of the 1e-4 slack is left (bit-identical constant rows may get U == score == 0)
    worst = int(margin.argmin())
    assert margin.min() >= 0 and np.all((margin >= 0.5e-4) | (sc == 0)), (margin.min(), worst, u[worst], sc[worst])
    decided = u <= 1.5
    assert decided.mean() > 0.6                     # the bound is not trivially "undecided"
    # constant / near-constant rows (k == 7, 8) and the 1e-12 amplitude rows are either undecided or bounded
    assert np.all(u[7::12] >= sc[7::12])


@pytest.mark.parametrize("N,max_lag", [(1440, 60), (1440, 0), (1440, 5000), (1026, 15), (1500, 300), (2048, 60), (2046, 1),
                                       (2050, 30), (4000, 240), (5000, 0), (10080, 240), (10080, 20000), (16384, 7),
                                       (480, 15), (300, 0), (512, 600), (1000, 60), (1024, 3),
                                       (1441, 60), (2047, 5), (1027, 0), (481, 15), (9999, 240), (2049, 30),
                                       (66, 3), (100, 10), (128, 0), (129, 200), (200, 15), (255, 7), (256, 30)])
def test_refined_bounds_bracket_exact_score(ctx, N, max_lag):
    """Fused second stage (fp32 inverse transform) on every series: lower <= exact score <= upper, a series
    declared outside the lag window really is, one declared inside really is; the fp32 error is reported."""
    rng = np.random.default_rng(11 * N + max_lag)
    S = 6000 if N <= 2048 else 1200
    Y = _adversarial(rng, S, N)
    ref = np.zeros(N)
    ref[N // 2 - 5:N // 2 + 5] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    b = mb.DeviceBatch(ctx, store, ref)
    up, lo = b.screen_bounds(refine=True, max_lag=max_lag)
    up = up.astype(np.float64)
    lo = lo.astype(np.float64)
    sc, lg = b.score_all()
    inside = np.abs(lg) <= max_lag
    out = up == -1.0
    assert not np.any(out & inside)                  # "certainly outside" is never wrong
    assert np.all(inside[lo >= 0])                   # "certainly inside" is never wrong
    dec = ~out
    assert np.all(up[dec] >= sc[dec] + 0.5e-4)       # upper bound with at least half of the slack left
    assert np.all(lo[lo >= 0] <= sc[lo >= 0] - 0.5e-4)
    tight = dec & (up <= 1.5)
    assert tight.sum() >= dec.sum() - S // 3         # only the huge-offset / tiny / constant / near-constant rows (4 kinds of 12) stay undecided
    # the refined bound is tight: within ~2 slacks of the exact score almost everywhere it was computed
    assert np.mean(up[tight] - sc[tight] <= 2.2e-4) > 0.99
    # most rows are decided one way or the other
    assert (out | (lo >= 0)).mean() > 0.5


@pytest.mark.parametrize("N", [1440, 2500, 10080, 480, 1000, 1441, 5001, 100, 250])
def test_grouped_screened_run_equals_exact_run(ctx, N):
    """Grouped runs on the fused kernels: every member refined, a group's best lower bound prunes its members,
    only the contenders are scored in fp64 -- the result must be the all-exact run's, bit for bit."""
    rng = np.random.default_rng(3 * N)
    S = 12000 if N <= 2048 else 4000
    Y = _adversarial(rng, S, N)
    ref = np.zeros(N)
    ref[N // 2 - 5:N // 2 + 5] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    graph = (np.arange(S) // 40).astype(np.int32)
    host = (np.arange(S) % 40).astype(np.int32)
    colo = rng.integers(0, 3, S).astype(np.int32)
    rnd = rng.integers(0, 1_500_000, S).astype(np.int32)      # hash-table path with singleton groups
    store = mb.DeviceStore(ctx, N, 4, S)
    store.append(Y, np.stack([graph, host, colo, rnd], axis=1))
    b = mb.DeviceBatch(ctx, store, ref)
    for cols in ([0], [1], [0, 2], [2], [3, 0]):
        for max_lag, top_n, thr in ((60, 100, 0.5), (15, 10, 0.0), (N, 2000, 0.2), (60, 3, 0.0), (N, 1, 0.9), (5, 7, 0.3)):
            e = b.run(cols, max_lag, top_n, thr, mode=mb.MODE_EXACT)
            s = b.run(cols, max_lag, top_n, thr, mode=mb.MODE_SCREEN)
            t = b.timing()
            assert t.mode == mb.MODE_SCREEN
            for x, y in zip(e, s):
                np.testing.assert_array_equal(x, y)
    # the point of it: far fewer fp64 scorings than series
    b.run([0], 60, 100, 0.5, mode=mb.MODE_SCREEN)
    assert b.timing().n_rescored < 0.6 * S
    if N > 2048:
        # n = 4096 .. 16384: a short top-N needs exact scores only for groups that can reach it (group_cut_find_kernel)
        b.run([3, 0], N, 2000, 0.0, mode=mb.MODE_SCREEN)
        many = b.timing().n_rescored
        b.run([3, 0], N, 5, 0.0, mode=mb.MODE_SCREEN)
        assert b.timing().n_rescored < many
    # sharded partials (F2: unfiltered group representatives) out of the screened path: every group whose representative
    # reaches the threshold is there unchanged; below it the screened path may name another member (or none) -- a member
    # whose bound is under the threshold is never scored, and such a group fails results.go:46-52 after any merge
    pe = b.run_partial([0, 2], 60, 100, 0.5, mode=mb.MODE_EXACT)
    ps = b.run_partial([0, 2], 60, 100, 0.5, mode=mb.MODE_SCREEN)
    np.testing.assert_array_equal(np.sort(pe[pe["score"] >= 0.5], order=["group_key"]), np.sort(ps[ps["score"] >= 0.5], order=["group_key"]))
    assert np.all(np.isin(ps["group_key"], pe["group_key"])) and np.all(ps["score"][~np.isin(ps["series_idx"], pe["series_idx"])] < 0.5)
    for top_n in (100, 5):
        for x, y in zip(mb.merge_partials(pe, 60, top_n, 0.5), mb.merge_partials(ps, 60, top_n, 0.5)):
            np.testing.assert_array_equal(x, y)
    # threshold 0: nothing may be left out
    pe = b.run_partial([0, 2], 60, 100, 0.0, mode=mb.MODE_EXACT)
    ps = b.run_partial([0, 2], 60, 100, 0.0, mode=mb.MODE_SCREEN)
    np.testing.assert_array_equal(np.sort(pe, order=["group_key"]), np.sort(ps, order=["group_key"]))


def test_fused_run_with_more_exact_candidates_than_the_launch_bound(ctx):
    """top_n above the store size: the cut-off never rises, every series reaches the exact kernel, and the
    list is longer than the fixed launch bound of the fused path (the overflow branch of run_select)."""
    N, S, seed = 1440, 50_000, 7
    store = mb.DeviceStore(ctx, N, 2, S)
    store.append_synthetic(S, seed, 0)
    ref = mb.synth_reference(seed, N)
    b = mb.DeviceBatch(ctx, store, ref)
    for max_lag, top_n, thr in ((N, 60_000, 0.0), (60, 45_000, 0.0)):
        e = b.run([], max_lag, top_n, thr, mode=mb.MODE_EXACT)
        s = b.run([], max_lag, top_n, thr, mode=mb.MODE_SCREEN)
        t = b.timing()
        assert t.mode == mb.MODE_SCREEN
        for x, y in zip(e, s):
            np.testing.assert_array_equal(x, y)
    assert len(e[0]) > 0


def test_screening_prunes_on_siggen_data(ctx):
    # on the benchmark's own data only a few percent may reach the exact kernel
    N, S, seed = 1440, 200_000, 20261018
    store = mb.DeviceStore(ctx, N, 2, S)
    store.append_synthetic(S, seed, 0)
    ref = mb.synth_reference(seed, N)
    b = mb.DeviceBatch(ctx, store, ref)
    e = b.run([], 60, 100, 0.5, mode=mb.MODE_EXACT)
    s = b.run([], 60, 100, 0.5, mode=mb.MODE_AUTO)
    t = b.timing()
    assert t.mode == mb.MODE_SCREEN
    for x, y in zip(e, s):
        np.testing.assert_array_equal(x, y)
    assert 100 <= t.n_rescored <= 0.01 * S        # the fused fp32 second stage leaves a few hundred
    assert t.n_refined <= 0.2 * S


def test_randomised_differential_screen_vs_exact(ctx):
    """Random shapes, windows, thresholds, groupings and pathological rows (NaN, Inf, constants, huge offsets,
    duplicates): the screened run must return exactly what the all-exact run returns, every time."""
    rng = np.random.default_rng(20261018)
    lengths = [258, 300, 480, 512, 700, 1000, 1024, 1026, 1440, 1600, 2048, 2050, 3000, 4096, 5000, 8192, 8200, 10080]
    for trial in range(36):
        N = int(lengths[trial % len(lengths)])
        S = int(rng.integers(200, 3000 if N <= 2048 else 700))
        Y = _adversarial(rng, S, N)
        # extra pathologies
        for _ in range(int(rng.integers(0, 6))):
            i = int(rng.integers(0, S))
            kind = int(rng.integers(0, 5))
            if kind == 0:
                Y[i, int(rng.integers(0, N))] = np.nan
            elif kind == 1:
                Y[i, int(rng.integers(0, N))] = np.inf
            elif kind == 2:
                Y[i] = Y[int(rng.integers(0, S))]             # exact duplicate: ties
            elif kind == 3:
                Y[i] = -Y[int(rng.integers(0, S))]            # mirrored: negative peak, same |score|
            else:
                Y[i] = 1e300 * rng.standard_normal(N)         # overflows fp32 and the fp64 variance
        ref = np.zeros(N)
        w = int(rng.integers(3, 40))
        c = int(rng.integers(N // 4, 3 * N // 4))
        ref[c:c + w] = rng.uniform(0.5, 3.0)
        ref += rng.uniform(0.0, 0.3) * (rng.random(N) - 0.5)
        nk = 3
        ids = np.stack([rng.integers(0, max(2, S // int(rng.integers(2, 60))), S),
                        rng.integers(0, 5, S), rng.integers(-1, 3, S)], axis=1).astype(np.int32)
        store = mb.DeviceStore(ctx, N, nk, S)
        store.append(Y, ids)
        b = mb.DeviceBatch(ctx, store, ref)
        for _ in range(3):
            max_lag = int(rng.choice([0, 1, 15, 60, 240, N // 2, N, 5 * N]))
            top_n = int(rng.choice([1, 4, 20, 100, S // 2 + 1, 2 * S]))
            thr = float(rng.choice([0.0, 0.2, 0.5, 0.9, 0.999]))
            sf = int(rng.choice([mb.SignFilter_ANY, mb.SignFilter_POS]))
            cols = [[], [], [0], [1], [0, 2], [2, 1, 0]][int(rng.integers(0, 6))]
            e = b.run(cols, max_lag, top_n, thr, sf, mode=mb.MODE_EXACT)
            s = b.run(cols, max_lag, top_n, thr, sf, mode=mb.MODE_SCREEN)
            assert b.timing().mode == mb.MODE_SCREEN
            for x, y in zip(e, s):
                np.testing.assert_array_equal(x, y, err_msg="N=%d S=%d lag=%d top=%d thr=%g cols=%s" % (N, S, max_lag, top_n, thr, cols))
            if not cols:
                pe = b.run_partial([], max_lag, top_n, thr, sf, mode=mb.MODE_EXACT)
                np.testing.assert_array_equal(pe["score"], e[0])
        b.close()
        store.close()


def test_scratch_pool_survives_batch_churn(ctx):
    """Batches created and destroyed in every order on one context share pooled scratch; results must not change
    when a batch inherits a smaller or larger set than its store needs."""
    rng = np.random.default_rng(5)
    stores, refs, want = [], [], []
    for S, N in ((500, 480), (20000, 1440), (3000, 1440), (40000, 480)):
        Y = _adversarial(rng, S, N)
        ref = np.zeros(N)
        ref[N // 2 - 5:N // 2 + 5] = 1.5
        ref += 0.1 * (rng.random(N) - 0.5)
        st = mb.DeviceStore(ctx, N, 1, S)
        st.append(Y, (np.arange(S) % 17).astype(np.int32)[:, None])
        stores.append(st)
        refs.append(ref)
        b = mb.DeviceBatch(ctx, st, ref)
        want.append((b.run([], 60, 50, 0.3), b.run([0], 60, 50, 0.3)))
        b.close()
    order = [3, 0, 1, 2, 0, 3, 2, 1, 1, 0]
    alive = []
    for k in order:
        b = mb.DeviceBatch(ctx, stores[k], refs[k])
        alive.append(b)
        for got, exp in zip((b.run([], 60, 50, 0.3), b.run([0], 60, 50, 0.3)), want[k]):
            for x, y in zip(got, exp):
                np.testing.assert_array_equal(x, y)
        if len(alive) > 2:
            alive.pop(0).close()
    for b in alive:
        b.close()


@pytest.mark.parametrize("N", [1440, 1030, 2048])
def test_one_pass_multi_query_run_equals_exact_runs(ctx, N):
    # muse_multi_run at FFT length 2048: the tensor-core path bounds ALL queries of a launch group (up to 256) in one bf16
    # contraction and refines them in one pass over the slab, then finishes their tails with one launch per stage.
    # Every query must return exactly what its own all-exact Batch.Run returns; a constant reference fails for itself only.
    rng = np.random.default_rng(N + 7)
    S, Q = 30000, 21
    Y = _adversarial(rng, S, N)
    refs = np.zeros((Q, N))
    for q in range(Q):
        m, w = int(rng.integers(N // 4, 3 * N // 4)), int(rng.integers(3, 21))
        refs[q, m:m + w] = 1.5
        refs[q] += 0.1 * (rng.random(N) - 0.5)
    refs[5] = -2.5                                         # sigma = 0 (muse_batch.go:38-41)
    refs[9] = np.sin(2 * np.pi * np.arange(N) / 37.0)      # matches the sinusoid rows at some lag
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    for max_lag, top_n, thr in ((60, 100, 0.5), (N, 40, 0.0), (5, 7000, 0.2)):
        got = mb.multi_run(store, refs, [], max_lag, top_n, thr, mode=mb.MODE_SCREEN)
        assert got[5] is None
        for q in range(Q):
            if q == 5:
                continue
            b = mb.DeviceBatch(ctx, store, refs[q])
            want = b.run([], max_lag, top_n, thr, mode=mb.MODE_EXACT)
            b.close()
            for g, w_ in zip(got[q], want):
                np.testing.assert_array_equal(g, w_)       # bit-identical scores, lags and indices
    # and the oracle agrees
    wsc, wlg, wix = co.batch_run(refs[0], Y, None, 60, 100, 0.5)
    sc, lg, ix = mb.multi_run(store, refs[:2], [], 60, 100, 0.5, mode=mb.MODE_SCREEN)[0]
    assert np.max(np.abs(sc - wsc), initial=0) <= 1e-9
    np.testing.assert_array_equal(lg, wlg)
    np.testing.assert_array_equal(ix, wix)


def test_multi_query_randomised_against_separate_runs(ctx):
    # random shapes around the tensor-core path's edges: query counts 2 .. 35 (one launch group each), store sizes that
    # do not divide by the warps of a block, top_n from 1 to a quarter of the store, thresholds from 0 to beyond every
    # score, windows from 0 to all lags.  Reference: the same queries as separate screened batches
    # (themselves pinned to the all-exact run by the tests above).
    rng = np.random.default_rng(2026)
    for case in range(8):
        N = int(rng.choice([1026, 1200, 1440, 1800, 2046, 2048]))
        S = int(rng.integers(16384, 23000))
        Q = int(rng.choice([2, 15, 16, 17, 18, 32, 33, 35]))
        Y = _adversarial(rng, S, N)
        refs = np.zeros((Q, N))
        for q in range(Q):
            kind = q % 4
            if kind == 0:
                m, w = int(rng.integers(10, N - 30)), int(rng.integers(2, 25))
                refs[q, m:m + w] = rng.uniform(0.5, 5)
            elif kind == 1:
                refs[q] = np.sin(2 * np.pi * np.arange(N) / rng.uniform(5, 200))
            elif kind == 2:
                refs[q] = Y[int(rng.integers(0, S))] if rng.random() < 0.5 else rng.standard_normal(N)
            else:
                refs[q] = 0.01 * np.arange(N) * rng.uniform(-1, 1)
            refs[q] += 0.05 * (rng.random(N) - 0.5)
        if Q > 4:
            refs[3] = 1.25                                     # constant: this query alone fails
        max_lag = int(rng.choice([0, 7, 60, N // 2, N]))
        top_n = int(rng.choice([1, 10, 100, S // 4]))
        thr = float(rng.choice([0.0, 0.2, 0.5, 0.9, 1.5]))
        store = mb.DeviceStore(ctx, N, 0, S)
        store.append(Y)
        got = mb.multi_run(store, refs, [], max_lag, top_n, thr, mode=mb.MODE_SCREEN)
        for q in range(Q):
            try:
                b = mb.DeviceBatch(ctx, store, refs[q])
            except mb.MuseError as e:
                assert e.code == mb.MUSE_ERR_STDDEV_ZERO and got[q] is None
                continue
            want = b.run([], max_lag, top_n, thr, mode=mb.MODE_SCREEN)
            b.close()
            assert got[q] is not None
            for g, w_ in zip(got[q], want):
                np.testing.assert_array_equal(g, w_, err_msg="case %d query %d N %d S %d Q %d" % (case, q, N, S, Q))
        store.close()
