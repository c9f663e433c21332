"""The hand-out of series to the warps of the n = 2048 screening kernel (score_screen_warp_kernel, claims of
consecutive series from a device counter): every series is visited exactly once whatever the store size, and neither
the size nor the layout of the store changes a result.  Needs a B200."""
import numpy as np
import pytest

import muse_b200 as mb

pytestmark = pytest.mark.gpu

SEED, N = 20261018, 1440      # N = 1440: n = 2048, the warp kernel


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _store(ctx, S, layout, n_keys=0):
    """The benchmark's rows (rect, line, noise by index mod 3; only rect rows reach the second stage).  layout "period3"
    keeps that order; "contiguous" puts all rect rows first, then the lines, then the noise."""
    store = mb.DeviceStore(ctx, N, n_keys, S)
    store.append_synthetic(S, SEED, 0)
    if layout == "period3":
        return store
    Y = store.read_rows(0, S)
    store.close()
    store = mb.DeviceStore(ctx, N, n_keys, S)
    for kind in range(3):
        if Y[kind::3].shape[0]:
            store.append(Y[kind::3])
    return store


@pytest.mark.parametrize("layout", ["period3", "contiguous"])
@pytest.mark.parametrize("S", [1, 100, 1775, 1776, 1777, 200_003])
def test_screened_run_equals_exact_run_at_every_store_size(ctx, S, layout):
    """Sizes around the 1776 warps of a 148-SM grid (12 per SM) and far above them; expensive rows at a period of 3
    (what a fixed stride of 1776 series aliases with) and in one block."""
    store = _store(ctx, S, layout)
    b = mb.DeviceBatch(ctx, store, mb.synth_reference(SEED, N))
    for max_lag, top_n, thr in ((60, 100, 0.5), (60, 1000, 0.0), (N, 20, 0.9)):
        e = b.run([], max_lag, top_n, thr, mode=mb.MODE_EXACT)
        s = b.run([], max_lag, top_n, thr, mode=mb.MODE_SCREEN)
        assert b.timing().mode == mb.MODE_SCREEN
        for x, y in zip(e, s):
            np.testing.assert_array_equal(x, y)      # bit-identical scores, lags and indices
    b.close()
    store.close()


@pytest.mark.parametrize("S", [3, 1001, 1777, 60_001])
def test_every_series_is_visited_exactly_once(S):
    """Refined bounds of every series (cut-off 0: every series takes the second stage) on two stores of the same size,
    one after the other in a context of their own: the second batch inherits the first one's bound arrays from the
    context's scratch pool.  The first store holds copies of the reference (lower bounds ~0.9999), the second the
    benchmark's rows (every score below 0.999), so a series the kernel skipped keeps a lower bound above its score.
    Sizes below the warps of the grid, and odd ones (not a whole number of two-series claims).  A grouped run with
    threshold 0 refines every series once: its refined count is the store size."""
    ctx = mb.Context(0)
    ref = mb.synth_reference(SEED, N)
    first = mb.DeviceStore(ctx, N, 0, S)
    first.append(np.tile(ref, (S, 1)))
    b = mb.DeviceBatch(ctx, first, ref)
    up, lo = b.screen_bounds(refine=True, max_lag=60)
    assert np.all(lo >= 0.999) and np.all(up >= 1.0)
    b.close()
    first.close()

    store = _store(ctx, S, "period3")
    b = mb.DeviceBatch(ctx, store, ref)
    up, lo = b.screen_bounds(refine=True, max_lag=60)
    up, lo = up.astype(np.float64), lo.astype(np.float64)
    sc, lg = b.score_all()
    assert sc.max() < 0.999
    inside = np.abs(lg) <= 60
    out = up == -1.0
    assert not np.any(out & inside)
    assert np.all(up[~out] >= sc[~out])
    assert np.all(inside[lo >= 0]) and np.all(lo[lo >= 0] <= sc[lo >= 0])
    b.close()
    store.close()

    store = _store(ctx, S, "period3", n_keys=1)
    store.set_synthetic_labels([7], [1000])
    b = mb.DeviceBatch(ctx, store, ref)
    e = b.run([0], 60, 100, 0.0, mode=mb.MODE_EXACT)
    s = b.run([0], 60, 100, 0.0, mode=mb.MODE_SCREEN)
    t = b.timing()
    assert t.mode == mb.MODE_SCREEN and t.n_refined == S
    for x, y in zip(e, s):
        np.testing.assert_array_equal(x, y)
    b.close()
    store.close()
    ctx.close()
