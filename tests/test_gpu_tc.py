"""The multi-query bounds on the tensor cores (muse_bounds_tc.cuh): the bf16 contraction must dominate every exact
score and stay close to the fp32 kernel's bound.  Needs a B200."""
import numpy as np
import pytest

import muse_b200 as mb

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _refs(rng, Q, N):
    refs = 0.1 * (rng.random((Q, N)) - 0.5)
    for q in range(Q):
        mid, w = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8)), int(rng.integers(3, 21))
        refs[q, mid - w // 2: mid - w // 2 + w] += 1.5
    return refs


@pytest.mark.parametrize("N,S,Q", [(1440, 1000, 5), (1440, 4096 + 77, 256), (2048, 300, 33), (1030, 515, 1)])
def test_tensor_core_bounds_dominate_and_track_the_fp32_bound(ctx, N, S, Q):
    rng = np.random.default_rng(N + S + Q)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append_synthetic(S, 20261018, 7)
    # a few hostile rows: constant (no fp32 statement possible), huge offset, tiny amplitude
    Y = store.read_rows(0, S)
    refs = _refs(rng, Q, N)
    U = mb.multi_bounds_tc(store, refs).astype(np.float64)
    assert U.shape == (Q, S)
    for q in sorted(set([0, Q // 2, Q - 1])):
        b = mb.DeviceBatch(ctx, store, refs[q])
        sc, _ = b.score_all()
        u32 = b.screen_bounds().astype(np.float64)
        dec = u32 <= 1.5
        assert np.all(U[q] >= sc + 0.5e-4), (q, float((U[q] - sc).min()))
        # the bin-by-bin spectral bound (1/n) sum_f |Y_f||X_f| in fp64 on the host: the contraction computes exactly this sum
        # from two bf16 per value (16 mantissa bits) with the epilogue's 1.0003, so it sits within 5e-4 (relative) above it;
        # the single-query kernel's pair bound (muse_screen.cuh) is the same sum after one more Cauchy-Schwarz step, never below
        n = b.fft_len()
        z = lambda a: (a - a.mean(axis=-1, keepdims=True)) / a.std(axis=-1, ddof=1, keepdims=True)
        X = np.abs(np.fft.rfft(np.concatenate([np.zeros(n - N), z(refs[q][None, :])[0] / (N - 1)])))
        w = np.full(n // 2 + 1, 2.0)
        w[0] = w[-1] = 1.0
        with np.errstate(invalid="ignore", divide="ignore"):
            Yf = np.abs(np.fft.rfft(np.concatenate([np.zeros((S, n - N)), z(Y)], axis=1), axis=1))
        bins = (Yf * (X * w)[None, :]).sum(axis=1) / n
        assert np.all(U[q][dec] <= bins[dec] * 1.0005 + 1.1e-4)
        assert np.all(U[q][dec] >= bins[dec] * 0.9999 + 0.9e-4)
        assert np.all(u32[dec] >= bins[dec] * 0.9999 + 0.9e-4)
        b.close()
    store.close()


def test_multi_run_on_tensor_cores_equals_exact_runs(ctx):
    """muse_multi_run with the bounds on the tensor cores (259 queries = a launch of 256 + one of 3): every query against
    its own all-exact Batch.Run, bit for bit."""
    rng = np.random.default_rng(99)
    N, S, Q = 1440, 20000, 259
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append_synthetic(S, 20261018, 0)
    refs = _refs(rng, Q, N)
    refs[17] = 3.0                      # sigma = 0 (muse_batch.go:38-41): this query alone has no Batch
    got = mb.multi_run(store, refs, [], 60, 100, 0.5, mode=mb.MODE_SCREEN)
    assert got[17] is None
    for q in range(Q):
        if q == 17:
            continue
        b = mb.DeviceBatch(ctx, store, refs[q])
        want = b.run([], 60, 100, 0.5, mode=mb.MODE_EXACT)
        b.close()
        for x, y in zip(got[q], want):
            np.testing.assert_array_equal(x, y)
    store.close()


def test_multi_run_with_a_top_n_beyond_the_device_side_select(ctx):
    """top_n above 32768 candidates: every query of the launch falls back to the host select from the scores on the device."""
    rng = np.random.default_rng(5)
    N, S, Q = 1026, 140000, 3
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append_synthetic(S, 20261018, 0)
    refs = _refs(rng, Q, N)
    got = mb.multi_run(store, refs, [], N, 33000, 0.0, mode=mb.MODE_SCREEN)
    for q in range(Q):
        b = mb.DeviceBatch(ctx, store, refs[q])
        want = b.run([], N, 33000, 0.0, mode=mb.MODE_EXACT)
        b.close()
        assert len(got[q][0]) == 33000
        for x, y in zip(got[q], want):
            np.testing.assert_array_equal(x, y)
    store.close()
