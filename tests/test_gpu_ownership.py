"""Every device and page-locked buffer of the library has one owner that frees it: after a scenario has closed every handle it
made, including its own context, muse_held_bytes is back to exactly where it started.  That holds on the error paths that free
half-built state too.  GPU tests need a B200; the argument check at the end runs without one."""
import contextlib
import ctypes as C
import gc

import numpy as np
import pytest

import muse_b200 as mb

gpu = pytest.mark.gpu
SEED = 20261018


def _held():
    dev, pinned = C.c_int64(-1), C.c_int64(-1)
    mb._check(mb.lib().muse_held_bytes(C.byref(dev), C.byref(pinned)))
    return dev.value, pinned.value


class _Scope:
    """A context of its own and the handles made on it, closed newest first and the context last."""

    def __init__(self):
        self.ctx = mb.Context(0)
        self.handles = []

    def add(self, h):
        self.handles.append(h)
        return h

    def close(self):
        for h in reversed(self.handles):
            h.close()
        self.ctx.close()


@contextlib.contextmanager
def _owned():
    gc.collect()      # handles of earlier tests that only a collection frees must not be freed during the scenario
    start = _held()
    s = _Scope()
    try:
        yield s
    finally:
        s.close()
    assert _held() == start


def _refs(Q, N, constant=()):
    rng = np.random.default_rng(3)
    R = 0.1 * (rng.random((Q, N)) - 0.5)
    for q in range(Q):
        m = int(rng.integers(N // 4, 3 * N // 4))
        R[q, m:m + 10] += 1.5
    for q in constant:
        R[q] = 7.0
    return R


def _synthetic(s, N, S, keys=2):
    st = s.add(mb.DeviceStore(s.ctx, N, keys, S))
    st.append_synthetic(S, SEED, 0)
    return st


@gpu
def test_store_create_append_roll_clear_destroy():
    N = 1440
    rng = np.random.default_rng(1)
    with _owned() as s:
        st = s.add(mb.DeviceStore(s.ctx, N, 2, 16))
        st.append(rng.random((1000, N)), rng.integers(0, 9, size=(1000, 2)).astype(np.int32))   # grows past the hint
        st.append_synthetic(3000, SEED, 1000)
        assert _held()[0] > 0 and _held()[1] > 0      # the slab, and the pinned staging ring of the pageable append
        st.roll(rng.random((4000, 7)))
        st.roll(rng.random((100, 300)), first=50)     # a larger roll buffer
        st.clear()
        st.append(rng.random((10, N)), np.zeros((10, 2), dtype=np.int32))
        assert st.size() == 10


@gpu
@pytest.mark.parametrize("N", [1440, 10080, 20000])      # FFT lengths 2048, 16384 and 32768 (the long path)
def test_batch_lifecycle(N):
    S = 4096 if N < 20000 else 64
    with _owned() as s:
        st = _synthetic(s, N, S)
        b = s.add(mb.DeviceBatch(s.ctx, st, mb.synth_reference(SEED, N)))
        for mode in (mb.MODE_EXACT, mb.MODE_SCREEN):
            b.run([], 60, 20, 0.3, mode=mode)
            b.run([0], 60, 20, 0.3, mode=mode)
            b.run([], 60, 20, 0.0, mode=mode, signed_scores=True)
        b.score_all()
        if N < 20000:
            b.screen_bounds(refine=True, max_lag=60)
        cc, zero = b.xcorr(5)
        assert not zero and cc.size == b.fft_len()
        # a second batch on the same context takes the scratch the first one gave back
        b.close()
        b2 = s.add(mb.DeviceBatch(s.ctx, st, mb.synth_row(SEED, 7, N)))
        b2.run([], 60, 20, 0.3)


@gpu
def test_multi_run_on_tensor_cores_with_a_constant_reference():
    N, S = 1440, 16384
    with _owned() as s:
        st = _synthetic(s, N, S, keys=0)
        got = mb.multi_run(st, _refs(3, N, constant=(1,)), [], 60, 20, 0.3)
        assert got[1] is None and got[0] is not None and got[2] is not None
        assert mb.multi_last_timing(s.ctx)[0] > 0     # the tensor-core path ran (its stage events exist only there)


@gpu
def test_multi_run_as_separate_batches_with_a_constant_reference():
    N, S = 1440, 4096
    with _owned() as s:
        st = _synthetic(s, N, S)
        got = mb.multi_run(st, _refs(3, N, constant=(2,)), [0], 60, 20, 0.3)
        assert got[2] is None and got[0] is not None and got[1] is not None
        assert mb.multi_last_timing(s.ctx) == (0.0, 0.0, 0.0, 0.0)


@gpu
def test_bounds_xcorr_and_one_rank_exchange():
    N, S, top_n = 1440, 4096, 20
    rng = np.random.default_rng(2)
    with _owned() as s:
        st = _synthetic(s, N, S, keys=0)
        assert mb.multi_bounds_tc(st, _refs(2, N)).shape == (2, S)
        for n in (64, 5000, 8192):      # direct sum, folded FFT, FFT of length n
            cc, _, _ = mb.xCorr(rng.random(n), rng.random(n // 2), n, True, ctx=s.ctx)
            assert cc.size == n
        ex = s.add(mb.Exchange(s.ctx, 256 * top_n))
        b = s.add(mb.DeviceBatch(s.ctx, st, mb.synth_reference(SEED, N)))
        ex.run(b, 60, top_n, 0.3)
        assert len(ex.run_many(st, _refs(3, N), 60, top_n, 0.3)) == 3


@gpu
def test_error_paths_free_what_they_built():
    N, S = 1440, 4096
    with _owned() as s:
        st = _synthetic(s, N, S)
        with pytest.raises(mb.MuseError) as e:
            mb.DeviceBatch(s.ctx, st, np.full(N, 7.0))
        assert e.value.code == mb.MUSE_ERR_STDDEV_ZERO
        with pytest.raises(mb.MuseError) as e:
            mb.DeviceBatch(s.ctx, st, np.ones(N + 1))
        assert e.value.code == mb.MUSE_ERR_LENGTH_MISMATCH
        with pytest.raises(mb.MuseError) as e:
            mb.multi_run(st, _refs(2, N + 1), [], 60, 20, 0.3)
        assert e.value.code == mb.MUSE_ERR_LENGTH_MISMATCH
        with pytest.raises(mb.MuseError) as e:
            mb.DeviceStore(s.ctx, N, 2, 10 ** 11)      # ~1 PB of slab
        assert e.value.code == mb.MUSE_ERR_OUT_OF_MEMORY
        with pytest.raises(mb.MuseError) as e:
            mb.Exchange(s.ctx, 1 << 40)
        assert e.value.code == mb.MUSE_ERR_OUT_OF_MEMORY
        b = s.add(mb.DeviceBatch(s.ctx, st, mb.synth_reference(SEED, N)))      # the context still works
        b.run([], 60, 20, 0.3)


def test_held_bytes_rejects_null_arguments():
    mb.build()
    x = C.c_int64(0)
    assert mb.lib().muse_held_bytes(None, C.byref(x)) == mb.MUSE_ERR_INVALID_ARG
    assert mb.lib().muse_held_bytes(C.byref(x), None) == mb.MUSE_ERR_INVALID_ARG
    assert mb.lib().muse_held_bytes(None, None) == mb.MUSE_ERR_INVALID_ARG
