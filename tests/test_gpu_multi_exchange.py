"""Many references against a sharded store: Exchange.run_many (muse_multi_run_exchange) and the device-side per-query merge
(muse_merge_partials_many) give exactly what muse_multi_run gives on one store holding every shard.  Needs a B200."""
import os
import subprocess
import sys

import numpy as np
import pytest

import muse_b200 as mb

pytestmark = pytest.mark.gpu

SEED = 20261018


@pytest.fixture(scope="module")
def ctx():
    return mb.default_context(0)


def _refs(Q, N, seed=3, constant=()):
    # rect mids / widths varied, as the many-reference benchmark shape
    rng = np.random.default_rng(seed)
    refs = np.zeros((Q, N))
    for q in range(Q):
        mid, w = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8)), int(rng.integers(3, 21))
        refs[q, mid - w // 2: mid - w // 2 + w] = 1.5
        refs[q] += 0.1 * (rng.random(N) - 0.5)
    for q in constant:
        refs[q] = 7.0
    return refs


def _assert_same(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if w is None:
            continue
        for a, b in zip(g, w):
            np.testing.assert_array_equal(a, b)


def _synthetic_store(ctx, S, N, first=0, variant=0):
    st = mb.DeviceStore(ctx, N, 0, max(S, 1))
    if S:
        st.append_synthetic(S, SEED, first, variant)
    st.set_global_offset(first)
    return st


def test_run_many_one_rank_tensor_core_shape(ctx):
    # N = 1440 (FFT length 2048), 20 000 series, 259 references: the tensor-core multi-query path, two exchange steps (256 + 3)
    S, N, Q, top_n = 20000, 1440, 259, 50
    store = _synthetic_store(ctx, S, N)
    refs = _refs(Q, N, constant=(7,))
    ex = mb.Exchange(ctx, 256 * top_n)
    want = mb.multi_run(store, refs, [], 60, top_n, 0.5)
    assert want[7] is None and sum(w is not None and len(w[0]) > 0 for w in want) > 200
    _assert_same(ex.run_many(store, refs, 60, top_n, 0.5), want)
    ex.close()
    store.close()


def test_run_many_one_rank_separate_batches_and_sign_filter(ctx):
    # N = 480: no one-pass kernel, the queries are separate batches on the store; then SIGN_NEG on the n = 2048 shape
    rng = np.random.default_rng(5)
    S, N, Q = 3000, 480, 5
    Y = 0.1 * (rng.random((S, N)) - 0.5)
    for i in range(0, S, 3):
        m = int(rng.integers(0, N - 20))
        Y[i, m:m + int(rng.integers(1, 20))] += rng.uniform(0.5, 40)
    store = mb.DeviceStore(ctx, N, 0, S)
    store.append(Y)
    refs = _refs(Q, N, seed=9, constant=(3,))
    ex = mb.Exchange(ctx, 64)
    for max_lag, top_n, thr in ((20, 15, 0.2), (5, 64, 0.0), (200, 1, 0.9)):
        _assert_same(ex.run_many(store, refs, max_lag, top_n, thr), mb.multi_run(store, refs, [], max_lag, top_n, thr))
    big = _synthetic_store(ctx, 20000, 1440)
    refs = _refs(6, 1440, seed=11)
    for sign in (mb.SignFilter_NEG, mb.SignFilter_POS):
        _assert_same(ex.run_many(big, refs, 60, 40, 0.3, sign), mb.multi_run(big, refs, [], 60, 40, 0.3, sign))
    ex.close()
    big.close()
    store.close()


def test_run_many_small_capacity_takes_several_steps(ctx):
    # capacity 3 x top_n: 10 references in 4 steps (3 + 3 + 3 + 1), both parities of the receive buffer twice
    S, N, Q, top_n = 20000, 1440, 10, 30
    store = _synthetic_store(ctx, S, N)
    refs = _refs(Q, N, seed=13, constant=(4,))
    ex = mb.Exchange(ctx, 3 * top_n)
    want = mb.multi_run(store, refs, [], 60, top_n, 0.5)
    for _ in range(2):
        _assert_same(ex.run_many(store, refs, 60, top_n, 0.5), want)
    ex.close()
    store.close()


def test_run_many_empty_store_and_argument_errors(ctx):
    N, top_n = 1440, 20
    empty = _synthetic_store(ctx, 0, N)
    refs = _refs(4, N, seed=17, constant=(2,))
    ex = mb.Exchange(ctx, 2 * top_n)
    got = ex.run_many(empty, refs, 60, top_n, 0.5)
    _assert_same(got, mb.multi_run(empty, refs, [], 60, top_n, 0.5))
    assert got[2] is None and all(len(got[q][0]) == 0 for q in (0, 1, 3))
    # argument errors come before the step begins: the next valid call still pairs with its peers' epochs
    store = _synthetic_store(ctx, 20000, N)
    with pytest.raises(mb.MuseError) as e:
        ex.run_many(store, refs, 60, 2 * top_n + 1, 0.5)
    assert e.value.code == mb.MUSE_ERR_INVALID_ARG
    with pytest.raises(mb.MuseError) as e:
        ex.run_many(store, refs[:, :1000], 60, top_n, 0.5)
    assert e.value.code == mb.MUSE_ERR_LENGTH_MISMATCH
    _assert_same(ex.run_many(store, refs, 60, top_n, 0.5), mb.multi_run(store, refs, [], 60, top_n, 0.5))
    ex.close()
    store.close()
    empty.close()


def _repeated_rows(S, N, period=97):
    # row i = synthetic row i % period: bit-identical rows, hence bit-identical scores, in every shard
    base = np.stack([mb.synth_row(SEED, i, N) for i in range(period)])
    return np.tile(base, (S // period + 1, 1))[:S]


def _rows_store(ctx, Y, lo, hi):
    st = mb.DeviceStore(ctx, Y.shape[1], 0, max(hi - lo, 1))
    if hi > lo:
        st.append(Y[lo:hi])
    st.set_global_offset(lo)
    return st


@pytest.mark.parametrize("data", ["mix", "rect", "repeated"])
def test_merge_partials_many_of_uneven_shards(ctx, data):
    # k = 3 uneven shards plus an empty one, each with its global offset; their multi_run lists stacked [k][Q][top_n] in
    # device memory and merged on the device == multi_run on the whole store == the host merge per query.  "rect"
    # (append_synthetic variant 1: every series a rect of one width) packs the scores closely; "repeated" (one period of 97
    # rows repeated over the store) makes equal scores certain, so the order by global index decides ties across shards.
    import torch
    S, N, Q, top_n, max_lag, thr = 20000, 1440, 24, 60, 60, 0.3
    bounds = [(0, 4100), (4100, 13000), (13000, S), (S, S)]
    if data == "repeated":
        Y = _repeated_rows(S, N)
        whole = _rows_store(ctx, Y, 0, S)
        shards = [_rows_store(ctx, Y, lo, hi) for lo, hi in bounds]
    else:
        variant = 1 if data == "rect" else 0
        whole = _synthetic_store(ctx, S, N, variant=variant)
        shards = [_synthetic_store(ctx, hi - lo, N, lo, variant) for lo, hi in bounds]
    refs = _refs(Q, N, seed=19 + len(data), constant=(5,))
    want = mb.multi_run(whole, refs, [], max_lag, top_n, thr)
    raws = [mb.multi_run(st, refs, [], max_lag, top_n, thr, raw=True) for st in shards]
    recs = np.stack([mb.multi_records(*r) for r in raws])                       # [k][Q][top_n]
    d = torch.from_numpy(recs.view(np.uint8).reshape(-1).copy()).cuda()
    torch.cuda.synchronize()
    sc, lg, ix, n = mb.merge_partials_many(ctx, d.data_ptr(), len(shards), Q, top_n)
    n = np.where(raws[0][3] < 0, -1, n)
    got = [None if n[q] < 0 else (sc[q, :n[q]], lg[q, :n[q]], ix[q, :n[q]]) for q in range(Q)]
    _assert_same(got, want)
    if data == "repeated":     # equal scores of series in different shards really are merged
        shard_of = lambda i: np.searchsorted([hi for _, hi in bounds], i, side="right")
        assert any(w is not None and np.any((np.diff(w[0]) == 0) & (np.diff(shard_of(w[2])) != 0)) for w in want)
    for q in range(Q):
        if want[q] is None:
            continue
        host = mb.merge_partials(recs[:, q, :].reshape(-1), max_lag, top_n, thr)
        for a, b in zip(host, want[q]):
            np.testing.assert_array_equal(a, b)
    for st in shards:
        st.close()
    whole.close()


def test_run_many_two_gpus():
    # two ranks, one per GPU (skipped on a one-GPU box): tools/multi_exchange_check.py compares Exchange.run_many with the
    # NCCL all-gather + device merge path and with multi_run on a store holding every shard, for several argument sets
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.join(root, "tools", "multi_exchange_check.py")],
                       env=dict(os.environ, CHECK_SERIES="60000"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ALL IDENTICAL" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
