"""Multi-where probe: what muse_multi_run_where costs against the two ways of getting the same results without it.

The store and references are C5's (bench.py --workload c5): 1 M x 1440 synthetic rows and 256 references, with synthetic label columns
i % 100, i % 10 and i % 2 (muse_group_set_synthetic_labels), so that one equality selects 1 %, 10 % and 50 % of the store as
interleaved (scattered) rows; no equality selects 100 %.  For each selection, alternated in one process:
  (a) muse_multi_run_where on the whole store;
  (b) muse_multi_run on a fresh store of the selected rows (100 %: the store itself); the fresh store is built once, by reading
      the rows back in chunks, gathering the selected ones on the device and muse_group_append_device, and that build is
      timed on its own;
  (c) a loop of 256 muse_batch_run_where, one batch per reference (batches created before the timing);
and whether (a) returns exactly what (b) returns.  Runs: ungrouped, AUTO, maxLag 60, top 100, threshold 0.5.  Times are
medians of --reps host-clock measurements from call to return (every call is complete when it returns) after warm-up, with
a 512 MB write before each measurement so that no run finds its rows in L2 (126 MB).  The card's name and power limit are
read in the same call.

usage: python tools/multi_where_probe.py [--reps R] [--out profiles/r03_multi_where.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "go-muse_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import muse_b200 as mb  # noqa: E402

SEED, N, MAX_LAG, TOP_N, THRESHOLD = 20261018, 1440, 60, 100, 0.5
SELECTIONS = [("1%", [0], [7]), ("10%", [1], [3]), ("50%", [2], [1]), ("100%", [], [])]
MODS = [100, 10, 2]


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, _, limit = q.stdout.strip().partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": limit.strip() or None}


_flush = None


def flush_l2():
    global _flush
    if _flush is None:
        _flush = torch.empty(64 << 20, dtype=torch.float64, device="cuda")
    _flush.fill_(1.0)
    torch.cuda.synchronize()


def timed(fn):
    flush_l2()
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def pinned(n_doubles):
    p = C.c_void_p()
    mb._check(mb.lib().muse_host_alloc(C.byref(p), max(1, n_doubles) * 8))
    return p, np.ctypeslib.as_array((C.c_double * max(1, n_doubles)).from_address(p.value))


def build_fresh(ctx, store, sel, S, chunk=1 << 16):
    """a store of the rows `sel` of `store`, in order: rows read back in chunks, the selected ones gathered on the device"""
    fresh = mb.DeviceStore(ctx, N, 0, max(1, len(sel)))
    hp, H = pinned(chunk * N)
    d_idx = torch.from_numpy(sel).cuda()
    for first in range(0, S, chunk):
        n = min(chunk, S - first)
        lo, hi = np.searchsorted(sel, [first, first + n])
        if hi == lo:
            continue
        store.read_rows(first, n, H[:n * N].reshape(n, N))
        rows = torch.from_numpy(H[:n * N].reshape(n, N)).cuda(non_blocking=False)
        part = rows.index_select(0, d_idx[lo:hi] - first).contiguous()
        torch.cuda.synchronize()
        fresh.append_device(part.data_ptr(), hi - lo, N)
    mb.lib().muse_host_free(hp)
    return fresh


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--series", type=int, default=1_000_000)
    ap.add_argument("--queries", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    S, Q = args.series, args.queries
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = mb.Context(0)
    ctx.set_stream(stream.cuda_stream)
    store = mb.DeviceStore(ctx, N, len(MODS), S)
    store.append_synthetic(S, SEED, 0)
    store.set_synthetic_labels([1] * len(MODS), MODS)
    ids = np.stack([np.arange(S) % m for m in MODS], axis=1)
    rng = np.random.default_rng(3)                       # bench.py --workload c5's references
    refs = np.zeros((Q, N))
    for q in range(Q):
        mid, w = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8)), int(rng.integers(3, 21))
        refs[q, mid - w // 2: mid - w // 2 + w] = 1.5
        refs[q] += 0.1 * (rng.random(N) - 0.5)
    batches = [mb.DeviceBatch(ctx, store, refs[q]) for q in range(Q)]
    res = {"gpu": card(), "series": S, "length": N, "queries": Q, "max_lag": MAX_LAG, "top_n": TOP_N, "threshold": THRESHOLD,
           "reps": args.reps, "selections": []}
    for share, cols, vals in SELECTIONS:
        sel = np.flatnonzero(np.all(ids[:, cols] == np.asarray(vals), axis=1)) if cols else np.arange(S)
        t0 = time.perf_counter()
        fresh = build_fresh(ctx, store, sel, S) if cols else store
        build_ms = (time.perf_counter() - t0) * 1e3
        a = lambda: mb.multi_run_where(store, refs, cols, vals, [], MAX_LAG, TOP_N, THRESHOLD, raw=True)
        b = lambda: mb.multi_run(fresh, refs, [], MAX_LAG, TOP_N, THRESHOLD, raw=True)
        c = lambda: [bt.run_where(cols, vals, [], MAX_LAG, TOP_N, THRESHOLD) for bt in batches]
        for fn in (a, b, c):
            fn()
        ta, tb, tc = [], [], []
        for _ in range(args.reps):
            ms, got = timed(a)
            ta.append(ms)
            stats, tim = mb.multi_last_stats(ctx), mb.multi_last_timing(ctx)
            ms, want = timed(b)
            tb.append(ms)
            tc.append(timed(c)[0])
        identical = bool(np.array_equal(got[3], want[3]) and all(
            np.array_equal(got[0][q, :k], want[0][q, :k]) and np.array_equal(got[1][q, :k], want[1][q, :k]) and
            np.array_equal(got[2][q, :k], sel[want[2][q, :k]]) for q, k in enumerate(np.maximum(got[3], 0))))
        rec = {"share": share, "rows": int(len(sel)), "multi_where_ms": float(np.median(ta)), "fresh_multi_run_ms": float(np.median(tb)),
               "fresh_build_ms": build_ms, "loop_run_where_ms": float(np.median(tc)),
               "multi_where_spread_ms": [float(min(ta)), float(max(ta))], "fresh_spread_ms": [float(min(tb)), float(max(tb))],
               "tensor_core_path": stats[0] > 0, "refined": stats[0], "rescored": stats[1],
               "last_group_stage_ms": list(tim), "identical_to_fresh": identical}
        print(json.dumps(rec), flush=True)
        res["selections"].append(rec)
        if fresh is not store:
            fresh.close()
    for bt in batches:
        bt.close()
    store.close()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
