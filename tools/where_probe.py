"""Where probe: what a filtered run (muse_batch_run_where) costs against a run on a store that holds only the selected rows.

On the C3 store (1 M x 1440 synthetic rows) and on an n = 512 store (3 M x 480), with synthetic labels chosen so that one
equality selects 50 %, 10 % and 1 % of the rows, in two layouts -- scattered rows (i % 2 == 1, i % 10 == 3, i % 100 == 3) and
contiguous blocks of 10 000 rows (i / 10000 % 2 == 1, % 10 == 7, % 100 == 7) -- it reports for every selection:
  * muse_batch_run_where on the whole store;
  * muse_batch_run_ex on a fresh store that holds only the selected rows (and whether the results are identical);
  * what building that fresh store costs: muse_group_clear + muse_group_append from page-locked host rows;
and the run of the whole store.  Runs: ungrouped, AUTO, maxLag 60, top 100, threshold 0.5.  Times are medians
of --reps host-clock measurements from call to return (every call is complete when it returns) after warm-up, with a 512 MB
write between measurements so that no run finds its rows in L2 (126 MB).  The card's name and power limit are read in the
same call.

usage: python tools/where_probe.py [--reps R] [--out profiles/r03_where.json]"""
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

SEED, TOP_N, THRESHOLD = 20261018, 100, 0.5
# per layout, three label columns (muse_group_set_synthetic_labels: id = (i / div) % mod) and the id each selects
LAYOUTS = {"scattered": (1, [("50%", 2, 1), ("10%", 10, 3), ("1%", 100, 3)]),
           "contiguous": (10000, [("50%", 2, 1), ("10%", 10, 7), ("1%", 100, 7)])}


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


def wall_ms(fn, warm, reps):
    for _ in range(warm):
        fn()
    out = []
    for _ in range(reps):
        flush_l2()
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out))


def pinned(n_doubles):
    p = C.c_void_p()
    mb._check(mb.lib().muse_host_alloc(C.byref(p), max(1, n_doubles) * 8))
    return p, np.ctypeslib.as_array((C.c_double * max(1, n_doubles)).from_address(p.value))


def probe(ctx, S, N, max_lag, reps):
    res = {"series": S, "length": N, "max_lag": max_lag, "top_n": TOP_N, "threshold": THRESHOLD, "selections": []}
    store = mb.DeviceStore(ctx, N, 3, S)
    store.append_synthetic(S, SEED, 0)
    ref = mb.synth_reference(SEED, N)
    b = mb.DeviceBatch(ctx, store, ref)
    full = lambda: b.run([], max_lag, TOP_N, THRESHOLD)
    res["full_ms"] = wall_ms(full, 2, reps)
    full()
    res["full_mode"] = b.timing().mode
    i = np.arange(S)
    m_max = max(int(np.count_nonzero((i // d) % m == v)) for d, sels in LAYOUTS.values() for _, m, v in sels)
    hp, H = pinned(m_max * N)
    fresh = mb.DeviceStore(ctx, N, 0, m_max)
    chunk = 1 << 16
    for layout, share, d, col, mod, v in [(lay, sh, d, c, mo, v) for lay, (d, sels) in LAYOUTS.items()
                                          for c, (sh, mo, v) in enumerate(sels)]:
        if col == 0:
            store.set_synthetic_labels([d] * 3, [mo for _, mo, _ in LAYOUTS[layout][1]])
        sel = np.flatnonzero((i // d) % mod == v)
        m = len(sel)
        # the selected rows, page-locked, in store order
        Hm = H[:m * N].reshape(m, N)
        k = 0
        for first in range(0, S, chunk):
            n = min(chunk, S - first)
            part = sel[(sel >= first) & (sel < first + n)] - first
            if len(part):
                Hm[k:k + len(part)] = store.read_rows(first, n)[part]
                k += len(part)
        build = lambda: (fresh.clear(), fresh.append_host_ptr(hp.value, m, N))
        build_ms = wall_ms(build, 1, max(3, reps // 3))
        bf = mb.DeviceBatch(ctx, fresh, ref)
        where = lambda: b.run_where([col], [v], [], max_lag, TOP_N, THRESHOLD)
        run_fresh = lambda: bf.run([], max_lag, TOP_N, THRESHOLD)
        where_ms = wall_ms(where, 2, reps)
        got = where()
        t_where = b.timing()
        fresh_ms = wall_ms(run_fresh, 2, reps)
        want = run_fresh()
        t_fresh = bf.timing()
        identical = (np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
                     and np.array_equal(got[2], sel[want[2]]) and t_where.mode == t_fresh.mode)
        rec = {"layout": layout, "share": share, "rows": m, "where_ms": where_ms, "fresh_run_ms": fresh_ms,
               "fresh_build_ms": build_ms, "where_minus_fresh_ms": where_ms - fresh_ms,
               "where_device_total_ms": t_where.total_ms, "fresh_device_total_ms": t_fresh.total_ms,
               "where_score_ms": t_where.score_ms, "fresh_score_ms": t_fresh.score_ms,
               "mode": t_where.mode, "identical_to_fresh": bool(identical)}
        print(json.dumps(rec), flush=True)
        res["selections"].append(rec)
        bf.close()
    fresh.close()
    mb.lib().muse_host_free(hp)
    b.close()
    store.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--c3-series", type=int, default=1_000_000)
    ap.add_argument("--n512-series", type=int, default=3_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = mb.Context(0)
    ctx.set_stream(stream.cuda_stream)
    out = {"gpu": card(), "c3": probe(ctx, args.c3_series, 1440, 60, args.reps),
           "n512": probe(ctx, args.n512_series, 480, 60, args.reps)}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
