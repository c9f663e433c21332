"""Roll probe: what muse_group_roll costs on the C3 store, against a device copy of the slab and against a full re-upload.

On the C3 store (1 M x 1440 synthetic rows, 11.5 GB, far larger than L2) it reports, in one process:
  * the device-to-device copy bandwidth (cudaMemcpyAsync of the slab's size, CUDA events);
  * the roll kernel alone (muse_group_roll_device) for k = 1, 60 and 1440: median of --reps after warm-up, CUDA events,
    its 2 S N 8 bytes over that time and that rate's share of the copy bandwidth;
  * muse_group_roll from page-locked and from pageable host blocks at k = 1 and 60, host clock from call to return;
  * muse_group_clear + muse_group_append of the same rows from page-locked memory;
  * the C3 Run (maxLag 60, top 100, threshold 0.5, ungrouped) before any roll and after the rolls (the store rolled back to
    its first rows by a k = N roll), with the results compared bit for bit.
Then it rolls a C4-sized store (1.25 M x 10080, 100.8 GB) and reports the device memory in use around the roll.

usage: python tools/roll_probe.py [--series S] [--c4-series S4] [--reps R] [--out FILE.json]"""
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


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, _, limit = q.stdout.strip().partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": limit.strip() or None}


def events_ms(fn, warm, reps):
    """Median device time of fn() between two events on the current stream (the library runs on it)."""
    for _ in range(warm):
        fn()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out))


def wall_ms(fn, warm, reps):
    """Median host time from call to return of fn() (every library call here is complete when it returns)."""
    for _ in range(warm):
        fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out))


def pinned(n_doubles):
    p = C.c_void_p()
    mb._check(mb.lib().muse_host_alloc(C.byref(p), n_doubles * 8))
    return p, np.ctypeslib.as_array((C.c_double * n_doubles).from_address(p.value))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--series", type=int, default=1_000_000)
    ap.add_argument("--c4-series", type=int, default=1_250_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    S, reps = args.series, args.reps
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = mb.Context(0)
    ctx.set_stream(stream.cuda_stream)
    res = {"gpu": card(), "series": S, "length": N}
    rng = np.random.default_rng(SEED)

    store = mb.DeviceStore(ctx, N, 2, S)
    store.append_synthetic(S, SEED, 0)
    slab_bytes = S * ((N + 15) // 16 * 16) * 8
    roll_bytes = 2 * S * N * 8
    src = torch.empty(slab_bytes // 8, dtype=torch.float64, device="cuda").normal_()
    dst = torch.empty_like(src)
    copy_ms = events_ms(lambda: dst.copy_(src), 3, reps)
    copy_bw = 2 * slab_bytes / copy_ms / 1e9          # TB/s (bytes read + written)
    res["copy"] = {"bytes": slab_bytes, "ms": copy_ms, "TB_per_s": copy_bw}
    del src, dst

    # the store's first rows, page-locked: the source of the clear + append comparison and of the roll back
    hp, H = pinned(S * N)
    store.read_rows_ptr(0, S, hp.value)
    H2 = H.reshape(S, N)
    store.roll(H2)          # the same rows, their statistics now from the roll kernel (as after every roll below)
    ref = mb.synth_reference(SEED, N)
    b = mb.DeviceBatch(ctx, store, ref)
    first = b.run([], MAX_LAG, TOP_N, THRESHOLD)
    res["run_before_ms"] = events_ms(lambda: b.run([], MAX_LAG, TOP_N, THRESHOLD), 3, reps)

    res["kernel"] = {}
    for k in (1, 60, N):
        X = torch.randn(S, k, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        ms = events_ms(lambda: store.roll_device(X.data_ptr(), 0, S, k), 3, reps)
        res["kernel"][str(k)] = {"ms": ms, "bytes": roll_bytes, "TB_per_s": roll_bytes / ms / 1e9,
                                 "share_of_copy": roll_bytes / ms / 1e9 / copy_bw}
        del X

    res["host"] = {}
    for k in (1, 60):
        Xh = rng.normal(size=(S, k))
        xp, Xp = pinned(S * k)
        Xp[:] = Xh.reshape(-1)
        Xp2 = Xp.reshape(S, k)
        res["host"][str(k)] = {"pinned_ms": wall_ms(lambda: store.roll(Xp2), 2, max(5, reps // 2)),
                               "pageable_ms": wall_ms(lambda: store.roll(Xh), 2, max(5, reps // 2)),
                               "sample_bytes": S * k * 8}
        mb.lib().muse_host_free(xp)

    # back to the first rows with one k = N roll from page-locked memory, then the same Run
    res["host"][str(N)] = {"pinned_ms": wall_ms(lambda: store.roll(H2), 0, 1), "sample_bytes": S * N * 8}
    after = b.run([], MAX_LAG, TOP_N, THRESHOLD)
    res["run_after_identical"] = all(np.array_equal(x, y) for x, y in zip(first, after))
    res["run_after_ms"] = events_ms(lambda: b.run([], MAX_LAG, TOP_N, THRESHOLD), 3, reps)

    ids = np.zeros((S, 2), dtype=np.int32)

    def reupload():
        store.clear()
        store.append_host_ptr(hp.value, S, N, ids.ctypes.data)
    res["clear_append_pinned_ms"] = wall_ms(reupload, 1, 3)
    b.close()
    store.close()
    mb.lib().muse_host_free(hp)
    torch.cuda.empty_cache()

    # C4-sized store: the roll needs no second slab
    S4, N4 = args.c4_series, 10080
    free0, total = torch.cuda.mem_get_info()
    big = mb.DeviceStore(ctx, N4, 3, S4)
    big.append_synthetic(S4, SEED, 0)
    X = torch.randn(S4, 60, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    ms = events_ms(lambda: big.roll_device(X.data_ptr(), 0, S4, 60), 1, 5)
    Xh = rng.normal(size=(S4, 1))
    host_ms = wall_ms(lambda: big.roll(Xh), 1, 3)
    free2, _ = torch.cuda.mem_get_info()
    res["c4"] = {"series": S4, "length": N4, "store_bytes": S4 * N4 * 8, "device_total": total, "in_use_before_store": total - free0,
                 "in_use_after_store_and_samples": total - free1, "added_by_the_rolls": free1 - free2,
                 "kernel_k60_ms": ms, "kernel_k60_TB_per_s": 2 * S4 * N4 * 8 / ms / 1e9, "pageable_k1_ms": host_ms}
    big.close()

    line = json.dumps(res, indent=1)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
