"""Remove probe: what muse_group_remove costs on the C3 store, against a device copy of the slab, a fresh store of the remaining
rows and a full re-upload of them.

On the C3 store (1 M x 1440 synthetic rows, 11.5 GB, far larger than L2) it reports, in one process, for removals of 1, 100,
10 k, 100 k and 500 k rows, scattered (uniform without replacement) and as one contiguous block in the middle of the store:
  * the rows moved (holes below the new size) and the bytes the kernel reads and writes (2 x moved x ld x 8);
  * the call from call to return (host clock, the call ends in a synchronise): median of --reps, the store rebuilt before each;
  * move_rows_kernel alone (torch.profiler, CUDA activities, a separate pass): mean over --reps removals, its rate and that
    rate's share of the device-to-device copy bandwidth measured in the same process;
  * muse_group_clear + muse_group_append of the remaining rows from page-locked memory (host clock), which builds a fresh store
    of the same rows in the same order;
  * the C3 Run (maxLag 60, top 100, threshold 0.5, ungrouped, AUTO) on the store after the removal and on that fresh store
    (CUDA events, median of --reps), results compared bit for bit.

usage: python tools/remove_probe.py [--series S] [--reps R] [--out FILE.json]"""
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
COUNTS = (1, 100, 10_000, 100_000, 500_000)


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


def pinned(n, ctype=C.c_double):
    p = C.c_void_p()
    mb._check(mb.lib().muse_host_alloc(C.byref(p), n * C.sizeof(ctype)))
    return p, np.ctypeslib.as_array((ctype * n).from_address(p.value))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--series", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    S, reps = args.series, args.reps
    ld = (N + 15) // 16 * 16
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = mb.Context(0)
    ctx.set_stream(stream.cuda_stream)
    res = {"gpu": card(), "series": S, "length": N, "reps": reps}
    rng = np.random.default_rng(SEED)

    slab_bytes = S * ld * 8
    src = torch.empty(slab_bytes // 8, dtype=torch.float64, device="cuda").normal_()
    dst = torch.empty_like(src)
    copy_ms = events_ms(lambda: dst.copy_(src), 3, 10)
    copy_bw = 2 * slab_bytes / copy_ms / 1e9          # TB/s (bytes read + written)
    res["copy"] = {"bytes": slab_bytes, "ms": copy_ms, "TB_per_s": copy_bw}
    del src, dst
    torch.cuda.empty_cache()

    store = mb.DeviceStore(ctx, N, 2, S)
    fresh = mb.DeviceStore(ctx, N, 2, S)
    ref = mb.synth_reference(SEED, N)

    def rebuild():
        store.clear()
        store.append_synthetic(S, SEED, 0)

    i = np.arange(S)
    ids0 = np.stack([i // 1000, i % 1000], axis=1).astype(np.int32)     # the synthetic label ids
    hp, H = pinned(S * N)
    ip, IDS = pinned(S * 2, C.c_int32)
    rebuild()
    store.remove([0])                                # warm: the context's pair buffer, the max-id pass
    rebuild()
    b = mb.DeviceBatch(ctx, store, ref)
    bf = mb.DeviceBatch(ctx, fresh, ref)
    res["run_full_store_ms"] = events_ms(lambda: b.run([], MAX_LAG, TOP_N, THRESHOLD), 3, reps)

    res["cases"] = []
    for kind in ("scattered", "block"):
        for n in COUNTS:
            if kind == "scattered":
                rows = np.sort(rng.choice(S, n, replace=False))
            else:
                rows = np.arange((S - n) // 2, (S - n) // 2 + n)
            case = {"kind": kind, "removed": n, "remaining": S - n}
            wall = []
            for _ in range(reps):
                rebuild()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                moved_from, moved_to = store.remove(rows)
                wall.append((time.perf_counter() - t0) * 1e3)
            case["moved"] = int(moved_from.size)
            case["kernel_bytes"] = 2 * int(moved_from.size) * ld * 8
            case["call_ms"] = float(np.median(wall))
            if moved_from.size:
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    for _ in range(reps):
                        rebuild()
                        store.remove(rows)
                    torch.cuda.synchronize()
                ks = [a for a in prof.key_averages() if "move_rows_kernel" in a.key]
                case["kernel_launches"] = sum(a.count for a in ks)
                case["kernel_ms"] = sum(a.device_time_total for a in ks) / max(1, case["kernel_launches"]) / 1e3
                case["kernel_TB_per_s"] = case["kernel_bytes"] / case["kernel_ms"] / 1e9
                case["kernel_share_of_copy"] = case["kernel_TB_per_s"] / copy_bw
            # the store as the removal leaves it, and a fresh store of the same rows in the same order
            rebuild()
            m = S - n
            ids = ids0.copy()
            ids[moved_to] = ids0[moved_from]
            store.read_rows_ptr(0, S, hp.value)
            Hr = H.reshape(S, N)
            Hr[moved_to] = Hr[moved_from]
            IDS[:] = ids.reshape(-1)
            store.remove(rows)

            def refill():
                fresh.clear()
                fresh.append_host_ptr(hp.value, m, N, ip.value)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            refill()
            case["clear_append_remaining_pinned_ms"] = (time.perf_counter() - t0) * 1e3
            got, want = b.run([], MAX_LAG, TOP_N, THRESHOLD), bf.run([], MAX_LAG, TOP_N, THRESHOLD)
            case["run_identical_to_fresh"] = all(np.array_equal(x, y) for x, y in zip(got, want))
            case["run_after_removal_ms"] = events_ms(lambda: b.run([], MAX_LAG, TOP_N, THRESHOLD), 2, reps)
            case["run_mode"] = int(b.timing().mode)
            case["run_fresh_ms"] = events_ms(lambda: bf.run([], MAX_LAG, TOP_N, THRESHOLD), 2, reps)
            case["run_fresh_mode"] = int(bf.timing().mode)
            res["cases"].append(case)
            print(json.dumps(case), flush=True)

    b.close()
    bf.close()
    store.close()
    fresh.close()
    mb.lib().muse_host_free(hp)
    mb.lib().muse_host_free(ip)
    line = json.dumps(res, indent=1)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
