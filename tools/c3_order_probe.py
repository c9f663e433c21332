"""C3 order probe: does the order of the rows in the store change the speed of the screening kernel?

Builds the C3 store (1 M x 1440 of the benchmark's generator, maxLag 60, top 100, threshold 0.5) three times from the
same rows: (a) in the benchmark's order (row kind = index mod 3: rect, line, noise), (b) in a seeded random permutation,
(c) sorted by kind, so that all rect rows -- the only ones that take the fused second stage -- form one contiguous block.
Then alternates Batch.Run on the three stores in one process and reports, per store, the screening kernel's time
(timing().score_ms), the step time (CUDA events around blocks of consecutive runs), the refined and re-scored counts,
and whether the results are the same series as (a)'s once mapped back through the permutation.

usage: python tools/c3_order_probe.py [--series S] [--rounds R] [--block K] [--out FILE.json]
Needs about 46 GB of device memory: three stores plus the staging copy of the rows."""
import argparse
import json
import os
import subprocess
import sys

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


def orders(S):
    kind = torch.arange(S) % 3
    return {
        "a_bench": None,
        "b_random": torch.randperm(S, generator=torch.Generator().manual_seed(SEED)),
        "c_by_kind": torch.argsort(kind, stable=True),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--series", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=8, help="alternations over the three stores")
    ap.add_argument("--block", type=int, default=5, help="consecutive runs per store and round")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    S = args.series

    ctx = mb.Context(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)      # the library's kernels and torch's copies on one stream
    src = mb.DeviceStore(ctx, N, 0, S)
    src.append_synthetic(S, SEED, 0)
    ctx.synchronize()
    rows = torch.empty((S, N), dtype=torch.float64, device="cuda")
    chunk = 65536
    host = torch.empty((chunk, N), dtype=torch.float64, pin_memory=True)
    for lo in range(0, S, chunk):
        n = min(chunk, S - lo)
        src.read_rows_ptr(lo, n, host.data_ptr())
        rows[lo:lo + n].copy_(host[:n])
    torch.cuda.synchronize()
    del host

    ref = mb.synth_reference(SEED, N)
    stores, perms = {}, orders(S)
    for name, perm in perms.items():
        if perm is None:
            stores[name] = src
            continue
        st = mb.DeviceStore(ctx, N, 0, S)
        moved = rows.index_select(0, perm.cuda())
        torch.cuda.synchronize()
        st.append_device(moved.data_ptr(), S, N)
        ctx.synchronize()
        del moved
        stores[name] = st
    del rows
    torch.cuda.empty_cache()
    batches = {k: mb.DeviceBatch(ctx, s, ref) for k, s in stores.items()}

    res = {k: {"score_ms": [], "ms_per_step": [], "n_refined": [], "n_rescored": []} for k in stores}
    last = {}
    for k, b in batches.items():            # warm-up: tables, scratch, module load
        for _ in range(3):
            last[k] = b.run([], MAX_LAG, TOP_N, THRESHOLD)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for k, b in batches.items():
            torch.cuda.synchronize()
            ev0.record(stream)
            for _ in range(args.block):
                last[k] = b.run([], MAX_LAG, TOP_N, THRESHOLD)
                tm = b.timing()
                res[k]["score_ms"].append(tm.score_ms)
                res[k]["n_refined"].append(tm.n_refined)
                res[k]["n_rescored"].append(tm.n_rescored)
            ev1.record(stream)
            torch.cuda.synchronize()
            res[k]["ms_per_step"].append(ev0.elapsed_time(ev1) / args.block)

    a_idx = last["a_bench"][2]
    out = {"config": "C3 order probe: %d series x %d, maxLag=%d, topN=%d, threshold=%g, %d rounds x %d runs per store"
                     % (S, N, MAX_LAG, TOP_N, THRESHOLD, args.rounds, args.block),
           "card": card(), "lib": os.path.basename(mb.LIB_PATH), "stores": {}}
    for k, r in res.items():
        perm = perms[k]
        idx = last[k][2] if perm is None else perm.numpy()[last[k][2]]
        sc = np.asarray(r["score_ms"])
        out["stores"][k] = {
            "score_ms_mean": float(sc.mean()), "score_ms_std": float(sc.std()),
            "score_ms_min": float(sc.min()), "score_ms_max": float(sc.max()), "runs": int(sc.size),
            "ms_per_step_mean": float(np.mean(r["ms_per_step"])), "ms_per_step_blocks": [round(x, 4) for x in r["ms_per_step"]],
            "n_refined_mean": float(np.mean(r["n_refined"])), "n_rescored_mean": float(np.mean(r["n_rescored"])),
            "same_series_as_a": bool(np.array_equal(np.sort(idx), np.sort(a_idx))),
            "same_scores_as_a": bool(np.array_equal(np.sort(last[k][0]), np.sort(last["a_bench"][0]))),
        }
    text = json.dumps(out, indent=1)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
