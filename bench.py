#!/usr/bin/env python
"""bench.py -- series-samples/s of Batch.Run on synthetic siggen-style data.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torchrun)
    python bench.py --impl reference ...                   (CPU arm: the oracle port)

Workload (BASELINE.json configs[2], "C3", the configuration the north-star target is
quoted on): S = 1,000,000 series x 1440 fp64 samples PER GPU (weak scaling: rank r owns
global series [r*S, (r+1)*S)), reference = Rect(1.5, 720, 10)+noise, maxLag 60, topN 100,
threshold 0.5, ungrouped.  A step is one Batch.Run over the resident slab; at N>1 each
rank runs its shard, the shard partials are all-gathered over NCCL and merged.

One JSON line is printed by rank 0 (see the repo prompt for the contract).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "go-muse_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "series-samples/sec (and % HBM roofline) for Batch.Run at 1/2/4/8 B200 vs host Go"
UNIT = "series-samples/s"
SEED = 20261018
DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: the result records of the last timed step, one float64 <path>/<name>.npy per field (lags and series
    indices are exact in float64), so that two builds can be compared output for output.  Above DUMP_BYTES in all, a
    fixed, seeded sample of the records is written, and the record numbers it kept go to sample_rows.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64).ravel() for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    keep = (DUMP_BYTES - 4096) // (8 * (len(arrays) + 1))         # 4096: room for the .npy headers
    if n * 8 * len(arrays) > DUMP_BYTES - 4096:
        rows = np.sort(np.random.default_rng(SEED).choice(n, keep, replace=False))
        arrays = dict({k: v[rows] for k, v in arrays.items()}, sample_rows=rows.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


def workload(args):
    if args.workload == "c4":
        name = ("C4 (%s): %d series x %d fp64 samples per GPU, maxLag=%d, topN=%d, threshold=%g, %s (BASELINE.json configs[3])"
                % ("full size" if args.series * max(1, args.gpus) >= 10_000_000 else "weak-scaled share", args.series, args.length,
                   args.max_lag, args.top_n, args.threshold,
                   "ungrouped" if args.ungrouped else "grouped by [graph, host] (100 series per group)"))
    else:
        name = ("C3: %d series x %d fp64 samples %s, maxLag=%d, topN=%d, threshold=%g, ungrouped "
                "(BASELINE.json configs[2])" % (args.series, args.length, "per GPU" if args.scaling == "weak" else "in total (sharded)",
                                                args.max_lag, args.top_n, args.threshold))
    return {
        "workload": name,
        "series_per_gpu": args.series if args.scaling == "weak" else args.series // max(1, args.gpus), "series_len": args.length, "fft_len": int(2 ** int(np.ceil(np.log2(args.length)))),
        "max_lag": args.max_lag, "top_n": args.top_n, "threshold": args.threshold,
        "group_by": ["graph", "host"] if args.workload == "c4" and not args.ungrouped else None,
        "mode": args.mode,
        "l2": "inputs (%.2f GB per GPU) are far larger than the 126 MB L2; no flush needed" % (args.series * args.length * 8 / 1e9),
    }


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.stop_flag = threading.Event()
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag.is_set():
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        if self.proc is not None:
            try:
                self.proc.kill()
            except Exception:
                pass
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_arm(args, Y, ref, steps, warmup, nthreads):
    """The reference algorithm on the host cores: the C oracle port of go-muse's Batch.Run path.
    Returns (series-samples/s, ms per step, the last step's (scores, lags, series indices))."""
    from oracle import c_oracle as co
    S, N = Y.shape
    for _ in range(max(0, warmup)):
        co.batch_run(ref, Y, None, args.max_lag, args.top_n, args.threshold, 0, nthreads)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = co.batch_run(ref, Y, None, args.max_lag, args.top_n, args.threshold, 0, nthreads)
    dt = (time.perf_counter() - t0) / steps
    return S * N / dt, dt * 1e3, out


def run_reference(args):
    """The reference arm maps nothing but oracle/: rows and reference come from oracle/synth_gen.c (the same
    counter-based generator as the device's, bit for bit), the timed loop is oracle/muse_oracle.c."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import c_oracle as co
    cores = co.max_threads()
    n_rows = min(args.series, args.cpu_sample)
    Y = co.synth_rows(SEED, 0, n_rows, args.length)
    ref = co.synth_reference(SEED, args.length)
    value, ms, out = cpu_arm(args, Y, ref, args.steps, args.warmup, cores)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"scores": out[0], "lags": out[1], "series_idx": out[2]})
    sample = "first %d of the %d series of the workload per step (bounded so the run ends in minutes)" % (n_rows, args.series)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "go-muse is Go and no Go toolchain exists in this image: this arm times oracle/muse_oracle.c, a C "
                "restatement of the reference path (pthreads, one worker per label group as muse_batch.go:104-128)",
    }
    print(json.dumps(line), flush=True)


def run_c5(args, mb, torch, dist, rank, local_rank, world, mode):
    """BASELINE.json configs[4]: Q reference queries against ONE store of --series series, sharded by series over
    the GPUs (strong scaling).  A step = muse_multi_run on the shard (bounds of all queries as one bf16 contraction on
    the tensor cores, one pass over the store for the second stages, one launch per stage for the tails) + one
    all-gather of the shards' per-query top-N + the per-query merge.  Not the headline line."""
    ctx = mb.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    S_total, N, Q, top_n = args.series, args.length, args.queries, args.top_n
    lo, hi = rank * S_total // world, (rank + 1) * S_total // world
    store = mb.DeviceStore(ctx, N, 2, hi - lo)
    store.append_synthetic(hi - lo, SEED, lo)
    store.set_global_offset(lo)
    rng = np.random.default_rng(3)
    refs = np.zeros((Q, N))
    for q in range(Q):                                   # rect mids / widths varied (SURVEY 8d C5)
        mid, w = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8)), int(rng.integers(3, 21))
        refs[q, mid - w // 2: mid - w // 2 + w] = 1.5
        refs[q] += 0.1 * (rng.random(N) - 0.5)

    def step():
        sc, lg, ix, n_out = mb.multi_run(store, refs, [], args.max_lag, top_n, args.threshold, 0, mode=mode, raw=True)
        if world == 1:
            return [(sc[q, :n_out[q]], lg[q, :n_out[q]], ix[q, :n_out[q]]) for q in range(Q)]
        # fixed-size records per query: (score, lag, global index), padded with score -1; one all-gather, then the
        # per-query merge (score desc, index asc: results.go:81-85) for all queries at once
        valid = np.arange(top_n)[None, :] < n_out[:, None]
        rec = np.stack([np.where(valid, sc, -1.0), lg.astype(np.float64), ix.astype(np.float64)], axis=-1)
        mine = torch.from_numpy(rec).cuda(non_blocking=True)
        allr = torch.empty((world,) + tuple(mine.shape), dtype=mine.dtype, device="cuda")
        dist.all_gather_into_tensor(allr, mine)
        # shards hold ascending global indices and each shard's list is already (score desc, index asc): a STABLE
        # sort by score over the rank-ordered concatenation breaks ties by index
        r = allr.permute(1, 0, 2, 3).reshape(Q, world * top_n, 3)
        order = torch.sort(-r[..., 0], dim=-1, stable=True).indices[:, :top_n]
        r = torch.gather(r, 1, order[..., None].expand(-1, -1, 3)).cpu().numpy()
        k = (r[..., 0] >= 0).sum(axis=1)
        return [(r[q, :k[q], 0], r[q, :k[q], 1].astype(np.int64), r[q, :k[q], 2].astype(np.int64)) for q in range(Q)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        out = step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.5)
    stage_ms = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        out = step()
        stage_ms.append(mb.multi_last_timing(ctx))
    ev1.record(stream)
    barrier()
    time.sleep(0.2)
    clocks = sampler.finish()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / args.steps
    if rank == 0:
        refined, rescored = mb.multi_last_stats(ctx)
        tc = os.environ.get("MUSE_MULTI_TC") != "0"
        st = np.mean(np.array(stage_ms), axis=0) if stage_ms else np.zeros(4)
        n_groups = (Q + 255) // 256
        # the contraction of ONE launch group on this rank: three bf16 MMAs (hi x hi, hi x lo, lo x hi) of [S_shard x 1024] x [1024 x 256]
        flops = 3 * 2.0 * (hi - lo) * min(Q, 256) * 1024
        bf16_peak, peak_src = 1405.2, "fallback"
        ppath = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(ppath):
            with open(ppath) as f:
                pk = json.load(f)
            bf16_peak, peak_src = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1405.2))), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        roofline = None
        if tc and st[1] > 0:
            ach = flops / (st[1] * 1e-3) / 1e12
            roofline = {"bound": "tensor", "achieved": ach, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach / bf16_peak, "traffic": None,
                        "peak_source": peak_src, "kernel": "bounds_tc_kernel (tcgen05.mma kind::f16, bf16 hi/lo split, fp32 in TMEM)",
                        "kernel_ms": float(st[1]), "flops_per_launch": flops,
                        "stage_ms": {"magnitudes": float(st[0]), "bounds_gemm": float(st[1]), "second_stages": float(st[2]), "tails": float(st[3])},
                        "note": "the contraction is the tensor-core kernel of the path; the step is dominated by the fp32 second stages "
                                "(refine_multi_kernel) of the %.1f %% of (series, query) pairs whose bound reaches their query's cut-off"
                                % (100.0 * refined / max(1.0, float(hi - lo) * Q))}
        cpu = None
        if world == 1 and not args.no_cpu:
            from oracle import c_oracle as co
            n_rows, n_q = min(hi - lo, 16384), min(Q, 8)
            Y = store.read_rows(0, n_rows)
            cores = co.max_threads()
            t0 = time.perf_counter()
            for q in range(n_q):
                co.batch_run(refs[q], Y, None, args.max_lag, top_n, args.threshold, 0, cores)
            dt = time.perf_counter() - t0
            cpu = {"value": n_q * n_rows * N / dt, "unit": "pair-samples/s", "cores": cores, "kind": "port",
                   "sample": "%d queries x first %d series, one NewBatch + Run each (muse_batch.go:23-52, :99-130) of oracle/muse_oracle.c "
                             "on %d threads, %.0f ms" % (n_q, n_rows, cores, dt * 1e3)}
        line = {
            "metric": "pair-samples/sec for Q reference queries against one sharded store (BASELINE.json configs[4])",
            "value": Q * S_total * N / (ms * 1e-3), "unit": "pair-samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C5: %d reference queries x %d series x %d fp64 samples, maxLag=%d, topN=%d, threshold=%g, "
                                   "ungrouped, store sharded by series over %d GPU(s)" % (Q, S_total, N, args.max_lag, top_n, args.threshold, world),
                       "queries": Q, "series_total": S_total, "series_len": N, "ms_per_query": ms / Q,
                       "refined_pairs_per_step": refined, "rescored_pairs_per_step": rescored,
                       "bounds": "bf16x2 tcgen05" if tc else "fp32",
                       "l2": "each shard (%.2f GB) is far larger than the 126 MB L2" % ((hi - lo) * N * 8 / 1e9)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": None,
            "gpu_launches": int(args.steps * n_groups * 12),
            "clocks": clocks, "top": {"score": float(out[0][0][0]) if len(out[0][0]) else None, "n": int(len(out[0][0]))},
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"query": np.concatenate([np.full(len(o[0]), q) for q, o in enumerate(out)]),
                                             "scores": np.concatenate([o[0] for o in out]),
                                             "lags": np.concatenate([o[1] for o in out]),
                                             "series_idx": np.concatenate([o[2] for o in out])})
        print(json.dumps(line), flush=True)
    store.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--queries", type=int, default=256, help="--workload c5: reference queries per step")
    ap.add_argument("--workload", default="c3", choices=["c3", "c4", "c5"],
                    help="c3 (default, the configuration the metric is quoted on) or c4: 1.25 M x 10080 per GPU, maxLag 240, "
                         "grouped by two labels (not a headline line: BASELINE.json configs[3]); c5: --queries references "
                         "against 1 M x 1440 series sharded over the GPUs (BASELINE.json configs[4], pair-samples/s)")
    ap.add_argument("--series", type=int, default=None)
    ap.add_argument("--length", type=int, default=None)
    ap.add_argument("--max-lag", type=int, default=None)
    ap.add_argument("--top-n", type=int, default=100)
    ap.add_argument("--threshold", type=float, default=0.5)
    ap.add_argument("--mode", default="auto", choices=["auto", "exact", "screen"])
    ap.add_argument("--cpu-sample", type=int, default=131072)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--nccl-exchange", action="store_true", help="N > 1: NCCL all-gather instead of the peer-memory push")
    ap.add_argument("--ungrouped", action="store_true", help="--workload c4: Run(nil) instead of Run([graph, host])")
    ap.add_argument("--data", default="mix", choices=["mix", "rect"],
                    help="mix: rect / line / noise rows (the benchmark); rect: every row a rect of the reference's width "
                         "(adversarial for the screening: nearly every score lies within the slack of the cut-off)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --series per GPU (the metric's configuration); strong: --series in total, sharded over the GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last one as DIR/<name>.npy (float64; a seeded "
                         "sample of them above 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    dflt = {"c3": (1_000_000, 1440, 60), "c4": (1_250_000, 10080, 240), "c5": (1_000_000, 1440, 60)}[args.workload]
    args.series = args.series if args.series is not None else dflt[0]
    args.length = args.length if args.length is not None else dflt[1]
    args.max_lag = args.max_lag if args.max_lag is not None else dflt[2]
    if args.workload == "c4":
        args.no_e2e = True        # 100.8 GB of pinned host rows per GPU: the end-to-end leg is measured on the C3 line only
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = max(args.warmup, 0)

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import muse_b200 as mb

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: muse_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    mode = {"auto": mb.MODE_AUTO, "exact": mb.MODE_EXACT, "screen": mb.MODE_SCREEN}[args.mode]
    if args.workload == "c5":
        run_c5(args, mb, torch, dist, rank, local_rank, world, mode)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    ctx = mb.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)          # library kernels and NCCL deps on one stream: one event bracket
    N = args.length
    strong = args.scaling == "strong"
    if strong:                                  # --series in total, sharded by series
        first, S = rank * args.series // world, (rank + 1) * args.series // world - rank * args.series // world
    else:                                       # --series per GPU (the metric's configuration)
        first, S = rank * args.series, args.series
    S_total = args.series if strong else world * args.series
    grouped = args.workload == "c4" and not args.ungrouped
    variant = 1 if args.data == "rect" else 0
    store = mb.DeviceStore(ctx, N, 3 if grouped else 2, S)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    store.append_synthetic(S, SEED, first, variant)      # rows AND their row statistics (mean, 1/std): one ingest kernel
    ctx.synchronize()
    ingest_ms = (time.perf_counter() - t0) * 1e3
    store.set_global_offset(first)
    cols = []
    if grouped:
        # SURVEY 8d C4: graph = i/10000 % 1000, host = i/100 % 100, colo = i % 100 -> (graph, host) groups of 100 series
        store.set_synthetic_labels([10000, 100, 1], [1000, 100, 100])
        cols = [0, 1]
    ref = mb.synth_reference(SEED, N)
    batch = mb.DeviceBatch(ctx, store, ref)
    exchange, exchange_kind = None, None
    if world > 1:
        exchange_kind = "nccl-allgather"
        if not args.nccl_exchange:
            try:
                # ungrouped: top_n records per shard; grouped: every group representative of the shard (100 series per group here)
                cap = max(1, args.top_n) if not grouped else max(args.top_n, S // 100 + 64)
                exchange = mb.Exchange(ctx, cap)      # all ranks succeed or all raise
                exchange_kind = "nvlink-peer-push + device merge"
            except mb.MuseError as e:
                if rank == 0:
                    print("bench: %s -> NCCL all-gather" % e, file=sys.stderr)

    def exchange_step(b):
        # the kernel that produces the shard's records stores them into every rank's receive buffer over NVLink peer
        # memory and releases a flag; one call = scores, push, wait for the peers, merge on the device, top_n records to
        # the host (same result on every rank).  None: some shard's list was too long for the device-side select ->
        # all ranks take the all-gather path together
        r = exchange.run(b, args.max_lag, args.top_n, args.threshold, 0, mode=mode, key_cols=cols) if exchange else None
        if r is None and grouped:
            parts = b.run_partial(cols, args.max_lag, args.top_n, args.threshold, 0, mode=mode)
            r = mb.allgather_merge(parts, args.max_lag, args.top_n, args.threshold, 0)
        elif r is None:
            r = mb.allgather_merge_device(b, args.max_lag, args.top_n, args.threshold, 0, mode=mode)
        return r

    def step():
        if world == 1:
            return batch.run(cols, args.max_lag, args.top_n, args.threshold, 0, mode=mode)
        return exchange_step(batch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the first Run on a freshly ingested store: nothing is cached across Runs but the store's row statistics, which the
    # ingest kernels produce with the rows -- so this "cold" figure holds no extra pass over the slab (tables, scratch
    # allocation and module load excluded by one throw-away run on a tiny store of the same shape)
    tiny = mb.DeviceStore(ctx, N, 3 if grouped else 2, 1024)
    tiny.append_synthetic(1024, SEED, 0, variant)
    if grouped:
        tiny.set_synthetic_labels([10000, 100, 1], [1000, 100, 100])
    tb = mb.DeviceBatch(ctx, tiny, ref)
    tb.run(cols, args.max_lag, min(args.top_n, 100), args.threshold, 0, mode=mb.MODE_SCREEN)
    tb.close()
    tiny.close()
    barrier()
    out = step()
    cold_run_ms = batch.timing().total_ms
    for _ in range(max(args.warmup, 3)):
        out = step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    score_ms, launches, n_rescored, n_refined, tail_ms = [], 0, 0, 0, []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        out = step()
        tm = batch.timing()
        score_ms.append(tm.score_ms)
        launches += tm.n_launches
        n_rescored += tm.n_rescored
        n_refined += tm.n_refined
        tail_ms.append(tm.total_ms - tm.score_ms)
    ev1.record(stream)
    barrier()
    time.sleep(0.2)
    clocks = sampler.finish()
    total_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = S_total * N / (ms_per_step * 1e-3)
    used_mode = {mb.MODE_EXACT: "exact", mb.MODE_SCREEN: "screen"}.get(batch.timing().mode, "?")

    # ---- end to end through the C ABI with HOST buffers (pinned), H2D inside the timed region ----
    e2e = None
    if not args.no_e2e:
        host = torch.empty((S, N), dtype=torch.float64, pin_memory=True)
        store.read_rows_ptr(0, S, host.data_ptr())          # same rows as the resident slab, now on the host
        ids = torch.zeros((S, 2), dtype=torch.int32, pin_memory=True)
        gidx = torch.arange(first, first + S, dtype=torch.int64)
        ids[:, 0] = (gidx // 1000).to(torch.int32)
        ids[:, 1] = (gidx % 1000).to(torch.int32)
        st2 = mb.DeviceStore(ctx, N, 2, S)

        def e2e_step():
            st2.clear()
            st2.append_host_ptr(host.data_ptr(), S, N, ids.data_ptr())     # Group.Add: H2D of the step's inputs (+ row statistics)
            st2.set_global_offset(first)
            b2 = mb.DeviceBatch(ctx, st2, ref)                               # NewBatch
            if world == 1:
                r = b2.run([], args.max_lag, args.top_n, args.threshold, 0, mode=mode)   # Run; results land on the host
            else:
                r = exchange_step(b2)
            b2.close()
            return r

        r = e2e_step()
        assert np.array_equal(r[2], out[2]) and np.array_equal(r[0], out[0]), "e2e result differs from the resident run"
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        barrier()
        dt = (time.perf_counter() - t0) / args.e2e_steps
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": S_total * N / dt, "unit": UNIT, "h2d_bytes_per_step": int(S * N * 8 + S * 2 * 4 + N * 8),
               "d2h_bytes_per_step": int(len(out[0]) * 24) if world == 1 else int(max(1, args.top_n) * 32), "ms_per_step": dt * 1e3, "steps": args.e2e_steps,
               "api": "muse_group_clear + muse_group_append(pinned host rows) + muse_batch_create + muse_batch_run"}
        st2.close()
        del host

    if rank == 0:
        hbm_peak, peak_src = peaks()
        alg_bytes = S * (8 * N + 16)
        k_ms = float(np.mean(score_ms))
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                with open(tpath) as f:
                    tj = json.load(f)
                key = used_mode if (args.workload, S, N) == ("c3", 1_000_000, 1440) and variant == 0 else \
                    ("c4_grouped" if grouped else "c4_ungrouped") if (args.workload, S, N) == ("c4", 1_250_000, 10080) else \
                    "n512" if (args.workload, S, N, used_mode) == ("c3", 3_000_000, 480, "screen") else None
                traffic = tj.get(key, {}).get("dram_bytes_per_launch") if key else None
            except Exception:
                traffic = None
        roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                    "traffic": traffic, "peak_source": peak_src,
                    "kernel": "score_exact_kernel" if used_mode == "exact" else
                              ("score_screen_warp_kernel" if 1024 < N <= 2048 else "score_screen_big_kernel" if N > 2048
                               else "score_screen_block_kernel" if os.environ.get("MUSE_BLOCK_SMALL")
                               else "score_screen_sub_kernel"),
                    "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes,
                    "frac_of_nominal_8TBps": achieved / 8000.0}
        cpu = None
        if world == 1 and not args.no_cpu:
            from oracle import c_oracle as co
            n_rows = min(S, args.cpu_sample if N <= 2048 else args.cpu_sample // 8)
            Y = store.read_rows(0, n_rows)
            gids = (np.arange(n_rows) // 100).astype(np.int64) if grouped else None
            cores = co.max_threads()
            co.batch_run(ref, Y, gids, args.max_lag, args.top_n, args.threshold, 0, cores)
            t0 = time.perf_counter()
            for _ in range(2):
                co.batch_run(ref, Y, gids, args.max_lag, args.top_n, args.threshold, 0, cores)
            ms = (time.perf_counter() - t0) / 2 * 1e3
            cpu = {"value": n_rows * N / (ms * 1e-3), "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "first %d of the %d series, 2 timed passes (%.0f ms each) of oracle/muse_oracle.c on %d threads"
                             % (n_rows, S, ms, cores)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": dict(workload(args), mode_used=used_mode,
                                                rescored_per_step=n_rescored / max(1, args.steps),
                                                refined_per_step=n_refined / max(1, args.steps),
                                                tail_ms=sum(tail_ms) / max(1, len(tail_ms)), exchange=exchange_kind,
                                                cold_run_ms=cold_run_ms, ingest_ms=ingest_ms,
                                                row_stats="mean and 1/std of every row are produced by the ingest kernels (synthetic rows: "
                                                          "in the generator; host / device appends: one kernel behind the copy), so no Run -- "
                                                          "the first one included (cold_run_ms) -- holds a separate pass over the slab",
                                                data_variant=args.data, series_total=S_total),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "top": {"score": float(out[0][0]) if len(out[0]) else None, "n": int(len(out[0]))},
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"scores": out[0], "lags": out[1], "series_idx": out[2]})
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        if exchange:
            exchange.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
