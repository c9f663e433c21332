"""C5 over a sharded store, two ways in the same process (torchrun --nproc-per-node N tools/c5_sharded.py; one GPU works too):
  - run_many:  Exchange.run_many -- muse_multi_run on the shard, the per-query lists pushed over peer memory, merged on the device;
  - allgather: bench.py's C5 step -- muse_multi_run on the shard, a torch all-gather, a stable torch.sort, a Python loop over the
               queries (restated here; bench.py's own step is not imported so that its arguments stay its own).
A third variant, multi_run alone, is the shard's scoring: variant - multi_run is the merge and transfer tail of each.
The variants alternate step by step after a warm-up; every step ends in a device synchronise and a barrier, and its time is the
maximum over the ranks.  The first timed step of the two full variants must give identical outputs.  One JSON file goes to --out."""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "go-muse_b200"))
import numpy as np, torch, torch.distributed as dist
import muse_b200 as mb

ap = argparse.ArgumentParser()
ap.add_argument("--series", type=int, default=1_000_000, help="series of the whole store, split over the ranks")
ap.add_argument("--length", type=int, default=1440)
ap.add_argument("--queries", type=int, default=256)
ap.add_argument("--max-lag", type=int, default=60)
ap.add_argument("--top-n", type=int, default=100)
ap.add_argument("--threshold", type=float, default=0.5)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--out", required=True, help="output directory")
args = ap.parse_args()

rank, local, world = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
SEED = 20261018
ctx = mb.Context(local)
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream); ctx.set_stream(stream.cuda_stream)
S_total, N, Q, top_n = args.series, args.length, args.queries, args.top_n
lo, hi = rank * S_total // world, (rank + 1) * S_total // world
store = mb.DeviceStore(ctx, N, 2, hi - lo)
store.append_synthetic(hi - lo, SEED, lo)
store.set_global_offset(lo)
rng = np.random.default_rng(3)
refs = np.zeros((Q, N))
for q in range(Q):                                       # bench.py's C5 references
    mid, w = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8)), int(rng.integers(3, 21))
    refs[q, mid - w // 2: mid - w // 2 + w] = 1.5
    refs[q] += 0.1 * (rng.random(N) - 0.5)
ex = mb.Exchange(ctx, min(Q, 256) * top_n)


def step_multi_run():
    return mb.multi_run(store, refs, [], args.max_lag, top_n, args.threshold, 0, raw=True)


def step_run_many():
    return [(np.zeros(0), np.zeros(0, np.int64), np.zeros(0, np.int64)) if o is None else o
            for o in ex.run_many(store, refs, args.max_lag, top_n, args.threshold)]


def step_allgather():
    sc, lg, ix, n_out = mb.multi_run(store, refs, [], args.max_lag, top_n, args.threshold, 0, raw=True)
    if world == 1:
        return [(sc[q, :n_out[q]], lg[q, :n_out[q]], ix[q, :n_out[q]]) for q in range(Q)]
    valid = np.arange(top_n)[None, :] < n_out[:, None]
    rec = np.stack([np.where(valid, sc, -1.0), lg.astype(np.float64), ix.astype(np.float64)], axis=-1)
    mine = torch.from_numpy(rec).cuda(non_blocking=True)
    allr = torch.empty((world,) + tuple(mine.shape), dtype=mine.dtype, device="cuda")
    dist.all_gather_into_tensor(allr, mine)
    r = allr.permute(1, 0, 2, 3).reshape(Q, world * top_n, 3)
    order = torch.sort(-r[..., 0], dim=-1, stable=True).indices[:, :top_n]
    r = torch.gather(r, 1, order[..., None].expand(-1, -1, 3)).cpu().numpy()
    k = (r[..., 0] >= 0).sum(axis=1)
    return [(r[q, :k[q], 0], r[q, :k[q], 1].astype(np.int64), r[q, :k[q], 2].astype(np.int64)) for q in range(Q)]


def sync():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


def timed(fn):
    sync()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    t = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return out, float(t.item())


variants = {"multi_run": step_multi_run, "run_many": step_run_many, "allgather": step_allgather}
for fn in variants.values():
    for _ in range(args.warmup):
        fn()
ms = {k: [] for k in variants}
first = {}
for i in range(args.steps):
    for k, fn in variants.items():
        out, t = timed(fn)
        ms[k].append(t)
        if i == 0:
            first[k] = out
identical = len(first["run_many"]) == len(first["allgather"]) == Q and all(
    len(a) == len(b) and all(np.array_equal(np.asarray(u), np.asarray(v)) for u, v in zip(a, b))
    for a, b in zip(first["run_many"], first["allgather"]))
flag = torch.tensor([1 if identical else 0], device="cuda")
if world > 1:
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    def smi(field):
        try:
            return subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=" + field, "--format=csv,noheader"],
                                  capture_output=True, text=True, timeout=30).stdout.strip() or None
        except Exception:
            return None
    med = {k: float(np.median(v)) for k, v in ms.items()}
    res = {
        "workload": "C5: %d reference queries x %d series x %d fp64 samples, maxLag=%d, topN=%d, threshold=%g, ungrouped, "
                    "store sharded by series over %d GPU(s)" % (Q, S_total, N, args.max_lag, top_n, args.threshold, world),
        "world": world, "gpu": torch.cuda.get_device_name(local), "power_limit": smi("power.limit"),
        "max_sm_clock": smi("clocks.max.sm"), "steps": args.steps, "warmup": args.warmup,
        "timing": "host clock around each step, ending in a device synchronise; max over ranks; variants alternate step by step",
        "median_ms": med, "per_step_ms": ms,
        "tail_ms": {"run_many": med["run_many"] - med["multi_run"], "allgather": med["allgather"] - med["multi_run"]},
        "first_step_outputs_identical": bool(flag.item() == 1),
        "results_first_step": int(sum(len(o[0]) for o in first["run_many"])),
    }
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "c5_sharded_n%d.json" % world)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("world", "gpu", "power_limit", "median_ms", "tail_ms", "first_step_outputs_identical")}), flush=True)
ex.close()
store.close()
if world > 1:
    dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
