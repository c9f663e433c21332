"""Multi-GPU check of many references against a sharded store (torchrun --nproc-per-node N tools/multi_exchange_check.py):
Exchange.run_many (peer-memory exchange) == allgather_merge_many (NCCL all-gather + device merge) == multi_run on rank 0 over
ONE store holding every shard, for several argument sets and shard layouts.  Prints ALL IDENTICAL when every set agrees."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "go-muse_b200"))
import numpy as np, torch, torch.distributed as dist
import muse_b200 as mb
rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
S, N, SEED = int(os.environ.get("CHECK_SERIES", "200000")), 1440, 20261018
ctx = mb.Context(local)
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream); ctx.set_stream(stream.cuda_stream)


def refs_of(Q, seed):
    rng = np.random.default_rng(seed)
    R = np.zeros((Q, N))
    for q in range(Q):
        mid, w = int(rng.integers(N // 2 - N // 8, N // 2 + N // 8)), int(rng.integers(3, 21))
        R[q, mid - w // 2: mid - w // 2 + w] = 1.5
        R[q] += 0.1 * (rng.random(N) - 0.5)
    R[Q // 2] = 3.0                                     # std == 0: None on every rank
    return R


def same(a, b):
    return len(a) == len(b) and all((x is None) == (y is None) and (x is None or all(np.array_equal(u, v) for u, v in zip(x, y)))
                                    for x, y in zip(a, b))


# shard layouts: even blocks of S each, and uneven blocks (rank r holds a share growing with r, the last may be small)
layouts = {"even": [(r * S, (r + 1) * S) for r in range(world)]}
cuts = [0] + [int(world * S * (r + 1) * (r + 2) / (world * (world + 1))) for r in range(world)]
layouts["uneven"] = [(cuts[r], cuts[r + 1]) for r in range(world)]
full = None
if rank == 0:                                           # rows of append_synthetic depend only on (seed, global index)
    full = mb.DeviceStore(ctx, N, 0, world * S); full.append_synthetic(world * S, SEED, 0)
ok = True
for name, bounds in layouts.items():
    lo, hi = bounds[rank]
    store = mb.DeviceStore(ctx, N, 0, max(hi - lo, 1))
    if hi > lo:
        store.append_synthetic(hi - lo, SEED, lo)
    store.set_global_offset(lo)
    for Q, max_lag, top_n, thr, cap, sign in ((40, 60, 100, 0.5, 256 * 100, 0), (300, 60, 50, 0.3, 256 * 50, 0),
                                              (9, 15, 10, 0.0, 30, 0), (5, 60, 64, 0.2, 64, -1), (3, 5, 1, 0.9, 1, 0)):
        R = refs_of(Q, 1000 + Q)
        ex = mb.Exchange(ctx, cap)
        got = ex.run_many(store, R, max_lag, top_n, thr, sign)
        dist.barrier()
        ex.close()
        gathered = mb.allgather_merge_many(store, R, max_lag, top_n, thr, sign)
        res = same(got, gathered)
        if rank == 0:
            want = mb.multi_run(full, R, [], max_lag, top_n, thr, sign)
            res = res and same(got, want)
            nres = sum(len(g[0]) for g in got if g is not None)
            print("%s shards %s, Q %d max_lag %d top_n %d thr %g sign %d capacity %d: %s (%d results)"
                  % (name, bounds, Q, max_lag, top_n, thr, sign, cap, "identical" if res else "MISMATCH", nres), flush=True)
        ok &= bool(res)
    store.close()
flag = torch.tensor([1 if ok else 0], device="cuda"); dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0: print("ALL IDENTICAL" if flag.item() == 1 else "FAILED", flush=True)
if full is not None: full.close()
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
