"""Query rounds of an address-sharded sketch at config C5's shape (DESIGN.md §6): get_median_count for every read of every rank,
the counters fetched from their owners over NVLink (route | offsets + push | lookup | pull | per-read statistics).

Counttable k=40 (MurmurHash3), 4 tables of 3.2e10 bins per GPU (128 GB of tables per GPU), 1 M synthetic 150 bp reads per GPU
and round.  The tables are filled by ingest rounds first; the query rounds then ask for the same reads.  One process per GPU:

    python -m torch.distributed.run --nproc-per-node N tools/bench_sharded_query.py

Prints one JSON line (rank 0).  Times are wall clock between barriers (each phase ends in a device synchronisation), max over
ranks.  At one GPU it also times the local sketch's own read_medians on the same tables (no exchange) and checks that both give
identical medians, averages and deviations.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import N_TABLES, READ_LEN, primes_near_x, synth_batch  # noqa: E402


def card(local_rank):
    """name and power limit of the GPU, read in the run that measures it"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:
        import torch
        return {"name": torch.cuda.get_device_name(local_rank), "power_limit": "unknown (%s)" % type(e).__name__}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=1_000_000, help="reads per GPU and round")
    ap.add_argument("--shard-x", type=float, default=0, help="bins per table (default 3.2e10 per GPU)")
    ap.add_argument("--fill", type=int, default=3, help="ingest rounds before the queries (all but the first are timed)")
    ap.add_argument("--steps", type=int, default=4, help="timed query rounds")
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    from khmer_b200 import cabi
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    k = 40
    x = int(args.shard_x) if args.shard_x else int(3.2e10) * world
    sizes = primes_near_x(N_TABLES, x)
    R = args.reads
    sh = cabi.Shard(cabi.BYTE, cabi.MURMUR, k, sizes, rank, world, device=local_rank, max_positions=R * READ_LEN)
    handles = np.ascontiguousarray(sh.ipc_export())
    if world > 1:
        t = torch.from_numpy(handles).to(dev)
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        handles = np.concatenate([p.cpu().numpy() for p in parts])
    sh.ipc_attach(handles)
    batches = [synth_batch(9000 * (rank + 1) + b, R, pinned=True) for b in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    ingest_s = 0.0
    for i in range(args.fill):
        buf, off, _ = batches[i % 2]
        t0 = time.perf_counter()
        for step in (lambda: sh.route((buf, off), clean=True), sh.offsets, sh.push, sh.apply, sh.count_new):
            step()
            barrier()
        if i:
            ingest_s += time.perf_counter() - t0

    def query(s, t):
        buf, off, _ = batches[s % 2]
        marks = [time.perf_counter()]
        for step in (lambda: sh.route((buf, off), clean=True), lambda: (sh.offsets(), barrier(), sh.push()), sh.lookup, sh.pull):
            step()
            barrier()
            marks.append(time.perf_counter())
        res = sh.read_medians()
        barrier()
        marks.append(time.perf_counter())
        for j in range(5):
            t[j] += marks[j + 1] - marks[j]
        return res

    t = [0.0] * 5
    for s in range(args.warmup):
        query(s, t)
    t = [0.0] * 5
    kmers = 0
    t0 = time.perf_counter()
    for s in range(args.steps):
        res = query(args.warmup + s, t)
        kmers += int(res[3].sum(dtype=np.uint64))
    dt = time.perf_counter() - t0
    last = (args.warmup + args.steps - 1) % 2

    ref = None
    if world == 1:
        # the same reads through the local sketch's own query path: no exchange, the 128 GB tables read in place
        buf, off, _ = batches[last]
        sh.local.read_medians((buf, off), clean=True)   # warm-up
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        loc = sh.local.read_medians((buf, off), clean=True)
        torch.cuda.synchronize()
        ref_s = time.perf_counter() - t1
        same = all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip(res, loc))
        ref = {"local_read_medians_ms": 1e3 * ref_s, "local_kmers_per_sec": float(loc[3].sum(dtype=np.uint64)) / ref_s,
               "identical_to_query_rounds": bool(same)}

    tt = torch.tensor([dt, float(kmers), ingest_s] + t, dtype=torch.float64, device=dev)
    mx, sm = tt.clone(), tt.clone()
    if world > 1:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    if rank == 0:
        per = lambda v: 1e3 * float(v) / args.steps   # noqa: E731
        line = {
            "metric": "queried_kmers_per_sec_counttable_k40_N4_address_sharded", "value": float(sm[1]) / float(mx[0]), "unit": "k-mers/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_query_round": per(mx[0]),
            "config": {"workload": "read_medians over Counttable k=40 (MurmurHash3) N=4, tables of %.3g bins cut across %d GPUs (%.1f GB of "
                                   "tables per GPU), synthetic 150bp 30x reads, %d reads per GPU and round, the reads the tables were "
                                   "filled with" % (x, world, sum(sizes) / world / 1e9, R),
                       "timing": "wall clock between barriers (each phase ends in a device synchronisation), max over ranks"},
            "phases_ms_per_round": {"route": per(mx[3]), "exchange (offsets + push)": per(mx[4]), "lookup": per(mx[5]), "pull": per(mx[6]),
                                    "stats (read_medians)": per(mx[7])},
            "ingest_round_ms": 1e3 * float(mx[2]) / max(args.fill - 1, 1),
            # a query record crosses NVLink twice (push, pull): 8 bytes each way per table, (world - 1) / world of them remote
            "nvlink_bytes_per_kmer": 2 * N_TABLES * 8.0 * (world - 1) / world,
            "gpu": card(local_rank),
        }
        if ref is not None:
            line["no_exchange_reference"] = ref
        print(json.dumps(line), flush=True)
    sh.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
