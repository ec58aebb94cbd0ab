"""Ingest rounds of an address-sharded sketch with bigcount off and on, at config C5's shape (DESIGN.md §6).

Counttable k=40 (MurmurHash3), 4 tables of 3.2e10 bins per GPU, 1 M reads of 150 bp per GPU and round.  The same reads go
through rounds with bigcount off and on, alternating in one process on one sketch (two sketches of 128 GB do not fit one GPU).
Two workloads: "ordinary" (synthetic 30x reads of a new genome every round: nearly no byte reaches 255, so a round with bigcount
on adds one flag check)
and "worst" (1 M reads of one 2 Mb genome per round, ~55 touches per k-mer and round: after the warm-up rounds every byte of
the genome's k-mers is 255 and every touch is an event).  A smaller genome concentrates more touches per round on a bucket
than the sharded apply's bucket regions hold, and the regions then grow every round until they no longer fit next to 128 GB
of tables.  One process per GPU:

    python -m torch.distributed.run --nproc-per-node N tools/bench_sharded_bigcount.py [--out profiles/sharded_bigcount_n1.json]

Prints one JSON line (rank 0) and writes it to --out.  Times are wall clock between barriers (each step ends in a device
synchronisation), max over ranks.  The apply step of a round with bigcount on includes the marking of saturated touches; the
events step is the pull of the marks, the fold and the aggregation per k-mer; the map step is the exchange and the map update.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import N_TABLES, READ_LEN, primes_near_x, synth_batch  # noqa: E402
from bench_sharded_query import card  # noqa: E402


def genome_reads(seed, n_reads, genome_len):
    """n_reads reads of 150 bp of one random genome of genome_len bases (the same for every seed), uniform start, random strand"""
    g = np.random.default_rng(1).integers(0, 4, genome_len, dtype=np.uint8)
    rng = np.random.default_rng(seed)
    starts = rng.integers(0, genome_len - READ_LEN, n_reads)
    strands = rng.integers(0, 2, n_reads).astype(bool)
    codes = g[starts[:, None] + np.arange(READ_LEN)[None, :]]
    codes[strands] = (3 - codes[strands])[:, ::-1]
    buf = np.frombuffer(b"ACGT", dtype=np.uint8)[codes].reshape(-1).copy()
    return buf, np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(READ_LEN)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=1_000_000, help="reads per GPU and round")
    ap.add_argument("--shard-x", type=float, default=0, help="bins per table (default 3.2e10 per GPU)")
    ap.add_argument("--steps", type=int, default=3, help="timed rounds per setting and workload")
    ap.add_argument("--warmup", type=int, default=3, help="untimed rounds per setting and workload")
    ap.add_argument("--genome", type=int, default=2_000_000, help="genome length of the worst-case workload")
    ap.add_argument("--out", default="")
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

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(obj):
        if world == 1:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    def used_bytes():
        free, total = torch.cuda.mem_get_info(dev)   # cudaMemGetInfo
        return total - free

    def run_workload(batches):
        sh = cabi.Shard(cabi.BYTE, cabi.MURMUR, k, sizes, rank, world, device=local_rank, max_positions=R * READ_LEN)
        handles = np.ascontiguousarray(sh.ipc_export())
        handles = np.concatenate([np.frombuffer(h, dtype=np.uint8) for h in gather(handles.tobytes())])
        sh.ipc_attach(handles)
        barrier()
        res = {}
        mem = {}
        t = {False: np.zeros(6), True: np.zeros(6)}
        ev = {False: [], True: []}
        for i in range(2 * (args.warmup + args.steps)):
            big = bool(i % 2)                       # off, on, off, on, ...
            sh.set_use_bigcount(big)
            buf, off = batches[i % len(batches)]
            marks = [time.perf_counter()]
            steps = [lambda: sh.route((buf, off), clean=True), lambda: (sh.offsets(), barrier(), sh.push()), sh.apply, sh.count_new]
            for step in steps:
                step()
                barrier()
                marks.append(time.perf_counter())
            n_ev = n_kmers = 0
            if big:
                hs, cs = sh.bigcount_events()
                barrier()
                marks.append(time.perf_counter())
                lists = gather((hs.tobytes(), cs.tobytes()))
                allh = np.concatenate([np.frombuffer(a, dtype=np.uint64) for a, _ in lists])
                allc = np.concatenate([np.frombuffer(b, dtype=np.uint32) for _, b in lists])
                sh.bigcount_apply(allh, allc)
                barrier()
                marks.append(time.perf_counter())
                n_ev, n_kmers = int(cs.sum(dtype=np.uint64)), len(hs)
            else:
                marks += [marks[-1], marks[-1]]
            if i >= 2 * args.warmup:
                t[big] += np.diff(marks)
                ev[big].append((n_ev, n_kmers))
            if i == 0 or big:   # off: before any round with bigcount on has allocated its buffers
                mem[big] = used_bytes()
        mx = t
        if world > 1:
            allt = gather({b: t[b].tolist() for b in t})
            mx = {b: np.max([a[b] for a in allt], axis=0) for b in t}
        names = ["route", "offsets + push", "apply (incl. marking)", "count_new", "events (pull + fold + aggregate)", "map exchange + apply"]
        for big in (False, True):
            per = mx[big] / args.steps * 1e3
            res["bigcount_" + ("on" if big else "off")] = {
                "round_ms": float(per.sum()), "steps_ms": {n: float(v) for n, v in zip(names, per) if big or n in names[:4]},
                "device_bytes_in_use": int(mem.get(big, 0)),
            }
        res["bigcount_on"]["events_per_round_this_rank"] = [e[0] for e in ev[True]]
        res["bigcount_on"]["distinct_kmers_per_round_this_rank"] = [e[1] for e in ev[True]]
        res["map_entries"] = int(len(sh.bigcounts()[0]))
        sh.close()
        torch.cuda.synchronize()
        return res

    # ordinary: fresh reads of a fresh genome every round, so that counts stay at 30x instead of adding up over the rounds
    ordinary = [synth_batch(9000 * (rank + 1) + b, R)[:2] for b in range(2 * (args.warmup + args.steps))]
    worst = [genome_reads(7000 + b, R, args.genome) for b in range(2)]
    out = {}
    out["ordinary"] = run_workload(ordinary)
    del ordinary
    out["worst"] = run_workload(worst)
    if rank == 0:
        line = {
            "metric": "sharded_ingest_round_ms_bigcount_off_vs_on", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "config": {"workload": "Counttable k=40 (MurmurHash3) N=4, tables of %.3g bins cut across %d GPUs (%.1f GB of tables per GPU), "
                                   "%d reads of 150 bp per GPU and round; ordinary: synthetic 30x reads; worst: reads of one %d-base genome; %d warm-up rounds per setting"
                                   % (x, world, sum(sizes) / world / 1e9, R, args.genome, args.warmup),
                       "timing": "wall clock between barriers (each step ends in a device synchronisation), max over ranks; rounds "
                                 "with bigcount off and on alternate on one sketch"},
            "results": out,
            "gpu": card(local_rank),
        }
        s = json.dumps(line)
        print(s, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(s + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
