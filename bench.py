#!/usr/bin/env python
"""bench.py — k-mers/s ingested into Countgraph (k=20, N=4) on B200, beside the reference CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # our arm
    python bench.py --impl reference [--gpus N] [--steps K] ...    # reference CPU arm (rank 0 only)

Workload (BASELINE.json metric; SURVEY.md §8d): Countgraph/ByteStorage k=20, N=4 tables of ~1e8 bytes
(get_n_primes_near_x(4, 1e8), 400 MB — larger than the 126 MB L2), bigcount on at N=1, synthetic 150 bp reads
sampled at 30x from a uniform random genome.  A step = one pass of the hot path over one batch of R reads.
P distinct batches are cycled; after every P steps the sketch is reset (one "job" = P batches), so no step
ever runs on saturated counters.

value  : k-mers/s with the packed batches already resident in HBM (kmgpu_consume_batch), device-timed with
         CUDA events on the library's own stream, max over ranks.
e2e    : the same through kmgpu_consume_reads with ASCII reads in pinned HOST memory: H2D copy, 2-bit packing
         on the device, ingestion, D2H of the per-chunk result block — all inside the timed region.
N > 1  : one process per GPU (torchrun), each ingests its own read shard into its own replica (weak scaling, no
         data-path collective per step); the replicas are merged once per job by the saturating-add NVLink
         reduction (reduce-scatter + all-gather over CUDA-IPC peer memory), inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 20
N_TABLES = 4
TABLE_X = int(1e8)
READ_LEN = 150
COVERAGE = 30
KMERS_PER_READ = READ_LEN - K + 1
ALGO_BYTES_PER_KMER = N_TABLES * 64          # 32 B sector in + 32 B sector out per counter update (SURVEY §8d)


def primes_near_x(n, x):
    """get_n_primes_near_x (include/oxli/hashtable.hh:99-123) — host-side sizing, same as khmer_args does."""
    def is_prime(v):
        if v < 2:
            return False
        if v % 2 == 0:
            return v == 2
        i = 3
        while i * i <= v:
            if v % i == 0:
                return False
            i += 2
        return True
    out = []
    c = x - 1
    if c % 2 == 0:
        c -= 1
    while len(out) < n and c > 0:
        if is_prime(c):
            out.append(c)
        c -= 2
    return out


def synth_batch(seed, n_reads, pinned=False):
    """R reads of exactly 150 bp, uniform start, random strand, genome G = 5R (30x) — SURVEY.md §8d."""
    rng = np.random.default_rng(seed)
    genome_len = max(READ_LEN + 1, n_reads * READ_LEN // COVERAGE)
    g = rng.integers(0, 4, genome_len, dtype=np.uint8)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    if pinned:
        import torch
        t = torch.empty(n_reads * READ_LEN, dtype=torch.uint8, pin_memory=True)
        buf = t.numpy()
    else:
        t = None
        buf = np.empty(n_reads * READ_LEN, dtype=np.uint8)
    view = buf.reshape(n_reads, READ_LEN)
    step = 1 << 18
    for i0 in range(0, n_reads, step):
        m = min(step, n_reads - i0)
        starts = rng.integers(0, genome_len - READ_LEN, m)
        strands = rng.integers(0, 2, m).astype(bool)
        codes = g[starts[:, None] + np.arange(READ_LEN)[None, :]]
        codes[strands] = (3 - codes[strands])[:, ::-1]
        view[i0:i0 + m] = lut[codes]
    off = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(READ_LEN)
    if pinned:   # the read offsets are part of the step's input: page-locked like the sequence bytes
        to = torch.empty(n_reads + 1, dtype=torch.int64, pin_memory=True)
        po = to.numpy().view(np.uint64)
        po[:] = off
        return buf, po, (t, to)
    return buf, off, t


class ClockSampler:
    """nvidia-smi clocks and throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md, MEASURED_PEAKS.json absent)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "ingest_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return None


# ---------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref when it was compiled, else the port)
# ---------------------------------------------------------------------------------------------------------
def cpu_reference_run(n_reads, threads, seed=4242, repeats=1):
    """k-mers/s of the reference's consume_seqfile on a FASTA of n_reads synthetic reads, T threads sharing one
    parser (scripts/load-into-counting.py:145-158).  Timer around the consume loop only."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    buf, off, _ = synth_batch(seed, n_reads)
    sizes = primes_near_x(N_TABLES, TABLE_X)
    kind = "reference" if ol.have_ref() else "port"
    times = []
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "reads.fa")
        if kind == "reference":
            with open(path, "wb") as fh:
                rows = buf.reshape(n_reads, READ_LEN)
                hdr = np.frombuffer(b">r\n", dtype=np.uint8)
                block = np.empty((n_reads, READ_LEN + 4), dtype=np.uint8)
                block[:, :3] = hdr
                block[:, 3:3 + READ_LEN] = rows
                block[:, -1] = ord("\n")
                fh.write(block.tobytes())
        for _ in range(repeats):
            if kind == "reference":
                sk = ol.Ref("Countgraph", K, sizes)
                sk.set_use_bigcount(True)
                t0 = time.perf_counter()
                _, kmers = sk.consume_seqfile(path, threads=threads)
                times.append(time.perf_counter() - t0)
            else:
                threads = 1
                sk = ol.Oracle("Countgraph", K, sizes)
                sk.set_use_bigcount(True)
                t0 = time.perf_counter()
                kmers = sk.L.ko_consume_reads(sk.h, buf.ctypes.data_as(ol.C.c_char_p), off.ctypes.data_as(ol.u64p),
                                              n_reads, 1, 0, 0, 0)
                times.append(time.perf_counter() - t0)
            del sk
    return kmers, times, kind, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_reads = args.ref_reads
    kmers, times, kind, threads = cpu_reference_run(n_reads, threads, repeats=args.steps + args.warmup)
    timed = times[args.warmup:]
    total = sum(timed)
    value = kmers * len(timed) / total
    sample = "%d synthetic 150 bp reads (%d k-mers) per step from a FASTA file, Countgraph k=%d N=%d x=%d" % (
        n_reads, kmers, K, N_TABLES, TABLE_X)
    line = {
        "impl": "reference", "metric": "kmers_per_sec_countgraph_k20_N4", "value": value, "unit": "k-mers/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(timed),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "load-into-counting Countgraph k=20 N=4 x=1e8 bigcount, synthetic 150bp 30x reads",
                   "reads_per_step": n_reads, "threads": threads},
        "cpu_baseline": {"value": value, "unit": "k-mers/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def table_md5s(sk):
    import hashlib
    return [hashlib.md5(sk.table(i).tobytes()).hexdigest() for i in range(N_TABLES)]


def parity_check(cabi, local_rank, n_reads, seed=31337):
    """One fixed batch into a fresh sketch through the same call the e2e leg times, compared with the reference at one
    thread (oracle/_ref; the oracle port when the compiled reference is absent): table images, n_occupied, n_unique_kmers.
    The checker is never the thing measured."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hashlib
    import oracle_lib as ol
    buf, off, _ = synth_batch(seed, n_reads)
    sizes = primes_near_x(N_TABLES, TABLE_X)
    sk = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, K, sizes, device=local_rank)
    sk.set_use_bigcount(True)
    kmers = sk.consume_reads((buf, off), clean=True)
    got = {"kmers": int(kmers), "n_occupied": int(sk.stats()[0]), "n_unique_kmers": int(sk.stats()[1]), "table_md5": table_md5s(sk)}
    sk.close()
    if ol.have_ref():
        kind = "reference"
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "reads.fa")
            rows = buf.reshape(n_reads, READ_LEN)
            block = np.empty((n_reads, READ_LEN + 4), dtype=np.uint8)
            block[:, :3] = np.frombuffer(b">r\n", dtype=np.uint8)
            block[:, 3:3 + READ_LEN] = rows
            block[:, -1] = ord("\n")
            with open(path, "wb") as fh:
                fh.write(block.tobytes())
            ref = ol.Ref("Countgraph", K, sizes)
            ref.set_use_bigcount(True)
            _, rk = ref.consume_seqfile(path, threads=1)
        want = {"kmers": int(rk), "n_occupied": int(ref.n_occupied()), "n_unique_kmers": int(ref.n_unique_kmers()),
                "table_md5": [hashlib.md5(ref.table(i).tobytes()).hexdigest() for i in range(N_TABLES)]}
    else:
        kind = "port"
        o = ol.Oracle("Countgraph", K, sizes)
        o.set_use_bigcount(True)
        rk = o.L.ko_consume_reads(o.h, buf.ctypes.data_as(ol.C.c_char_p), off.ctypes.data_as(ol.u64p), n_reads, 1, 0, 0, 0)
        want = {"kmers": int(rk), "n_occupied": int(o.n_occupied()), "n_unique_kmers": int(o.n_unique_kmers()),
                "table_md5": [hashlib.md5(o.table(i).tobytes()).hexdigest() for i in range(N_TABLES)]}
    ok = got == want
    return {"ok": ok, "checker": kind, "reads": n_reads, "kmers": got["kmers"], "n_unique_kmers": got["n_unique_kmers"],
            "n_occupied": got["n_occupied"], "table_md5_0": got["table_md5"][0],
            "mismatch": None if ok else {"got": got, "want": want}}


def file_leg(args, local_rank, repeats=3):
    """k-mers/s of khmer_b200.Countgraph(20, 1e8, 4).consume_seqfile(fasta) — wall clock around the call (it returns when the table
    is final), best of `repeats`, file in the page cache like the reference arm's."""
    import khmer_b200
    os.environ.setdefault("KMGPU_DEVICE", str(local_rank))
    n_reads = args.reads
    buf, off, _ = synth_batch(777, n_reads)
    td = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    path = os.path.join(td, "reads.fa")
    try:
        rows = buf.reshape(n_reads, READ_LEN)
        block = np.empty((n_reads, READ_LEN + 4), dtype=np.uint8)
        block[:, :3] = np.frombuffer(b">r\n", dtype=np.uint8)
        block[:, 3:3 + READ_LEN] = rows
        block[:, -1] = ord("\n")
        with open(path, "wb") as fh:
            fh.write(block.tobytes())
        del block
        # one table for all passes (the first pass is the warm-up: device workspaces and pinned batches are allocated once per
        # table); counts simply keep growing, 4 passes of 26x stay far below 255
        t = khmer_b200.Countgraph(K, TABLE_X, N_TABLES)
        best = None
        for i in range(repeats + 1):
            t0 = time.perf_counter()
            reads, kmers = t.consume_seqfile(path)
            dt = time.perf_counter() - t0
            assert reads == n_reads and kmers == n_reads * KMERS_PER_READ
            if i:
                best = dt if best is None else min(best, dt)
        # compressed input (the reference's own benchmark file is a .fq.gz): FASTA of the first 500 k reads as ordinary gzip (one
        # sequential inflate, done ahead by a thread of its own) and as BGZF (bgzip's block-compressed gzip, inflated by all
        # parser threads)
        comp = {}
        n_c = min(n_reads, 500_000)
        with open(path, "rb") as fh:
            data = fh.read(n_c * (READ_LEN + 4))
        import gzip
        import struct
        import zlib
        gz_path, bg_path = os.path.join(td, "reads.fa.gz"), os.path.join(td, "reads.bgzf.fa.gz")
        with open(gz_path, "wb") as fh:
            fh.write(gzip.compress(data, 1))
        with open(bg_path, "wb") as fh:
            for o in list(range(0, len(data), 65280)) + [None]:
                chunk = b"" if o is None else data[o:o + 65280]
                c = zlib.compressobj(1, zlib.DEFLATED, -15)
                body = c.compress(chunk) + c.flush()
                fh.write(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, 12 + 6 + len(body) + 8 - 1))
                fh.write(body + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))
        del data
        for name, pth in (("gzip", gz_path), ("bgzf", bg_path)):
            bc = None
            for i in range(3):
                t0 = time.perf_counter()
                reads, km = t.consume_seqfile(pth)
                dt = time.perf_counter() - t0
                assert reads == n_c and km == n_c * KMERS_PER_READ
                if i:
                    bc = dt if bc is None else min(bc, dt)
            comp[name] = {"value": km / bc, "unit": "k-mers/s", "reads": n_c, "file_bytes": os.path.getsize(pth), "seconds": bc}
        del t
        return {"value": kmers / best, "unit": "k-mers/s", "api": "khmer_b200.Countgraph.consume_seqfile(path)", "reads": n_reads,
                "file_bytes": os.path.getsize(path), "format": "FASTA, uncompressed", "parser_threads": min(16, os.cpu_count() or 1),
                "seconds": best, "timing": "wall clock (perf_counter) around the call, best of %d after one warm-up" % repeats,
                "compressed": comp}
    finally:
        for f in ("reads.fa", "reads.fa.gz", "reads.bgzf.fa.gz"):
            try:
                os.unlink(os.path.join(td, f))
            except OSError:
                pass
        try:
            os.rmdir(td)
        except OSError:
            pass


def file_leg_subprocess(args, local_rank):
    """The file leg in a process of its own, as a user's script would run it (load-into-counting.py is one process per file):
    `python bench.py --file-leg` prints file_leg()'s dictionary."""
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--file-leg", "--reads", str(args.reads)],
                       env=dict(os.environ, KMGPU_DEVICE=str(local_rank)), capture_output=True, text=True, timeout=1200)
    for ln in reversed(r.stdout.strip().split("\n")):
        if ln.startswith("{"):
            d = json.loads(ln)
            d["process"] = "separate process (python bench.py --file-leg)"
            return d
    sys.stderr.write("[bench] file leg failed: %s\n" % r.stderr[-2000:])
    return {"value": None, "error": r.stderr[-500:]}


def secondary_legs(cabi, sk, host, dev, local_rank, n_query=400_000):
    """The read-side queries on the table the timed legs left behind (not the headline metric): per-read medians
    (Hashtable::get_median_count, hashtable.cc:299-328) and the abundance histogram (hashtable.cc:451-493), wall clock around the
    C-ABI calls with host buffers."""
    buf, off, _ = host[0]
    sk.reset()
    sk.consume_batch(dev[0])
    q = (buf[: n_query * READ_LEN], off[: n_query + 1])
    sk.read_medians(q)                                              # warm-up (workspaces grow to the query's size)
    t0 = time.perf_counter()
    med, _, _, nk = sk.read_medians(q)
    t_med = time.perf_counter() - t0
    # the same query over a batch already resident in HBM: device time (CUDA events) of the count + select kernels and the
    # copy of the medians back to the host
    sk.batch_read_medians(dev[1], stats=False)
    sk.timer_start()
    med_r = sk.batch_read_medians(dev[1], stats=False)[0]
    ms_res = sk.timer_stop()
    n_res = len(med_r)
    sizes = primes_near_x(N_TABLES, TABLE_X)
    tracking = cabi.Sketch(cabi.BIT, cabi.TWOBIT, K, sizes, device=local_rank)
    sk.abundance_distribution((buf, off), tracking)                 # warm-up: the tracking filter's workspaces are allocated here
    tracking.reset()
    t0 = time.perf_counter()
    hist = sk.abundance_distribution((buf, off), tracking)
    t_ab = time.perf_counter() - t0
    n_all = (len(off) - 1) * KMERS_PER_READ
    out = {"medians": {"reads_per_s": n_query / t_med, "kmers_per_s": n_query * KMERS_PER_READ / t_med, "reads": n_query,
                       "median_of_medians": float(np.median(med))},
           "medians_resident": {"reads_per_s": n_res / ms_res * 1e3, "kmers_per_s": n_res * KMERS_PER_READ / ms_res * 1e3, "reads": n_res,
                                "timing": "CUDA events around kmgpu_batch_read_medians (batch in HBM, medians copied out)"},
           "abundance_distribution": {"kmers_per_s": n_all / t_ab, "kmers": n_all, "distinct": int(hist.sum())},
           "timing": "wall clock around kmgpu_read_medians / kmgpu_abundance_distribution, host ASCII in, results out"}
    tracking.close()
    return out


DUMP_SAMPLE_PER_TABLE = 1 << 21
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(sk, kmers, out_dir, seed=20240601):
    """What the last timed step handed its caller, as .npy files for comparing two builds output for output: the k-mers it
    ingested; n_occupied, n_unique_kmers and the number of bigcount entries; the four counter tables (a histogram of every
    counter, plus the counters at fixed seeded positions: the full tables are 400 MB); and the bigcount map itself when it
    has entries (at the bench's 30x coverage no counter reaches 255, so it stays empty)."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(seed)
    keys, vals = sk.bigcounts()
    out = {"kmers": np.array([kmers], dtype=np.float64),
           "stats": np.array(list(sk.stats()) + [len(keys)], dtype=np.float64)}
    for i in range(N_TABLES):
        t = sk.table(i)
        out["table%d_histogram" % i] = np.bincount(t, minlength=256).astype(np.float64)
        idx = np.sort(rng.choice(len(t), size=min(len(t), DUMP_SAMPLE_PER_TABLE), replace=False))
        out["table%d_sample" % i] = t[idx].astype(np.float32)
        del t
    if len(keys):
        order = np.argsort(keys, kind="stable")
        out["bigcount_keys"] = keys[order].astype(np.float64)   # 2-bit hashes of k = 20: below 2**40, exact in float64
        out["bigcount_values"] = vals[order].astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_MAX_BYTES))
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def merge_check(cabi, dist, torch, group_cls, rank, world, local_rank, n_reads=125_000):
    """N > 1: every rank ingests its own fixed batch into a fresh replica, the replicas are merged over NVLink exactly as in
    the timed region; all ranks must then hold identical tables, and rank 0 compares them with ONE sketch fed every rank's
    batch (saturating add is associative, so the images must be byte-identical)."""
    import hashlib
    sizes = primes_near_x(N_TABLES, TABLE_X)
    sk = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, K, sizes, device=local_rank)
    sk.set_use_bigcount(False)
    buf, off, _ = synth_batch(555000 + rank, n_reads)
    sk.consume_reads((buf, off), clean=True)
    grp = group_cls(sk, dist, device=torch.device("cuda", local_rank))
    grp.attach()
    grp.merge()
    mine = hashlib.md5("".join(table_md5s(sk)).encode()).digest()
    occ = sk.stats()[0]
    t = torch.tensor(list(mine) + [occ % 251], dtype=torch.int64, device="cuda")
    gathered = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(gathered, t)
    same = all(bool((g == gathered[0]).all().item()) for g in gathered)
    res = {"ok": same, "ranks_identical": same, "reads_per_rank": n_reads}
    if rank == 0:
        one = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, K, sizes, device=local_rank)
        one.set_use_bigcount(False)
        for r in range(world):
            b, o, _ = synth_batch(555000 + r, n_reads)
            one.consume_reads((b, o), clean=True)
        single = hashlib.md5("".join(table_md5s(one)).encode()).digest()
        res["equals_single_sketch"] = single == mine and one.stats()[0] == occ
        res["ok"] = bool(same and res["equals_single_sketch"])
        res["n_occupied"] = int(occ)
        one.close()
    grp.detach()
    sk.close()
    return res


# ---------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from khmer_b200 import cabi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if cabi.device_count() == 0:
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    R = args.reads
    P = args.batches
    sizes = primes_near_x(N_TABLES, TABLE_X)
    sk = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, K, sizes, device=local_rank)
    bigcount = world == 1     # replicated sketches cannot keep bigcount exact (SURVEY.md §8e)
    sk.set_use_bigcount(bigcount)

    # synthetic batches: pinned host ASCII (e2e leg) and device-resident packed (value leg)
    host = []
    dev = []
    for b in range(P):
        buf, off, keep = synth_batch(1000 * (rank + 1) + b, R, pinned=True)
        host.append((buf, off, keep))
        dev.append(cabi.Batch((buf, off), K, clean=True, device=local_rank))

    # the same batches as the host read feed hands them over (kmgpu_consume_packed): cleaned, 2 bits per base, pinned
    packed = []
    code_of = np.zeros(256, dtype=np.uint64)
    for ch, v in ((b"T", 1), (b"C", 2), (b"G", 3)):
        code_of[ch[0]] = v
    shifts = np.uint64(62) - np.uint64(2) * np.arange(32, dtype=np.uint64)
    for buf, off, _ in host:
        n_words = (len(buf) + 31) // 32 + 2
        tw = torch.zeros(n_words, dtype=torch.int64, pin_memory=True)
        w = tw.numpy().view(np.uint64)
        step = 32 << 20
        for o in range(0, len(buf), step):
            c = code_of[buf[o:o + step]]
            if len(c) % 32:
                c = np.concatenate([c, np.zeros(32 - len(c) % 32, dtype=np.uint64)])
            w[o // 32: o // 32 + len(c) // 32] = (c.reshape(-1, 32) << shifts).sum(axis=1, dtype=np.uint64)
        packed.append((w, off, tw))

    from khmer_b200.multigpu import ReplicaGroup
    group = ReplicaGroup(sk, dist if world > 1 else None, device=torch.device("cuda", local_rank))
    group.attach()

    def merge_replicas():
        group.merge()

    def job_boundary(step):
        """after every P steps: fold the replicas (N > 1), then start a new job on empty tables"""
        if (step + 1) % P == 0:
            merge_replicas()
            sk.reset()

    def run_steps(n, leg, first):
        kmers = 0
        for s in range(first, first + n):
            if leg == "hbm":
                kmers += sk.consume_batch(dev[s % P])
            elif leg == "e2e_packed":
                w, off, _ = packed[s % P]
                kmers += sk.consume_packed(w, off)
            else:
                buf, off, _ = host[s % P]
                kmers += sk.consume_reads((buf, off), clean=True)
            job_boundary(s)
        return kmers

    results = {}
    clocks = None
    for leg in ("hbm", "e2e", "e2e_packed"):
        sk.reset()
        run_steps(args.warmup, leg, 0)
        # start the timed region on a job boundary so every timed step sees the same table states
        first = ((args.warmup + P - 1) // P) * P
        run_steps(first - args.warmup, leg, args.warmup)
        sampler = ClockSampler(local_rank) if leg == "hbm" and rank == 0 else None
        if sampler:
            sampler.start()
            time.sleep(0.25)
        barrier()                      # all ranks enter the timed region together
        sk.profile_reset()
        t0 = time.time()
        sk.timer_start()
        kmers = run_steps(args.steps, leg, first)
        if args.steps % P != 0:
            merge_replicas()
        ms = sk.timer_stop()
        barrier()
        t1 = time.time()
        if sampler:
            clocks = sampler.stop(t0, t1)
        kern_ms, kern_launches, all_launches = sk.profile_get()
        print("[bench rank %d] leg=%s device_ms=%.2f wall_ms=%.2f ingest_kernel_ms=%.2f launches=%d" % (
            rank, leg, ms, 1e3 * (t1 - t0), kern_ms, all_launches), file=sys.stderr, flush=True)
        results[leg] = {"ms": max_over_ranks(ms), "kmers": sum_over_ranks(kmers), "kern_ms": kern_ms,
                        "kern_launches": kern_launches, "launches": all_launches, "local_kmers": kmers,
                        "wall_ms": 1e3 * (t1 - t0)}

    # the same device-timed leg with bigcount off (what every N > 1 run uses): the N = 1 denominator of a scaling ratio
    value_nobig = None
    if world == 1:
        sk.set_use_bigcount(False)
        sk.reset()
        run_steps(P, "hbm", 0)
        barrier()
        sk.timer_start()
        kk = run_steps(P, "hbm", P)
        ms_nb = sk.timer_stop()
        value_nobig = kk / (ms_nb * 1e-3)
        sk.set_use_bigcount(True)
        sk.reset()

    # end to end from a FILE through the host layer's reference-named call, khmer_b200.Countgraph.consume_seqfile(path): mmap + parser
    # threads (clean + 2-bit pack) + pinned batches + H2D + ingest, all inside the timed region — what the reference arm's
    # consume_seqfile<FastxReader> does on the CPU
    e2e_file = None
    secondary = None
    if world == 1 and not args.no_file:
        e2e_file = file_leg_subprocess(args, local_rank)
        secondary = secondary_legs(cabi, sk, host, dev, local_rank)

    checks = {}
    if not args.no_check:
        if rank == 0:
            checks["parity_check"] = parity_check(cabi, local_rank, args.check_reads)
        if world > 1:
            checks["merge_check"] = merge_check(cabi, dist, torch, ReplicaGroup, rank, world, local_rank)

    hbm, e2e = results["hbm"], results["e2e"]
    value = hbm["kmers"] / (hbm["ms"] * 1e-3)
    e2e_value = e2e["kmers"] / (e2e["ms"] * 1e-3)
    peak, peak_src = measured_peak()
    # the ingest kernel group (hash, group by bucket, apply in shared memory); algorithmic bytes of the timed
    # launches = k-mers ingested x N x 64 B, divided by the summed group durations (CUDA events on the library's stream)
    kmers_per_launch = hbm["local_kmers"] / max(1, hbm["kern_launches"])
    avg_launch_ms = hbm["kern_ms"] / max(1, hbm["kern_launches"])
    achieved = hbm["local_kmers"] * ALGO_BYTES_PER_KMER / (hbm["kern_ms"] * 1e-3) / 1e9
    traffic = ncu_traffic()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic["dram_bytes_per_kmer"] * kmers_per_launch if traffic else None,
                "kernel": ("ingest kernel group per chunk: k_part (fused hash + grouping) + k_apply2<BYTE> + k_popc (grouped path, KMGPU_PREFER_BINS=0)"
                           if os.environ.get("KMGPU_PREFER_BINS") == "0" else
                           "ingest kernel group per chunk: k_hashbins + k_bucketize + k_apply<BYTE> + k_popc (bins path, the default for this shape)"),
                "kernel_ms_per_launch": avg_launch_ms, "kernel_launches": int(hbm["kern_launches"]),
                "kmers_per_launch": kmers_per_launch, "algorithmic_bytes_per_launch": kmers_per_launch * ALGO_BYTES_PER_KMER,
                "algorithmic_bytes_per_kmer": ALGO_BYTES_PER_KMER,
                "peak_source": peak_src, "kernel_share_of_step": hbm["kern_ms"] / hbm["ms"] if world == 1 else None,
                "traffic_source": traffic.get("source") if traffic else None,
                # frac above is the distance to the spec's random-sector model (SURVEY 8d: N x 64 B per k-mer); dram_frac is
                # real DRAM utilisation: bytes ncu saw the group move per k-mer x the measured k-mer rate / peak
                "dram_frac": (traffic["dram_bytes_per_kmer"] * hbm["local_kmers"] / (hbm["kern_ms"] * 1e-3) / 1e9 / peak) if traffic else None,
                "dram_bytes_per_kmer": traffic["dram_bytes_per_kmer"] if traffic else None}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        kmers_c, times, kind, threads = cpu_reference_run(args.cpu_reads, threads)
        cpu = {"value": kmers_c / times[0], "unit": "k-mers/s", "cores": threads, "kind": kind,
               "sample": "%d synthetic 150 bp reads (%d k-mers), same table shape, one timed consume_seqfile with %d "
                         "threads sharing one parser" % (args.cpu_reads, kmers_c, threads)}

    if args.dump_outputs and rank == 0:
        # the tables the last timed step of the hbm leg left behind: replay its job up to that step on an empty sketch
        last = ((args.warmup + P - 1) // P) * P + args.steps - 1
        sk.reset()
        for s in range(last - last % P, last + 1):
            kmers_last = sk.consume_batch(dev[s % P])
        dump_outputs(sk, kmers_last, args.dump_outputs)

    if rank == 0:
        bases = R * READ_LEN
        line = {
            "metric": "kmers_per_sec_countgraph_k20_N4", "value": value, "unit": "k-mers/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": hbm["ms"] / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "load-into-counting Countgraph k=20 N=4 x=1e8 (4 x ~100 MB byte tables), synthetic "
                                   "150bp 30x reads", "reads_per_step_per_gpu": R, "kmers_per_step_per_gpu": R * KMERS_PER_READ,
                       "batches_per_job": P, "bigcount": bigcount, "l2": "tables (400 MB) larger than L2 (126 MB); no flush",
                       "parallelism": "replicated sketch per GPU, disjoint read shards, saturating-add NVLink merge per job"
                       if world > 1 else "single GPU"},
            "roofline": roofline, "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "k-mers/s", "h2d_bytes_per_step": bases + 8 * (R + 1),
                    "d2h_bytes_per_step": 64 * ((bases + (32 << 20) - 1) // (32 << 20)), "ms_per_step": e2e["ms"] / args.steps},
            "gpu_launches": int(hbm["launches"]), "clocks": clocks,
        }
        pk = results["e2e_packed"]
        line["e2e_packed"] = {"value": pk["kmers"] / (pk["ms"] * 1e-3), "unit": "k-mers/s", "h2d_bytes_per_step": bases // 4 + 8 * (R + 1),
                              "api": "kmgpu_consume_packed: host buffers as the read feed's parser threads leave them (cleaned, 2 bits per base)"}
        if value_nobig is not None:
            line["value_bigcount_off"] = value_nobig
        if e2e_file is not None:
            line["e2e_file"] = e2e_file
        if secondary is not None:
            line["secondary"] = secondary
        line.update(checks)
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    bad = [k for k, v in checks.items() if not v.get("ok")]
    if bad:
        print("[bench] FAILED checks: %s" % ", ".join(bad), file=sys.stderr, flush=True)
        raise SystemExit(3)


# ---------------------------------------------------------------------------------------------------------
# address-sharded mode (config C5): Counttable k=40 (Murmur), tables cut across the ranks, k-mer all-to-all over NVLink
# ---------------------------------------------------------------------------------------------------------
def run_sharded(args):
    import torch
    import torch.distributed as dist
    from khmer_b200 import cabi
    from khmer_b200.multigpu import ShardedGroup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    k = 40
    # C5: 4 tables of 2.56e11 bytes over 8 GPUs = 128 GB per GPU; other world sizes keep 32 GB per table and GPU unless told otherwise
    x = int(args.shard_x) if args.shard_x else int(3.2e10) * world
    sizes = primes_near_x(N_TABLES, x)
    R = args.shard_reads
    max_pos = R * READ_LEN
    sh = cabi.Shard(cabi.BYTE, cabi.MURMUR, k, sizes, rank, world, device=local_rank, max_positions=max_pos)
    grp = ShardedGroup(sh, dist if world > 1 else None, device=dev)
    grp.attach()
    batches = [synth_batch(9000 * (rank + 1) + b, R, pinned=True) for b in range(2)]
    kmers_per_read = READ_LEN - k + 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(s, t):
        buf, off, _ = batches[s % 2]
        t0 = time.perf_counter()
        n = sh.route((buf, off), clean=True)
        barrier()
        ta = time.perf_counter()
        sh.offsets()
        barrier()
        sh.push()
        barrier()
        t1 = time.perf_counter()
        sh.apply()
        barrier()
        t2 = time.perf_counter()
        sh.count_new()
        barrier()
        t3 = time.perf_counter()
        t[0] += ta - t0
        t[1] += t2 - t1
        t[2] += t3 - t2
        t[3] += t1 - ta
        return n

    t = [0.0, 0.0, 0.0, 0.0]
    for s in range(args.warmup):
        step(s, t)
    barrier()
    t = [0.0, 0.0, 0.0, 0.0]
    t0 = time.perf_counter()
    kmers = 0
    for s in range(args.steps):
        kmers += step(args.warmup + s, t)
    barrier()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt, float(kmers)] + t, dtype=torch.float64, device=dev)
    if world > 1:
        mx = tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tt.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    else:
        mx, sm = tt, tt
    occ, uniq = grp.stats()
    _, _, store_bytes = sh.stats()
    if rank == 0:
        total_kmers = float(sm[1])
        line = {
            "metric": "kmers_per_sec_counttable_k40_N4_address_sharded", "value": total_kmers / float(mx[0]), "unit": "k-mers/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(mx[0]) / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "mode": "sharded",
            "config": {"workload": "Counttable k=40 (MurmurHash3) N=4, tables of %.3g bytes cut across %d GPUs (%.1f GB of tables per GPU), "
                                   "synthetic 150bp 30x reads, %d reads per GPU and round" % (x, world, sum(sizes) / world / 1e9, R),
                       "table_bytes_per_gpu": sum(sizes) // world, "receive_store_bytes_per_gpu": store_bytes,
                       "timing": "wall clock between barriers (each phase ends in a device synchronisation), max over ranks"},
            "phases_ms_per_step": {"route (hash + group locally)": 1e3 * float(mx[2]) / args.steps,
                                   "exchange (offsets + push over NVLink)": 1e3 * float(mx[5]) / args.steps,
                                   "apply": 1e3 * float(mx[3]) / args.steps, "count_new": 1e3 * float(mx[4]) / args.steps},
            # every counter update is an 8-byte record written into its owner's HBM; (world - 1) / world of them cross NVLink
            "nvlink_bytes_per_kmer": N_TABLES * 8.0 * (world - 1) / world,
            "n_occupied": occ, "n_unique_kmers": uniq, "gpu_launches": int(sh.local.profile_get()[2]),
        }
        emit(line)
    sh.close()
    if world > 1:
        dist.destroy_process_group()


def emit(line):
    """The one JSON line goes to the real stdout; everything else a library prints (NCCL banners ...) was
    diverted to stderr by divert_stdout()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def divert_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def main():
    divert_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=2_000_000, help="reads per step per GPU")
    ap.add_argument("--batches", type=int, default=4, help="distinct batches cycled (= steps per job)")
    ap.add_argument("--cpu-reads", type=int, default=1_000_000, help="sample size of the cpu_baseline leg")
    ap.add_argument("--ref-reads", type=int, default=250_000, help="reads per step of --impl reference")
    ap.add_argument("--mode", default="replicated", choices=["replicated", "sharded"], help="sharded: config C5's address-sharded sketch")
    ap.add_argument("--shard-x", type=float, default=0, help="sharded: bins per table (default 3.2e10 per GPU)")
    ap.add_argument("--shard-reads", type=int, default=1_000_000, help="sharded: reads per GPU and round")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip parity_check / merge_check")
    ap.add_argument("--no-file", action="store_true", help="skip the e2e_file and secondary legs")
    ap.add_argument("--check-reads", type=int, default=250_000, help="reads of the parity_check batch")
    ap.add_argument("--file-leg", action="store_true", help="internal: run the e2e_file leg alone and print its dictionary")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.file_leg:
        emit(file_leg(args, int(os.environ.get("KMGPU_DEVICE", "0"))))
    elif args.impl == "reference":
        run_reference(args)
    elif args.mode == "sharded":
        run_sharded(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
