"""Bit-exact ingestion at production table shapes, with the default knobs: the delta path at a dozen blocks, two-level
grouping with the super-bucket shift planned for the table sizes, k_apply2 split 2 and split 4, k_apply_sparse, 64-bit bins
and mod_magic with a divisor above 2^32, chunks of more than 2^28 positions in which counters cross 255.  Each shape is
compared after every call with tests/golden/shape_golden.json, what the reference's ingestion computes for the same inputs
(written on the CPU by tests/golden/make_shape_golden.py from the oracle port, which tests/test_oracle.py pins to the
reference): k-mers consumed, n_occupied, n_unique_kmers, a digest of every 256 MiB block of every table, the bigcount map,
and k-mer counts, medians and median_at_least over a probe of 20 k reads.

Each GPU test runs its shape in a subprocess with KMGPU_DEBUG=1 and asserts, from the one line ingest_chunk prints per
chunk, that the shape reached the kernels it is meant to cover: a change of path selection that moves a shape elsewhere
fails here instead of leaving the test green and the form unchecked.

    python tests/test_gpu_shapes.py S3      # one shape on the GPU: its record as one JSON line on stdout"""
import concurrent.futures
import hashlib
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
from test_gpu_benchscale import READ_LEN, _batch, bigcount_md5

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden", "shape_golden.json")

BLOCK = 256 << 20          # bytes per digested block of a table image
N_PROBE = 20_000           # reads of the query probe: the first reads of the shape's last call

# calls: (seed, reads, genome length) per consume_reads call, in order; coverage = reads * 150 / genome length.
# expect: per call, what every chunk of it must show in its KMGPU_DEBUG line (n_pos_min: the largest chunk of the call at least)
SHAPES = {
    # C2: 165 M bases per call against 152 M-position chunks: two chunks, each through 12 delta blocks (3 per table)
    "S1": dict(cls="Nodegraph", k=32, n=4, x=1e9, bigcount=False, cutoffs=(1, 2),
               calls=[(101, 1_100_000, 3_000_000)],
               expect=[dict(path="delta", delta_blocks=12, chunks=2)]),
    # 12 208 buckets per table: two levels, 128 buckets per super-bucket
    "S2": dict(cls="SmallCountgraph", k=31, n=4, x=4e8, bigcount=False, cutoffs=(3, 6),
               calls=[(102, 600_000, 18_000_000)],
               expect=[dict(path="grouped", levels=2, sb_shift=7)]),
    # C3-like: a 30x call, then 270 M bases at 300x in one chunk (more than 2^28 positions, ~4400 records per bucket: split 2),
    # in which most counters cross 255 (k_bigscan2 on a two-level chunk).  Two tables, not C3's four: with four, the 270 M-position
    # chunk holds 60 GB of device memory (measured on a B200), with two about half; the kernels and their loads are the same
    "S3": dict(cls="Countgraph", k=20, n=2, x=2e9, bigcount=True, cutoffs=(100, 256),
               calls=[(103, 300_000, 1_500_000), (104, 1_800_000, 900_000)],
               expect=[dict(path="grouped", levels=2, sb_shift=8, apply="sparse"),
                       dict(path="grouped", levels=2, sb_shift=8, apply="split2", n_pos_min=1 << 28)]),
    # C4-like: 8e9 nibbles per table (bins past 2^32), 270 M positions: ~1100 records per bucket, split 4
    "S4": dict(cls="SmallCountgraph", k=31, n=2, x=8e9, bigcount=False, cutoffs=(2, 3),
               calls=[(105, 1_800_000, 100_000_000)],
               expect=[dict(path="grouped", levels=2, sb_shift=9, apply="split4", n_pos_min=1 << 28)]),
    # C5-like: two calls of 30 M bases (~200 records per bucket: k_hash64 + k_apply_sparse), then 180 M bases at 360x
    # (split 4, counters past 255)
    "S5": dict(cls="Counttable", k=40, n=2, x=5e9, bigcount=True, cutoffs=(100, 256),
               calls=[(106, 200_000, 10_000_000), (107, 200_000, 10_000_000), (108, 1_200_000, 500_000)],
               expect=[dict(path="grouped", levels=2, sb_shift=9, apply="sparse"),
                       dict(path="grouped", levels=2, sb_shift=9, apply="sparse"),
                       dict(path="grouped", levels=2, sb_shift=9, apply="split4", n_pos_min=170_000_000)]),
    # BitStorage on 5e9-bin tables: 4 KB slices in k_apply2, 64-bit bins
    "S6": dict(cls="Nodegraph", k=25, n=2, x=5e9, bigcount=False, cutoffs=(1, 2),
               calls=[(109, 1_200_000, 20_000_000)],
               expect=[dict(path="grouped", levels=2, sb_shift=9, apply="split4", n_pos_min=170_000_000)]),
    # address-sharded, world 3 emulated on one GPU: slices of 4.4e9-bin tables (rank 2 owns bins 2.9e9 to 4.4e9, past 2^32);
    # each call is fed as rounds of SHARD_RUN reads per rank taken in read order, so the rounds' stream order is the reads'
    # order; the second call is one round at 300x in which counters cross 255 from the three senders' k-mers
    "S7": dict(cls="Countgraph", k=20, n=2, x=4.4e9, bigcount=True, cutoffs=(100, 256), world=3,
               calls=[(110, 450_000, 20_000_000), (111, 150_000, 75_000)],
               expect=None),
}
SHARD_RUN = 50_000         # reads per rank and round of S7: 7.5 M bases, within the shards' 8 Mi positions per round
PARAMS = ("cls", "k", "n", "x", "bigcount", "cutoffs", "calls", "world")


def shape_params(sid):
    """what the golden records of a shape's definition (JSON-shaped: lists, not tuples)"""
    s = SHAPES[sid]
    return json.loads(json.dumps({p: s.get(p) for p in PARAMS}))


def call_reads(call):
    seed, n_reads, genome_len = call
    return _batch(seed, n_reads, genome_len)


def _block_stats(a):
    return hashlib.md5(memoryview(a)).hexdigest(), int(np.count_nonzero(a)), int(a.sum(dtype=np.uint64))


def table_record(blocks, pool):
    """blocks: the table image in BLOCK-byte pieces, in order -> md5 per block, md5 of their concatenation, nonzero bytes and
    byte sum.  Blocks are hashed on the pool (hashlib and numpy's reductions release the GIL) while the next is produced."""
    futs = []
    for b in blocks:
        futs.append(pool.submit(_block_stats, b))
        if len(futs) > 8:
            futs[-9].result()   # at most ~2 GB of blocks waiting
    st = [f.result() for f in futs]
    digests = [s[0] for s in st]
    return {"blocks": digests, "digest": hashlib.md5("".join(digests).encode()).hexdigest(),
            "nonzero": sum(s[1] for s in st), "sum": sum(s[2] for s in st)}


def probe_record(med, avg, sd, counts, at_least, cutoffs):
    def h(a, dt):
        return hashlib.md5(np.ascontiguousarray(a, dtype=dt).tobytes()).hexdigest()
    return {"kmer_counts_md5": h(counts, "<u2"), "kmer_counts_sum": int(np.asarray(counts, dtype=np.uint64).sum()),
            "medians_md5": h(med, "<u2"), "medians_sum": int(np.asarray(med, dtype=np.uint64).sum()),
            "averages_md5": h(avg, "<f4"), "deviations_md5": h(sd, "<f4"),
            "median_at_least": {str(c): h(a, "u1") for c, a in zip(cutoffs, at_least)}}


def run_shape(sid, sk, pool, log=None):
    """Feed shape `sid` to `sk` (an adapter: OracleShape, GpuShape or ShardedShape) and record what the golden holds."""
    s = SHAPES[sid]
    out = dict(shape_params(sid), sizes=list(sk.sizes), after_call=[])
    for ci, call in enumerate(s["calls"]):
        buf, off = call_reads(call)
        if log:
            log(ci)
        kmers = sk.consume(buf, off)
        occ, uniq = sk.stats()
        rec = {"kmers": int(kmers), "n_occupied": int(occ), "n_unique_kmers": int(uniq),
               "tables": [table_record(sk.table_blocks(i), pool) for i in range(len(sk.sizes))]}
        if s["bigcount"]:
            keys, vals = sk.bigcount_arrays()
            order = np.argsort(keys, kind="stable")
            rec["bigcounts"] = {"n": int(len(keys)), "md5": bigcount_md5(keys[order], vals[order])}
        out["after_call"].append(rec)
    q = (buf[:N_PROBE * READ_LEN], off[:N_PROBE + 1])
    out["probe"] = sk.probe(q, s["cutoffs"])
    return out


class OracleShape:
    """the oracle port behind run_shape's interface (CPU, single-threaded)"""

    def __init__(self, sid):
        s = SHAPES[sid]
        self.sizes = ol.primes_near_x(s["n"], s["x"])
        self.o = ol.Oracle(s["cls"], s["k"], self.sizes)
        if s["bigcount"]:
            self.o.set_use_bigcount(True)

    def consume(self, buf, off):
        o = self.o
        return o.L.ko_consume_reads(o.h, buf.ctypes.data_as(ol.C.c_char_p), off.ctypes.data_as(ol.u64p), len(off) - 1, 1, 0, 0, 0)

    def stats(self):
        return self.o.n_occupied(), self.o.n_unique_kmers()

    def table_blocks(self, i):
        L, h = self.o.L, self.o.h
        view = np.ctypeslib.as_array(L.ko_table(h, i), shape=(L.ko_table_nbytes(h, i),))
        return (view[lo:lo + BLOCK] for lo in range(0, len(view), BLOCK))

    def bigcount_arrays(self):
        m = self.o.bigcounts()
        return np.array(list(m.keys()), dtype=np.uint64), np.array(list(m.values()), dtype=np.uint16)

    def probe(self, q, cutoffs):
        buf, off = q
        reads = [buf[off[j]:off[j + 1]].tobytes() for j in range(len(off) - 1)]
        med, avg, sd = zip(*(self.o.median(r) for r in reads))
        counts = np.concatenate([self.o.kmer_counts(r) for r in reads])
        al = [[int(self.o.median_at_least(r, c)) for r in reads] for c in cutoffs]
        return probe_record(med, avg, sd, counts, al, cutoffs)


class GpuShape:
    """a cabi.Sketch behind run_shape's interface; tables are downloaded a block at a time"""

    def __init__(self, sid):
        from khmer_b200 import cabi
        self.cabi = cabi
        s = SHAPES[sid]
        kind, hk, _ = ol.CLASSES[s["cls"]]
        self.sizes = ol.primes_near_x(s["n"], s["x"])
        self.g = cabi.Sketch(kind, hk, s["k"], self.sizes)
        if s["bigcount"]:
            self.g.set_use_bigcount(True)

    def consume(self, buf, off):
        return self.g.consume_reads((buf, off), clean=True)

    def stats(self):
        return self.g.stats()

    def table_blocks(self, i):
        n = self.g.table_nbytes(i)
        for lo in range(0, n, BLOCK):
            b = np.empty(min(BLOCK, n - lo), dtype=np.uint8)
            self.cabi.check(self.cabi.lib().kmgpu_download_table(self.g.h, i, self.cabi._ptr(b), lo, len(b)))
            yield b

    def bigcount_arrays(self):
        return self.g.bigcounts()

    def probe(self, q, cutoffs):
        med, avg, sd, nk = self.g.read_medians(q)
        assert (nk == READ_LEN - self.g.ksize + 1).all()
        return probe_record(med, avg, sd, self.g.kmer_counts(q), [self.g.median_at_least(q, c) for c in cutoffs], cutoffs)

    def close(self):
        self.g.close()


class ShardedShape:
    """address-sharded ranks (cabi.Shard, emulated in one process) behind run_shape's interface: a call is fed in rounds of
    SHARD_RUN reads per rank (rank r of round j: reads [(world j + r) SHARD_RUN, ...)), tables are the slices concatenated in
    rank order"""

    def __init__(self, sid):
        from khmer_b200 import cabi
        s = SHAPES[sid]
        kind, hk, _ = ol.CLASSES[s["cls"]]
        self.sizes = ol.primes_near_x(s["n"], s["x"])
        self.shards = [cabi.Shard(kind, hk, s["k"], self.sizes, r, s["world"]) for r in range(s["world"])]
        cabi.attach_local_shards(self.shards)
        for sh in self.shards:
            sh.set_use_bigcount(s["bigcount"])
        self.events = []   # bigcount events per round

    def _rounds(self, off):
        w = len(self.shards)
        n = len(off) - 1
        for j0 in range(0, n, w * SHARD_RUN):
            yield [off[min(n, j0 + r * SHARD_RUN): min(n, j0 + (r + 1) * SHARD_RUN) + 1] for r in range(w)]

    def consume(self, buf, off):
        kmers = 0
        for runs in self._rounds(off):
            for sh, o in zip(self.shards, runs):
                kmers += sh.route((buf, o))
            for step in ("offsets", "push", "apply", "count_new"):
                for sh in self.shards:
                    getattr(sh, step)()
            ev = [sh.bigcount_events() for sh in self.shards]
            hs, cs = np.concatenate([e[0] for e in ev]), np.concatenate([e[1] for e in ev])
            for sh in self.shards:
                sh.bigcount_apply(hs, cs)
            self.events.append(int(cs.sum()))
        return kmers

    def stats(self):
        return sum(sh.stats()[0] for sh in self.shards), sum(sh.stats()[1] for sh in self.shards)

    def table_blocks(self, i):
        pending = []
        for sh in self.shards:
            pending.append(sh.slice_bytes(i))
            while sum(len(p) for p in pending) >= BLOCK:
                cat = np.concatenate(pending)
                yield cat[:BLOCK]
                pending = [cat[BLOCK:]]
        if pending and sum(len(p) for p in pending):
            yield np.concatenate(pending)

    def bigcount_arrays(self):
        k0, v0 = self.shards[0].bigcounts()
        for r, sh in enumerate(self.shards[1:], 1):
            k, v = sh.bigcounts()
            assert np.array_equal(k, k0) and np.array_equal(v, v0), "rank %d holds another bigcount map than rank 0" % r
        return k0, v0

    def probe(self, q, cutoffs):
        buf, off = q
        w, n = len(self.shards), len(off) - 1
        for r, sh in enumerate(self.shards):
            sh.route((buf, off[r * n // w: (r + 1) * n // w + 1]))
        for step in ("offsets", "push", "lookup", "pull"):
            for sh in self.shards:
                getattr(sh, step)()
        med, avg, sd, _ = (np.concatenate(x) for x in zip(*(sh.read_medians() for sh in self.shards)))
        counts = np.concatenate([sh.kmer_counts() for sh in self.shards])
        al = [np.concatenate([sh.median_at_least(c) for sh in self.shards]) for c in cutoffs]
        return probe_record(med, avg, sd, counts, al, cutoffs)

    def close(self):
        for sh in self.shards:
            sh.close()


def load_golden():
    with open(GOLDEN) as fh:
        return json.load(fh)


def table_nbytes(cls, size):
    kind = ol.CLASSES[cls][0]
    return size if kind == ol.BYTE else size // 2 + 1 if kind == ol.NIBBLE else size // 8 + 1


# ---- CPU: the golden matches the shape definitions ---------------------------------------------------------------------
def test_shape_golden_matches_definitions():
    """every shape of shape_golden.json was generated from the current definitions: table sizes are primes_near_x of the
    shape, the calls, classes, k and cutoffs are the ones defined here, and each table has one digest per 256 MiB block"""
    want = load_golden()
    assert want["block_bytes"] == BLOCK and want["probe_reads"] == N_PROBE and want["read_len"] == READ_LEN
    assert sorted(want["shapes"]) == sorted(SHAPES)
    for sid in SHAPES:
        w = want["shapes"][sid]
        assert {p: w[p] for p in PARAMS} == shape_params(sid), sid
        assert w["sizes"] == ol.primes_near_x(SHAPES[sid]["n"], SHAPES[sid]["x"]), sid
        assert len(w["after_call"]) == len(SHAPES[sid]["calls"]), sid
        for rec in w["after_call"]:
            assert [len(t["blocks"]) for t in rec["tables"]] == [-(-table_nbytes(w["cls"], s) // BLOCK) for s in w["sizes"]], sid
            assert ("bigcounts" in rec) == w["bigcount"], sid


# ---- GPU ----------------------------------------------------------------------------------------------------------------
CHUNK_RE = re.compile(r"\[kmgpu\] chunk: path=(\w+) delta_blocks=(\d+) levels=(\d) sb_shift=(\d+) apply=(\S+) n_pos=(\d+)")


def _run_child(sid, env_extra=None):
    env = dict(os.environ, KMGPU_DEBUG="1", **(env_extra or {}))
    r = subprocess.run([sys.executable, os.path.abspath(__file__), sid], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-5000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    calls = []   # per call, the chunk lines it printed
    for line in r.stderr.splitlines():
        if line.startswith("[shape] call "):
            calls.append([])
        m = CHUNK_RE.search(line)
        if m and calls:
            p, blocks, levels, shift, apply, n_pos = m.groups()
            calls[-1].append(dict(path=p, delta_blocks=int(blocks), levels=int(levels), sb_shift=int(shift), apply=apply, n_pos=int(n_pos)))
    print("%s%s: %s" % (sid, " " + str(env_extra) if env_extra else "", got["device"]))
    for ci, ch in enumerate(calls):
        print("  call %d: %d chunks; %s" % (ci, len(ch), ch[0] if len(ch) == 1 else ch))
    return got, calls


def _check_paths(sid, calls):
    s = SHAPES[sid]
    assert len(calls) == len(s["calls"]), "%s: %d calls logged" % (sid, len(calls))
    for ci, (exp, chunks) in enumerate(zip(s["expect"], calls)):
        assert chunks, "%s call %d: no chunk line (KMGPU_DEBUG)" % (sid, ci)
        for ch in chunks:
            for key in ("path", "delta_blocks", "levels", "sb_shift", "apply"):
                if key in exp:
                    assert ch[key] == exp[key], "%s call %d: %s is %r, the shape is meant to reach %r (%s)" % (sid, ci, key, ch[key], exp[key], ch)
        if "chunks" in exp:
            assert len(chunks) == exp["chunks"], "%s call %d: %d chunks" % (sid, ci, len(chunks))
        if "n_pos_min" in exp:
            assert max(c["n_pos"] for c in chunks) >= exp["n_pos_min"], "%s call %d: chunks of %s positions" % (sid, ci, [c["n_pos"] for c in chunks])


def _compare(sid, got):
    want = load_golden()["shapes"][sid]
    assert {p: got[p] for p in PARAMS} == {p: want[p] for p in PARAMS} and got["sizes"] == want["sizes"], sid
    per = {ol.BYTE: 1, ol.NIBBLE: 2, ol.BIT: 8}[ol.CLASSES[want["cls"]][0]]
    for ci, (w, g) in enumerate(zip(want["after_call"], got["after_call"])):
        where = "%s after call %d" % (sid, ci)
        assert g["kmers"] == w["kmers"], where + ": k-mers consumed"
        for i, (wt, gt) in enumerate(zip(w["tables"], g["tables"])):
            bad = [b for b, (x, y) in enumerate(zip(wt["blocks"], gt["blocks"])) if x != y]
            assert not bad and wt["digest"] == gt["digest"], (
                "%s: table %d differs from the reference in block %d (bins [%d, %d)) and %d other blocks; nonzero bytes %d (want %d), "
                "byte sum %d (want %d)" % (where, i, bad[0], bad[0] * BLOCK * per, min(want["sizes"][i], (bad[0] + 1) * BLOCK * per),
                                           len(bad) - 1, gt["nonzero"], wt["nonzero"], gt["sum"], wt["sum"]))
            assert (gt["nonzero"], gt["sum"]) == (wt["nonzero"], wt["sum"]), where
        assert (g["n_occupied"], g["n_unique_kmers"]) == (w["n_occupied"], w["n_unique_kmers"]), where + ": (n_occupied, n_unique_kmers)"
        assert g.get("bigcounts") == w.get("bigcounts"), where + ": bigcount map"
    for key, wv in want["probe"].items():
        assert got["probe"][key] == wv, "%s: probe %s" % (sid, key)


def _shape_test(sid, env_extra=None):
    got, calls = _run_child(sid, env_extra)
    if not env_extra:
        _check_paths(sid, calls)
    _compare(sid, got)


@pytest.mark.gpu
def test_S1_nodegraph_c2_delta_path_two_chunks():
    """C2 (Nodegraph k=32, 4 x 1e9 bits): the delta path at 12 blocks (red.or into L2-sized blocks, k_fold), a call cut into two
    full-size chunks"""
    _shape_test("S1")


@pytest.mark.gpu
def test_S2_smallcountgraph_two_level_planned_shift():
    """SmallCountgraph k=31, 4 x 4e8 nibbles: the two-level grouped path with the super-bucket shift plan_group picks for
    these sizes (7), not a forced one"""
    _shape_test("S2")


@pytest.mark.gpu
def test_S3_countgraph_c3_split2_chunk_past_2_28_crossing_255():
    """C3-like (Countgraph k=20, bigcount, 2 x 2e9 bytes): two levels; a 270 M-position chunk applied by k_apply2 split 2 in which
    counters cross 255 (k_bigscan2 rehashes the two-level chunk); the bigcount map and probe counts above 255"""
    _shape_test("S3")


@pytest.mark.gpu
def test_S4_smallcountgraph_c4_64bit_bins_split4():
    """C4-like (SmallCountgraph k=31, 2 x 8e9 nibbles): bins past 2^32 (64-bit bins in k_part MODE 1, mod_magic with a divisor
    above 2^32) applied by k_apply2 split 4"""
    _shape_test("S4")


@pytest.mark.gpu
def test_S5_counttable_c5_murmur_sparse_then_split4():
    """C5-like (Counttable k=40, MurmurHash3, bigcount, 2 x 5e9 bytes): small calls through k_hash64 + k_apply_sparse on
    64-bit bins, then a large call through k_apply2 split 4 whose counters cross 255"""
    _shape_test("S5")


@pytest.mark.gpu
def test_S6_nodegraph_bit_storage_64bit_bins():
    """Nodegraph k=25, 2 x 5e9 bits: BitStorage on 64-bit bins, 4 KB slices in k_apply2 (split 4)"""
    _shape_test("S6")


@pytest.mark.gpu
def test_S7_sharded_world3_slices_past_2_32_bigcount_across_senders():
    """address-sharded Countgraph k=20 with bigcount, world 3 emulated on one GPU, 2 x 4.4e9 bins: slices of tables past 2^32
    bins (the last rank's ends beyond it); a 300x round in which the three senders' k-mers drive counters past 255; the
    concatenated slices, n_unique_kmers, the bigcount map of every rank and a query round (counts, medians, median_at_least)
    equal the oracle fed the rounds in stream order"""
    got, _ = _run_child("S7")
    s = SHAPES["S7"]
    world, sizes = s["world"], ol.primes_near_x(s["n"], s["x"])
    for i, size in enumerate(sizes):
        assert got["slices"][0][i][0] == 0 and got["slices"][-1][i][1] == size
        assert all(got["slices"][r][i][1] == got["slices"][r + 1][i][0] for r in range(world - 1))
        assert got["slices"][-1][i][0] < 1 << 32 < got["slices"][-1][i][1], "the last rank's slice is meant to cross 2^32 bins"
    assert got["round_events"][-1] > 0, "the 300x round is meant to bring k-mers whose counters are all 255"
    _compare("S7", got)


@pytest.mark.gpu
@pytest.mark.parametrize("sid", ["S2", "S6"])
def test_chunking_does_not_change_answers(sid):
    """S2 and S6 with 16 Mi-base chunks instead of the default, which for two-level shapes depends on the device memory free
    at the time: the same golden"""
    _shape_test(sid, {"KMGPU_CHUNK_BASES": str(1 << 24)})


def _device_main(sid):
    import torch
    s = SHAPES[sid]
    free0, total = torch.cuda.mem_get_info(0)
    sizes = ol.primes_near_x(s["n"], s["x"])
    tables = sum(table_nbytes(s["cls"], x) for x in sizes)
    # sketch_chunk_bases: chunks of two-level sketches grow to what half of the free memory holds at (21 x tables + 16) B a position
    need = tables + 2 * (21 * s["n"] + 16) * max(n * READ_LEN for _, n, _ in s["calls"])
    if "KMGPU_CHUNK_BASES" not in os.environ and s["expect"] and s["expect"][0]["path"] == "grouped" and free0 < need:
        raise SystemExit("%s needs %.1f GB of free device memory for its chunks to cover its calls; %.1f GB are free" % (sid, need / 1e9, free0 / 1e9))
    peak = [0]

    def log(ci):
        peak[0] = max(peak[0], free0 - torch.cuda.mem_get_info(0)[0])
        print("[shape] call %d" % ci, file=sys.stderr, flush=True)

    sk = ShardedShape(sid) if s.get("world") else GpuShape(sid)
    with concurrent.futures.ThreadPoolExecutor(8) as pool:
        out = run_shape(sid, sk, pool, log)
    peak[0] = max(peak[0], free0 - torch.cuda.mem_get_info(0)[0])
    if s.get("world"):
        out["slices"] = [[list(sh.slice(i)) for i in range(s["n"])] for sh in sk.shards]
        out["round_events"] = sk.events
    sk.close()
    out["device"] = "%s, %.1f GB held by the sketch at most (sampled between calls)" % (torch.cuda.get_device_name(0), peak[0] / 1e9)
    print(json.dumps(out))


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _device_main(sys.argv[1])
