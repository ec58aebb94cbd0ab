"""Query rounds on address-sharded sketches (route | offsets | push | lookup | pull): per-k-mer counts, medians, median_at_least,
trimming and the abundance histogram equal a single sketch fed the same reads and the oracle.  Ranks are emulated in one process
on one GPU (peer pointers are then ordinary device pointers); with >= 2 GPUs the one-process-per-GPU form runs as well."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
from common import synth_reads

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAXPOS = 20000
EMPTY = (np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64))


def _sizes(world):
    return ol.primes_near_x(4, 70000) if world < 8 else [1009, 997, 991, 64]     # tiny tables: some ranks own nothing


def _runs(reads, world):
    """per rank: its reads (shard_range) as the runs of its rounds, and the index of its first read"""
    from khmer_b200 import cabi
    from khmer_b200.multigpu import shard_range, split_by_bases
    out = []
    for r in range(world):
        lo, hi = shard_range(len(reads), r, world)
        buf, off = cabi.as_reads(reads[lo:hi])
        out.append([(buf, off[a:b + 1]) for a, b in split_by_bases(buf, off, MAXPOS)])
    return out


def _round(shards, runs, i, clean, query):
    for s, rr in zip(shards, runs):
        s.route(rr[i] if i < len(rr) else EMPTY, clean=clean)
    for s in shards:
        s.offsets()
    for s in shards:
        s.push()
    for s in shards:
        s.lookup() if query else s.apply()
    for s in shards:
        s.pull() if query else s.count_new()


def _ingest(shards, reads):
    runs = _runs(reads, len(shards))
    for i in range(max(len(rr) for rr in runs)):
        _round(shards, runs, i, True, False)


def _query(shards, reads, clean):
    """every getter over the query reads, concatenated in read order (rank 0's reads first)"""
    runs = _runs(reads, len(shards))
    got = {"counts": [], "med": [], "avg": [], "sd": [], "nk": [], "trim": []}
    parts = [[] for _ in shards]
    for i in range(max(len(rr) for rr in runs)):
        _round(shards, runs, i, clean, True)
        for r, s in enumerate(shards):
            m, a, sd, nk = s.read_medians()
            one = {"counts": s.kmer_counts(), "med": m, "avg": a, "sd": sd, "nk": nk}
            for c in (1, 2, 20, 255):
                one["al%d" % c] = s.median_at_least(c)
            for ab in (2, 3):
                for below in (False, True):
                    one["tr%d%d" % (ab, below)] = s.trim(ab, below)
            parts[r].append(one)
    out = {}
    for key in parts[0][0]:
        out[key] = np.concatenate([p[key] for pr in parts for p in pr])
    return out


def _query_reads(seed, k, murmur_unclean):
    q = synth_reads(seed, 300, 130, 6000, err=0.01, with_n=True)      # same genome as the ingested reads
    q += synth_reads(seed + 1000, 100, 120, 5000)                        # k-mers never seen
    q += ["", "ACG", "A" * (k - 1), "A" * k, "A" * 300, "A" * 300, "ACGTNACGTACGTTTGCA" * 10, "G" * 90]
    if murmur_unclean:      # the Murmur hash of an uncleaned sequence holding N is not computed (KMGPU_ENONACGT)
        q = [r for r in q if "N" not in r]
    return q


def _check_queries(shards, single, o, reads, clean, k):
    got = _query(shards, reads, clean)
    want_counts = single.kmer_counts(reads, clean=clean)
    assert np.array_equal(got["counts"], want_counts)
    seqs = [ol.clean(r) for r in reads] if clean else reads
    assert np.array_equal(got["counts"], np.concatenate([o.kmer_counts(s) for s in seqs] + [np.zeros(0, np.uint16)]))
    med, avg, sd, nk = single.read_medians(reads, clean=clean)
    for key, want in (("med", med), ("avg", avg), ("sd", sd), ("nk", nk)):
        assert np.array_equal(got[key].view(np.uint8), want.view(np.uint8)), key     # bit for bit
    for j, s in enumerate(seqs):
        if len(s) >= k:
            assert (int(got["med"][j]), float(got["avg"][j]), float(got["sd"][j])) == o.median(s), j
        else:
            assert got["nk"][j] == 0
    for c in (1, 2, 20, 255):
        assert np.array_equal(got["al%d" % c], single.median_at_least(reads, c, clean=clean)), c
    for ab in (2, 3):
        for below in (False, True):
            assert np.array_equal(got["tr%d%d" % (ab, below)], single.trim_batch(reads, ab, below=below, clean=clean)), (ab, below)


def _state(shards):
    return [(s.stats()[:2], [s.slice_bytes(i).copy() for i in range(4)]) for s in shards]


def _same_state(a, b):
    return all(x[0] == y[0] and all(np.array_equal(p, q) for p, q in zip(x[1], y[1])) for x, y in zip(a, b))


@pytest.mark.parametrize("cls,k", [("Countgraph", 20), ("SmallCountgraph", 17), ("Nodegraph", 31), ("Counttable", 40),
                                   ("SmallCounttable", 33), ("Nodetable", 21)])
@pytest.mark.parametrize("world", [1, 3, 8])
def test_sharded_queries_equal_single_sketch(cls, k, world):
    from khmer_b200 import cabi
    kind, hk, _ = ol.CLASSES[cls]
    sizes = _sizes(world)
    seed = world * 7 + k
    reads = synth_reads(seed, 900, 130, 6000, err=0.01, with_n=True) + ["A" * 300] * 40 + ["", "ACG"]
    shards = [cabi.Shard(kind, hk, k, sizes, r, world, max_positions=MAXPOS) for r in range(world)]
    cabi.attach_local_shards(shards)
    single = cabi.Sketch(kind, hk, k, sizes)
    o = ol.Oracle(cls, k, sizes)
    for half in (reads[: len(reads) // 2], reads[len(reads) // 2:]):       # ingest -> query -> ingest -> query
        _ingest(shards, half)
        single.consume_reads(half)
        o.consume_reads(half)
        before = _state(shards)
        for clean in (True, False):
            _check_queries(shards, single, o, _query_reads(seed, k, hk == cabi.MURMUR and not clean), clean, k)
        assert _same_state(before, _state(shards)), "a query round changed the sketch"
    # the tables are still those of one sketch (the queries left nothing behind)
    for i in range(4):
        assert np.array_equal(np.concatenate([s.slice_bytes(i) for s in shards]), single.table(i)), i
    for s in shards:
        s.close()


@pytest.mark.parametrize("cls,k,track", [("Countgraph", 20, "Nodegraph"), ("SmallCountgraph", 31, "Nodegraph"),
                                         ("Counttable", 40, "Nodetable")])
@pytest.mark.parametrize("world", [1, 3, 8])
def test_sharded_abundance_distribution(cls, k, track, world):
    from khmer_b200 import cabi
    kind, hk, _ = ol.CLASSES[cls]
    sizes = _sizes(world)
    reads = synth_reads(world + k, 1200, 140, 8000, err=0.01, with_n=True) + ["A" * 300] * 30 + ["", "AC"]
    counts = [cabi.Shard(kind, hk, k, sizes, r, world, max_positions=MAXPOS) for r in range(world)]
    tracking = [cabi.Shard(cabi.BIT, hk, k, sizes, r, world, max_positions=MAXPOS) for r in range(world)]
    cabi.attach_local_shards(counts)
    cabi.attach_local_shards(tracking)
    _ingest(counts, reads)
    o = ol.Oracle(cls, k, sizes)
    o.consume_reads(reads)
    ot = ol.Oracle(track, k, sizes)
    runs = _runs(reads, world)
    hist = np.zeros(65536, dtype=np.uint64)
    want = np.zeros(65536, dtype=np.uint64)
    for i in range(max(len(rr) for rr in runs)):
        _round(tracking, runs, i, True, False)
        _round(counts, runs, i, True, True)
        for c, t in zip(counts, tracking):
            cabi.shard_abundance_hist(c, t, hist)
        for rr in runs:                           # the stream order of the round: run i of rank 0, of rank 1, ...
            if i < len(rr):
                buf, off = rr[i]
                part = [bytes(buf[off[j]:off[j + 1]]).decode() for j in range(len(off) - 1)]
                want += o.abundance_distribution(part, ot)
    assert np.array_equal(hist, want)
    assert hist.sum() == sum(t.stats()[1] for t in tracking)
    for s in counts + tracking:
        s.close()


def test_shard_query_calls_are_refused_out_of_order():
    from khmer_b200 import cabi
    sizes = _sizes(2)
    a = [cabi.Shard(cabi.BYTE, cabi.TWOBIT, 20, sizes, r, 2, max_positions=MAXPOS) for r in range(2)]
    b = [cabi.Shard(cabi.BIT, cabi.TWOBIT, 20, sizes, r, 2, max_positions=MAXPOS) for r in range(2)]
    m = [cabi.Shard(cabi.BIT, cabi.MURMUR, 20, sizes, r, 2, max_positions=MAXPOS) for r in range(2)]
    other = [cabi.Shard(cabi.BIT, cabi.TWOBIT, 20, sizes, r, 2, max_positions=2 * MAXPOS) for r in range(2)]
    for g in (a, b, m, other):
        cabi.attach_local_shards(g)
    reads = synth_reads(3, 50, 100, 2000)
    runs = [[cabi.as_reads(reads[:20])], [cabi.as_reads(reads[20:])]]
    with pytest.raises(cabi.KmgpuError, match="pulled"):
        a[0].read_medians()                       # nothing routed and answered yet
    _round(a, runs, 0, True, True)
    _round(b, runs, 0, True, False)
    _round(other, runs, 0, True, False)
    _round(m, runs, 0, True, False)
    assert len(a[0].read_medians()[0]) == 20
    with pytest.raises(cabi.KmgpuError) as e:
        cabi.shard_abundance_hist(a[0], other[0])
    assert e.value.code == 1 and "max_positions" in str(e.value)
    with pytest.raises(cabi.KmgpuError) as e:
        cabi.shard_abundance_hist(a[0], m[0])
    assert e.value.code == 1
    with pytest.raises(cabi.KmgpuError) as e:
        cabi.shard_abundance_hist(a[0], b[1])     # b[1] routed rank 1's reads
    assert e.value.code == 1 and "different reads" in str(e.value)
    assert cabi.shard_abundance_hist(a[0], b[0]).sum() > 0
    _round(b, runs, 0, True, True)                # a query round leaves no new positions behind to count
    with pytest.raises(cabi.KmgpuError) as e:
        cabi.shard_abundance_hist(a[0], b[0])
    assert e.value.code == 1
    with pytest.raises(cabi.KmgpuError) as e:     # Murmur without cleaning: a byte outside ACGT is refused
        m[0].route(cabi.as_reads(["ACGTNACGTACGTACGTACGTACGT"]), clean=False)
    assert e.value.code == 5
    for s in a + b + m + other:
        s.close()


def test_sharded_group_queries_world1():
    """ShardedGroup's collective calls on one rank: the rounds of consume_reads, answers in read order"""
    from khmer_b200 import cabi
    from khmer_b200.multigpu import ShardedGroup
    sizes = _sizes(1)
    reads = synth_reads(11, 700, 130, 6000, err=0.01) + ["A" * 300] * 20 + ["", "ACG"]
    g = ShardedGroup(cabi.Shard(cabi.BYTE, cabi.TWOBIT, 20, sizes, 0, 1, max_positions=MAXPOS))
    t = ShardedGroup(cabi.Shard(cabi.BIT, cabi.TWOBIT, 20, sizes, 0, 1, max_positions=MAXPOS))
    g.attach()
    t.attach()
    g.consume_reads(reads)
    single = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, 20, sizes)
    single.consume_reads(reads)
    q = reads[::3] + synth_reads(12, 100, 120, 5000)
    assert np.array_equal(g.kmer_counts(q), single.kmer_counts(q))
    for x, y in zip(g.read_medians(q), single.read_medians(q)):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert np.array_equal(g.median_at_least(q, 3), single.median_at_least(q, 3))
    assert np.array_equal(g.trim(q, 2, below=True), single.trim_batch(q, 2, below=True))
    assert all(len(x) == 0 for x in g.read_medians([]))
    tr = cabi.Sketch(cabi.BIT, cabi.TWOBIT, 20, sizes)
    assert np.array_equal(g.abundance_distribution(t, reads), single.abundance_distribution(reads, tr))


REFUSE = r'''
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np
from khmer_b200 import cabi
import oracle_lib as ol
from common import synth_reads
sizes = ol.primes_near_x(4, 3000000)
shards = [cabi.Shard(cabi.BYTE, cabi.TWOBIT, 20, sizes, r, 2, max_positions=200000) for r in range(2)]
cabi.attach_local_shards(shards)
big = synth_reads(1, 1000, 150, 40000)
small = synth_reads(2, 3, 150, 40000)
def round_(reads_by_rank, query):
    errs = []
    for r in range(2):
        shards[r].route(cabi.as_reads(reads_by_rank[r]))
    for r in range(2):
        shards[r].offsets()
    for r in range(2):
        shards[r].push()
    for step in ("lookup", "pull") if query else ("apply", "count_new"):
        for r in range(2):
            try:
                getattr(shards[r], step)()
            except cabi.KmgpuError as e:
                assert "arena" in str(e) and e.code == 4, str(e)
                errs.append((step, r))
    return errs
assert round_([small, small], False) == []
state = [(s.stats()[:2], [s.slice_bytes(i).copy() for i in range(4)]) for s in shards]
# 2 x 131 k k-mers x 4 tables against arenas of 20000 records: both owners refuse to answer, both senders get no counts
assert round_([big, big], True) == [("lookup", 0), ("lookup", 1), ("pull", 0), ("pull", 1)]
try:
    shards[0].read_medians()
    raise AssertionError("a refused round has no counts")
except cabi.KmgpuError as e:
    assert e.code == 1
assert round_([small, small], True) == []     # the next round is exact
single = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, 20, sizes)
single.consume_reads(small); single.consume_reads(small)
for r in range(2):
    for x, y in zip(shards[r].read_medians(), single.read_medians(small)):
        assert np.array_equal(x, y)
    assert np.array_equal(shards[r].kmer_counts(), single.kmer_counts(small))
assert all(a[0] == b[0] and all(np.array_equal(p, q) for p, q in zip(a[1], b[1]))
           for a, b in zip(state, [(s.stats()[:2], [s.slice_bytes(i) for i in range(4)]) for s in shards]))
print("REFUSE-OK")
'''


def test_sharded_query_round_larger_than_the_arena_is_refused(tmp_path):
    script = tmp_path / "refuse.py"
    script.write_text(REFUSE % {"root": ROOT})
    r = subprocess.run([sys.executable, str(script)], env=dict(os.environ, KMGPU_SHARD_ARENA="20000"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "REFUSE-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np, torch, torch.distributed as dist
from khmer_b200 import cabi
from khmer_b200.multigpu import ShardedGroup, shard_range, split_by_bases
import oracle_lib as ol
from common import synth_reads
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
sizes = ol.primes_near_x(4, 3000000)
reads = synth_reads(5, 6000, 150, 40000) + ["AC" * 100] * 300 + ["", "ACG"]
lo, hi = shard_range(len(reads), rank, world)
for cls, k, track in (("Countgraph", 20, "Nodegraph"), ("Counttable", 40, "Nodetable")):
    kind, hk, _ = ol.CLASSES[cls]
    g = ShardedGroup(cabi.Shard(kind, hk, k, sizes, rank, world, device=rank, max_positions=200000), dist, device=dev)
    t = ShardedGroup(cabi.Shard(cabi.BIT, hk, k, sizes, rank, world, device=rank, max_positions=200000), dist, device=dev)
    g.attach()
    t.attach()
    g.consume_reads(reads[lo:hi])
    o = ol.Oracle(cls, k, sizes)
    o.consume_reads(reads)
    med, avg, sd, nk = g.read_medians(reads[lo:hi])
    for j, r in enumerate(reads[lo:hi]):
        if len(r) >= k:
            assert (int(med[j]), float(avg[j]), float(sd[j])) == o.median(r), (cls, rank, j)
        else:
            assert nk[j] == 0
    hist = g.abundance_distribution(t, reads[lo:hi])
    ot = ol.Oracle(track, k, sizes)
    runs = []
    for r in range(world):
        a, b = shard_range(len(reads), r, world)
        buf, off = cabi.as_reads(reads[a:b])
        runs.append([(a + x, a + y) for x, y in split_by_bases(buf, off, 200000)])
    want = np.zeros(65536, dtype=np.uint64)
    for i in range(max(len(x) for x in runs)):
        for r in range(world):
            if i < len(runs[r]):
                want += o.abundance_distribution(reads[runs[r][i][0]:runs[r][i][1]], ot)
    assert np.array_equal(hist, want), cls
    dist.barrier()
    g.shard.close()
    t.shard.close()
if rank == 0:
    print("SHARDED-QUERY-IPC-OK")
dist.destroy_process_group()
'''


def test_sharded_queries_one_process_per_gpu(tmp_path):
    from khmer_b200 import cabi
    if cabi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT})
    n = min(cabi.device_count(), 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr",
                        "127.0.0.1", "--master-port", "29631", str(script)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "SHARDED-QUERY-IPC-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
