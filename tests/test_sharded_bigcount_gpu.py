"""Bigcount on address-sharded sketches: owners mark the touches that found their byte at 255 (kmgpu_shard_apply), senders list
their k-mers whose N bytes were all saturated (kmgpu_shard_bigcount_events), every rank applies all ranks' lists in rank order
(kmgpu_shard_bigcount_apply).  Tables, counters and the bigcount map — its entries, values and iteration order — equal ONE sketch
fed the rounds in stream order, and the oracle.  Ranks are emulated in one process on one GPU, as in test_sharded_query_gpu.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
from common import synth_reads

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAXPOS = 8192
EMPTY = (np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64))


def _sizes(world):
    return ol.primes_near_x(4, 70000) if world < 8 else [1009, 997, 991, 64]     # tiny tables: almost everything saturates


def _reads(seed):
    """a background that stays below 255, a 150-base genome read ~500 times over (its k-mers cross 255 in the middle of the
    stream) and "A" * 300 repeated past 65535 events; shuffled so that every rank and round holds some of each"""
    reads = synth_reads(seed, 500, 130, 4000, err=0.005)
    reads += synth_reads(seed + 1, 800, 100, 150)
    reads += ["A" * 300] * 260 + ["", "ACG"]
    order = np.random.default_rng(seed).permutation(len(reads))
    return [reads[i] for i in order]


def _runs(reads, world):
    from khmer_b200 import cabi
    from khmer_b200.multigpu import shard_range, split_by_bases
    out = []
    for r in range(world):
        lo, hi = shard_range(len(reads), r, world)
        buf, off = cabi.as_reads(reads[lo:hi])
        out.append([(buf, off[a:b + 1]) for a, b in split_by_bases(buf, off, MAXPOS)])
    return out


def _round(shards, runs, i, query=False):
    for s, rr in zip(shards, runs):
        s.route(rr[i] if i < len(rr) else EMPTY)
    for s in shards:
        s.offsets()
    for s in shards:
        s.push()
    for s in shards:
        s.lookup() if query else s.apply()
    for s in shards:
        s.pull() if query else s.count_new()
    if not query and shards[0].get_use_bigcount():
        ev = [s.bigcount_events() for s in shards]
        hs, cs = np.concatenate([e[0] for e in ev]), np.concatenate([e[1] for e in ev])
        for s in shards:
            s.bigcount_apply(hs, cs)
        return sum(len(e[0]) for e in ev)
    return 0


def _stream(runs, i):
    """the reads of round i in stream order: run i of rank 0, of rank 1, ..."""
    return [[bytes(buf[off[j]:off[j + 1]]).decode() for j in range(len(off) - 1)] for rr in runs if i < len(rr) for buf, off in [rr[i]]]


def _feed(shards, single, o, runs, i):
    """round i on the shards; the same reads, in stream order, into the single sketch and the oracle"""
    n = _round(shards, runs, i)
    for part in _stream(runs, i):
        single.consume_reads(part)
        o.consume_reads(part)
    return n


def _check_state(shards, single, o):
    for i in range(4):
        cat = np.concatenate([s.slice_bytes(i) for s in shards])
        assert np.array_equal(cat, single.table(i)), i
        assert np.array_equal(cat, o.table(i)), i
    occ = sum(s.stats()[0] for s in shards)
    uniq = sum(s.stats()[1] for s in shards)
    assert (occ, uniq) == single.stats() == (o.n_occupied(), o.n_unique_kmers())
    want_k, want_v = single.bigcounts()
    for r, s in enumerate(shards):
        k, v = s.bigcounts()
        assert np.array_equal(k, want_k) and np.array_equal(v, want_v), "rank %d: map differs (in order) from the single sketch's" % r
    assert dict(zip(want_k.tolist(), want_v.tolist())) == o.bigcounts()
    return want_k, want_v


def _make(cls, k, world, big=True):
    from khmer_b200 import cabi
    kind, hk, _ = ol.CLASSES[cls]
    sizes = _sizes(world)
    shards = [cabi.Shard(kind, hk, k, sizes, r, world, max_positions=MAXPOS) for r in range(world)]
    cabi.attach_local_shards(shards)
    single = cabi.Sketch(kind, hk, k, sizes)
    o = ol.Oracle(cls, k, sizes)
    for x in shards + [single, o]:
        x.set_use_bigcount(big)
    return shards, single, o


@pytest.mark.parametrize("cls,k", [("Countgraph", 20), ("Counttable", 40)])
@pytest.mark.parametrize("world", [1, 3, 8])
def test_sharded_bigcount_ingest_equals_single_sketch(cls, k, world):
    shards, single, o = _make(cls, k, world)
    reads = _reads(world * 5 + k)
    runs = _runs(reads, world)
    n_rounds = max(len(rr) for rr in runs)
    assert n_rounds >= 4
    with_events = 0
    for i in range(n_rounds):
        with_events += _feed(shards, single, o, runs, i) > 0
    assert with_events >= 2
    keys, vals = _check_state(shards, single, o)
    assert len(keys) > 10 and vals.max() == 65535 and (vals < 65535).any()
    for s in shards:
        s.close()


def _check_queries(shards, single, o, reads, k):
    runs = _runs(reads, len(shards))
    got = {}
    for i in range(max(len(rr) for rr in runs)):
        _round(shards, runs, i, query=True)
        for s in shards:
            m, a, sd, nk = s.read_medians()
            one = {"counts": s.kmer_counts(), "med": m, "avg": a, "sd": sd, "nk": nk}
            for c in (20, 255, 300, 1000):
                one["al%d" % c] = s.median_at_least(c)
            for ab in (2, 300):
                for below in (False, True):
                    one["tr%d%d" % (ab, below)] = s.trim(ab, below)
            got.setdefault(s.rank, []).append(one)
    cat = {key: np.concatenate([p[key] for r in sorted(got) for p in got[r]]) for key in got[0][0]}
    assert np.array_equal(cat["counts"], single.kmer_counts(reads))
    assert cat["counts"].max() == 65535 and ((cat["counts"] > 255) & (cat["counts"] < 65535)).any()
    seqs = [ol.clean(r) for r in reads]
    assert np.array_equal(cat["counts"], np.concatenate([o.kmer_counts(s) for s in seqs] + [np.zeros(0, np.uint16)]))
    for key, want in zip(("med", "avg", "sd", "nk"), single.read_medians(reads)):
        assert np.array_equal(cat[key].view(np.uint8), want.view(np.uint8)), key     # bit for bit
    for j, s in enumerate(seqs):
        if len(s) >= k:
            assert (int(cat["med"][j]), float(cat["avg"][j]), float(cat["sd"][j])) == o.median(s), j
    for c in (20, 255, 300, 1000):
        assert np.array_equal(cat["al%d" % c], single.median_at_least(reads, c)), c
    for ab in (2, 300):
        for below in (False, True):
            assert np.array_equal(cat["tr%d%d" % (ab, below)], single.trim_batch(reads, ab, below=below)), (ab, below)


@pytest.mark.parametrize("cls,k,track", [("Countgraph", 20, "Nodegraph"), ("Counttable", 40, "Nodetable")])
@pytest.mark.parametrize("world", [1, 3])
def test_sharded_bigcount_queries(cls, k, track, world):
    from khmer_b200 import cabi
    shards, single, o = _make(cls, k, world)
    reads = _reads(world + k)
    runs = _runs(reads, world)
    for i in range(max(len(rr) for rr in runs)):
        _feed(shards, single, o, runs, i)
    before = [(s.stats()[:2], [s.slice_bytes(i).copy() for i in range(4)], s.bigcounts()) for s in shards]
    q = reads[::4] + ["A" * 300, "A" * 40] + synth_reads(99, 50, 120, 5000)
    _check_queries(shards, single, o, q, k)
    after = [(s.stats()[:2], [s.slice_bytes(i) for i in range(4)], s.bigcounts()) for s in shards]
    for x, y in zip(before, after):
        assert x[0] == y[0] and all(np.array_equal(p, q) for p, q in zip(x[1], y[1]))
        assert np.array_equal(x[2][0], y[2][0]) and np.array_equal(x[2][1], y[2][1]), "a query round changed the map"
    # the abundance histogram, bins above 255 included
    kind, hk, _ = ol.CLASSES[cls]
    tracking = [cabi.Shard(cabi.BIT, hk, k, _sizes(world), r, world, max_positions=MAXPOS) for r in range(world)]
    cabi.attach_local_shards(tracking)
    qruns = _runs(q, world)
    hist = np.zeros(65536, dtype=np.uint64)
    for i in range(max(len(rr) for rr in qruns)):
        _round(tracking, qruns, i)
        _round(shards, qruns, i, query=True)
        for c, t in zip(shards, tracking):
            cabi.shard_abundance_hist(c, t, hist)
    tr = cabi.Sketch(cabi.BIT, hk, k, _sizes(world))
    ot = ol.Oracle(track, k, _sizes(world))
    want = np.zeros(65536, dtype=np.uint64)
    want_single = np.zeros(65536, dtype=np.uint64)
    for i in range(max(len(rr) for rr in qruns)):
        for part in _stream(qruns, i):
            want += o.abundance_distribution(part, ot)
            want_single += single.abundance_distribution(part, tr)
    assert np.array_equal(hist, want)
    assert np.array_equal(hist, want_single)
    assert hist[256:].sum() > 0 and hist[65535] > 0
    for s in shards + tracking:
        s.close()


def test_sharded_bigcount_switched_on_between_rounds():
    shards, single, o = _make("Countgraph", 20, 3, big=False)
    reads = _reads(31)
    runs = _runs(reads, 3)
    n_rounds = max(len(rr) for rr in runs)
    for i in range(n_rounds):
        if i == n_rounds // 2:      # the single sketch and the oracle take the same switch at the same point of the stream
            for x in shards + [single, o]:
                x.set_use_bigcount(True)
        _feed(shards, single, o, runs, i)
        if i < n_rounds // 2:
            assert all(len(s.bigcounts()[0]) == 0 for s in shards)
    keys, _ = _check_state(shards, single, o)
    assert len(keys) > 0
    for s in shards:
        s.close()


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
single = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, 20, sizes)
for x in shards + [single]:
    x.set_use_bigcount(True)
small = ["A" * 300] * 4
big = synth_reads(1, 1000, 150, 40000)
def round_(reads_by_rank):
    errs = []
    for r in range(2):
        shards[r].route(cabi.as_reads(reads_by_rank[r]))
    for r in range(2):
        shards[r].offsets()
    for r in range(2):
        shards[r].push()
    for step in ("apply", "count_new", "bigcount_events"):
        for r in range(2):
            try:
                getattr(shards[r], step)()
            except cabi.KmgpuError as e:
                assert "arena" in str(e) and e.code == 4, str(e)
                errs.append((step, r))
    return errs
def events_apply():
    ev = [s.bigcount_events() for s in shards]
    for s in shards:
        s.bigcount_apply(np.concatenate([e[0] for e in ev]), np.concatenate([e[1] for e in ev]))
assert round_([small, small]) == []
events_apply()
single.consume_reads(small); single.consume_reads(small)
maps = [s.bigcounts() for s in shards]
assert len(maps[0][0]) == 1
# 2 x 131 k k-mers x 4 tables against arenas of 20000 records: both owners refuse, both senders get no events
assert round_([big, big]) == [("apply", 0), ("apply", 1), ("bigcount_events", 0), ("bigcount_events", 1)]
for s, m in zip(shards, maps):
    k, v = s.bigcounts()
    assert np.array_equal(k, m[0]) and np.array_equal(v, m[1])
# a sender that sent the refusing owner nothing still gets its (empty) list
assert round_([small, small]) == []
events_apply()
single.consume_reads(small); single.consume_reads(small)
for s in shards:
    for a, b in zip(s.bigcounts(), single.bigcounts()):
        assert np.array_equal(a, b)
print("REFUSE-OK")
'''


def test_sharded_bigcount_refused_round_leaves_the_map(tmp_path):
    script = tmp_path / "refuse.py"
    script.write_text(REFUSE % {"root": ROOT})
    r = subprocess.run([sys.executable, str(script)], env=dict(os.environ, KMGPU_SHARD_ARENA="20000"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "REFUSE-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_sharded_group_bigcount_world1():
    """ShardedGroup with bigcount on, one rank: the events of every round reach the map"""
    from khmer_b200 import cabi
    from khmer_b200.multigpu import ShardedGroup
    sizes = _sizes(1)
    reads = _reads(7)
    g = ShardedGroup(cabi.Shard(cabi.BYTE, cabi.TWOBIT, 20, sizes, 0, 1, max_positions=MAXPOS))
    g.attach()
    g.set_use_bigcount(True)
    g.consume_reads(reads)
    single = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, 20, sizes)
    single.set_use_bigcount(True)
    for run in g._runs(reads):
        single.consume_reads(run)
    for a, b in zip(g.bigcounts(), single.bigcounts()):
        assert np.array_equal(a, b)
    q = reads[::5]
    assert np.array_equal(g.kmer_counts(q), single.kmer_counts(q))
    g.shard.close()


WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np, torch, torch.distributed as dist
from khmer_b200 import cabi
from khmer_b200.multigpu import ShardedGroup, shard_range
import oracle_lib as ol
from common import synth_reads
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
sizes = ol.primes_near_x(4, 3000000)
reads = synth_reads(5, 4000, 150, 40000) + synth_reads(6, 1500, 100, 150) + ["A" * 300] * 260
reads = [reads[i] for i in np.random.default_rng(3).permutation(len(reads))]
lo, hi = shard_range(len(reads), rank, world)
for cls, k in (("Countgraph", 20), ("Counttable", 40)):
    kind, hk, _ = ol.CLASSES[cls]
    g = ShardedGroup(cabi.Shard(kind, hk, k, sizes, rank, world, device=rank, max_positions=50000), dist, device=dev)
    g.attach()
    g.set_use_bigcount(True)
    g.consume_reads(reads[lo:hi])
    o = ol.Oracle(cls, k, sizes)
    o.set_use_bigcount(True)
    o.consume_reads(reads)
    keys, vals = g.bigcounts()
    assert dict(zip(keys.tolist(), vals.tolist())) == o.bigcounts(), (cls, rank)
    mine = keys.tobytes() + vals.tobytes()
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    assert all(p == parts[0] for p in parts), (cls, "the ranks' maps differ")
    dist.barrier()
    g.shard.close()
if rank == 0:
    print("SHARDED-BIGCOUNT-IPC-OK")
dist.destroy_process_group()
'''


def test_sharded_bigcount_one_process_per_gpu(tmp_path):
    from khmer_b200 import cabi
    if cabi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT})
    n = min(cabi.device_count(), 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr",
                        "127.0.0.1", "--master-port", "29641", str(script)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "SHARDED-BIGCOUNT-IPC-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
