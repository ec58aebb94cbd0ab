"""Host-side protocol of query rounds on address-sharded sketches, without a GPU: a stub shard, world 2 over SocketComm.
A query round is route | offsets | push | lookup | pull, every phase finished on all ranks before the next starts."""
import os
import sys

import numpy as np
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class StubShard:
    """Logs the phases ShardedGroup asks for; its getters answer with the lengths of the reads of the last route."""

    def __init__(self, rank, log, max_positions, name="counts"):
        self.rank, self.log, self.max_positions, self.name = rank, log, max_positions, name
        self.routed = []
        self.off = np.zeros(1, dtype=np.uint64)

    def _w(self, what):
        with open(self.log, "a") as fh:
            fh.write("%d %s %s\n" % (self.rank, self.name, what))

    def ipc_export(self):
        return np.full(64 * 5, self.rank + 1, dtype=np.uint8)

    def ipc_attach(self, handles):
        pass

    def route(self, reads, clean=True):
        buf, off = reads
        self.off = np.asarray(off, dtype=np.uint64)
        self.routed.append(len(off) - 1)
        self._w("route")
        return int(off[-1] - off[0])

    def offsets(self):
        self._w("offsets")

    def push(self):
        self._w("push")

    def apply(self):
        self._w("apply")

    def count_new(self):
        self._w("count_new")

    def lookup(self):
        self._w("lookup")

    def pull(self):
        self._w("pull")

    def _lens(self):
        return (self.off[1:] - self.off[:-1]).astype(np.int64)

    def kmer_counts(self):
        return np.concatenate([np.full(max(n - 3, 0), n, dtype=np.uint16) for n in self._lens()] + [np.zeros(0, np.uint16)])

    def read_medians(self):
        n = self._lens()
        return n.astype(np.uint16), n.astype(np.float32), np.zeros(len(n), np.float32), n.astype(np.uint32)

    def median_at_least(self, cutoff):
        return (self._lens() >= cutoff).astype(np.uint8)

    def trim(self, abund, below=False):
        return np.minimum(self._lens(), abund).astype(np.uint32)


def _worker(rank, world, port, log, out):
    from khmer_b200 import cabi
    from khmer_b200.multigpu import ShardedGroup, SocketComm

    def fake_hist(counts, tracking, hist=None):   # one entry per read of the run, at the rank's index
        hist[10 + counts.rank] += len(counts.off) - 1
        return hist

    cabi.shard_abundance_hist = fake_hist
    comm = SocketComm(rank=rank, world=world, addr="127.0.0.1", port=port)
    sh = StubShard(rank, log, max_positions=1000)
    g = ShardedGroup(sh, comm)
    g.attach()
    # rank 0: 30 reads of 100 bases in three rounds; rank 1: 8 reads, one round, then two rounds of empty input
    n_reads = 30 if rank == 0 else 8
    reads = [("ACGT" * 25)[: 90 + (i % 11)] for i in range(n_reads)]
    lens = np.array([len(r) for r in reads])
    med, avg, sd, nk = g.read_medians(reads)
    assert sh.routed == ([10, 10, 10] if rank == 0 else [8, 0, 0])
    assert np.array_equal(med, lens) and np.array_equal(nk, lens) and med.dtype == np.uint16 and avg.dtype == np.float32
    assert np.array_equal(g.median_at_least(reads, 95), lens >= 95)
    assert np.array_equal(g.trim(reads, 93), np.minimum(lens, 93))
    kc = g.kmer_counts(reads)
    assert kc.dtype == np.uint16 and np.array_equal(kc, np.concatenate([np.full(n - 3, n) for n in lens]))
    # a rank without reads at all still takes part in every round and gets empty answers
    none = g.kmer_counts([] if rank == 1 else reads)
    assert len(none) == (0 if rank == 1 else len(kc))
    assert [len(x) for x in g.read_medians([] if rank == 1 else reads)] == [0 if rank == 1 else n_reads] * 4
    tracking = ShardedGroup(StubShard(rank, log, max_positions=1000, name="tracking"), comm)
    hist = g.abundance_distribution(tracking, reads)
    want = np.zeros(65536, dtype=np.uint64)
    want[10], want[11] = 30, 8
    assert hist.dtype == np.uint64 and np.array_equal(hist, want)
    comm.close()
    if rank == 0:
        open(out, "w").write("ok")


def test_sharded_query_protocol_world2(tmp_path):
    log, out = str(tmp_path / "log"), str(tmp_path / "out")
    port = 33500 + (os.getpid() % 500)
    mp.spawn(_worker, args=(2, port, log, out), nprocs=2, join=True)
    assert open(out).read() == "ok"
    lines = [ln.split() for ln in open(log).read().split("\n") if ln]
    ops = [(name, op) for _, name, op in lines]
    query = [("counts", p) for p in ("route", "offsets", "push", "lookup", "pull")]
    ingest = [("tracking", p) for p in ("route", "offsets", "push", "apply", "count_new")]
    want = []
    for rounds in (3, 3, 3, 3, 3, 3):        # read_medians, median_at_least, trim, kmer_counts, and the two calls with rank 1 empty
        for _ in range(rounds):
            for phase in query:
                want += [phase, phase]   # both ranks log a phase before either logs the next one
    for _ in range(3):                    # abundance_distribution: per round, the tracking shards ingest, then the counts answer
        for phase in ingest + query:
            want += [phase, phase]
    assert ops == want
    by_rank = {}
    for r, name, op in lines:
        by_rank.setdefault(r, []).append((name, op))
    assert by_rank["0"] == by_rank["1"] == want[::2]
