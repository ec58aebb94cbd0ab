"""Host-side protocol of bigcount on address-sharded sketches, without a GPU: stub shards, world 3 over SocketComm.  Every rank
applies the concatenation of all ranks' event lists in rank order; the switch is collective; bigcount off adds no collective."""
import os
import sys

import numpy as np
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class StubShard:
    """Its events of a round: one entry per read of at least 240 bases, hash = 1000 * rank + round, count = the read's length.
    The lists it is asked to apply are kept."""

    def __init__(self, rank):
        self.rank, self.max_positions = rank, 1000
        self.big, self.round, self.n_reads = False, 0, 0
        self.applied = []

    def ipc_export(self):
        return np.full(64 * 5, self.rank + 1, dtype=np.uint8)

    def ipc_attach(self, handles):
        pass

    def set_use_bigcount(self, on):
        self.big = bool(on)

    def get_use_bigcount(self):
        return self.big

    def route(self, reads, clean=True):
        buf, off = reads
        self.off = np.asarray(off, dtype=np.uint64)
        self.round += 1
        return int(off[-1] - off[0])

    def offsets(self):
        pass

    def push(self):
        pass

    def apply(self):
        pass

    def count_new(self):
        pass

    def bigcount_events(self):
        lens = (self.off[1:] - self.off[:-1]).astype(np.uint32)
        lens = lens[lens >= 240]
        return np.full(len(lens), 1000 * self.rank + self.round, dtype=np.uint64), lens

    def bigcount_apply(self, hashes, counts):
        self.applied.append((np.asarray(hashes).tolist(), np.asarray(counts).tolist()))


def _worker(rank, world, port, out):
    from khmer_b200.multigpu import ShardedGroup, SocketComm

    class CountingComm(SocketComm):
        calls = 0

        def all_gather_bytes(self, b):
            CountingComm.calls += 1
            return super().all_gather_bytes(b)

    comm = CountingComm(rank=rank, world=world, addr="127.0.0.1", port=port)
    sh = StubShard(rank)
    g = ShardedGroup(sh, comm)
    g.attach()
    # rank 0: 12 reads in three rounds, all with events; rank 1: 5 reads in one round, none with events; rank 2: no reads
    reads = {0: ["A" * (240 + i) for i in range(12)], 1: ["C" * (200 + i) for i in range(5)], 2: []}[rank]

    # bigcount off: the five barriers of an ingest round and the round count of _runs, nothing more
    before = CountingComm.calls
    g.consume_reads(reads)
    assert CountingComm.calls - before == 1 + 3 * 5, CountingComm.calls - before
    assert sh.applied == []

    # ranks that disagree: every rank raises, nothing changes
    try:
        g.set_use_bigcount(rank != 1)
        raise AssertionError("disagreeing set_use_bigcount did not raise")
    except ValueError as e:
        assert "disagree" in str(e)
    assert not sh.get_use_bigcount()

    g.set_use_bigcount(True)
    assert sh.get_use_bigcount()
    first = sh.round
    before = CountingComm.calls
    g.consume_reads(reads)
    # per round: three barriers, the apply's refusal count, the list lengths and the lists
    assert CountingComm.calls - before == 1 + 3 * 6, CountingComm.calls - before
    # every rank applies rank 0's list of every round (the only rank with events), also the ranks without reads in it
    assert sh.applied == [([first + i + 1] * 4, [240 + 4 * i + j for j in range(4)]) for i in range(3)], sh.applied
    # rounds in which no rank has events (rank 1's reads, two rounds) exchange the list lengths only
    sh.applied = []
    before = CountingComm.calls
    g.consume_reads(reads if rank == 1 else [])
    assert sh.applied == [] and CountingComm.calls - before == 1 + 2 * 5, CountingComm.calls - before
    comm.close()
    with open(out + str(rank), "w") as fh:
        fh.write("ok")


def test_sharded_bigcount_protocol_world3(tmp_path):
    out = str(tmp_path / "out")
    port = 34100 + (os.getpid() % 500)
    mp.spawn(_worker, args=(3, port, out), nprocs=3, join=True)
    assert all(open(out + str(r)).read() == "ok" for r in range(3))
