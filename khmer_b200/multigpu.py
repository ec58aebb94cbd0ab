"""Multi-GPU plumbing for replicated and address-sharded sketches (SURVEY.md §8e): one process per GPU.

The table data never goes through this module — the kernels read and write the peers' HBM directly over NVLink (CUDA IPC).
What the ranks need from each other on the host is tiny: 64-byte IPC handles once, barriers between phases, a few integers.
`SocketComm` does that over plain TCP on 127.0.0.1 (no dependency); `TorchComm` wraps an initialised torch.distributed process
group for callers that already have one (bench.py: the launch contract is torchrun + NCCL).
"""
import os
import socket
import struct
import time

import numpy as np


def shard_range(n_items, rank, world):
    """Contiguous, rank-ordered shard [lo, hi) of n_items (rank order == stream order, so that "first toucher"
    arguments carry over: the lowest rank that touched a bin holds its first toucher)."""
    per, rem = divmod(n_items, world)
    lo = rank * per + min(rank, rem)
    return lo, lo + per + (1 if rank < rem else 0)


# ---------------------------------------------------------------------------------------------------------------------
# communicators: rank, world, barrier(), all_gather_bytes(b) -> [bytes per rank], all_reduce_sum(int) -> int
# ---------------------------------------------------------------------------------------------------------------------
class SocketComm:
    """Star over TCP: rank 0 listens, the others connect; every collective is a gather to rank 0 and a broadcast back."""

    def __init__(self, rank=None, world=None, addr=None, port=None, timeout=120.0):
        self.rank = int(os.environ.get("RANK", "0")) if rank is None else rank
        self.world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else world
        addr = addr or os.environ.get("MASTER_ADDR", "127.0.0.1")
        port = int(port if port is not None else int(os.environ.get("MASTER_PORT", "29400")) + 17)
        self.peers = []
        self.sock = None
        if self.world == 1:
            return
        if self.rank == 0:
            srv = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
            srv.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
            srv.bind((addr, port))
            srv.listen(self.world)
            srv.settimeout(timeout)
            conns = {}
            while len(conns) < self.world - 1:
                c, _ = srv.accept()
                c.setsockopt(socket.IPPROTO_TCP, socket.TCP_NODELAY, 1)
                r, = struct.unpack("<i", self._recv(c, 4))
                conns[r] = c
            srv.close()
            self.peers = [conns[r] for r in range(1, self.world)]
        else:
            deadline = time.time() + timeout
            while True:
                try:
                    s = socket.create_connection((addr, port), timeout=5.0)
                    break
                except OSError:
                    if time.time() > deadline:
                        raise
                    time.sleep(0.05)
            s.setsockopt(socket.IPPROTO_TCP, socket.TCP_NODELAY, 1)
            s.settimeout(timeout)
            s.sendall(struct.pack("<i", self.rank))
            self.sock = s

    @staticmethod
    def _recv(s, n):
        buf = bytearray()
        while len(buf) < n:
            chunk = s.recv(n - len(buf))
            if not chunk:
                raise ConnectionError("peer closed the rendezvous socket")
            buf += chunk
        return bytes(buf)

    def _send_msg(self, s, b):
        s.sendall(struct.pack("<q", len(b)) + b)

    def _recv_msg(self, s):
        n, = struct.unpack("<q", self._recv(s, 8))
        return self._recv(s, n)

    def all_gather_bytes(self, b):
        b = bytes(b)
        if self.world == 1:
            return [b]
        if self.rank == 0:
            parts = [b] + [self._recv_msg(c) for c in self.peers]
            blob = b"".join(struct.pack("<q", len(p)) + p for p in parts)
            for c in self.peers:
                self._send_msg(c, blob)
            return parts
        self._send_msg(self.sock, b)
        blob = self._recv_msg(self.sock)
        parts, at = [], 0
        for _ in range(self.world):
            n, = struct.unpack_from("<q", blob, at)
            parts.append(blob[at + 8: at + 8 + n])
            at += 8 + n
        return parts

    def barrier(self):
        self.all_gather_bytes(b"")

    def all_reduce_sum(self, x):
        return sum(struct.unpack("<q", p)[0] for p in self.all_gather_bytes(struct.pack("<q", int(x))))

    def close(self):
        for c in self.peers:
            c.close()
        if self.sock:
            self.sock.close()
        self.peers, self.sock = [], None


class TorchComm:
    """The same four operations on an initialised torch.distributed process group."""

    def __init__(self, dist, device=None):
        self.dist, self.device = dist, device
        self.rank, self.world = dist.get_rank(), dist.get_world_size()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def all_gather_bytes(self, b):
        import torch
        t = torch.from_numpy(np.frombuffer(bytes(b), dtype=np.uint8).copy())
        if self.device is not None:
            t = t.to(self.device)
        gathered = [torch.empty_like(t) for _ in range(self.world)]   # equal lengths on every rank (handles, integers)
        self.dist.all_gather(gathered, t)
        return [g.cpu().numpy().tobytes() for g in gathered]

    def all_reduce_sum(self, x):
        import torch
        t = torch.tensor([int(x)], dtype=torch.int64, device=self.device if self.device is not None else "cpu")
        self.dist.all_reduce(t)
        return int(t.item())

    def close(self):
        pass


class _Single:
    rank, world = 0, 1

    def barrier(self):
        pass

    def all_gather_bytes(self, b):
        return [bytes(b)]

    def all_reduce_sum(self, x):
        return int(x)

    def close(self):
        pass


def _as_comm(comm, device):
    if comm is None:
        return _Single()
    if hasattr(comm, "all_gather_bytes"):
        return comm
    return TorchComm(comm, device)      # a torch.distributed module


class ReplicaGroup:
    """The replicas of one sketch across ranks.  `comm`: a SocketComm / TorchComm, a torch.distributed module, or None.

    exact_unique: keep the first-touch log (kmgpu_first_touch_log) so that merge() leaves n_unique_kmers equal to ONE sketch
    fed rank 0's reads, then rank 1's, ... (SURVEY.md §8e); costs one extra pass over the positions marked new per chunk."""

    def __init__(self, sketch, comm=None, device=None, exact_unique=False):
        self.sketch = sketch
        self.comm = _as_comm(comm, device)
        self.rank, self.world = self.comm.rank, self.comm.world
        self.attached = False
        self.exact_unique = exact_unique
        self.base_unique = 0

    def barrier(self):
        self.comm.barrier()

    def attach(self):
        """Exchange the CUDA-IPC handles of every rank's tables and map the peers (collective)."""
        if self.exact_unique:
            self.base_unique = self.sketch.n_unique_kmers()
            self.sketch.first_touch_log(True)
        if self.world == 1:
            return
        mine = np.ascontiguousarray(self.sketch.ipc_export(), dtype=np.uint8)
        parts = self.comm.all_gather_bytes(mine.tobytes())
        allh = np.frombuffer(b"".join(parts), dtype=np.uint8).copy()
        self.sketch.ipc_attach(self.rank, self.world, allh)
        self.attached = True
        self.barrier()

    def merge(self):
        """All replicas become the saturating sum (OR for Bloom filters) of all replicas (collective)."""
        if self.world == 1:
            if self.exact_unique:
                self.sketch.first_touch_resolve()
                self.base_unique = self.sketch.n_unique_kmers()
            return
        if not self.attached:
            self.attach()
        self.barrier()                       # every rank has finished ingesting
        total_new = None
        if self.exact_unique:                # against the peers' tables as they are BEFORE anything is merged
            n_new, _ = self.sketch.first_touch_resolve()
            total_new = self.comm.all_reduce_sum(n_new)   # (also a barrier: nobody merges before everybody has resolved)
        self.sketch.reduce_scatter_peers()   # rank r folds slice r of all peers into its own copy
        self.barrier()                       # all slices final before anyone copies them
        self.sketch.all_gather_peers()       # rank r pulls the other slices from their owners
        self.barrier()
        if total_new is not None:
            self.base_unique += total_new
            self.sketch.set_stats(self.sketch.n_occupied(), self.base_unique)

    def abundance_distribution(self, counts, reads, clean=True):
        """Hashtable::abundance_distribution over this rank's read shard with `self.sketch` as the tracking filter (log on):
        returns the histogram of ONE tracking filter fed all ranks' shards in rank order (collective; the tracking replicas are
        left unmerged)."""
        assert self.exact_unique, "needs the first-touch log (exact_unique=True)"
        counts.abundance_distribution(reads, self.sketch, clean=clean)
        self.barrier()
        hist = np.zeros(65536, dtype=np.uint64)
        self.sketch.first_touch_resolve(hist=hist)
        parts = self.comm.all_gather_bytes(hist.tobytes())
        self.barrier()
        return np.sum([np.frombuffer(p, dtype=np.uint64) for p in parts], axis=0).astype(np.uint64)

    def detach(self):
        if self.attached:
            self.barrier()
            self.sketch.ipc_detach()
            self.attached = False


def split_by_bases(buf, off, max_bases):
    """Cut (buffer, offsets) into runs of whole reads of at most max_bases bases each (a single longer read gets
    its own run: callers create their shards with max_positions >= the longest read)."""
    runs = []
    n = len(off) - 1
    r = 0
    while r < n:
        r1 = r + 1
        while r1 < n and int(off[r1 + 1]) - int(off[r]) <= max_bases:
            r1 += 1
        runs.append((r, r1))
        r = r1
    return runs


class ShardedGroup:
    """An address-sharded sketch across ranks: every rank hashes its own reads and groups the counter updates by the owners'
    super-buckets (route), the owners lay out their receive arenas (offsets), the senders write their runs into the owners' HBM
    over NVLink peer memory (push), owners apply what they received (apply); every rank counts which of its k-mers were new
    (count_new).  A query round takes the same first three steps, then the owners answer every record with its counter in place
    (lookup) and the senders read the answers back, keeping the minimum over the tables per k-mer (pull).  Only the barriers
    between the phases come from `comm`.

    With bigcount on (set_use_bigcount, ByteStorage), an ingest round also lists, on every rank, its k-mers whose N bytes were
    all 255 before they arrived (bigcount_events); the ranks exchange the lists and every rank applies all of them in rank order,
    so every rank holds the bigcount map of one sketch fed the rounds in stream order."""

    def __init__(self, shard, comm=None, device=None):
        self.shard = shard
        self.comm = _as_comm(comm, device)
        self.rank, self.world = self.comm.rank, self.comm.world
        get = getattr(shard, "get_use_bigcount", None)
        self.bigcount = bool(get()) if get else False   # the ranks' common setting (set_use_bigcount)

    def barrier(self):
        self.comm.barrier()

    def attach(self):
        mine = np.ascontiguousarray(self.shard.ipc_export(), dtype=np.uint8)
        parts = self.comm.all_gather_bytes(mine.tobytes())
        self.shard.ipc_attach(np.frombuffer(b"".join(parts), dtype=np.uint8).copy())
        self.barrier()

    def _runs(self, reads):
        """This rank's reads as the runs of its rounds (collective): runs of whole reads of at most max_positions bases, then
        empty runs up to the number of rounds of the rank with the most — a rank without reads left still takes part."""
        from . import cabi
        buf, off = cabi.as_reads(reads)
        runs = split_by_bases(buf, off, self.shard.max_positions)
        rounds = max(int.from_bytes(p, "little") for p in self.comm.all_gather_bytes(len(runs).to_bytes(8, "little")))
        empty = (np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64))
        return [(buf, off[r0:r1 + 1]) for r0, r1 in runs] + [empty] * (rounds - len(runs))

    def set_use_bigcount(self, on):
        """Collective: bigcount on or off for the whole sketch from the next round on.  Every rank must pass the same value;
        if they disagree, every rank raises and nothing changes."""
        on = bool(on)
        votes = [bool(p[0]) for p in self.comm.all_gather_bytes(bytes([on]))]
        if len(set(votes)) > 1:
            raise ValueError("set_use_bigcount: the ranks disagree (%s)" % ", ".join("rank %d: %s" % (r, v) for r, v in enumerate(votes)))
        self.shard.set_use_bigcount(on)
        self.bigcount = on

    def bigcounts(self):
        """The bigcount map, identical on every rank, in its iteration order (that of a .ct file's trailer): (hashes, counts)."""
        return self.shard.bigcounts()

    def _ingest_round(self, run, clean):
        n = self.shard.route(run, clean=clean)
        self.barrier()          # every owner knows what it will be sent
        self.shard.offsets()
        self.barrier()          # every sender can read where its runs go
        self.shard.push()
        self.barrier()          # every update of this round sits in its owner's arena
        if not self.bigcount:
            self.shard.apply()
            self.barrier()      # every owner has marked the new positions of the round
            self.shard.count_new()
            self.barrier()      # nobody reads a peer's bitmap or store any more: the next round may start
            return n
        from . import cabi
        err = None
        try:
            self.shard.apply()
        except cabi.KmgpuError as e:
            err = e
        # (also the barrier after apply: every owner has marked the new positions and the saturated touches of the round)
        if self.comm.all_reduce_sum(err is not None):
            raise err or cabi.KmgpuError(4, "another rank's arena could not hold this round")
        self.shard.count_new()
        self._exchange_bigcount()
        return n

    def _exchange_bigcount(self):
        """every rank's events of the round -> every rank, applied in rank order.  The exchange is also the barrier that ends
        the round: nobody reads a peer's store any more."""
        from . import cabi
        hashes, counts = np.zeros(0, np.uint64), np.zeros(0, np.uint32)
        err = None
        try:
            hashes, counts = self.shard.bigcount_events()
        except cabi.KmgpuError as e:
            err = e
        heads = [struct.unpack("<qq", p) for p in self.comm.all_gather_bytes(struct.pack("<qq", len(hashes), err is not None))]
        if any(failed for _, failed in heads):
            raise err or cabi.KmgpuError(4, "another rank could not read the bigcount marks of this round")
        most = max(n for n, _ in heads)
        if most == 0:
            return
        # equal lengths on every rank (TorchComm gathers equal-sized tensors)
        blob = hashes.tobytes() + counts.tobytes()
        parts = self.comm.all_gather_bytes(blob + bytes(12 * most - len(blob)))
        hs = [np.frombuffer(p, dtype=np.uint64, count=n) for p, (n, _) in zip(parts, heads)]
        cs = [np.frombuffer(p, dtype=np.uint32, count=n, offset=8 * n) for p, (n, _) in zip(parts, heads)]
        self.shard.bigcount_apply(np.concatenate(hs), np.concatenate(cs))

    def _query_round(self, run, clean):
        """route | offsets | push | lookup | pull: afterwards the shard's getters answer for `run`.  A round an owner refused
        raises on every rank, so that no rank runs on into the next collective alone."""
        from . import cabi
        self.shard.route(run, clean=clean)
        self.barrier()
        self.shard.offsets()
        self.barrier()
        self.shard.push()
        self.barrier()          # every query of this round sits in its owner's arena
        err = None
        try:
            self.shard.lookup()
        except cabi.KmgpuError as e:
            err = e
        self.barrier()          # every record is answered
        if err is None:
            try:
                self.shard.pull()
            except cabi.KmgpuError as e:
                err = e
        # (also the barrier after pull: no owner's arena or refusal flag is rewritten before every sender has read it)
        if self.comm.all_reduce_sum(err is not None):
            raise err or cabi.KmgpuError(4, "another rank's arena could not hold this query round")

    def _query(self, reads, clean, get, dtypes):
        parts = []
        for run in self._runs(reads):
            self._query_round(run, clean)
            got = get()
            parts.append(got if isinstance(got, tuple) else (got,))
        out = tuple(np.concatenate([p[i] for p in parts]) if parts else np.zeros(0, dtype=dt) for i, dt in enumerate(dtypes))
        return out if len(out) > 1 else out[0]

    def consume_reads(self, reads, clean=True):
        """Collective: every rank passes its own shard of the reads; returns the k-mers this rank hashed."""
        return sum(self._ingest_round(run, clean) for run in self._runs(reads))

    # -- queries (collective): every rank passes its own reads and gets the answers for them, in read order.  The reads go in the
    #    same rounds as consume_reads would take them.
    def kmer_counts(self, reads, clean=False):
        """Hashtable::get_kmer_counts over all of this rank's reads: counts of read 0's k-mers, then read 1's, ..."""
        return self._query(reads, clean, self.shard.kmer_counts, (np.uint16,))

    def read_medians(self, reads, clean=False):
        """Hashtable::get_median_count per read: (median uint16, average float32, stddev float32, n_kmers uint32)"""
        return self._query(reads, clean, self.shard.read_medians, (np.uint16, np.float32, np.float32, np.uint32))

    def median_at_least(self, reads, cutoff, clean=False):
        """Hashtable::median_at_least per read: 0 / 1, 2 for a read without k-mers"""
        return self._query(reads, clean, lambda: self.shard.median_at_least(cutoff), (np.uint8,))

    def trim(self, reads, abund, below=False, clean=False):
        """trim_on_abundance (below=False) / trim_below_abundance (below=True) per read: the length each read keeps"""
        return self._query(reads, clean, lambda: self.shard.trim(abund, below), (np.uint32,))

    def abundance_distribution(self, tracking_group, reads, clean=True):
        """Hashtable::abundance_distribution with this group's sketch as the counts and `tracking_group`'s (a Bloom filter of the
        same hash kind, on the same devices and ranks) as the tracking filter: returns the histogram summed over the ranks, which
        equals ONE abundance_distribution fed the rounds in stream order (run i of rank 0, of rank 1, ..., then run i + 1)."""
        from . import cabi
        hist = np.zeros(65536, dtype=np.uint64)
        for run in self._runs(reads):
            tracking_group._ingest_round(run, clean)
            self._query_round(run, clean)
            cabi.shard_abundance_hist(self.shard, tracking_group.shard, hist)
        parts = self.comm.all_gather_bytes(hist.tobytes())
        return np.sum([np.frombuffer(p, dtype=np.uint64) for p in parts], axis=0).astype(np.uint64)

    def stats(self):
        """(n_occupied, n_unique_kmers) of the whole sketch (collective)."""
        occ, uniq, _ = self.shard.stats()
        return self.comm.all_reduce_sum(occ), self.comm.all_reduce_sum(uniq)
