"""Shared parity checks: run one golden case (tests/golden/golden.json, produced by the compiled reference)
through an implementation and compare every recorded output bit for bit."""
import hashlib
import json
import os
import struct

import numpy as np

import oracle_lib as ol

HERE = os.path.dirname(os.path.abspath(__file__))
DATA = os.path.join(HERE, "golden", "data")

_reads_cache = {}


def reads_of(fn):
    if fn not in _reads_cache:
        _reads_cache[fn] = ol.read_fastx(os.path.join(DATA, fn))
    return _reads_cache[fn]


def md5(b):
    return hashlib.md5(bytes(b)).hexdigest()


def load_port_golden():
    """tests/golden/port_golden.json: the reference's outputs for inputs beyond golden.json, written by
    tests/golden/make_port_golden.py"""
    with open(os.path.join(HERE, "golden", "port_golden.json")) as fh:
        return json.load(fh)


def f32(hexstr):
    return struct.unpack("<f", bytes.fromhex(hexstr))[0]


def synth_reads(seed, n_reads, read_len, genome_len, err=0.0, with_n=False):
    """Same generator as tests/golden/make_golden.py (SURVEY.md §8d)."""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, genome_len, dtype=np.uint8)
    comp = np.array([3, 2, 1, 0], dtype=np.uint8)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    starts = rng.integers(0, genome_len - read_len, n_reads)
    strands = rng.integers(0, 2, n_reads)
    out = []
    for s, st in zip(starts, strands):
        r = g[s:s + read_len]
        if st:
            r = comp[r[::-1]]
        r = lut[r].copy()
        if err:
            m = rng.random(read_len) < err
            r[m] = lut[rng.integers(0, 4, int(m.sum()))]
        if with_n and rng.random() < 0.05:
            r[rng.integers(0, read_len)] = ord("N")
        out.append(r.tobytes().decode())
    return out


def synth_buffer(seed, n_reads, read_len, genome_len):
    """Vectorised variant for large inputs: returns (uint8 ASCII buffer, uint64 offsets)."""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, genome_len, dtype=np.uint8)
    starts = rng.integers(0, genome_len - read_len, n_reads)
    strands = rng.integers(0, 2, n_reads).astype(bool)
    idx = starts[:, None] + np.arange(read_len)[None, :]
    codes = g[idx]
    codes[strands] = (3 - codes[strands])[:, ::-1]
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    buf = lut[codes].reshape(-1)
    off = (np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(read_len))
    return np.ascontiguousarray(buf), off


class OracleImpl:
    """Adapter giving the oracle port the same surface as khmer_b200.cabi.Sketch for check_case."""

    def __init__(self, cls, k, sizes):
        self.o = ol.Oracle(cls, k, sizes)

    def set_use_bigcount(self, on):
        self.o.set_use_bigcount(on)

    def consume_reads(self, reads, clean=True):
        return self.o.consume_reads(reads, clean=clean)

    def stats(self):
        return self.o.n_occupied(), self.o.n_unique_kmers()

    def table(self, i):
        return self.o.table(i)

    def read_medians(self, reads, clean=False):
        med, avg, sd, nk = [], [], [], []
        for r in reads:
            n = max(0, len(r) - self.o.k + 1)
            nk.append(n)
            if n == 0:
                med.append(0); avg.append(0.0); sd.append(0.0)
                continue
            m, a, s = self.o.median(r)
            med.append(m); avg.append(a); sd.append(s)
        return (np.array(med, dtype=np.uint16), np.array(avg, dtype=np.float32), np.array(sd, dtype=np.float32),
                np.array(nk, dtype=np.uint32))

    def median_at_least(self, reads, cutoff, clean=False):
        return np.array([2 if len(r) < self.o.k else int(self.o.median_at_least(r, cutoff)) for r in reads],
                        dtype=np.uint8)

    def kmer_counts(self, reads, clean=False):
        return np.concatenate([self.o.kmer_counts(r) for r in reads]) if reads else np.zeros(0, np.uint16)

    def kmer_hashes(self, reads, clean=False):
        return np.concatenate([self.o.kmer_hashes(r) for r in reads]) if reads else np.zeros(0, np.uint64)

    def abundance_distribution(self, reads, tracking, clean=True):
        return self.o.abundance_distribution(reads, tracking.o, clean=clean)

    def bigcounts(self):
        d = self.o.bigcounts()
        return np.array(list(d.keys()), dtype=np.uint64), np.array(list(d.values()), dtype=np.uint16)


def check_case(make, rec, light=False):
    """make(cls, k, sizes) -> implementation object.  Compares with the reference's recorded outputs."""
    cls, k, sizes = rec["cls"], rec["k"], rec["sizes"]
    reads = reads_of(rec["file"])
    sk = make(cls, k, sizes)
    if rec["bigcount"] is not None:
        sk.set_use_bigcount(rec["bigcount"])
    kmers = sk.consume_reads(reads, clean=True)
    assert len(reads) == rec["reads"]
    assert kmers == rec["kmers"]
    occ, uniq = sk.stats()
    assert occ == rec["n_occupied"], "n_occupied"
    assert uniq == rec["n_unique"], "n_unique_kmers"
    for i in range(len(sizes)):
        assert md5(sk.table(i)) == rec["table_md5"][i], "table %d bytes differ" % i
    cleaned = [ol.clean(r) for r in reads[:len(rec["medians"])]]
    ok = [i for i, m in enumerate(rec["medians"]) if m is not None]
    if ok:
        sub = [cleaned[i] for i in ok]
        med, avg, sd, nk = sk.read_medians(sub)
        al2 = sk.median_at_least(sub, 2)
        al5 = sk.median_at_least(sub, 5)
        for j, i in enumerate(ok):
            m = rec["medians"][i]
            assert int(med[j]) == m[0], "median of read %d" % i
            assert np.float32(avg[j]).tobytes() == bytes.fromhex(m[1]), "average of read %d" % i
            assert np.float32(sd[j]).tobytes() == bytes.fromhex(m[2]), "stddev of read %d" % i
            assert int(al2[j]) == m[3] and int(al5[j]) == m[4], "median_at_least of read %d" % i
    if "counts0" in rec:
        c0 = ol.clean(reads[0])
        assert sk.kmer_counts([c0]).tolist() == rec["counts0"]
        assert [int(x) for x in sk.kmer_hashes([c0])] == rec["hashes0"]
    if "abund" in rec and not light:
        track_cls = "Nodegraph" if cls.endswith("graph") else "Nodetable"
        tracking = make(track_cls, k, sizes)
        dist = sk.abundance_distribution(reads, tracking, clean=True)
        got = {str(i): int(v) for i, v in enumerate(dist) if v}
        assert got == rec["abund"], "abundance distribution"
        assert tracking.stats()[1] == rec["tracking_unique"]
    return sk
