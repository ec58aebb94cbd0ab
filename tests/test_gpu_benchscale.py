"""Parity at the scale bench.py runs: 1 M x 150 bp reads at 30x (131 M k-mers) into Countgraph k=20, primes(4, 1e8), bigcount on,
default chunking (one 150 M-position chunk per call, uploaded in parts: the same grouped path and bucket loads as the bench's chunks),
compared with tests/golden/port_golden.json — what the reference's ingestion computes at one thread for the same batches (written by
tests/golden/make_port_golden.py from the oracle port, which tests/test_oracle.py pins to the reference): the four table images,
n_occupied, n_unique_kmers, and — after a second, 300x batch that drives counters through 255 on every chunk — the bigcount map
the reference writes into its .ct file.  -m gpu."""
import os

import numpy as np
import pytest

import oracle_lib as ol
from common import load_port_golden, md5

pytestmark = pytest.mark.gpu

K = 20
READ_LEN = 150
N_READS = 1_000_000
# 1. the bench's workload: 30x coverage of a 5 Mbp genome
# 2. then 300x coverage of a 0.5 Mbp genome: every 20-mer of it is seen ~260 times, counters cross 255 inside both chunks
BATCHES = ((4242, 30, "30x"), (77, 300, "300x"))


def _batch(seed, n_reads, genome_len):
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, genome_len, dtype=np.uint8)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
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
    return buf, off


def bigcount_arrays(m):
    """a {hash: count} bigcount map as (hashes, counts) sorted by hash: the map has no order of its own"""
    keys = np.array(sorted(m), dtype=np.uint64)
    return keys, np.array([m[k] for k in keys.tolist()], dtype=np.uint16)


def bigcount_md5(keys, vals):
    return md5(keys.astype("<u8").tobytes() + vals.astype("<u2").tobytes())


def test_bench_scale_parity_grouped_path(tmp_path):
    """the same comparison with the fused grouping kernel (k_part + k_apply2) instead of bins[] + k_bucketize + k_apply"""
    import subprocess
    import sys
    env = dict(os.environ, KMGPU_PREFER_BINS="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k",
                        "test_bench_scale_parity_with_compiled_reference"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def test_bench_scale_parity_with_compiled_reference(tmp_path):
    from khmer_b200 import cabi
    want = load_port_golden()["benchscale"]
    sizes = ol.primes_near_x(4, 1e8)
    assert sizes == want["sizes"] and want["n_reads"] == N_READS
    g = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, K, sizes)
    g.set_use_bigcount(True)
    for seed, coverage, tag in BATCHES:
        buf, off = _batch(seed, N_READS, N_READS * READ_LEN // coverage)
        assert g.consume_reads((buf, off), clean=True) == N_READS * (READ_LEN - K + 1)
        w = want["batches"][tag]
        assert g.stats() == (w["n_occupied"], w["n_unique_kmers"]), tag
        for i in range(4):
            assert md5(g.table(i)) == w["table_md5"][i], "%s: table %d differs from the reference" % (tag, i)
        if tag == "30x":
            assert g.bigcounts()[0].size == 0
    gk, gv = g.bigcounts()
    order = np.argsort(gk)
    assert want["bigcounts"]["n"] > 1000
    assert (len(gk), bigcount_md5(gk[order], gv[order])) == (want["bigcounts"]["n"], want["bigcounts"]["md5"])
    g.close()
