"""Streaming trim-low-abund on the device (kmgpu_trim_low_abund_pass1 / pass2, khmer_b200.trimming.Trimmer) against the serial
loop: the reference script's pinned md5s, the oracle's per-read outcomes and tables for every sketch class (pairs, --diginorm
on both sides of trim_at_coverage, reads shorter than k), tiny windows, 1 M reads, and the refusals.  -m gpu."""
import hashlib
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import oracle_lib as ol
import trim_low_abund_oracle as tla
from common import synth_reads, synth_buffer
from test_oracle import TRIM_MD5

pytestmark = pytest.mark.gpu

DIGINORM_MD5 = ((0, 20, "942e9024c25a8d85033d755d86aba4a3"), (0, 15, "0d1b4b9d4c76cb8cdeee5a98f6e70163"),
                (2, 15, "fa09d094a9e623639a34f772b04d766c"))


def make_gpu(cls, k, sizes):
    from khmer_b200 import cabi
    kind, hk, _ = ol.CLASSES[cls]
    return cabi.Sketch(kind, hk, k, sizes)


def _same(g, o, n_tables):
    assert g.stats() == (o.n_occupied(), o.n_unique_kmers())
    for i in range(n_tables):
        assert np.array_equal(g.table(i), o.table(i)), "table %d" % i


@pytest.mark.parametrize("batch", [None, 7, 300])
def test_trimmer_reference_script_md5s(datadir, batch):
    """scripts/trim-low-abund.py -k 21 -M 1e7 on simple-genome-reads.fa (tests/test_script_output.py:73-182): all nine pinned
    outputs through Trimmer, the whole file per device call and 7 / 300 reads per call"""
    from khmer_b200 import _oxli
    from khmer_b200.trimming import Trimmer
    recs, name = [], None
    for ln in open(os.path.join(datadir, "simple-genome-reads.fa")).read().split("\n"):
        if ln.startswith(">"):
            name = ln[1:]
        elif ln:
            recs.append((name, ln, None))
    settings = [dict(cutoff=c, variable_coverage=v, trim_at_coverage=z, want=w) for (c, v, z), w in TRIM_MD5.items()]
    settings += [dict(cutoff=c, diginorm_coverage=d, want=w) for c, d, w in DIGINORM_MD5]
    for s in settings:
        want = s.pop("want")
        t = Trimmer(_oxli.Countgraph(21, 1e7 / 4, 4), batch_reads=batch or len(recs), **s)
        out = list(t.pass1(recs)) + list(t.pass2())
        text = "".join(">%s\n%s\n" % (n, q) for n, q, _ in out)
        assert hashlib.md5(text.encode()).hexdigest() == want, s
        assert t.n_saved > 0


def _settings(kind):
    """(Z, C, [D...]) per storage: D off, D <= Z, D > Z"""
    if kind == ol.BYTE:
        return 12, 2, [None, 8, 16]
    if kind == ol.NIBBLE:
        return 5, 2, [None, 3, 8]
    return 1, 1, [None, 1, 2]


def _body(cls):
    kind, hk, _ = ol.CLASSES[cls]
    k = 21 if hk == ol.TWOBIT else 35
    sizes = ol.primes_near_x(3, 60000)
    z, c, ds = _settings(kind)
    for paired_case in (False, True):
        for d in ds:
            g, o = make_gpu(cls, k, sizes), ol.Oracle(cls, k, sizes)
            if kind == ol.BYTE:
                g.set_use_bigcount(True)
                o.set_use_bigcount(True)
            saved, saved_pw = [], []
            n_trim = 0
            for part in range(3):
                # deep coverage of a small genome with 1 % errors: most bundles are judged against a table the window changes
                reads = synth_reads(200 + part, 3000, 100, 2500, err=0.01) + ["ACGT", "", "A" * 60, "ACGTTGCA" * 20]
                reads[17:17] = ["ACGTACGTAC"]
                paired = None
                if paired_case:
                    paired = np.zeros(len(reads), dtype=np.uint8)
                    paired[0:len(reads) - 6:4] = 1
                act, pos, kmers = g.trim_low_abund_pass1(reads, z, c, d, paired=paired)
                oact, opos, okmers = tla.pass1(o, reads, z, c, d, paired=paired)
                assert np.array_equal(act, oact), "actions differ (%s, D=%s, part %d)" % (cls, d, part)
                assert np.array_equal(pos[act == 3], opos[oact == 3])
                assert kmers == okmers
                _same(g, o, 3)
                n_trim += int((act == 3).sum())
                for i in np.flatnonzero(act == 2):
                    saved.append(reads[i])
                    saved_pw.append(int(paired is not None and paired[i] and act[i + 1] == 2))
            if d is None or d > z:
                assert n_trim > 0, (cls, d)
            spw = np.array(saved_pw, dtype=np.uint8) if paired_case else None
            for variable in (False, True):
                act2, pos2 = g.trim_low_abund_pass2(saved, z, c, variable, paired=spw)
                oact2, opos2 = tla.pass2(o, saved, z, c, variable, paired=spw)
                assert np.array_equal(act2, oact2) and np.array_equal(pos2, opos2), (cls, d, variable)
            _same(g, o, 3)
            if kind == ol.BYTE:
                gk, gv = g.bigcounts()
                assert dict(zip(gk.tolist(), gv.tolist())) == o.bigcounts()


@pytest.mark.parametrize("cls", list(ol.CLASSES))
@pytest.mark.parametrize("window", [None, 7, 300])
def test_trim_low_abund_vs_oracle(cls, window):
    if window is None:
        _body(cls)
        return
    env = dict(os.environ, KMGPU_NORM_WINDOW=str(window), KMGPU_TLA_CLS=cls)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k", "test_trim_low_abund_inner"],
                       env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def test_trim_low_abund_inner():
    cls = os.environ.get("KMGPU_TLA_CLS")
    if not cls:
        pytest.skip("run by test_trim_low_abund_vs_oracle under a fixed window")
    _body(cls)


def with_errors(buf, rate, seed):
    """substitutions at `rate` per base (a base drawn from ACGT, so about 3/4 of them change it)"""
    rng = np.random.default_rng(seed)
    buf = buf.copy()
    m = np.flatnonzero(rng.random(len(buf)) < rate)
    buf[m] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, len(m))]
    return buf


def test_trim_low_abund_one_million_reads():
    """1 M reads of 150 bp, 30x of a 5 Mbp genome with 1 % errors, Countgraph k=20 on 4 x 4e7 B; Z=20, C=2"""
    buf, off = synth_buffer(2025, 1_000_000, 150, 5_000_000)
    buf = with_errors(buf, 0.01, 7)
    sizes = ol.primes_near_x(4, 4e7)
    g, o = make_gpu("Countgraph", 20, sizes), ol.Oracle("Countgraph", 20, sizes)
    g.trim_low_abund_pass1((buf[:150 * 300_000], off[:300_001]), 20, 2)   # warm-up: device workspaces
    g.reset()
    t0 = time.perf_counter()
    act, pos, kmers = g.trim_low_abund_pass1((buf, off), 20, 2)
    t1 = time.perf_counter() - t0
    saved = np.flatnonzero(act == 2)
    sbuf = buf.reshape(-1, 150)[saved].reshape(-1)
    soff = np.arange(len(saved) + 1, dtype=np.uint64) * np.uint64(150)
    t0 = time.perf_counter()
    act2, pos2 = g.trim_low_abund_pass2((sbuf, soff), 20, 2)
    t2 = time.perf_counter() - t0
    t0 = time.perf_counter()
    oact, opos, okmers = tla.pass1(o, (buf, off), 20, 2)
    oact2, opos2 = tla.pass2(o, (sbuf, soff), 20, 2)
    t_cpu = time.perf_counter() - t0
    print("trim-low-abund 1M reads: pass 1 %.2f s (%.2f M reads/s), pass 2 %.2f s over %d saved reads, serial oracle %.1f s; "
          "trimmed now %d" % (t1, 1.0 / t1, t2, len(saved), t_cpu, (act == 3).sum()))
    assert np.array_equal(act, oact)
    assert np.array_equal(pos, opos)
    assert kmers == okmers
    assert np.array_equal(act2, oact2) and np.array_equal(pos2, opos2)
    assert 0 < len(saved) < 1_000_000 and (act == 3).sum() > 0 and (pos[act == 3] < 150).sum() > 0
    _same(g, o, 4)


def test_trim_low_abund_refusals():
    from khmer_b200 import cabi
    sizes = ol.primes_near_x(2, 10000)
    g = make_gpu("Countgraph", 21, sizes)
    g.set_use_bigcount(True)
    reads = synth_reads(3, 10, 100, 1000)
    for z, c, d in ((256, 2, None), (20, 256, None), (20, 2, 256)):
        with pytest.raises(cabi.KmgpuError) as e:
            g.trim_low_abund_pass1(reads, z, c, d)
        assert e.value.code == 7
    paired = np.zeros(len(reads), dtype=np.uint8)
    paired[-1] = 1
    with pytest.raises(cabi.KmgpuError) as e:
        g.trim_low_abund_pass1(reads, 20, 2, paired=paired)
    assert e.value.code == 1
    with pytest.raises(cabi.KmgpuError) as e:
        g.trim_low_abund_pass2(reads, 20, 2, paired=paired)
    assert e.value.code == 1
    long_read = "ACGT" * (152_000_000 // 16 + 1)    # longer than a window (a quarter of a device chunk)
    with pytest.raises(cabi.KmgpuError) as e:
        g.trim_low_abund_pass1([long_read], 20, 2)
    assert e.value.code == 7
    assert g.stats() == (0, 0)
