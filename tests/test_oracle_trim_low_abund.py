"""The serial trim-low-abund passes over the oracle port (tests/trim_low_abund_oracle.c) against the reference's pinned script md5s and
against the restatement of the script in test_oracle._trim_low_abund.  CPU only."""
import hashlib
import os

import numpy as np

import oracle_lib as ol
import trim_low_abund_oracle as tla
from common import synth_reads
from test_oracle import TRIM_MD5, _trim_low_abund

DIGINORM_MD5 = ((0, 20, "942e9024c25a8d85033d755d86aba4a3"), (0, 15, "0d1b4b9d4c76cb8cdeee5a98f6e70163"),
                (2, 15, "fa09d094a9e623639a34f772b04d766c"))


def oracle_trim(o, recs, k, cutoff, z=20, variable=False, diginorm=None):
    """records written by the two serial passes of the oracle, in the script's order"""
    cleaned = [s.upper().replace("N", "A") for _, s in recs]
    act, pos, _ = tla.pass1(o, cleaned, z, cutoff, diginorm)
    out, saved = [], []
    for (name, seq), a, t in zip(recs, act, pos):
        if a == 3 and t >= k:
            out.append((name, seq if t == len(seq) else seq[:t]))
        elif a == 2:
            saved.append((name, seq))
    act2, pos2 = tla.pass2(o, [s.upper().replace("N", "A") for _, s in saved], z, cutoff, variable)
    for (name, seq), a, t in zip(saved, act2, pos2):
        if a == 4:
            out.append((name, seq))
        elif a == 3 and t >= k:
            out.append((name, seq if t == len(seq) else seq[:t]))
    return out


def _records(datadir):
    recs, name = [], None
    for ln in open(os.path.join(datadir, "simple-genome-reads.fa")).read().split("\n"):
        if ln.startswith(">"):
            name = ln[1:]
        elif ln:
            recs.append((name, ln))
    return recs


def _md5(out):
    return hashlib.md5("".join(">%s\n%s\n" % r for r in out).encode()).hexdigest()


def test_oracle_passes_reproduce_script_md5s(datadir):
    recs = _records(datadir)
    sizes = ol.primes_near_x(4, int(1e7 / 4))
    for (cutoff, variable, z), want in TRIM_MD5.items():
        out = oracle_trim(ol.Oracle("Countgraph", 21, sizes), recs, 21, cutoff, z, variable)
        assert _md5(out) == want, (cutoff, variable, z)
    for cutoff, dn, want in DIGINORM_MD5:
        out = oracle_trim(ol.Oracle("Countgraph", 21, sizes), recs, 21, cutoff, 20, False, diginorm=dn)
        assert _md5(out) == want, (cutoff, dn)


def test_oracle_passes_equal_restatement_with_errors():
    """deep coverage with 1 % errors (and reads shorter than k, which the script's reader drops), every setting family:
    records and the final tables equal those of the per-read restatement"""
    k = 21
    sizes = ol.primes_near_x(3, 60000)
    reads = synth_reads(7, 3000, 100, 2500, err=0.01, with_n=True)
    reads[5:5] = ["ACGT", "A" * 15]
    recs = [("r%d" % i, s) for i, s in enumerate(reads)]
    long_recs = [r for r in recs if len(r[1]) >= k]
    for cutoff, z, variable, dn in ((2, 20, False, None), (3, 12, True, None), (2, 12, False, 8), (2, 8, False, 16),
                                    (0, 20, False, 15)):
        o1, o2 = ol.Oracle("Countgraph", k, sizes), ol.Oracle("Countgraph", k, sizes)
        o1.set_use_bigcount(True)
        o2.set_use_bigcount(True)
        got = oracle_trim(o1, recs, k, cutoff, z, variable, dn)
        want = _trim_low_abund(o2, long_recs, k, cutoff, z, variable, dn)
        assert got == want, (cutoff, z, variable, dn)
        assert 0 < len(got) < len(recs)
        assert (o1.n_occupied(), o1.n_unique_kmers()) == (o2.n_occupied(), o2.n_unique_kmers())
        for i in range(len(sizes)):
            assert np.array_equal(o1.table(i), o2.table(i))
        assert o1.bigcounts() == o2.bigcounts()
