"""The oracle port (oracle/khmer_oracle.c) against the reference's own known answers (SURVEY.md §8c) and
against golden vectors produced by the compiled, unmodified reference (tests/golden/make_golden.py).
CPU only."""
import os

import numpy as np
import pytest

import oracle_lib as ol
from common import OracleImpl, check_case, load_port_golden, reads_of, md5


@pytest.fixture(scope="module")
def port_golden():
    return load_port_golden()


# ---- known answers held by the reference's own tests ------------------------------------------------
def test_twobit_known_answers():
    # tests/test_functions.py:51-85
    assert ol.hash_twobit("AAAA")[1] == 0 and ol.hash_twobit("TTTT")[1] == 85
    assert ol.hash_twobit("CCCC")[1] == 170 and ol.hash_twobit("GGGG")[1] == 255
    assert ol.hash_twobit("GGGG")[0] == 170           # forward_hash('GGGG', 4) == 170 (canonical: CCCC)
    assert ol.hash_twobit("AAAA")[0] == 0 and ol.hash_twobit("TTTT")[0] == 0
    assert ol.hash_twobit("GGTTGACGGGGCTCAGGGGGCGGCTGACTCCG")[0] == 13607885392109549066
    assert ol.hash_twobit("G" * 12)[0] == 11184810   # tests/test_countgraph.py:266-267
    # tests/test_countgraph.py:123-146
    assert ol.hash_twobit("AAACGTATGACT")[0] == 184777
    assert ol.hash_twobit("AAATACCGAGCG")[0] == 76603
    assert ol.hash_twobit("AAACGTATCGAG")[0] == 184755
    assert ol.hash_twobit("ATGGCAGTAGCAGTGAGCTG")[0] == 135513300199   # SURVEY.md §8c probe


def test_revhash_known_answers():
    # tests/test_functions.py:88-99
    assert [ol.revhash(h, 4) for h in (0, 85, 170, 255)] == ["AAAA", "TTTT", "CCCC", "GGGG"]


def test_murmur_known_answers():
    # tests/test_functions.py:148-171
    assert ol.hash_murmur("AAAA")[0] == 526240128537019279 == ol.hash_murmur("TTTT")[0]
    assert ol.hash_murmur("CCCC")[0] == 14391997331386449225 == ol.hash_murmur("GGGG")[0]
    assert ol.hash_murmur("AAAA")[1] == 5231866503566620412
    assert ol.hash_murmur("TTTT")[1] == 5753003579327329651
    assert ol.hash_murmur("CCCC")[1] == 3789793362494378039
    assert ol.hash_murmur("GGGG")[1] == 17519752047064575358
    # tests/test_counttable.py:42-60
    assert ol.hash_murmur("AAAC")[0] == 11898086063751343884
    assert ol.hash_murmur("AAAG")[0] == 10548630838975263317
    # SURVEY.md §8c probe
    assert ol.hash_murmur("CAGGCGCCCACCACCGTGCCCTCCAACCTGATGGTCAGGC")[0] == 650813168330713391


def test_murmur_revcomp_invariant():
    rng = np.random.default_rng(1)
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    for k in (5, 16, 21, 33, 40):
        s = "".join("ACGT"[i] for i in rng.integers(0, 4, k))
        rc = "".join(comp[c] for c in reversed(s))
        assert ol.hash_murmur(s)[0] == ol.hash_murmur(rc)[0]


def test_hashes_against_reference(golden):
    for s, c, f, r in golden["hash_twobit"]:
        assert ol.hash_twobit(s) == (c, f, r), s
    for s, c, f, r in golden["hash_murmur"]:
        assert ol.hash_murmur(s) == (c, f, r), s


def test_primes_against_reference(golden):
    for key, want in golden["primes"].items():
        n, x = map(int, key.split(","))
        assert ol.primes_near_x(n, x) == want, key
    assert ol.primes_near_x(4, 100000000) == [99999989, 99999971, 99999959, 99999941]   # SURVEY.md a7


def test_clean():
    assert ol.clean("ACGTacgtNnXx-*") == "ACGTACGTAAAAAA"


def test_band_interval():
    lo, hi = ol.band_interval(4, 1)
    assert lo == (2 ** 64 - 1) // 4 and hi == 2 * ((2 ** 64 - 1) // 4)
    with pytest.raises(ValueError):
        ol.band_interval(4, 5)


def test_occupancy_known_answers():
    # tests/test_nodegraph.py:222-260, tests/test_countgraph.py:633-666 (random-20-a.fa)
    reads = reads_of("random-20-a.fa")
    for cls in ("Nodegraph", "Countgraph"):
        o = ol.Oracle(cls, 20, ol.primes_near_x(3, 100000))
        o.consume_reads(reads)
        assert (o.n_occupied(), o.n_unique_kmers()) == (3884, 3960)
        o = ol.Oracle(cls, 20, ol.primes_near_x(3, 10000))
        o.consume_reads(reads)
        assert (o.n_occupied(), o.n_unique_kmers()) == (3269, 3916)
    o = ol.Oracle("Countgraph", 12, ol.primes_near_x(4, 100000))
    o.consume_reads(reads)
    assert o.n_occupied() == 3886


def test_abundance_known_answers():
    # tests/test_countgraph.py:669-692: sum(dist) == 3966 on random-20-a k=12; all-A file -> one distinct k-mer
    reads = reads_of("random-20-a.fa")
    sizes = ol.primes_near_x(4, 100000)
    o = ol.Oracle("Countgraph", 12, sizes)
    o.consume_reads(reads)
    t = ol.Oracle("Nodegraph", 12, sizes)
    d = o.abundance_distribution(reads, t)
    assert int(d.sum()) == 3966 and int(d[0]) == 0
    reads = reads_of("all-A.fa")
    o = ol.Oracle("Countgraph", 4, ol.primes_near_x(4, 100000))
    o.consume_reads(reads)
    t = ol.Oracle("Nodegraph", 4, ol.primes_near_x(4, 100000))
    d = o.abundance_distribution(reads, t)
    assert int(d.sum()) == 1 and int(d[0]) == 0


def test_bigcount_known_answers():
    # tests/test_countgraph.py:890-1036: 255 cap, beyond with bigcount, 65535 ceiling
    o = ol.Oracle("Countgraph", 4, ol.primes_near_x(4, 4 ** 4))
    for _ in range(1000):
        o.add("GGTT")
    assert o.get("GGTT") == 255
    o = ol.Oracle("Countgraph", 4, ol.primes_near_x(4, 4 ** 4))
    o.set_use_bigcount(True)
    for _ in range(1000):
        o.add("GGTT")
    assert o.get("GGTT") == 1000
    for _ in range(70000):
        o.add("GGTT")
    assert o.get("GGTT") == 65535
    with pytest.raises(ValueError):
        ol.Oracle("Nodegraph", 4, [17]).set_use_bigcount(True)


def test_abund2_bigcount_dist(golden):
    # tests/test_scripts.py:1313-1441 (abundance-dist on test-abund-read-2.fa, k=17): rows "1,96,96,0.98" and
    # "1001,2,98,1.0" with bigcount, "255,2,98,1.0" without.
    rec = next(c for c in golden["cases"] if c["name"] == "ab2-cg-big")
    assert rec["abund"] == {"1": 96, "1001": 2}
    rec = next(c for c in golden["cases"] if c["name"] == "ab2-cg-nobig")
    assert rec["abund"] == {"1": 96, "255": 2}


def test_nibble_known_answers():
    # tests/test_nibblestorage.py:69-95: clamp at 15, neighbours untouched
    o = ol.Oracle("SmallCounttable", 4, [5, 7])
    h = 3
    for _ in range(20):
        o.add(h)
    assert o.get(h) == 15
    assert o.get(4) == 0 and o.get(2) == 0
    t = o.table(0)
    assert t[1] == 0x0F and t[0] == 0 and t[2] == 0     # bin 3 of a 5-bin table: low nibble of byte 1


def test_median_known_answers():
    # tests/test_countgraph.py:285-330 test_simple_median
    o = ol.Oracle("Countgraph", 20, ol.primes_near_x(2, 1e6))
    o.consume("ATGGACAGTAGCAGTGAGC" + "A")          # one 20-mer
    m, a, s = o.median("ATGGACAGTAGCAGTGAGC" + "A")
    assert (m, a, s) == (1, 1.0, 0.0)
    o2 = ol.Oracle("Countgraph", 4, ol.primes_near_x(2, 1e5))
    o2.consume("AAAAAA")
    assert o2.median("AAAAAA")[0] == 3 and o2.median_at_least("AAAAAA", 3)
    assert not o2.median_at_least("AAAAAA", 4)
    with pytest.raises(ValueError):
        o2.median("AAA")


# ---- golden cases produced by the compiled reference -------------------------------------------------
def _case_ids(golden_path=os.path.join(os.path.dirname(__file__), "golden", "golden.json")):
    import json
    with open(golden_path) as fh:
        return [c["name"] for c in json.load(fh)["cases"]]


@pytest.mark.parametrize("name", _case_ids())
def test_oracle_matches_reference_golden(golden, name):
    rec = next(c for c in golden["cases"] if c["name"] == name)
    check_case(OracleImpl, rec)


def test_oracle_saved_file_matches_reference(golden, tmp_path):
    for name in ("r20-cg-1e5", "r20-ng-1e5", "r20-scg-1e4", "syn-ct-k40", "syn-scg-k31"):
        rec = next(c for c in golden["cases"] if c["name"] == name)
        o = ol.Oracle(rec["cls"], rec["k"], rec["sizes"])
        if rec["bigcount"] is not None:
            o.set_use_bigcount(rec["bigcount"])
        o.consume_reads(reads_of(rec["file"]))
        p = str(tmp_path / "t.ct")
        o.save(p)
        assert os.path.getsize(p) == rec["file_size"]
        if not o.bigcounts():
            assert md5(open(p, "rb").read()) == rec["file_md5"], name


def test_test_parser_matches_reference_parser(golden):
    for fn, want in golden["parse"].items():
        if "error" in want or fn.endswith(".bz2.x"):
            continue
        seqs = [ol.clean(s) for s in reads_of(fn)]
        assert len(seqs) == want["n"], fn
        assert md5("\n".join(seqs).encode()) == want["md5"], fn


def random_trials():
    """six fresh random inputs beyond the committed goldens: (class, k, table sizes, reads)"""
    from common import synth_reads
    rng = np.random.default_rng(99)
    for trial in range(6):
        cls = ["Countgraph", "SmallCountgraph", "Nodegraph", "Counttable", "SmallCounttable", "Nodetable"][trial]
        k = int(rng.integers(5, 33))
        sizes = ol.primes_near_x(int(rng.integers(1, 5)), int(rng.integers(500, 20000)))
        yield cls, k, sizes, synth_reads(100 + trial, 300, 80, 2000, err=0.02, with_n=True)


def random_trial_outputs(cls, k, sizes, reads):
    """what the oracle port computes for one trial: k-mers consumed, n_unique_kmers, n_occupied, md5 of every table"""
    o = ol.Oracle(cls, k, sizes)
    if cls in ("Countgraph", "Counttable"):
        o.set_use_bigcount(True)
    kmers = o.consume_reads(reads)
    return {"kmers": int(kmers), "n_unique_kmers": int(o.n_unique_kmers()), "n_occupied": int(o.n_occupied()),
            "table_md5": [md5(o.table(i)) for i in range(len(sizes))]}, o


def test_oracle_vs_live_reference_random(tmp_path, port_golden):
    """Differential run against the reference on fresh random inputs (beyond the committed goldens): the reference's outputs
    stored in tests/golden/port_golden.json, and the live reference too where oracle/_ref is built."""
    want = port_golden["random"]
    trials = list(random_trials())
    assert len(want) == len(trials)
    for trial, ((cls, k, sizes, reads), w) in enumerate(zip(trials, want)):
        got, o = random_trial_outputs(cls, k, sizes, reads)
        assert (cls, k, sizes) == (w["cls"], w["k"], w["sizes"])
        assert got == {key: w[key] for key in got}, cls
        if not ol.have_ref():
            continue
        p = str(tmp_path / ("t%d.fa" % trial))
        with open(p, "w") as fh:
            for i, r in enumerate(reads):
                fh.write(">%d\n%s\n" % (i, r))
        ref = ol.Ref(cls, k, sizes)
        if cls in ("Countgraph", "Counttable"):
            ref.set_use_bigcount(True)
        assert ref.consume_seqfile(p)[1] == got["kmers"]
        assert ref.n_unique_kmers() == o.n_unique_kmers() and ref.n_occupied() == o.n_occupied()
        for i in range(len(sizes)):
            assert np.array_equal(ref.table(i), o.table(i))


def test_diginorm_reproduces_reference_script_md5s(datadir):
    """tests/test_script_output.py:51-70: normalize-by-median.py -k 21 -M 1e7 on simple-genome-reads.fa writes files with these
    md5s at -C 20 / -C 15.  The serial loop of the oracle (ko_normalize_reads) driven the way the script drives the table
    (Countgraph(21, 1e7 / 4, 4); cleaned_seq = upper, N -> A; kept records written as >name\\nsequence\\n) reproduces both."""
    import hashlib
    recs, name = [], None
    for ln in open(os.path.join(datadir, "simple-genome-reads.fa")):
        ln = ln.rstrip("\n")
        if ln.startswith(">"):
            name = ln[1:]
        else:
            recs.append((name, ln))
    cleaned = [s.upper().replace("N", "A") for _, s in recs]
    for cutoff, want in ((20, "942e9024c25a8d85033d755d86aba4a3"), (15, "0d1b4b9d4c76cb8cdeee5a98f6e70163")):
        o = ol.Oracle("Countgraph", 21, ol.primes_near_x(4, int(1e7 / 4)))
        keep, _ = o.normalize_reads(cleaned, cutoff)
        out = "".join(">%s\n%s\n" % (n, s) for (n, s), k in zip(recs, keep) if k)
        assert hashlib.md5(out.encode()).hexdigest() == want


HLL_SHAPES = ((20, 14), (32, 10), (41, 16), (5, 4))


def hll_outputs(datadir):
    """the restatement's HLL registers on random-20-a.fa for every (k, p) of HLL_SHAPES: the whole file cleaned, and its first
    50 reads fed one by one — (reads, k-mers, md5 of the registers) each"""
    reads = ol.read_fastx(os.path.join(datadir, "random-20-a.fa"))
    out = []
    for k, p in HLL_SHAPES:
        regs, n = ol.hll_consume(reads, k, p, clean=True)
        regs2, n2 = ol.hll_consume(reads[:50], k, p, clean=True)
        out.append({"k": k, "p": p, "reads": len(reads), "kmers": int(n), "md5": md5(regs), "kmers_50": int(n2), "md5_50": md5(regs2)})
    return out


def test_hll_registers_restatement_equals_reference(datadir, port_golden):
    """ko_hll_consume (the restatement of HLLCounter::add / consume_string) against the reference's HLLCounter: identical
    registers on random-20-a.fa (consume_seqfile cleans the reads) and on strings fed one by one — the reference's registers
    as stored in tests/golden/port_golden.json, and the compiled reference itself where oracle/_ref is built"""
    assert hll_outputs(datadir) == port_golden["hll"]
    if not ol.have_ref():
        return
    reads = ol.read_fastx(os.path.join(datadir, "random-20-a.fa"))
    for k, p in HLL_SHAPES:
        ref = ol.RefHLL(p, k)
        nr, nk = ref.consume_seqfile(os.path.join(datadir, "random-20-a.fa"))
        regs, n = ol.hll_consume(reads, k, p, clean=True)
        assert (nr, nk) == (len(reads), n)
        assert np.array_equal(regs, ref.counters())
        ref2 = ol.RefHLL(p, k)
        tot = sum(ref2.consume_string(ol.clean(r)) for r in reads[:50])
        regs2, n2 = ol.hll_consume(reads[:50], k, p, clean=True)
        assert tot == n2 and np.array_equal(regs2, ref2.counters())
    # the estimate stays with the reference: registers computed elsewhere are handed over with set_counters
    ref3 = ol.RefHLL(14, 20)
    ref3.set_counters(ol.hll_consume(reads, 20, 14)[0])
    ref4 = ol.RefHLL(14, 20)
    ref4.consume_seqfile(os.path.join(datadir, "random-20-a.fa"))
    assert ref3.estimate() == ref4.estimate() > 0


def _trim_low_abund(o, recs, k, cutoff, trim_at_coverage=20, variable=False, diginorm=None):
    """scripts/trim-low-abund.py:196-271 (Trimmer.pass1 / pass2) with khmer/trimming.py:36-66 (trim_record) and
    Hashtable::trim_on_abundance (src/oxli/hashtable.cc:504-530), unpaired reads: records written, in the script's order"""
    def trim_at(seq):
        c = o.kmer_counts(seq)
        if len(c) <= 1 or c[0] < cutoff:
            return 0
        for i in range(1, len(c)):
            if c[i] < cutoff:
                return k + i - 1
        return len(seq)

    def trim_record(name, seq, cleaned):
        if variable and not o.median_at_least(cleaned, trim_at_coverage):
            return (name, seq)
        t = trim_at(cleaned)
        if t < k:
            return None
        return (name, seq if t == len(seq) else seq[:t])

    out, saved = [], []
    for name, seq in recs:
        cleaned = seq.upper().replace("N", "A")
        med = o.median(cleaned)[0]
        if diginorm is not None and med >= diginorm:      # --diginorm: pass 1 drops reads at or above that coverage
            continue
        if med >= trim_at_coverage:
            r = trim_record(name, seq, cleaned)
            if r:
                out.append(r)
        else:
            o.consume(cleaned)
            saved.append((name, seq))
    for name, seq in saved:
        cleaned = seq.upper().replace("N", "A")
        if not variable or o.median_at_least(cleaned, trim_at_coverage):
            r = trim_record(name, seq, cleaned)
            if r:
                out.append(r)
        else:
            out.append((name, seq))
    return out


TRIM_MD5 = {(2, False, 20): "9495801b282ff6b08961b685d12a954c", (3, False, 20): "da36ec64e7d001470c04dc19af5b8635",
            (4, False, 20): "65596253b87ed8d5aeb14dc8cf5a7406", (4, True, 20): "324871db807839f8bddd43548abcbeda",
            (4, True, 25): "6ec4f9874262f3eaf98cab4910c428f5", (4, True, 15): "393805ac92e8bed31a374de9ee89ead8"}


def test_trim_low_abund_script_md5s(datadir):
    """the output md5s the reference pins for trim-low-abund.py -k 21 -M 1e7 on simple-genome-reads.fa
    (tests/test_script_output.py:73-182: -C 2 / 3 / 4, -V, -V -Z 25, -V -Z 15 and the --diginorm forms), reproduced by the oracle's counts, medians and
    consume under a restatement of the script's two passes"""
    import hashlib
    recs, name = [], None
    for ln in open(os.path.join(datadir, "simple-genome-reads.fa")).read().split("\n"):
        if ln.startswith(">"):
            name = ln[1:]
        elif ln:
            recs.append((name, ln))
    for (cutoff, variable, z), want in TRIM_MD5.items():
        o = ol.Oracle("Countgraph", 21, ol.primes_near_x(4, int(1e7 / 4)))
        out = _trim_low_abund(o, recs, 21, cutoff, z, variable)
        text = "".join(">%s\n%s\n" % r for r in out)
        assert hashlib.md5(text.encode()).hexdigest() == want, (cutoff, variable, z)
    # --diginorm (tests/test_script_output.py:73-112): -C 0 with coverage 20 / 15 equals normalize-by-median's output; -C 2, 15
    for cutoff, dn, want in ((0, 20, "942e9024c25a8d85033d755d86aba4a3"), (0, 15, "0d1b4b9d4c76cb8cdeee5a98f6e70163"),
                             (2, 15, "fa09d094a9e623639a34f772b04d766c")):
        o = ol.Oracle("Countgraph", 21, ol.primes_near_x(4, int(1e7 / 4)))
        out = _trim_low_abund(o, recs, 21, cutoff, 20, False, diginorm=dn)
        text = "".join(">%s\n%s\n" % r for r in out)
        assert hashlib.md5(text.encode()).hexdigest() == want, (cutoff, dn)


def test_count_median_script_rows(datadir):
    """tests/test_scripts.py:465-481: count-median.py on test-abund-read-2.fa after load-into-counting -x 1e7 -N 2 -k 8 (bigcount):
    rows 'seq,1001,1001.0,0.0,18' and '895:1:37:17593:9954/1,1,103.803741455,303.702941895,114' — median, and the float mean /
    stddev rounded to nine places as the script prints them"""
    reads = ol.read_fastx(os.path.join(datadir, "test-abund-read-2.fa"))
    o = ol.Oracle("Countgraph", 8, ol.primes_near_x(2, int(1e7)))
    o.set_use_bigcount(True)
    o.consume_reads(reads, clean=True)
    rows = set()
    for r in (reads[0], reads[1]):
        seq = r.upper().replace("N", "A")
        med, avg, sd = o.median(seq)
        rows.add("%d,%s,%s,%d" % (med, round(float(avg), 9), round(float(sd), 9), len(seq)))
    assert rows == {"1001,1001.0,0.0,18", "1,103.803741455,303.702941895,114"}


def test_filter_abund_script_expectations(datadir):
    """tests/test_filter_abund.py:42-66, :171-186: filter-abund(-single).py -k 17 (cutoff 2) on test-abund-read-2.fa: 98 unique k-mers;
    every read kept is cut down to GGTTGACGGGGCTCAGGG (Hashtable::trim_on_abundance, src/oxli/hashtable.cc:504-530)"""
    reads = ol.read_fastx(os.path.join(datadir, "test-abund-read-2.fa"))
    k = 17
    o = ol.Oracle("Countgraph", k, ol.primes_near_x(2, int(1e7)))
    o.set_use_bigcount(True)
    o.consume_reads(reads, clean=True)
    assert o.n_unique_kmers() == 98
    seqs = set()
    for r in reads:
        seq = r.upper().replace("N", "A")
        c = o.kmer_counts(seq)
        if len(c) <= 1 or c[0] < 2:
            t = 0
        else:
            t = len(seq)
            for i in range(1, len(c)):
                if c[i] < 2:
                    t = k + i - 1
                    break
        if t >= k:
            seqs.add(r[:t])
    assert seqs == {"GGTTGACGGGGCTCAGGG"}
