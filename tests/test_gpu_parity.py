"""Parity of the CUDA path (through the C ABI) with the oracle and with the reference's goldens.  -m gpu."""
import json
import os

import numpy as np
import pytest

import oracle_lib as ol
from common import check_case, reads_of, synth_reads, md5, OracleImpl

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _cases():
    with open(os.path.join(HERE, "golden", "golden.json")) as fh:
        return [c["name"] for c in json.load(fh)["cases"]]


def make_gpu(cls, k, sizes):
    from khmer_b200 import cabi
    kind, hk, _ = ol.CLASSES[cls]
    return cabi.Sketch(kind, hk, k, sizes)


@pytest.mark.parametrize("name", _cases())
def test_gpu_matches_reference_golden(golden, name):
    rec = next(c for c in golden["cases"] if c["name"] == name)
    check_case(make_gpu, rec)


def test_gpu_golden_cases_grouped_path():
    """All reference goldens through the grouped path (fused hash + grouping), the small tables included; by default these
    shapes take the bins[] + k_bucketize path or the delta passes."""
    import subprocess, sys
    env = dict(os.environ, KMGPU_PREFER_BINS="0", KMGPU_GROUP_MIN_BUCKETS="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k",
                        "test_gpu_matches_reference_golden"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def test_gpu_golden_cases_no_delta_plan():
    """All reference goldens with delta blocks so small that no table has a delta plan: the shapes the bins path could take
    go to the grouped path instead, since the bins path needs the delta passes for a bucket that overflows."""
    import subprocess, sys
    env = dict(os.environ, KMGPU_DELTA_BLOCK_BINS="256", KMGPU_DELTA_MAX_PASSES="1", KMGPU_CHUNK_BASES="65536")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k",
                        "test_gpu_matches_reference_golden and not C1 and not 25k"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def test_gpu_golden_cases_delta_many_blocks():
    """All reference goldens through the delta+fold path with ~2k-bin blocks (many blocks per table)."""
    import subprocess, sys
    env = dict(os.environ, KMGPU_DELTA_BLOCK_BINS="2048", KMGPU_DELTA_MAX_PASSES="1000000", KMGPU_CHUNK_BASES="65536",
               KMGPU_COLD_MIN_NEW="64", KMGPU_BUCKETS="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k",
                        "test_gpu_matches_reference_golden and not C1 and not 25k"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def _same_state(g, o, n_tables):
    assert g.stats() == (o.n_occupied(), o.n_unique_kmers())
    for i in range(n_tables):
        assert np.array_equal(g.table(i), o.table(i)), "table %d" % i


@pytest.mark.parametrize("cls", list(ol.CLASSES))
@pytest.mark.parametrize("chunk", [None, 4096, "bins-no-delta", "bins-no-delta-parts", "delta-blocks", "delta-cold", "delta-cold-stamps", "buckets",
                                   "buckets-overflow", "buckets-whole", "group", "group-whole", "group-regroup", "group-two",
                                   "group-two-regroup", "group-turns", "group-t16k", "count-passes"])
def test_gpu_vs_oracle_random(cls, chunk, monkeypatch):
    """Fresh seeded inputs, incremental calls (state carried across calls), tiny device chunks so that reads
    straddle chunks (the chunk size is read once per process: exercised through a subprocess for != None)."""
    if chunk is not None:
        import subprocess, sys
        env = dict(os.environ, KMGPU_TEST_CLS=cls)
        if chunk == "bins-no-delta":   # tables the bins path could take, too many delta blocks for its overflow fallback: grouped path
            env.update(KMGPU_DELTA_BLOCK_BINS="256", KMGPU_DELTA_MAX_PASSES="1", KMGPU_CHUNK_BASES="16384")
        elif chunk == "bins-no-delta-parts":   # same, host input in 16 parts per chunk (every chunk of a call keeps the grouped path)
            env.update(KMGPU_DELTA_BLOCK_BINS="256", KMGPU_DELTA_MAX_PASSES="1", KMGPU_CHUNK_BASES="16384", KMGPU_PART_BASES="1000")
        elif chunk == "delta-cold":   # delta+fold path, per-block ("cold chunk") ranked-bitmap resolution forced
            env.update(KMGPU_DELTA_BLOCK_BINS="2000", KMGPU_COLD_MIN_NEW="1", KMGPU_CHUNK_BASES="32768", KMGPU_BUCKETS="0")
        elif chunk == "buckets":   # bucket path (records grouped by 32 Ki-bin bucket, applied in shared memory)
            env.update(KMGPU_CHUNK_BASES="16384", KMGPU_PART_BASES="1000")   # host input in 16 parts per chunk
        elif chunk == "buckets-whole":   # bucket path, every chunk uploaded in one piece
            env.update(KMGPU_CHUNK_BASES="16384", KMGPU_PARTS="0")
        elif chunk == "buckets-overflow":   # bucket path with buckets far too small: every chunk falls back to the delta passes
            env.update(KMGPU_CHUNK_BASES="16384", KMGPU_BUCKET_CAP="64", KMGPU_PART_BASES="3000")
        elif chunk == "delta-cold-stamps":   # same, through the stamp hash tables (blocks beyond 2^26 bins take this form)
            env.update(KMGPU_DELTA_BLOCK_BINS="2000", KMGPU_COLD_MIN_NEW="1", KMGPU_CHUNK_BASES="32768", KMGPU_COLD_RANK="0",
                       KMGPU_BUCKETS="0")
        elif chunk == "delta-blocks":   # delta+fold path with many blocks per table
            env.update(KMGPU_DELTA_BLOCK_BINS="1000", KMGPU_DELTA_MAX_PASSES="100000", KMGPU_CHUNK_BASES="16384", KMGPU_BUCKETS="0")
        elif isinstance(chunk, str) and chunk.startswith("group"):
            # grouped path (fused hash + grouping, apply in shared memory) forced on these tiny tables
            env.update(KMGPU_GROUP_MIN_BUCKETS="0", KMGPU_CHUNK_BASES="16384", KMGPU_PART_BASES="1000")
            if chunk == "group-whole":      # every chunk uploaded in one piece
                env.update(KMGPU_PARTS="0")
            elif chunk == "group-regroup":  # regions far too small: every chunk is regrouped with exact offsets
                env.update(KMGPU_BUCKET_CAP="64")
            elif chunk == "group-two":      # two-level grouping (super-buckets first)
                env.update(KMGPU_FORCE_TWO_LEVEL="1")
            elif chunk == "group-two-regroup":
                env.update(KMGPU_FORCE_TWO_LEVEL="1", KMGPU_SB_CAP="200", KMGPU_BUCKET_CAP="64")
            elif chunk == "group-turns":    # record store too small for all tables at once: one table per turn
                env.update(KMGPU_GROUP_MAX_RECORDS="20000")
            elif chunk == "group-t16k":
                env.update(KMGPU_PART_T="16384")
        else:
            env.update(KMGPU_CHUNK_BASES=str(chunk))
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__),
                            "-k", "test_gpu_vs_oracle_random_inner"], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
        return
    _random_body(cls)


def test_gpu_vs_oracle_random_inner():
    cls = os.environ.get("KMGPU_TEST_CLS")
    if not cls:
        pytest.skip("driver-invoked only")
    _random_body(cls)


def _random_body(cls):
    rng = np.random.default_rng(hash(cls) % 1000)
    kind, hk, _ = ol.CLASSES[cls]
    for trial in range(3):
        k = int(rng.integers(4, 33)) if hk == ol.TWOBIT else int(rng.choice([5, 16, 17, 31, 32, 33, 40, 47, 48, 64, 65, 100]))
        nt = int(rng.integers(1, 6))
        sizes = ol.primes_near_x(nt, int(rng.integers(300, 30000)))
        g = make_gpu(cls, k, sizes)
        o = ol.Oracle(cls, k, sizes)
        if kind == ol.BYTE:
            g.set_use_bigcount(True)
            o.set_use_bigcount(True)
        for part in range(3):
            reads = synth_reads(1000 * trial + part, 400, int(rng.integers(k, 300)), 3000, err=0.02, with_n=True)
            reads += ["", "A", "ACGT" * 70, "N" * 50, "acgtn" * 30]
            # a read far longer than the small device chunks of the subprocess variants: it continues across chunks
            reads.insert(7, "".join("ACGT"[i] for i in rng.integers(0, 4, 21000)))
            assert g.consume_reads(reads, clean=True) == o.consume_reads(reads, clean=True)
            _same_state(g, o, nt)
        probe = synth_reads(7, 50, 120, 3000)
        probe = [p for p in probe if len(p) >= k]
        hs = np.concatenate([o.kmer_hashes(p) for p in probe])
        assert np.array_equal(g.kmer_hashes(probe), hs)
        want = np.array([o.get(int(h)) for h in hs], dtype=np.uint16)
        assert np.array_equal(g.get_counts(hs), want)
        assert np.array_equal(g.kmer_counts(probe), want)
        if kind == ol.BYTE:
            gk, gv = g.bigcounts()
            assert dict(zip(gk.tolist(), gv.tolist())) == o.bigcounts()


def test_offsets_need_not_start_at_zero():
    """reads are seqs[offsets[r] .. offsets[r+1]): a window into a larger buffer works as is."""
    from khmer_b200 import cabi
    reads = synth_reads(77, 300, 90, 2000)
    buf, off = cabi.as_reads(reads)
    g, o = make_gpu("Countgraph", 19, [7919, 7927]), ol.Oracle("Countgraph", 19, [7919, 7927])
    assert g.consume_reads((buf, off[100:201])) == o.consume_reads(reads[100:200])
    _same_state(g, o, 2)


def test_raw_mode_twobit_matches_consume_string():
    """consume(str) does not clean (hashtable.cc:280-294): non-ATC bytes code as G, lower case too."""
    g = make_gpu("Countgraph", 11, [1009, 1013, 1019])
    o = ol.Oracle("Countgraph", 11, [1009, 1013, 1019])
    for s in ["ACGTNNNNACGTACGTAAAN", "acgtacgtacgtacgt", "ACGTTGCAAAGGTCCAXYZACGT" * 3]:
        assert g.consume_reads([s], clean=False) == o.consume(s)
    _same_state(g, o, 3)


def test_murmur_raw_non_acgt_is_refused():
    from khmer_b200 import cabi
    g = make_gpu("Counttable", 11, [1009, 1013])
    with pytest.raises(cabi.KmgpuError) as e:
        g.consume_reads(["ACGTNNNNACGTACGTAAAN"], clean=False)
    assert e.value.code == 5


def test_add_hashes_is_new_and_bigcount_limits():
    # tests/test_countgraph.py:890-1036
    g = make_gpu("Countgraph", 4, ol.primes_near_x(4, 4 ** 4))
    o = ol.Oracle("Countgraph", 4, ol.primes_near_x(4, 4 ** 4))
    h = o.hash("GGTT")
    assert g.add_hashes([h], want_new=True).tolist() == [1]
    assert g.add_hashes([h] * 999, want_new=True).sum() == 0
    assert g.get_counts([h]).tolist() == [255]
    g2 = make_gpu("Countgraph", 4, ol.primes_near_x(4, 4 ** 4))
    g2.set_use_bigcount(True)
    g2.add_hashes([h] * 1000)
    assert g2.get_counts([h]).tolist() == [1000]
    g2.add_hashes([h] * 70000)
    assert g2.get_counts([h]).tolist() == [65535]
    rng = np.random.default_rng(3)
    hs = rng.integers(0, 2 ** 63, 5000, dtype=np.uint64)
    hs = np.concatenate([hs, hs[:2500], hs[:100]])
    rng.shuffle(hs)
    g3 = make_gpu("SmallCounttable", 21, [257, 263])
    o3 = ol.Oracle("SmallCounttable", 21, [257, 263])
    want = np.array([o3.add(int(x)) for x in hs], dtype=np.uint8)
    assert np.array_equal(g3.add_hashes(hs, want_new=True), want)
    _same_state(g3, o3, 2)


def test_bigcount_not_supported_for_other_storages():
    from khmer_b200 import cabi
    for cls in ("Nodegraph", "SmallCountgraph"):
        with pytest.raises(cabi.KmgpuError):
            make_gpu(cls, 8, [101]).set_use_bigcount(True)


def test_banding(datadir):
    reads = synth_reads(5, 500, 100, 5000)
    for band in range(4):
        lo, hi = ol.band_interval(4, band)
        g = make_gpu("Countgraph", 21, [5003, 5009])
        o = ol.Oracle("Countgraph", 21, [5003, 5009])
        assert g.consume_reads(reads, band=(lo, hi)) == o.consume_reads(reads, band=(lo, hi))
        _same_state(g, o, 2)


def test_merge_and_update_from():
    reads_a = synth_reads(11, 300, 90, 2000)
    reads_b = synth_reads(12, 300, 90, 2000)
    # Nodegraph.update (storage.cc:63-96)
    sizes = [4001, 4003]
    ga, gb = make_gpu("Nodegraph", 15, sizes), make_gpu("Nodegraph", 15, sizes)
    oa, ob = ol.Oracle("Nodegraph", 15, sizes), ol.Oracle("Nodegraph", 15, sizes)
    for s, r in ((ga, reads_a), (gb, reads_b), (oa, reads_a), (ob, reads_b)):
        s.consume_reads(r)
    ga.merge(gb)
    oa.update(ob)
    assert ga.n_occupied() == oa.n_occupied()
    for i in range(2):
        assert np.array_equal(ga.table(i), oa.table(i))
    # counting storages: merged replicas == one sketch fed everything (saturating add is associative)
    for cls in ("Countgraph", "SmallCountgraph"):
        lowc = ["A" * 150] * 300
        g1, g2, gall = (make_gpu(cls, 15, sizes) for _ in range(3))
        g1.consume_reads(reads_a + lowc)
        g2.consume_reads(reads_b + lowc)
        gall.consume_reads(reads_a + lowc + reads_b + lowc)
        g1.merge(g2)
        for i in range(2):
            assert np.array_equal(g1.table(i), gall.table(i))
        assert g1.n_occupied() == gall.n_occupied()
    with pytest.raises(Exception):
        ga.merge(make_gpu("Nodegraph", 15, [4001, 4007]))


def test_packed_and_batch_paths_match_ascii():
    from khmer_b200 import cabi
    reads = synth_reads(21, 700, 150, 4000) + ["ACGT", "", "ACGTACGTACGTACGTACGTAC"]
    sizes = ol.primes_near_x(4, 20000)
    ref = make_gpu("Countgraph", 20, sizes)
    n = ref.consume_reads(reads)
    # host-side 2-bit packing as the read feed produces it
    code = np.zeros(256, dtype=np.uint64)
    for ch, c in zip(b"ATCGatcg", [0, 1, 2, 3, 0, 1, 2, 3]):
        code[ch] = c
    buf, off = cabi.as_reads(reads)
    codes = code[buf]
    nw = (len(codes) + 31) // 32 + 1
    padded = np.zeros(nw * 32, dtype=np.uint64)
    padded[:len(codes)] = codes
    shifts = np.uint64(62) - np.uint64(2) * (np.arange(32, dtype=np.uint64))
    words = (padded.reshape(nw, 32) << shifts[None, :]).sum(axis=1, dtype=np.uint64)
    g = make_gpu("Countgraph", 20, sizes)
    assert g.consume_packed(words, off) == n
    b = cabi.Batch(reads, 20)
    g2 = make_gpu("Countgraph", 20, sizes)
    assert g2.consume_batch(b) == n
    for i in range(4):
        assert np.array_equal(g.table(i), ref.table(i)) and np.array_equal(g2.table(i), ref.table(i))
    assert g.stats() == ref.stats() == g2.stats()


def test_upload_download_roundtrip_and_recount():
    o = ol.Oracle("SmallCountgraph", 9, [1009, 1013])
    o.consume_reads(synth_reads(31, 200, 60, 800))
    g = make_gpu("SmallCountgraph", 9, [1009, 1013])
    for i in range(2):
        g.upload_table(i, o.table(i))
        assert np.array_equal(g.table(i), o.table(i))
    g.recount_occupied()
    assert g.n_occupied() == o.n_occupied()


def test_empty_and_short_inputs():
    g = make_gpu("Countgraph", 20, [1009])
    assert g.consume_reads([]) == 0
    assert g.consume_reads(["", "ACGT", "A" * 19]) == 0
    assert g.stats() == (0, 0)
    med, avg, sd, nk = g.read_medians(["ACGT", "A" * 25])
    assert nk.tolist() == [0, 6] and med.tolist() == [0, 0]
    assert g.median_at_least(["ACGT", "A" * 25], 1).tolist() == [2, 0]


def test_full_size_properties_C1():
    """BASELINE config C1 at full table size (4 x ~1e8 bytes): properties that do not need an oracle run —
    idempotent table image under replay of n_kmers, sum of table-0 bytes == number of k-mers (no saturation,
    25k.fq.gz), merging a sketch with an empty one is the identity."""
    sizes = ol.primes_near_x(4, 1e8)
    reads = reads_of("25k.fq.gz")
    g = make_gpu("Countgraph", 20, sizes)
    n = g.consume_reads(reads)
    assert n == 1248896
    t0 = g.table(0)
    assert int(t0.sum(dtype=np.uint64)) == n
    assert int(np.count_nonzero(t0)) == g.n_occupied() == 1238304
    e = make_gpu("Countgraph", 20, sizes)
    e.merge(g)
    assert md5(e.table(0)) == md5(t0) and e.n_occupied() == g.n_occupied()


@pytest.mark.parametrize("cls", list(ol.CLASSES))
def test_bucket_path_many_buckets(cls):
    """Tables of ~70 buckets each, chunks small enough for the bucket path: counters, n_occupied, n_unique_kmers and the
    bigcount map against the oracle, state carried across calls (the second call meets occupied and saturating bins)."""
    kind, hk, _ = ol.CLASSES[cls]
    k = 21 if hk == ol.TWOBIT else 35
    sizes = ol.primes_near_x(4, 2300000)
    g = make_gpu(cls, k, sizes)
    o = ol.Oracle(cls, k, sizes)
    if kind == ol.BYTE:
        g.set_use_bigcount(True)
        o.set_use_bigcount(True)
    for part in range(3):
        reads = synth_reads(50 + part, 3000, 150, 20000, err=0.01, with_n=True) + ["ACGTTGCA" * 40] * 150
        assert g.consume_reads(reads) == o.consume_reads(reads)
        _same_state(g, o, 4)
    if kind == ol.BYTE:
        gk, gv = g.bigcounts()
        want = o.bigcounts()
        assert len(want) > 0 and dict(zip(gk.tolist(), gv.tolist())) == want
    g.close()


@pytest.mark.parametrize("variant", ["dense", "sparse", "sparse-two", "dense-two", "regroup", "sparse-regroup", "sparse-two-regroup", "turns", "t16k"])
def test_group_path_many_buckets(variant):
    """test_bucket_path_many_buckets (six classes, ~70 buckets per table, state carried across calls, bigcount map) with the
    grouped path forced on and steered into each of its forms."""
    import subprocess, sys
    env = dict(os.environ, KMGPU_GROUP_MIN_BUCKETS="0")
    if variant == "sparse":        # ~230 records per bucket and chunk: k_apply_sparse
        env.update(KMGPU_CHUNK_BASES="16384")
    elif variant == "sparse-two":
        env.update(KMGPU_CHUNK_BASES="16384", KMGPU_FORCE_TWO_LEVEL="1")
    elif variant == "dense-two":
        env.update(KMGPU_FORCE_TWO_LEVEL="1")
    elif variant == "regroup":     # regions of 500 records against ~6.7 K expected: exact offsets, dense apply with clamping rounds
        env.update(KMGPU_BUCKET_CAP="500")
    elif variant == "sparse-regroup":   # sparse plan whose regions overflow: exact offsets, k_apply_sparse + the heavily loaded buckets by list
        env.update(KMGPU_CHUNK_BASES="16384", KMGPU_BUCKET_CAP="40", KMGPU_REGROUP_SPARSE_MAX="300")
    elif variant == "sparse-two-regroup":
        env.update(KMGPU_CHUNK_BASES="16384", KMGPU_FORCE_TWO_LEVEL="1", KMGPU_BUCKET_CAP="40", KMGPU_SB_CAP="3000", KMGPU_REGROUP_SPARSE_MAX="300")
    elif variant == "turns":
        env.update(KMGPU_GROUP_MAX_RECORDS="900000")
    elif variant == "t16k":
        env.update(KMGPU_PART_T="16384")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k",
                        "test_bucket_path_many_buckets"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
