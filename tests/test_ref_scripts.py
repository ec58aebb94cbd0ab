"""The reference's scripts, UNCHANGED and read in place from a khmer source tree, on top of khmer_b200._oxli
(tests/ref_scripts_harness.py).  Pinned outputs are the reference's own: tests/test_scripts.py:65-90, :1313-1330, :521-533.

Needs a khmer source tree, named by KHMER_REFERENCE_DIR; the two script runs need a CUDA device as well.  Without the tree every test
here skips: the reference's scripts and test data are not part of this repository."""
import hashlib
import os

import pytest

REF = os.environ.get("KHMER_REFERENCE_DIR", "")
HERE = os.path.dirname(os.path.abspath(__file__))
have_ref = bool(REF) and os.path.isdir(os.path.join(REF, "scripts")) and os.path.isdir(os.path.join(REF, "khmer"))


@pytest.mark.skipif(not have_ref, reason="no khmer source tree at KHMER_REFERENCE_DIR")
def test_reference_python_layer_imports_on_this_backend():
    """every name khmer/__init__.py, khmer_args.py, kfile.py, utils.py and oxli/ import from the compiled modules resolves, and the
    three scripts get as far as their argument parsers (--version exits 0) — no device needed"""
    import ref_scripts_harness as hz
    kh = hz.install(REF)
    assert kh.Countgraph is not None and kh.Nodegraph is not None and callable(kh.calc_expected_collisions)
    import khmer.khmer_args, khmer.kfile, khmer.utils, oxli.functions      # noqa: F401  (the reference's files)
    for script in ("load-into-counting.py", "abundance-dist.py", "load-graph.py"):
        rc, out, err = hz.run_script(REF, script, ["--version"])
        assert rc == 0, (script, out, err)


@pytest.mark.gpu
@pytest.mark.skipif(not have_ref, reason="no khmer source tree at KHMER_REFERENCE_DIR")
def test_load_into_counting_and_abundance_dist_unchanged(tmp_path):
    import ref_scripts_harness as hz
    data = os.path.join(REF, "tests", "test-data")
    # tests/test_scripts.py:65-76
    out = str(tmp_path / "out.ct")
    rc, so, se = hz.run_script(REF, "load-into-counting.py", ["-x", "1e3", "-N", "2", "-k", "20", out, os.path.join(data, "test-abund-read-2.fa")])
    assert rc == 0, se
    assert "Total number of unique k-mers: 94" in se, se
    assert os.path.exists(out)
    # tests/test_scripts.py:1313-1330
    hist = str(tmp_path / "out.hist")
    ct = str(tmp_path / "abund.ct")
    rc, so, se = hz.run_script(REF, "load-into-counting.py", ["-x", "1e7", "-N", "2", "-k", "17", ct, os.path.join(data, "test-abund-read-2.fa")])
    assert rc == 0, se
    rc, so, se = hz.run_script(REF, "abundance-dist.py", ["-z", ct, os.path.join(data, "test-abund-read-2.fa"), hist])
    assert rc == 0, se
    rows = [ln.strip() for ln in open(hist)]
    assert rows[1] == "1,96,96,0.98" and rows[2] == "1001,2,98,1.0", rows[:4]
    # config C1: the .ct of data/25k.fq.gz (SURVEY.md §8c golden, regenerated from the compiled reference)
    c1 = str(tmp_path / "c1.ct")
    rc, so, se = hz.run_script(REF, "load-into-counting.py", ["-k", "20", "-N", "4", "-x", "1e8", c1, os.path.join(REF, "data", "25k.fq.gz")])
    assert rc == 0, se
    assert hashlib.md5(open(c1, "rb").read()).hexdigest() == "2c1668c9e986170d3319f8d001b1f2d3"


@pytest.mark.gpu
@pytest.mark.skipif(not have_ref, reason="no khmer source tree at KHMER_REFERENCE_DIR")
def test_load_graph_unchanged(tmp_path):
    import ref_scripts_harness as hz
    data = os.path.join(REF, "tests", "test-data")
    base = str(tmp_path / "out")
    # tests/test_scripts.py:521-533 (3960 unique k-mers), default path with the tagset
    rc, so, se = hz.run_script(REF, "load-graph.py", ["-x", "1e7", "-N", "2", "-k", "20", base, os.path.join(data, "random-20-a.fa")])
    assert rc == 0, se
    assert "Total number of unique k-mers: 3960" in se, se
    assert os.path.exists(base) and os.path.exists(base + ".tagset")
    rc, so, se = hz.run_script(REF, "load-graph.py", ["-x", "1e7", "-N", "2", "-k", "20", "--no-build-tagset", base + "2", os.path.join(data, "random-20-a.fa")])
    assert rc == 0, se
    assert not os.path.exists(base + "2.tagset")
