#!/usr/bin/env python
"""Generate tests/golden/port_golden.json: the reference's outputs for the inputs of the tests that once compared with a live
compiled reference (oracle/_ref), computed by the oracle port (oracle/khmer_oracle.c), which tests/test_oracle.py pins to
the reference's own answers and to golden.json.  CPU only, a few minutes and about 1 GB of memory.

  benchscale  tests/test_gpu_benchscale.py: after each of its two bench-scale batches, n_occupied, n_unique_kmers and the md5
              of every table image; after both, the bigcount map (entries, md5 of the hash-sorted (hash, count) arrays)
  random      tests/test_oracle.py::test_oracle_vs_live_reference_random: per random trial, k-mers, counts and table md5s
  hll         tests/test_oracle.py::test_hll_registers_restatement_equals_reference: HLL registers per (k, p)

    python tests/golden/make_port_golden.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as ol  # noqa: E402
import test_gpu_benchscale as tb  # noqa: E402
import test_oracle as to  # noqa: E402
from common import md5  # noqa: E402


def benchscale():
    sizes = ol.primes_near_x(4, 1e8)
    o = ol.Oracle("Countgraph", tb.K, sizes)
    o.set_use_bigcount(True)
    out = {"sizes": sizes, "n_reads": tb.N_READS, "batches": {}}
    for seed, coverage, tag in tb.BATCHES:
        buf, off = tb._batch(seed, tb.N_READS, tb.N_READS * tb.READ_LEN // coverage)
        kmers = o.L.ko_consume_reads(o.h, buf.ctypes.data_as(ol.C.c_char_p), off.ctypes.data_as(ol.u64p), tb.N_READS, 1, 0, 0, 0)
        assert kmers == tb.N_READS * (tb.READ_LEN - tb.K + 1)
        out["batches"][tag] = {"n_occupied": int(o.n_occupied()), "n_unique_kmers": int(o.n_unique_kmers()),
                               "table_md5": [md5(o.table(i)) for i in range(len(sizes))]}
    keys, vals = tb.bigcount_arrays(o.bigcounts())
    out["bigcounts"] = {"n": int(len(keys)), "md5": tb.bigcount_md5(keys, vals)}
    return out


def random():
    out = []
    for cls, k, sizes, reads in to.random_trials():
        got, _ = to.random_trial_outputs(cls, k, sizes, reads)
        out.append(dict(cls=cls, k=k, sizes=sizes, **got))
    return out


def main():
    out = {"benchscale": benchscale(), "random": random(), "hll": to.hll_outputs(os.path.join(HERE, "data"))}
    with open(os.path.join(HERE, "port_golden.json"), "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    main()
