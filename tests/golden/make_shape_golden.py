#!/usr/bin/env python
"""Generate tests/golden/shape_golden.json: what the reference's ingestion computes for the production-size shapes of
tests/test_gpu_shapes.py (the shapes, their inputs and the record are defined there), computed by the oracle port
(oracle/khmer_oracle.c), which tests/test_oracle.py pins to the reference.  CPU only, about three minutes on 8 cores: the
shapes run in three processes, so that at most three of the large ones (S3, S4, S5, S7: 8 to 10 GB of tables each) are held
at once, under 30 GB.

    python tests/golden/make_shape_golden.py
"""
import concurrent.futures
import json
import multiprocessing
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import test_gpu_shapes as ts  # noqa: E402

ORDER = ("S3", "S5", "S4", "S7", "S1", "S2", "S6")   # longest first


def one(sid):
    t0 = time.time()
    with concurrent.futures.ThreadPoolExecutor(4) as pool:
        rec = ts.run_shape(sid, ts.OracleShape(sid), pool)
    print("%s: %.0f s" % (sid, time.time() - t0), file=sys.stderr, flush=True)
    return sid, rec


def main():
    assert sorted(ORDER) == sorted(ts.SHAPES)
    with concurrent.futures.ProcessPoolExecutor(3, mp_context=multiprocessing.get_context("spawn")) as ex:
        shapes = dict(ex.map(one, ORDER))
    out = {"block_bytes": ts.BLOCK, "probe_reads": ts.N_PROBE, "read_len": ts.READ_LEN, "shapes": {s: shapes[s] for s in sorted(shapes)}}
    with open(os.path.join(HERE, "shape_golden.json"), "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    main()
