"""Streaming trim-low-abund on one GPU (kmgpu_trim_low_abund_pass1 / pass2): config C3's table shape (Countgraph k=20, 4 x 2e9 B)
and the headline shape (4 x 1e8 B), 4 M synthetic 150 bp reads at 30x with 1 % substitutions (without errors nothing is trimmed),
Z=20, C=2.

Per shape: wall clock of pass 1 over the whole input and of pass 2 over the reads pass 1 saved (reads/s, k-mers/s), with the
KMGPU_DEBUG phase split of pass 1.  On the same call: the per-read host loop (get_median_count, trim_on_abundance, consume per
read through the host layer, as tests/test_host_gpu.py drives the script) on a prefix of 20 k reads, whose per-read outcomes must
equal the batch run's on that prefix, and the oracle's serial loop on a prefix.  Prints one JSON line with the card's name and
power limit.

    python tools/bench_trim_low_abund.py [--reads 4000000] [--prefix 20000] [--oracle-prefix 200000]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

READ_LEN, K, Z, CUT = 150, 20, 20, 2


def card():
    """name and power limit of GPU 0, read in the run that measures it"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:
        return {"name": "unknown", "power_limit": "unknown (%s)" % type(e).__name__}


def reads_with_errors(n, seed=2026):
    from common import synth_buffer
    buf, off = synth_buffer(seed, n, READ_LEN, n * READ_LEN // 30)
    rng = np.random.default_rng(seed + 1)
    m = np.flatnonzero(rng.random(len(buf)) < 0.01)
    buf[m] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, len(m))]
    return buf, off


class StderrTap:
    """the library's KMGPU_DEBUG lines (written to fd 2) of the calls inside the block"""

    def __enter__(self):
        self.f = tempfile.TemporaryFile(mode="w+b")
        sys.stderr.flush()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *exc):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read().decode(errors="replace")
        self.f.close()


def per_read_loop(g, seqs):
    """the script's pass 1 read by read through the host layer: actions and trim lengths as the batch entry reports them"""
    act = np.zeros(len(seqs), dtype=np.uint8)
    pos = np.zeros(len(seqs), dtype=np.uint32)
    for i, s in enumerate(seqs):
        if g.get_median_count(s)[0] >= Z:
            act[i] = 3
            pos[i] = g.trim_on_abundance(s, CUT)[1]
        else:
            g.consume(s)
            act[i] = 2
    return act, pos


def run_shape(name, x, buf, off, prefix, oracle_prefix):
    from khmer_b200 import cabi, _oxli
    import oracle_lib as ol
    import trim_low_abund_oracle as tla
    n = len(off) - 1
    sizes = ol.primes_near_x(4, x)
    g = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, K, sizes)
    g.trim_low_abund_pass1((buf[:READ_LEN * 200_000], off[:200_001]), Z, CUT)   # warm-up: device workspaces
    g.reset()
    with StderrTap() as tap:
        t0 = time.perf_counter()
        act, pos, kmers = g.trim_low_abund_pass1((buf, off), Z, CUT)
        t1 = time.perf_counter() - t0
    saved = np.flatnonzero(act == 2)
    sbuf = np.ascontiguousarray(buf.reshape(-1, READ_LEN)[saved].reshape(-1))
    soff = np.arange(len(saved) + 1, dtype=np.uint64) * np.uint64(READ_LEN)
    t0 = time.perf_counter()
    act2, pos2 = g.trim_low_abund_pass2((sbuf, soff), Z, CUT)
    t2 = time.perf_counter() - t0
    n_kmers = n * (READ_LEN - K + 1)
    out = {"shape": name, "table_bytes": [int(s) for s in sizes], "reads": n,
           "pass1_s": round(t1, 3), "pass1_reads_per_s": round(n / t1), "pass1_kmers_per_s": round(n_kmers / t1),
           "pass2_reads": len(saved), "pass2_s": round(t2, 3), "pass2_reads_per_s": round(len(saved) / t2) if t2 else None,
           "pass2_kmers_per_s": round(len(saved) * (READ_LEN - K + 1) / t2) if t2 else None,
           "saved": len(saved), "trimmed_now": int((act == 3).sum()), "cut_now": int(((act == 3) & (pos < READ_LEN)).sum()),
           "kmers_consumed": int(kmers), "pass1_debug": [ln for ln in tap.text.splitlines() if "trim_low_abund_pass1" in ln]}
    m = re.search(r"(\d+) refined positions", tap.text)
    out["refined_positions"] = int(m.group(1)) if m else None
    # per-read host loop and the batch entry on the same prefix, from empty tables
    seqs = [bytes(buf[i * READ_LEN:(i + 1) * READ_LEN]).decode() for i in range(prefix)]
    hg = _oxli.Countgraph(K, 1, 1, primes=sizes)
    t0 = time.perf_counter()
    lact, lpos = per_read_loop(hg, seqs)
    tl = time.perf_counter() - t0
    g2 = cabi.Sketch(cabi.BYTE, cabi.TWOBIT, K, sizes)
    bact, bpos, _ = g2.trim_low_abund_pass1(seqs, Z, CUT)
    out["per_read_loop_reads_per_s"] = round(prefix / tl)
    out["prefix_outcomes_equal"] = bool(np.array_equal(bact, lact) and np.array_equal(bpos[bact == 3], lpos[lact == 3]))
    del g2, hg
    # the oracle's serial loop
    o = ol.Oracle("Countgraph", K, sizes)
    t0 = time.perf_counter()
    oact, opos, _ = tla.pass1(o, (buf[:READ_LEN * oracle_prefix], off[:oracle_prefix + 1]), Z, CUT)
    to = time.perf_counter() - t0
    out["oracle_reads_per_s"] = round(oracle_prefix / to)
    out["oracle_prefix_outcomes_equal"] = bool(np.array_equal(act[:oracle_prefix], oact) and np.array_equal(pos[:oracle_prefix], opos))
    del o
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000)
    ap.add_argument("--prefix", type=int, default=20_000, help="reads of the per-read host loop")
    ap.add_argument("--oracle-prefix", type=int, default=200_000, help="reads of the oracle's serial loop")
    args = ap.parse_args()
    os.environ["KMGPU_DEBUG"] = "1"
    buf, off = reads_with_errors(args.reads)
    res = {"bench": "trim_low_abund", "card": card(), "reads": args.reads, "read_len": READ_LEN, "coverage": 30, "error_rate": 0.01,
           "k": K, "trim_at_coverage": Z, "cutoff": CUT,
           "shapes": [run_shape("C3 4x2e9", 2e9, buf, off, args.prefix, args.oracle_prefix),
                      run_shape("headline 4x1e8", 1e8, buf, off, args.prefix, args.oracle_prefix)]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
