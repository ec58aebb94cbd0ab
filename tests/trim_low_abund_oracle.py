"""ctypes binding for the serial trim-low-abund loop over the oracle port (tests/trim_low_abund_oracle.c; TEST INFRASTRUCTURE
ONLY).  The library is compiled next to libkhmer_oracle.so on first use and linked against it."""
import ctypes as C
import os
import subprocess

import numpy as np

import oracle_lib as ol

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "trim_low_abund_oracle.c")
SO = os.path.join(os.path.dirname(ol.ORACLE_SO), "libtla_oracle.so")

_lib = None


def lib():
    global _lib
    if _lib is None:
        base = ol.build_oracle()
        if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(base)):
            tmp = "%s.%d.tmp" % (SO, os.getpid())
            subprocess.check_call(["cc", "-O2", "-std=gnu11", "-fPIC", "-shared", "-Wall", "-o", tmp, SRC, "-L" + os.path.dirname(base),
                                   "-lkhmer_oracle", "-Wl,-rpath,$ORIGIN"])
            os.replace(tmp, SO)
        ol.oracle_lib()
        L = C.CDLL(SO)
        L.tla_pass1.restype = C.c_int64
        L.tla_pass1.argtypes = [C.c_void_p, C.c_int, C.c_char_p, ol.u64p, C.c_uint64, C.c_void_p, C.c_uint, C.c_uint, C.c_uint,
                                C.c_void_p, C.c_void_p]
        L.tla_pass2.restype = None
        L.tla_pass2.argtypes = [C.c_void_p, C.c_int, C.c_char_p, ol.u64p, C.c_uint64, C.c_void_p, C.c_uint, C.c_uint, C.c_int,
                                C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _reads_and_pairs(reads, paired):
    if isinstance(reads, tuple):
        buf, off = reads
        seqs = buf.tobytes() if hasattr(buf, "tobytes") else bytes(buf)
        off = np.ascontiguousarray(off, dtype=np.uint64)
    else:
        seqs, off = ol.pack_reads(reads)
    pw = np.ascontiguousarray(paired, dtype=np.uint8) if paired is not None else None
    return seqs, off, pw


def pass1(o, reads, trim_at_coverage, cutoff, diginorm=None, paired=None):
    """serial pass 1 on the oracle sketch `o` (oracle_lib.Oracle), cleaned reads: (actions, trim lengths, k-mers consumed);
    actions as KMGPU_TLA_* (0 drop, 1 skip, 2 save, 3 trim)"""
    seqs, off, pw = _reads_and_pairs(reads, paired)
    n = len(off) - 1
    act = np.zeros(max(n, 1), dtype=np.uint8)
    pos = np.zeros(max(n, 1), dtype=np.uint32)
    kmers = lib().tla_pass1(o.h, o.k, seqs, off.ctypes.data_as(ol.u64p), n, pw.ctypes.data if pw is not None else None,
                            int(trim_at_coverage), int(cutoff), int(diginorm or 0), act.ctypes.data, pos.ctypes.data)
    return act[:n], pos[:n], kmers


def pass2(o, reads, trim_at_coverage, cutoff, variable=False, paired=None):
    """serial pass 2 on the saved (cleaned) reads: (actions, trim lengths); 3 trim, 4 keep untrimmed; the sketch is not changed"""
    seqs, off, pw = _reads_and_pairs(reads, paired)
    n = len(off) - 1
    act = np.zeros(max(n, 1), dtype=np.uint8)
    pos = np.zeros(max(n, 1), dtype=np.uint32)
    lib().tla_pass2(o.h, o.k, seqs, off.ctypes.data_as(ol.u64p), n, pw.ctypes.data if pw is not None else None,
                    int(trim_at_coverage), int(cutoff), int(bool(variable)), act.ctypes.data, pos.ctypes.data)
    return act[:n], pos[:n]
