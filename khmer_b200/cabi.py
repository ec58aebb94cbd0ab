"""ctypes view of the C ABI in include/kmgpu.h (libkmgpu.so).

Thin and literal: one Python method per C entry point, numpy arrays in and out.  The library is
built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no fallback: if the shared
library is missing, or no CUDA device is present, calls raise.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkmgpu.so")

BYTE, NIBBLE, BIT = 0, 1, 2
TWOBIT, MURMUR = 0, 1
CLEAN = 1

u8p = C.POINTER(C.c_uint8)
u16p = C.POINTER(C.c_uint16)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
f32p = C.POINTER(C.c_float)

# every symbol include/kmgpu.h declares (tests check the library exports all of them)
SYMBOLS = [
    "kmgpu_last_error", "kmgpu_abi_version", "kmgpu_device_count", "kmgpu_create", "kmgpu_destroy",
    "kmgpu_set_use_bigcount", "kmgpu_get_use_bigcount", "kmgpu_consume_reads", "kmgpu_consume_packed",
    "kmgpu_batch_create", "kmgpu_batch_destroy", "kmgpu_batch_info", "kmgpu_consume_batch", "kmgpu_batch_read_medians", "kmgpu_add_hashes",
    "kmgpu_get_counts", "kmgpu_kmer_counts", "kmgpu_kmer_hashes", "kmgpu_read_medians", "kmgpu_median_at_least",
    "kmgpu_abundance_distribution", "kmgpu_trim_batch", "kmgpu_normalize_batch", "kmgpu_consume_reads_new", "kmgpu_first_touch_log",
    "kmgpu_first_touch_resolve", "kmgpu_stats", "kmgpu_set_stats", "kmgpu_shape", "kmgpu_set_ksize",
    "kmgpu_table_nbytes", "kmgpu_download_table", "kmgpu_upload_table", "kmgpu_bigcount_size",
    "kmgpu_bigcount_export", "kmgpu_bigcount_import", "kmgpu_merge", "kmgpu_recount_occupied", "kmgpu_ipc_export",
    "kmgpu_ipc_attach", "kmgpu_ipc_detach", "kmgpu_reduce_scatter_peers", "kmgpu_all_gather_peers",
    "kmgpu_reduce_replicas", "kmgpu_attach_replicas", "kmgpu_profile_reset", "kmgpu_profile_get", "kmgpu_sync", "kmgpu_reset",
    "kmgpu_timer_start", "kmgpu_timer_stop", "kmgpu_slice_range", "kmgpu_alloc_pinned", "kmgpu_free_pinned",
    "kmgpu_shard_create", "kmgpu_shard_destroy", "kmgpu_shard_local", "kmgpu_shard_slice", "kmgpu_shard_ipc_export",
    "kmgpu_shard_ipc_attach", "kmgpu_shard_attach_local", "kmgpu_shard_route", "kmgpu_shard_offsets", "kmgpu_shard_push", "kmgpu_shard_apply",
    "kmgpu_shard_count_new", "kmgpu_shard_stats", "kmgpu_shard_lookup", "kmgpu_shard_pull", "kmgpu_shard_kmer_counts",
    "kmgpu_shard_read_medians", "kmgpu_shard_median_at_least", "kmgpu_shard_trim", "kmgpu_shard_abundance_hist",
    "kmgpu_shard_bigcount_events", "kmgpu_shard_bigcount_apply", "kmgpu_hll_create", "kmgpu_hll_destroy", "kmgpu_hll_consume",
    "kmgpu_hll_get_registers", "kmgpu_hll_merge_registers", "kmgpu_trim_low_abund_pass1", "kmgpu_trim_low_abund_pass2",
]

# per-read outcomes of the streaming trimmer (KMGPU_TLA_*)
TLA_DROP, TLA_SKIP, TLA_SAVE, TLA_TRIM, TLA_KEEP = 0, 1, 2, 3, 4


class Band(C.Structure):
    _fields_ = [("lo", C.c_uint64), ("hi", C.c_uint64)]


class Mask(C.Structure):
    _fields_ = [("mask", C.c_void_p), ("threshold", C.c_uint32), ("consume_masked", C.c_int)]


class KmgpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("kmgpu error %d: %s" % (code, msg))
        self.code = code
        self.msg = msg


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.kmgpu_last_error.restype = C.c_char_p
        L.kmgpu_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, u64p, C.c_int, C.POINTER(C.c_void_p)]
        L.kmgpu_destroy.argtypes = [C.c_void_p]
        L.kmgpu_set_use_bigcount.argtypes = [C.c_void_p, C.c_int]
        L.kmgpu_get_use_bigcount.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        L.kmgpu_consume_reads.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(Band),
                                          C.POINTER(Mask), u64p]
        L.kmgpu_consume_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(Band),
                                           C.POINTER(Mask), u64p]
        L.kmgpu_batch_create.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int,
                                         C.POINTER(C.c_void_p)]
        L.kmgpu_batch_destroy.argtypes = [C.c_void_p]
        L.kmgpu_batch_info.argtypes = [C.c_void_p, u64p, u64p, u64p]
        L.kmgpu_consume_batch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Band), C.POINTER(Mask), u64p]
        L.kmgpu_hll_create.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.kmgpu_hll_destroy.argtypes = [C.c_void_p]
        L.kmgpu_hll_consume.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, u64p]
        L.kmgpu_hll_get_registers.argtypes = [C.c_void_p, C.c_void_p]
        L.kmgpu_hll_merge_registers.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.kmgpu_batch_read_medians.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kmgpu_add_hashes.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.kmgpu_get_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.kmgpu_kmer_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, u64p]
        L.kmgpu_kmer_hashes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, u64p]
        L.kmgpu_read_medians.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
        L.kmgpu_median_at_least.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                            C.c_void_p]
        L.kmgpu_abundance_distribution.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                                   C.c_uint32, C.c_void_p]
        L.kmgpu_trim_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
        L.kmgpu_normalize_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32,
                                            C.c_void_p, u64p, u64p]
        L.kmgpu_trim_low_abund_pass1.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32,
                                                 C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, u64p]
        L.kmgpu_trim_low_abund_pass2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32,
                                                 C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
        L.kmgpu_consume_reads_new.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, u64p, u64p]
        L.kmgpu_first_touch_log.argtypes = [C.c_void_p, C.c_int]
        L.kmgpu_first_touch_resolve.argtypes = [C.c_void_p, u64p, u64p, C.c_void_p]
        L.kmgpu_stats.argtypes = [C.c_void_p, u64p, u64p]
        L.kmgpu_set_stats.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
        L.kmgpu_shape.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_int), u64p]
        L.kmgpu_set_ksize.argtypes = [C.c_void_p, C.c_int]
        L.kmgpu_table_nbytes.argtypes = [C.c_void_p, C.c_int, u64p]
        L.kmgpu_download_table.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64]
        L.kmgpu_upload_table.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64]
        L.kmgpu_bigcount_size.argtypes = [C.c_void_p, u64p]
        L.kmgpu_bigcount_export.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.kmgpu_bigcount_import.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.kmgpu_merge.argtypes = [C.c_void_p, C.c_void_p]
        L.kmgpu_recount_occupied.argtypes = [C.c_void_p]
        L.kmgpu_ipc_export.argtypes = [C.c_void_p, C.c_void_p]
        L.kmgpu_ipc_attach.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.kmgpu_ipc_detach.argtypes = [C.c_void_p]
        L.kmgpu_reduce_scatter_peers.argtypes = [C.c_void_p]
        L.kmgpu_all_gather_peers.argtypes = [C.c_void_p]
        L.kmgpu_reduce_replicas.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        L.kmgpu_attach_replicas.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        L.kmgpu_profile_reset.argtypes = [C.c_void_p]
        L.kmgpu_profile_get.argtypes = [C.c_void_p, C.POINTER(C.c_double), u64p, u64p]
        L.kmgpu_sync.argtypes = [C.c_void_p]
        L.kmgpu_reset.argtypes = [C.c_void_p]
        L.kmgpu_timer_start.argtypes = [C.c_void_p]
        L.kmgpu_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.kmgpu_device_count.argtypes = [C.POINTER(C.c_int)]
        L.kmgpu_slice_range.argtypes = [C.c_uint64, C.c_int, C.c_int, u64p, u64p]
        L.kmgpu_shard_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, u64p, C.c_int, C.c_int, C.c_int, C.c_uint64,
                                         C.POINTER(C.c_void_p)]
        L.kmgpu_shard_destroy.argtypes = [C.c_void_p]
        L.kmgpu_shard_local.restype = C.c_void_p
        L.kmgpu_shard_local.argtypes = [C.c_void_p]
        L.kmgpu_shard_slice.argtypes = [C.c_void_p, C.c_int, u64p, u64p]
        L.kmgpu_shard_ipc_export.argtypes = [C.c_void_p, C.c_void_p]
        L.kmgpu_shard_ipc_attach.argtypes = [C.c_void_p, C.c_void_p]
        L.kmgpu_shard_attach_local.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        L.kmgpu_shard_route.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, u64p]
        L.kmgpu_shard_apply.argtypes = [C.c_void_p]
        L.kmgpu_shard_offsets.argtypes = [C.c_void_p]
        L.kmgpu_shard_push.argtypes = [C.c_void_p]
        L.kmgpu_shard_count_new.argtypes = [C.c_void_p, u64p]
        L.kmgpu_shard_stats.argtypes = [C.c_void_p, u64p, u64p, u64p]
        L.kmgpu_shard_lookup.argtypes = [C.c_void_p]
        L.kmgpu_shard_pull.argtypes = [C.c_void_p]
        L.kmgpu_shard_kmer_counts.argtypes = [C.c_void_p, C.c_void_p, u64p]
        L.kmgpu_shard_read_medians.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kmgpu_shard_median_at_least.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.kmgpu_shard_trim.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_void_p]
        L.kmgpu_shard_abundance_hist.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.kmgpu_shard_bigcount_events.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, u64p]
        L.kmgpu_shard_bigcount_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise KmgpuError(rc, lib().kmgpu_last_error().decode(errors="replace"))


def device_count():
    n = C.c_int()
    rc = lib().kmgpu_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def as_reads(reads):
    """list of str/bytes, or (uint8 buffer, uint64 offsets) -> (np.uint8 buffer, np.uint64 offsets)."""
    if isinstance(reads, tuple):
        buf, off = reads
        if not isinstance(buf, np.ndarray):
            buf = np.frombuffer(buf, dtype=np.uint8)
        return buf, np.ascontiguousarray(off, dtype=np.uint64)
    bs = [r if isinstance(r, (bytes, bytearray)) else r.encode() for r in reads]
    off = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        off[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    buf = np.frombuffer(b"".join(bs), dtype=np.uint8) if bs else np.zeros(0, dtype=np.uint8)
    return buf, off


def _band(band):
    return C.byref(Band(band[0], band[1])) if band is not None else None


def _mask(mask):
    if mask is None:
        return None
    sk, thr, ge = mask
    return C.byref(Mask(sk.h, thr, int(ge)))


class Batch:
    """Device-resident packed reads (kmgpu_batch_*)."""

    def __init__(self, reads, ksize, clean=True, device=0):
        buf, off = as_reads(reads)
        self.h = C.c_void_p()
        check(lib().kmgpu_batch_create(device, _ptr(buf), _ptr(off), len(off) - 1, CLEAN if clean else 0, ksize,
                                       C.byref(self.h)))

    def info(self):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_batch_info(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def close(self):
        if self.h:
            lib().kmgpu_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HLL:
    """HyperLogLog registers on the device (kmgpu_hll_*): the ingest of the reference's HLLCounter."""

    def __init__(self, ksize, p, device=0):
        self.p, self.ksize = p, ksize
        self.h = C.c_void_p()
        check(lib().kmgpu_hll_create(device, ksize, p, C.byref(self.h)))

    def consume_reads(self, reads, clean=True):
        buf, off = as_reads(reads)
        n = C.c_uint64()
        check(lib().kmgpu_hll_consume(self.h, _ptr(buf), _ptr(off), len(off) - 1, CLEAN if clean else 0, C.byref(n)))
        return n.value

    def registers(self):
        out = np.zeros(1 << self.p, dtype=np.uint8)
        check(lib().kmgpu_hll_get_registers(self.h, _ptr(out)))
        return out

    def merge_registers(self, regs, replace=False):
        regs = np.ascontiguousarray(regs, dtype=np.uint8)
        assert len(regs) == 1 << self.p
        check(lib().kmgpu_hll_merge_registers(self.h, _ptr(regs), int(replace)))

    def close(self):
        if self.h:
            lib().kmgpu_hll_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Sketch:
    """One kmgpu_t handle."""

    def __init__(self, storage, hashkind, ksize, sizes, device=0):
        self.sizes = [int(s) for s in sizes]
        arr = (C.c_uint64 * len(self.sizes))(*self.sizes)
        self.h = C.c_void_p()
        self.storage, self.hashkind, self.ksize = storage, hashkind, ksize
        check(lib().kmgpu_create(storage, hashkind, ksize, len(self.sizes), arr, device, C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            lib().kmgpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- config
    def set_use_bigcount(self, on):
        check(lib().kmgpu_set_use_bigcount(self.h, int(on)))

    def get_use_bigcount(self):
        v = C.c_int()
        check(lib().kmgpu_get_use_bigcount(self.h, C.byref(v)))
        return bool(v.value)

    def set_ksize(self, k):
        check(lib().kmgpu_set_ksize(self.h, k))
        self.ksize = k

    # -- ingestion
    def consume_reads(self, reads, clean=True, band=None, mask=None):
        buf, off = as_reads(reads)
        n = C.c_uint64()
        check(lib().kmgpu_consume_reads(self.h, _ptr(buf), _ptr(off), len(off) - 1, CLEAN if clean else 0, _band(band),
                                        _mask(mask), C.byref(n)))
        return n.value

    def consume_packed(self, words, offsets, band=None, mask=None):
        words = np.ascontiguousarray(words, dtype=np.uint64)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = C.c_uint64()
        check(lib().kmgpu_consume_packed(self.h, _ptr(words), len(words), _ptr(offsets), len(offsets) - 1, _band(band),
                                         _mask(mask), C.byref(n)))
        return n.value

    def consume_batch(self, batch, band=None, mask=None):
        n = C.c_uint64()
        check(lib().kmgpu_consume_batch(self.h, batch.h, _band(band), _mask(mask), C.byref(n)))
        return n.value

    def add_hashes(self, hashes, want_new=False):
        hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
        out = np.zeros(len(hashes), dtype=np.uint8) if want_new else None
        check(lib().kmgpu_add_hashes(self.h, _ptr(hashes), len(hashes), _ptr(out)))
        return out

    # -- queries
    def get_counts(self, hashes):
        hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
        out = np.zeros(len(hashes), dtype=np.uint16)
        check(lib().kmgpu_get_counts(self.h, _ptr(hashes), len(hashes), _ptr(out)))
        return out

    def _n_kmers(self, off):
        lens = (off[1:] - off[:-1]).astype(np.int64)
        return int(np.maximum(lens - self.ksize + 1, 0).sum())

    def kmer_counts(self, reads, clean=False):
        buf, off = as_reads(reads)
        out = np.zeros(max(self._n_kmers(off), 1), dtype=np.uint16)
        n = C.c_uint64()
        check(lib().kmgpu_kmer_counts(self.h, _ptr(buf), _ptr(off), len(off) - 1, CLEAN if clean else 0, _ptr(out),
                                      C.byref(n)))
        return out[:n.value]

    def kmer_hashes(self, reads, clean=False):
        buf, off = as_reads(reads)
        out = np.zeros(max(self._n_kmers(off), 1), dtype=np.uint64)
        n = C.c_uint64()
        check(lib().kmgpu_kmer_hashes(self.h, _ptr(buf), _ptr(off), len(off) - 1, CLEAN if clean else 0, _ptr(out),
                                      C.byref(n)))
        return out[:n.value]

    def read_medians(self, reads, clean=False):
        buf, off = as_reads(reads)
        nr = len(off) - 1
        med = np.zeros(nr, dtype=np.uint16)
        avg = np.zeros(nr, dtype=np.float32)
        sd = np.zeros(nr, dtype=np.float32)
        nk = np.zeros(nr, dtype=np.uint32)
        check(lib().kmgpu_read_medians(self.h, _ptr(buf), _ptr(off), nr, CLEAN if clean else 0, _ptr(med), _ptr(avg),
                                       _ptr(sd), _ptr(nk)))
        return med, avg, sd, nk

    def batch_read_medians(self, batch, stats=True):
        """read_medians over a device-resident Batch (no upload inside the call); stats=False: medians only"""
        nr = batch.info()[0]
        med = np.zeros(nr, dtype=np.uint16)
        avg = np.zeros(nr, dtype=np.float32) if stats else None
        sd = np.zeros(nr, dtype=np.float32) if stats else None
        nk = np.zeros(nr, dtype=np.uint32) if stats else None
        check(lib().kmgpu_batch_read_medians(self.h, batch.h, _ptr(med), _ptr(avg), _ptr(sd), _ptr(nk)))
        return med, avg, sd, nk

    def median_at_least(self, reads, cutoff, clean=False):
        buf, off = as_reads(reads)
        nr = len(off) - 1
        out = np.zeros(nr, dtype=np.uint8)
        check(lib().kmgpu_median_at_least(self.h, _ptr(buf), _ptr(off), nr, CLEAN if clean else 0, cutoff, _ptr(out)))
        return out

    def abundance_distribution(self, reads, tracking, clean=True, hist=None):
        buf, off = as_reads(reads)
        if hist is None:
            hist = np.zeros(65536, dtype=np.uint64)
        check(lib().kmgpu_abundance_distribution(self.h, tracking.h, _ptr(buf), _ptr(off), len(off) - 1,
                                                 CLEAN if clean else 0, _ptr(hist)))
        return hist

    def trim_batch(self, reads, abund, below=False, clean=False):
        """trim_on_abundance (below=False) / trim_below_abundance (below=True) per read: the length each read keeps"""
        buf, off = as_reads(reads)
        nr = len(off) - 1
        out = np.zeros(max(nr, 1), dtype=np.uint32)
        check(lib().kmgpu_trim_batch(self.h, _ptr(buf), _ptr(off), nr, CLEAN if clean else 0, int(abund), int(below), _ptr(out)))
        return out[:nr]

    def consume_reads_new(self, reads, clean=True):
        """consume + one flag per base: 1 where the k-mer starting there was new in stream order (Storage::add's bool).
        Returns (n_kmers, n_new, flags uint8[n_bases])."""
        buf, off = as_reads(reads)
        nb = int(off[-1] - off[0]) if len(off) > 1 else 0
        bits = np.zeros((nb + 31) // 32 + 1, dtype=np.uint32)
        n, nn = C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_consume_reads_new(self.h, _ptr(buf), _ptr(off), len(off) - 1, CLEAN if clean else 0, _ptr(bits),
                                            C.byref(n), C.byref(nn)))
        flags = np.unpackbits(bits.view(np.uint8), bitorder="little")[:nb]
        return n.value, nn.value, flags

    def first_touch_log(self, on=True):
        check(lib().kmgpu_first_touch_log(self.h, int(on)))

    def first_touch_resolve(self, hist=None):
        """(globally new occurrences of this rank, its rank-local count); hist (uint64[65536]) is accumulated when given"""
        a, b = C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_first_touch_resolve(self.h, C.byref(a), C.byref(b), _ptr(hist) if hist is not None else None))
        return a.value, b.value

    def normalize_batch(self, reads, cutoff, paired=None, clean=False):
        """Digital normalization of a batch in stream order (scripts/normalize-by-median.py:155-179): returns the keep flags
        (uint8 per read) and the number of k-mers consumed.  `paired`: optional uint8 per read, 1 = forms a pair with the next."""
        buf, off = as_reads(reads)
        nr = len(off) - 1
        keep = np.zeros(max(nr, 1), dtype=np.uint8)
        pw = None
        if paired is not None:
            pw = np.ascontiguousarray(paired, dtype=np.uint8)
            assert len(pw) == nr
        kept, kmers = C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_normalize_batch(self.h, _ptr(buf), _ptr(off), nr, CLEAN if clean else 0,
                                          _ptr(pw) if pw is not None else None, int(cutoff), _ptr(keep), C.byref(kept),
                                          C.byref(kmers)))
        return keep[:nr], kmers.value

    def trim_low_abund_pass1(self, reads, trim_at_coverage, cutoff, diginorm_coverage=None, paired=None, clean=False):
        """Pass 1 of trim-low-abund (scripts/trim-low-abund.py:196-238) on a batch in stream order: per-read actions (TLA_*), trim
        lengths (for TLA_TRIM) and the number of k-mers consumed.  `paired` as in normalize_batch."""
        buf, off = as_reads(reads)
        nr = len(off) - 1
        act = np.zeros(max(nr, 1), dtype=np.uint8)
        pos = np.zeros(max(nr, 1), dtype=np.uint32)
        pw = None
        if paired is not None:
            pw = np.ascontiguousarray(paired, dtype=np.uint8)
            assert len(pw) == nr
        kmers = C.c_uint64()
        check(lib().kmgpu_trim_low_abund_pass1(self.h, _ptr(buf), _ptr(off), nr, CLEAN if clean else 0, _ptr(pw), int(trim_at_coverage),
                                               int(cutoff), int(diginorm_coverage or 0), _ptr(act), _ptr(pos), C.byref(kmers)))
        return act[:nr], pos[:nr], kmers.value

    def trim_low_abund_pass2(self, reads, trim_at_coverage, cutoff, variable_coverage=False, paired=None, clean=False):
        """Pass 2 (scripts/trim-low-abund.py:240-271) over saved reads: per-read actions (TLA_TRIM / TLA_KEEP / TLA_DROP) and trim
        lengths.  The table is not changed."""
        buf, off = as_reads(reads)
        nr = len(off) - 1
        act = np.zeros(max(nr, 1), dtype=np.uint8)
        pos = np.zeros(max(nr, 1), dtype=np.uint32)
        pw = None
        if paired is not None:
            pw = np.ascontiguousarray(paired, dtype=np.uint8)
            assert len(pw) == nr
        check(lib().kmgpu_trim_low_abund_pass2(self.h, _ptr(buf), _ptr(off), nr, CLEAN if clean else 0, _ptr(pw), int(trim_at_coverage),
                                               int(cutoff), int(bool(variable_coverage)), _ptr(act), _ptr(pos)))
        return act[:nr], pos[:nr]

    # -- state
    def stats(self):
        a, b = C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_stats(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_stats(self, n_occupied, n_unique):
        check(lib().kmgpu_set_stats(self.h, n_occupied, n_unique))

    def n_occupied(self):
        return self.stats()[0]

    def n_unique_kmers(self):
        return self.stats()[1]

    def table_nbytes(self, i):
        n = C.c_uint64()
        check(lib().kmgpu_table_nbytes(self.h, i, C.byref(n)))
        return n.value

    def table(self, i):
        n = self.table_nbytes(i)
        out = np.zeros(n, dtype=np.uint8)
        check(lib().kmgpu_download_table(self.h, i, _ptr(out), 0, n))
        return out

    def upload_table(self, i, data):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        check(lib().kmgpu_upload_table(self.h, i, _ptr(data), 0, len(data)))

    def bigcounts(self):
        n = C.c_uint64()
        check(lib().kmgpu_bigcount_size(self.h, C.byref(n)))
        keys = np.zeros(max(n.value, 1), dtype=np.uint64)
        vals = np.zeros(max(n.value, 1), dtype=np.uint16)
        check(lib().kmgpu_bigcount_export(self.h, _ptr(keys), _ptr(vals), n.value))
        return keys[:n.value], vals[:n.value]

    def bigcount_import(self, keys, vals):
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        vals = np.ascontiguousarray(vals, dtype=np.uint16)
        check(lib().kmgpu_bigcount_import(self.h, _ptr(keys), _ptr(vals), len(keys)))

    def merge(self, other):
        check(lib().kmgpu_merge(self.h, other.h))

    def recount_occupied(self):
        check(lib().kmgpu_recount_occupied(self.h))

    # -- multi-GPU
    def ipc_export(self):
        out = np.zeros(64 * len(self.sizes), dtype=np.uint8)
        check(lib().kmgpu_ipc_export(self.h, _ptr(out)))
        return out

    def ipc_attach(self, rank, world, all_handles):
        all_handles = np.ascontiguousarray(all_handles, dtype=np.uint8)
        check(lib().kmgpu_ipc_attach(self.h, rank, world, _ptr(all_handles)))

    def ipc_detach(self):
        check(lib().kmgpu_ipc_detach(self.h))

    def reduce_scatter_peers(self):
        check(lib().kmgpu_reduce_scatter_peers(self.h))

    def all_gather_peers(self):
        check(lib().kmgpu_all_gather_peers(self.h))

    # -- measurement
    def profile_reset(self):
        check(lib().kmgpu_profile_reset(self.h))

    def profile_get(self):
        ms, a, b = C.c_double(), C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_profile_get(self.h, C.byref(ms), C.byref(a), C.byref(b)))
        return ms.value, a.value, b.value

    def sync(self):
        check(lib().kmgpu_sync(self.h))

    def reset(self):
        check(lib().kmgpu_reset(self.h))

    def timer_start(self):
        check(lib().kmgpu_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_double()
        check(lib().kmgpu_timer_stop(self.h, C.byref(ms)))
        return ms.value


SHARD_IPC_HANDLES = 5


class Shard:
    """One rank's part of an address-sharded sketch (kmgpu_shard_*)."""

    def __init__(self, storage, hashkind, ksize, full_sizes, rank, world, device=0, max_positions=8 << 20):
        self.full_sizes = [int(x) for x in full_sizes]
        arr = (C.c_uint64 * len(self.full_sizes))(*self.full_sizes)
        self.h = C.c_void_p()
        self.storage, self.rank, self.world, self.max_positions = storage, rank, world, max_positions
        self.ksize = ksize
        self._routed = np.zeros(1, dtype=np.uint64)   # offsets of the reads of the last route call
        check(lib().kmgpu_shard_create(storage, hashkind, ksize, len(self.full_sizes), arr, device, rank, world, max_positions,
                                       C.byref(self.h)))
        # the local sketch is owned by the shard: wrap it without taking ownership
        self.local = Sketch.__new__(Sketch)
        self.local.h = C.c_void_p(lib().kmgpu_shard_local(self.h))
        self.local.sizes = [max(hi - lo, 1) for lo, hi in (self.slice(i) for i in range(len(self.full_sizes)))]
        self.local.storage, self.local.hashkind, self.local.ksize = storage, hashkind, ksize
        self.local.close = lambda: None

    def close(self):
        if getattr(self, "h", None):
            self.local.h = None
            lib().kmgpu_shard_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def slice(self, table):
        lo, hi = C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_shard_slice(self.h, table, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def ipc_export(self):
        out = np.zeros(64 * SHARD_IPC_HANDLES, dtype=np.uint8)
        check(lib().kmgpu_shard_ipc_export(self.h, _ptr(out)))
        return out

    def ipc_attach(self, all_handles):
        all_handles = np.ascontiguousarray(all_handles, dtype=np.uint8)
        check(lib().kmgpu_shard_ipc_attach(self.h, _ptr(all_handles)))

    def route(self, reads, clean=True):
        buf, off = as_reads(reads)
        n = C.c_uint64()
        self._routed = off
        check(lib().kmgpu_shard_route(self.h, _ptr(buf), _ptr(off), len(off) - 1, CLEAN if clean else 0, C.byref(n)))
        return n.value

    def offsets(self):
        check(lib().kmgpu_shard_offsets(self.h))

    def push(self):
        check(lib().kmgpu_shard_push(self.h))

    def apply(self):
        check(lib().kmgpu_shard_apply(self.h))

    def count_new(self):
        """after every rank has applied the round: how many k-mers of THIS rank's reads were new"""
        n = C.c_uint64()
        check(lib().kmgpu_shard_count_new(self.h, C.byref(n)))
        return n.value

    # -- bigcount (ByteStorage): the switch and the map are the local sketch's; every rank must use the same setting
    def set_use_bigcount(self, on):
        self.local.set_use_bigcount(on)

    def get_use_bigcount(self):
        return self.local.get_use_bigcount()

    def bigcount_events(self):
        """after every rank has applied the round (and before the next route): this rank's k-mers whose N bytes were all 255
        before they arrived, one per distinct hash in the order of its first event -> (hashes uint64, event counts uint32)"""
        n = C.c_uint64()
        check(lib().kmgpu_shard_bigcount_events(self.h, None, None, 0, C.byref(n)))
        keys = np.zeros(max(n.value, 1), dtype=np.uint64)
        counts = np.zeros(max(n.value, 1), dtype=np.uint32)
        check(lib().kmgpu_shard_bigcount_events(self.h, _ptr(keys), _ptr(counts), n.value, C.byref(n)))
        return keys[:n.value], counts[:n.value]

    def bigcount_apply(self, hashes, counts):
        """apply every rank's events of the round, concatenated in rank order, to this rank's bigcount map"""
        hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
        counts = np.ascontiguousarray(counts, dtype=np.uint32)
        check(lib().kmgpu_shard_bigcount_apply(self.h, _ptr(hashes), _ptr(counts), len(hashes)))

    def bigcounts(self):
        """the bigcount map (the same on every rank), in its iteration order: (hashes uint64, counts uint16)"""
        return self.local.bigcounts()

    # -- query rounds: route, offsets, push, then lookup and pull; the getters answer for this rank's reads of the last route
    def lookup(self):
        """owner: answer every record this rank was sent with the counter it addresses (tables are not changed)"""
        check(lib().kmgpu_shard_lookup(self.h))

    def pull(self):
        """sender: read the answers back; count per k-mer = the minimum over the tables"""
        check(lib().kmgpu_shard_pull(self.h))

    def kmer_counts(self):
        off = self._routed
        lens = (off[1:] - off[:-1]).astype(np.int64)
        out = np.zeros(max(int(np.maximum(lens - self.ksize + 1, 0).sum()), 1), dtype=np.uint16)
        n = C.c_uint64()
        check(lib().kmgpu_shard_kmer_counts(self.h, _ptr(out), C.byref(n)))
        return out[:n.value]

    def read_medians(self):
        nr = len(self._routed) - 1
        med = np.zeros(nr, dtype=np.uint16)
        avg = np.zeros(nr, dtype=np.float32)
        sd = np.zeros(nr, dtype=np.float32)
        nk = np.zeros(nr, dtype=np.uint32)
        check(lib().kmgpu_shard_read_medians(self.h, _ptr(med), _ptr(avg), _ptr(sd), _ptr(nk)))
        return med, avg, sd, nk

    def median_at_least(self, cutoff):
        out = np.zeros(len(self._routed) - 1, dtype=np.uint8)
        check(lib().kmgpu_shard_median_at_least(self.h, int(cutoff), _ptr(out)))
        return out

    def trim(self, abund, below=False):
        out = np.zeros(len(self._routed) - 1, dtype=np.uint32)
        check(lib().kmgpu_shard_trim(self.h, int(abund), int(below), _ptr(out)))
        return out

    def stats(self):
        """(n_occupied of this rank's slices, this rank's share of n_unique_kmers, bytes of the receive store)"""
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(lib().kmgpu_shard_stats(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def slice_bytes(self, table):
        """This rank's part of the table image: concatenating the parts of all ranks in rank order gives the
        table a single sketch would hold (slices start on a byte boundary of every storage kind)."""
        lo, hi = self.slice(table)
        if hi <= lo:
            return np.zeros(0, dtype=np.uint8)
        t = self.local.table(table)
        last = hi == self.full_sizes[table]
        if self.storage == BYTE:
            return t[: hi - lo]
        if self.storage == NIBBLE:
            return t if last else t[: (hi - lo) // 2]
        return t if last else t[: (hi - lo) // 8]


def shard_abundance_hist(counts, tracking, hist=None):
    """abundance_distribution over the run both shards last routed: `tracking` ingested it (up to count_new), `counts` answered it
    (pull).  Accumulates into hist (uint64[65536])."""
    if hist is None:
        hist = np.zeros(65536, dtype=np.uint64)
    check(lib().kmgpu_shard_abundance_hist(counts.h, tracking.h, _ptr(hist)))
    return hist


def attach_local_shards(shards):
    arr = (C.c_void_p * len(shards))(*[s.h for s in shards])
    check(lib().kmgpu_shard_attach_local(arr, len(shards)))


def slice_range(n_words, world, rank):
    a, b = C.c_uint64(), C.c_uint64()
    check(lib().kmgpu_slice_range(n_words, world, rank, C.byref(a), C.byref(b)))
    return a.value, b.value


def attach_replicas(sketches):
    arr = (C.c_void_p * len(sketches))(*[s.h for s in sketches])
    check(lib().kmgpu_attach_replicas(arr, len(sketches)))


def reduce_replicas(sketches):
    arr = (C.c_void_p * len(sketches))(*[s.h for s in sketches])
    check(lib().kmgpu_reduce_replicas(arr, len(sketches)))
