"""Streaming abundance trimming: the two passes of khmer's scripts/trim-low-abund.py (Trimmer.pass1 / pass2, :196-271, with
khmer/trimming.py:36-66) over a table on the device, a batch of reads per device call.

    from khmer_b200 import Countgraph
    from khmer_b200.trimming import Trimmer
    t = Trimmer(Countgraph(20, 2e9, 4), cutoff=2, trim_at_coverage=20)
    for name, seq, qual in t.pass1(records):     # records: (name, sequence, quality or None)
        ...
    for name, seq, qual in t.pass2():
        ...
"""

DROP, SKIP, SAVE, TRIM, KEEP = 0, 1, 2, 3, 4   # per-read actions (KMGPU_TLA_* in include/kmgpu.h)


class Trimmer:
    """trim-low-abund.py's Trimmer over a khmer_b200 table (`graph`: any class of the host layer, e.g. Countgraph).

    Pass 1 judges every read bundle against the table as it is when the bundle arrives, as the script does read by read: a bundle
    whose minimum median k-mer count is at least `diginorm_coverage` (when set) is dropped; otherwise one at or above
    `trim_at_coverage` is trimmed at once (each read cut before its first k-mer with a count below `cutoff`); any other is consumed
    into the table and saved, in host memory, for pass 2.  Pass 2 trims the saved reads against the final table; with
    `variable_coverage` a bundle is trimmed only if every read of it has median_at_least(trim_at_coverage), and written whole
    otherwise.  Reads shorter than k are dropped, as the script's reader does, and take no part in their bundle's coverage.
    Sequences are judged cleaned (upper case, anything but ACGT as A) and written as given, truncated at the trim length
    (quality too).

    `paired` (pass1): optional flags parallel to the records, 1 = the record forms a bundle with the next one.  A pair's coverage
    in pass 1 is the minimum over its reads, as ReadBundle does.  Its pass-2 test with `variable_coverage` follows
    ReadBundle.coverages_at_least over the pair; only the script's unpaired outputs are pinned by the reference's md5s, so the
    paired form rests on the script's code alone.

    Counters, as the script keeps them: n_reads and n_bp over the reads of both passes, trimmed_reads (cut or dropped by the trim),
    n_saved (pass 1), n_skipped and bp_skipped (pass 2 reads written untrimmed under variable coverage)."""

    def __init__(self, graph, cutoff=2, trim_at_coverage=20, variable_coverage=False, diginorm_coverage=None, batch_reads=1 << 18):
        self.graph = graph
        self.k = graph.ksize()
        self.cutoff = int(cutoff)
        self.trim_at_coverage = int(trim_at_coverage)
        self.variable_coverage = bool(variable_coverage)
        self.diginorm_coverage = int(diginorm_coverage) if diginorm_coverage else 0
        self.batch_reads = max(1, int(batch_reads))
        self.saved, self.saved_paired = [], []
        self.n_reads = self.n_bp = self.trimmed_reads = self.n_saved = self.n_skipped = self.bp_skipped = 0

    def _batches(self, records, paired):
        """batches of (records, pair flags) that never cut a pair"""
        flags = iter(paired) if paired is not None else None
        recs, pw = [], []
        for rec in records:
            recs.append(rec)
            pw.append(int(next(flags)) if flags is not None else 0)
            if len(recs) >= self.batch_reads and not pw[-1]:
                yield recs, pw
                recs, pw = [], []
        if recs:
            yield recs, pw

    def _trimmed(self, rec, t):
        """trim_record (khmer/trimming.py:36-66) given the trim length: the record to write, or None"""
        name, seq, qual = rec
        if t < self.k:
            self.trimmed_reads += 1
            return None
        if t == len(seq):
            return rec
        self.trimmed_reads += 1
        return (name, seq[:t], qual[:t] if qual is not None else None)

    def _count(self, rec):
        self.n_reads += 1
        self.n_bp += len(rec[1])

    def pass1(self, records, paired=None):
        """yields the records pass 1 writes; keeps the saved ones for pass2()"""
        for recs, pw in self._batches(records, paired):
            act, pos, _ = self.graph.trim_low_abund_pass1([r[1] for r in recs], self.trim_at_coverage, self.cutoff, self.diginorm_coverage,
                                                          pw if paired is not None else [], True)
            for i, (rec, a, t) in enumerate(zip(recs, act, pos)):
                if a == DROP:
                    continue
                self._count(rec)
                if a == TRIM:
                    out = self._trimmed(rec, t)
                    if out is not None:
                        yield out
                elif a == SAVE:
                    self.saved.append(rec)
                    self.saved_paired.append(int(pw[i] and act[i + 1] == SAVE))   # a read the reader drops leaves its mate single
                    self.n_saved += 1

    def pass2(self):
        """yields the records pass 2 writes, from the saved reads in their order"""
        paired = self.saved_paired if any(self.saved_paired) else None
        saved, self.saved, self.saved_paired = self.saved, [], []
        for recs, pw in self._batches(saved, paired):
            act, pos = self.graph.trim_low_abund_pass2([r[1] for r in recs], self.trim_at_coverage, self.cutoff, self.variable_coverage,
                                                       pw if paired is not None else [], True)
            for rec, a, t in zip(recs, act, pos):
                if a == DROP:
                    continue
                self._count(rec)
                if a == KEEP:
                    self.n_skipped += 1
                    self.bp_skipped += len(rec[1])
                    yield rec
                else:
                    out = self._trimmed(rec, t)
                    if out is not None:
                        yield out
