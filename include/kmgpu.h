/*
 * kmgpu.h — C ABI of the B200-native k-mer ingestion backend for khmer's sketches.
 *
 * This is the drop-in boundary: a storage backend that sits behind liboxli's
 * oxli::Storage / oxli::Hashtable interface (reference: include/oxli/storage.hh:56-78,
 * include/oxli/hashtable.hh:127-433).  Plain pointers and sizes only; no C++ or torch types.
 * Every entry point names the reference interface it replaces.  A handle is one sketch
 * (N tables + counters) resident in the HBM of one GPU.
 *
 * Conventions
 *   - All functions return 0 on success or a KMGPU_E* code; kmgpu_last_error() gives the
 *     thread-local message (the C++ host layer rethrows it as oxli_exception /
 *     oxli_file_exception, khmer/_oxli/oxli_exception_convert.cc:9-31).
 *   - Handles are internally locked: several host threads may call into the same handle
 *     (the reference's scripts run T threads in consume_seqfile on one table,
 *     scripts/load-into-counting.py:145-158); calls are applied in arrival order and each
 *     call is applied as if its k-mers were consumed one after another in stream order —
 *     results equal the reference at ONE thread, bit for bit.
 *   - "reads" are passed as one concatenated ASCII buffer plus offsets[n_reads + 1]
 *     (read r = seqs[offsets[r] .. offsets[r+1])), all HOST pointers unless a function
 *     says otherwise.
 *   - There is no CPU fallback: without a CUDA device every call fails with KMGPU_ENODEV.
 */
#ifndef KMGPU_H
#define KMGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMGPU_ABI_VERSION 2 /* 2: batch normalization / trimming / new-flags, first-touch log, HLL registers, five-step sharded rounds */

/* storage kinds — include/oxli/storage.hh: ByteStorage :480, NibbleStorage :241, BitStorage :92 */
enum { KMGPU_BYTE = 0, KMGPU_NIBBLE = 1, KMGPU_BIT = 2 };
/* hash kinds — TwoBitKmerHashIterator (_hash, src/oxli/kmer_hash.cc:65-95, k <= 32) and
 * MurmurKmerHashIterator (_hash_murmur, src/oxli/kmer_hash.cc:177-198) */
enum { KMGPU_TWOBIT = 0, KMGPU_MURMUR = 1 };

/* flags for sequence inputs */
#define KMGPU_CLEAN 1u /* bulk-loader cleaning: ACGT kept, acgt upper-cased, anything else 'A'
                          (Read::set_clean_seq, include/oxli/read_parsers.hh:128-133).  Without it
                          sequences are taken as consume_string takes them (no cleaning,
                          src/oxli/hashtable.cc:280-294): 2-bit code A=0 T=1 C=2 else 3. */

enum {
    KMGPU_OK = 0,
    KMGPU_EINVAL = 1,   /* bad argument                         -> oxli_value_exception */
    KMGPU_ENODEV = 2,   /* no CUDA device / driver              -> oxli_exception       */
    KMGPU_ECUDA = 3,    /* CUDA runtime error                   -> oxli_exception       */
    KMGPU_ENOMEM = 4,   /* device or host allocation failed     -> oxli_exception       */
    KMGPU_ENONACGT = 5, /* Murmur hashing of an uncleaned sequence holding non-ACGT bytes */
    KMGPU_ESHAPE = 6,   /* sketches of different shape          -> oxli_exception       */
    KMGPU_EUNSUPPORTED = 7
};

typedef struct kmgpu_sketch kmgpu_t;
typedef struct kmgpu_batch kmgpu_batch_t;

/* optional hash-band predicate: consume only k-mers with lo <= hash < hi
 * (Hashtable::consume_seqfile_banding, src/oxli/hashtable.cc:192-232; compute_band_interval
 * src/oxli/kmer_hash.cc:262-276) */
typedef struct {
    uint64_t lo, hi;
} kmgpu_band_t;

/* optional mask predicate: consume only k-mers whose count in `mask` is <= threshold
 * (or >= threshold when consume_masked != 0) — Hashtable::consume_seqfile_with_mask,
 * src/oxli/hashtable.cc:152-190 */
typedef struct {
    kmgpu_t* mask;
    uint32_t threshold;
    int consume_masked;
} kmgpu_mask_t;

const char* kmgpu_last_error(void);
int kmgpu_abi_version(void);
int kmgpu_device_count(int* n);
/* page-locked host memory for read batches (uploads from it are asynchronous and run at PCIe speed) */
int kmgpu_alloc_pinned(size_t nbytes, void** out);
int kmgpu_free_pinned(void* p);

/* ---- lifetime -------------------------------------------------------------------------
 * Replaces: ByteStorage/NibbleStorage/BitStorage constructors + _allocate_counters
 * (include/oxli/storage.hh:118-130, :283-297, :501-523) and the Hashtable/MurmurHashtable choice of
 * hash function (include/oxli/hashtable.hh:143-172, :494-520).  `sizes` are the table sizes in BINS
 * (bytes / nibbles / bits), normally get_n_primes_near_x (hashtable.hh:99-123). */
int kmgpu_create(int storage, int hash, int ksize, int n_tables, const uint64_t* sizes, int device,
                 kmgpu_t** out);
int kmgpu_destroy(kmgpu_t* h);
/* back to the freshly constructed state: zero tables, counters and bigcount map (what constructing a new
 * Hashtable does, without re-allocating) */
int kmgpu_reset(kmgpu_t* h);

/* Storage::set_use_bigcount / get_use_bigcount (src/oxli/storage.cc:50-61): only ByteStorage. */
int kmgpu_set_use_bigcount(kmgpu_t* h, int on);
int kmgpu_get_use_bigcount(kmgpu_t* h, int* on);

/* ---- bulk ingestion --------------------------------------------------------------------
 * Replaces the per-read loop of Hashtable::consume_seqfile (src/oxli/hashtable.cc:126-150) minus the
 * file parsing: clean (flag), iterate k-mers (KmerIterator, src/oxli/kmer_hash.cc:278-343), store->add
 * (storage.hh:571-624 / :320-359 / :172-199).  n_kmers_out receives the number of k-mers consumed
 * (= sum over reads of max(0, len - k + 1), or the number passing band/mask). */
int kmgpu_consume_reads(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads,
                        uint32_t flags, const kmgpu_band_t* band, const kmgpu_mask_t* mask,
                        uint64_t* n_kmers_out);

/* kmgpu_consume_reads that also returns, per base of [offsets[0], offsets[n_reads]), whether the k-mer starting there was NEW —
 * the bool Storage::add / test_and_set_bits returns for it in stream order (storage.hh:172-199, :564-569, :571-624).  Replaces the
 * per-k-mer `store->test_and_set_bits(kmer)` of Hashgraph::consume_sequence_and_tag (src/oxli/hashgraph.cc:200-271): the tag scan over
 * these bits stays on the host.  newbits_out holds ceil((offsets[n_reads] - offsets[0]) / 32) words, bit b of word w = base 32 w + b. */
int kmgpu_consume_reads_new(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                            uint32_t* newbits_out, uint64_t* n_kmers_out, uint64_t* n_new_out);

/* Same, from 2-bit packed host buffers as produced by the host read feed: 64-bit words, 32 bases per
 * word, first base in the two most significant bits, code A=0 T=1 C=2 G=3
 * (include/oxli/kmer_hash.hh:70-72); reads are concatenated without padding, offsets in bases. */
int kmgpu_consume_packed(kmgpu_t* h, const uint64_t* words, uint64_t n_words, const uint64_t* offsets,
                         uint64_t n_reads, const kmgpu_band_t* band, const kmgpu_mask_t* mask,
                         uint64_t* n_kmers_out);

/* Device-resident read batches (inputs already in HBM): upload once, consume many times. */
int kmgpu_batch_create(int device, const char* seqs, const uint64_t* offsets, uint64_t n_reads,
                       uint32_t flags, int ksize, kmgpu_batch_t** out);
int kmgpu_batch_destroy(kmgpu_batch_t* b);
int kmgpu_batch_info(const kmgpu_batch_t* b, uint64_t* n_reads, uint64_t* n_bases, uint64_t* device_bytes);
int kmgpu_consume_batch(kmgpu_t* h, const kmgpu_batch_t* b, const kmgpu_band_t* band,
                        const kmgpu_mask_t* mask, uint64_t* n_kmers_out);
/* kmgpu_read_medians over a device-resident batch (no upload inside the call): one entry per read of the batch in the four
 * output arrays (each may be NULL).  Fails with KMGPU_EUNSUPPORTED when the batch holds a read longer than a device chunk. */
int kmgpu_batch_read_medians(kmgpu_t* h, const kmgpu_batch_t* b, uint16_t* median_out, float* average_out, float* stddev_out,
                             uint32_t* n_kmers_out);

/* Hashtable::add(HashIntoType) / count (hashtable.hh:222-237): add already-hashed k-mers in order;
 * is_new_out[i] (nullable) = the bool Storage::add returns for the i-th hash. */
int kmgpu_add_hashes(kmgpu_t* h, const uint64_t* hashes, uint64_t n, uint8_t* is_new_out);

/* ---- queries ---------------------------------------------------------------------------
 * Storage::get_count (storage.hh:627-649 / :362-379 / :207-219) for n hashed k-mers. */
int kmgpu_get_counts(kmgpu_t* h, const uint64_t* hashes, uint64_t n, uint16_t* counts_out);

/* Hashtable::get_kmer_counts (src/oxli/hashtable.cc:403-413) for a set of reads: counts of all k-mers
 * of read 0, then read 1, ... ; counts_out must hold sum(max(0, len_r - k + 1)) entries. */
int kmgpu_kmer_counts(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads,
                      uint32_t flags, uint16_t* counts_out, uint64_t* n_kmers_out);

/* Hashtable::get_kmer_hashes (src/oxli/hashtable.cc:377-386). */
int kmgpu_kmer_hashes(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads,
                      uint32_t flags, uint64_t* hashes_out, uint64_t* n_kmers_out);

/* Hashtable::get_median_count (src/oxli/hashtable.cc:299-328) per read: median = sorted[n/2], float mean,
 * float population stddev.  n_kmers_out[r] == 0 marks reads with no k-mer (the reference throws). */
int kmgpu_read_medians(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads,
                       uint32_t flags, uint16_t* median_out, float* average_out, float* stddev_out,
                       uint32_t* n_kmers_out);

/* Hashtable::median_at_least (src/oxli/hashtable.cc:333-364) per read; out[r] in {0,1}, 2 = no k-mers. */
int kmgpu_median_at_least(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads,
                          uint32_t flags, uint32_t cutoff, uint8_t* out);

/* Hashtable::trim_on_abundance (below == 0: cut at the first k-mer with count < abund) / trim_below_abundance (below != 0: at the
 * first with count > abund) for a batch (src/oxli/hashtable.cc:504-560): trim_pos_out[r] = the length read r keeps. */
int kmgpu_trim_batch(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                     uint32_t abund, int below, uint32_t* trim_pos_out);

/* Hashtable::abundance_distribution (src/oxli/hashtable.cc:451-493): for every k-mer in stream order,
 * if `tracking` does not hold it, add it there and bump hist[count in `counts`].  hist (65536 entries)
 * is ACCUMULATED into, so a file can be fed in several calls. */
int kmgpu_abundance_distribution(kmgpu_t* counts, kmgpu_t* tracking, const char* seqs,
                                 const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                 uint64_t* hist);

/* Digital normalization, the loop of scripts/normalize-by-median.py:155-179 (Normalizer.__call__) with khmer/utils.py:178-180
 * (ReadBundle.coverages_at_least) for a batch of reads in stream order: a bundle (one read, or a read and the next one when
 * pair_with_next[r] != 0; pair_with_next may be NULL) is kept iff NOT every read of it has median_at_least(cutoff)
 * (src/oxli/hashtable.cc:333-364) in the table as it is when the bundle arrives, and a kept bundle is consumed
 * (Hashtable::consume_string) before the next bundle is looked at.  keep_out[r] = 1 for kept reads.  Reads without a k-mer never
 * make their bundle kept (the script drops them before this loop).  Results equal the serial loop bit for bit: keep flags,
 * tables, n_occupied, n_unique_kmers, bigcount map.  Cutoffs above 255 on a bigcount ByteStorage are not supported. */
int kmgpu_normalize_batch(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                          const uint8_t* pair_with_next, uint32_t cutoff, uint8_t* keep_out, uint64_t* n_kept_out,
                          uint64_t* n_kmers_out);

/* per-read outcome of the streaming trimmer (kmgpu_trim_low_abund_pass1 / pass2) */
enum { KMGPU_TLA_DROP = 0,   /* no k-mer (shorter than k): the script's reader removes it; never makes its bundle consumed */
       KMGPU_TLA_SKIP = 1,   /* pass 1, --diginorm: med >= D */
       KMGPU_TLA_SAVE = 2,   /* pass 1: consumed, saved for pass 2 */
       KMGPU_TLA_TRIM = 3,   /* trim_pos_out[r] = the length trim_on_abundance(read, C) keeps */
       KMGPU_TLA_KEEP = 4 }; /* pass 2 with variable coverage: written untrimmed */

/* The first pass of scripts/trim-low-abund.py:196-238 (Trimmer.pass1) for a batch of reads in stream order, bundles as in
 * kmgpu_normalize_batch.  With med = the bundle's minimum get_median_count in the table as it is when the bundle arrives:
 * med >= diginorm_coverage (0 = off) -> SKIP; else med >= trim_at_coverage -> TRIM against the table at arrival with cutoff;
 * else every read of the bundle is consumed and SAVEd.  May be called on consecutive batches of one stream.  Results equal the
 * serial loop: actions, trim lengths, tables, n_occupied, n_unique_kmers, bigcount map.  n_kmers_out: k-mers consumed.
 * Cutoffs above 255 on a bigcount ByteStorage are not supported. */
int kmgpu_trim_low_abund_pass1(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                               const uint8_t* pair_with_next, uint32_t trim_at_coverage, uint32_t cutoff,
                               uint32_t diginorm_coverage /* 0 = off */, uint8_t* action_out, uint32_t* trim_pos_out,
                               uint64_t* n_kmers_out);

/* The second pass (Trimmer.pass2, scripts/trim-low-abund.py:240-271) over the saved reads against the current table: TRIM, or
 * with variable_coverage != 0, TRIM a bundle whose every read has median_at_least(trim_at_coverage) and KEEP the others.
 * The table is not changed. */
int kmgpu_trim_low_abund_pass2(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                               const uint8_t* pair_with_next, uint32_t trim_at_coverage, uint32_t cutoff, int variable_coverage,
                               uint8_t* action_out, uint32_t* trim_pos_out);

/* ---- state -----------------------------------------------------------------------------
 * Storage::n_occupied / n_unique_kmers / n_tables / get_tablesizes (storage.hh:65-74). */
int kmgpu_stats(kmgpu_t* h, uint64_t* n_occupied, uint64_t* n_unique_kmers);
int kmgpu_set_stats(kmgpu_t* h, uint64_t n_occupied, uint64_t n_unique_kmers);
int kmgpu_shape(kmgpu_t* h, int* storage, int* hash, int* ksize, int* n_tables, uint64_t* sizes /*>=n_tables or NULL*/);
int kmgpu_set_ksize(kmgpu_t* h, int ksize);

/* Storage::get_raw_tables (storage.hh:74) and the table payload of save/load
 * (src/oxli/storage.cc:99-136, :582-638, :772-803): byte-exact table images. */
int kmgpu_table_nbytes(kmgpu_t* h, int table, uint64_t* nbytes);
int kmgpu_download_table(kmgpu_t* h, int table, uint8_t* dst, uint64_t offset, uint64_t nbytes);
int kmgpu_upload_table(kmgpu_t* h, int table, const uint8_t* src, uint64_t offset, uint64_t nbytes);

/* ByteStorage::_bigcounts (storage.hh:513): entries in the iteration order of the
 * std::unordered_map the reference writes to .ct files (src/oxli/storage.cc:623-632). */
int kmgpu_bigcount_size(kmgpu_t* h, uint64_t* n);
int kmgpu_bigcount_export(kmgpu_t* h, uint64_t* hashes, uint16_t* counts, uint64_t cap);
int kmgpu_bigcount_import(kmgpu_t* h, const uint64_t* hashes, const uint16_t* counts, uint64_t n);

/* BitStorage::update_from (src/oxli/storage.cc:63-96) generalised: dst |= src (bits),
 * dst = min(cap, dst + src) per counter (bytes: 255, nibbles: 15); n_occupied is recomputed from
 * table 0.  Shapes must match (KMGPU_ESHAPE otherwise). */
int kmgpu_merge(kmgpu_t* dst, kmgpu_t* src);
int kmgpu_recount_occupied(kmgpu_t* h);

/* ---- multi-GPU (no reference counterpart; SURVEY.md §8e) -----------------------------------
 * Replicated sketches, one per GPU / process, merged over NVLink peer memory.  Each rank exports the
 * IPC handles of its tables, the caller exchanges them (any transport), every rank attaches its
 * peers, then:  reduce_scatter (rank r folds slice r of every peer into its own tables with the
 * saturating add / OR above, reading peers over NVLink)  ->  caller barrier  ->  all_gather (rank r
 * pulls every other slice from its owner)  ->  caller barrier.
 * The merge folds table bytes only; n_occupied is recounted.  A ByteStorage with bigcount on is refused (KMGPU_EUNSUPPORTED): which
 * replica saw a counter's 255th touch is lost, so neither the bigcount map nor counts above 255 could be exact.  n_unique_kmers stays
 * each replica's own count unless the first-touch log is used (below). */
#define KMGPU_IPC_HANDLE_BYTES 64
int kmgpu_ipc_export(kmgpu_t* h, uint8_t* handles /* n_tables * 64 bytes */);
int kmgpu_ipc_attach(kmgpu_t* h, int rank, int world, const uint8_t* all_handles /* world * n_tables * 64 */);
int kmgpu_ipc_detach(kmgpu_t* h);
int kmgpu_reduce_scatter_peers(kmgpu_t* h);
int kmgpu_all_gather_peers(kmgpu_t* h);
/* single-process variant: fold sketches living on different GPUs of this process into replicas[0..n)
 * (peer access enabled internally). */
int kmgpu_reduce_replicas(kmgpu_t** replicas, int n);
/* the attach step of kmgpu_reduce_replicas alone (replica r becomes rank r of n; kmgpu_ipc_detach undoes it): lets a single process
 * call kmgpu_first_touch_resolve on every replica before it merges them */
int kmgpu_attach_replicas(kmgpu_t** replicas, int n);
/* the 32-bit-word range [*w0, *w1) of a table of n_words words that rank `rank` of `world` owns in the
 * reduce-scatter / all-gather above (pure arithmetic, no device needed) */
int kmgpu_slice_range(uint64_t n_words, int world, int rank, uint64_t* w0, uint64_t* w1);

/* Replicated sketches, exact n_unique_kmers and abundance_distribution across ranks (SURVEY.md §8e: "a bin's global first toucher
 * lives on the lowest rank that touched it").  With the first-touch log on, a sketch records, per newly occupied bin, which k-mer
 * occurrence occupied it (and, when it is the tracking filter of kmgpu_abundance_distribution, that k-mer's count).
 * kmgpu_first_touch_resolve — called on every rank of an attached group after all ranks have ingested and BEFORE the tables are
 * merged — returns how many of this rank's occurrences are new when the ranks' read shards are taken in rank order (an occurrence
 * is dropped when every bin it was first to occupy locally is occupied on a lower rank), accumulates their counts into hist
 * (nullable), returns the rank-local number for comparison, and empties the log.  The sum over ranks equals the n_unique_kmers
 * (the histogram) of ONE sketch fed rank 0's reads, then rank 1's, ...  All replicas must start the epoch from the same state
 * (freshly reset, or just merged).  Sketches with the log on always take the grouped path. */
int kmgpu_first_touch_log(kmgpu_t* h, int on);
int kmgpu_first_touch_resolve(kmgpu_t* h, uint64_t* n_new_out, uint64_t* n_local_out, uint64_t* hist);

/* ---- multi-GPU, address-sharded sketches (SURVEY.md §8e, config C5) ---------------------------------
 * For tables too large to replicate: rank r holds the bins [r*S_i, (r+1)*S_i) of table i (S_i: a whole number of super-buckets
 * of 2^(15+s) bins, see kmgpu_shard_slice) as an ordinary local sketch.  A round of the k-mer exchange:
 *     kmgpu_shard_route    every rank hashes its own reads, groups the counter updates by super-bucket of the FULL tables
 *                          (64-bit bins) in its own HBM and posts the per-super-bucket record counts to the owners
 *     kmgpu_shard_offsets  every owner lays out its receive arena exactly (per super-bucket, the senders' runs side by side)
 *     kmgpu_shard_push     every sender writes its runs — contiguous, hundreds of KB each — straight into the owners' arenas over
 *                          NVLink peer memory (plain stores from a copy kernel; no NCCL, no staging on the receiving side)
 *     kmgpu_shard_apply    every owner groups what it received by 32 Ki-bin bucket and applies it in shared memory like a chunk
 *     kmgpu_shard_count_new
 * with a barrier (provided by the caller) after each step; every rank takes part in every round, with zero reads if it has
 * none left.  Positions are global across the ranks of a round (rank * max_positions + position in the rank's reads, i.e. the
 * stream order is rank 0's reads, then rank 1's, ...), so the first toucher of a bin is decided across ranks and n_unique_kmers
 * is exact: it equals one sketch fed the rounds in that order.  Heavily repeated k-mers cannot overflow anything (regions are
 * exact); a round is refused (KMGPU_ENOMEM from kmgpu_shard_apply on that rank, nothing applied there) only if one owner is sent
 * more than 1.5 x what its share of the bins receives on average in a full round.
 * Table bytes and n_occupied are exact (concatenated slices / summed counters equal the single sketch); n_unique_kmers is the
 * sum of the ranks' shares (kmgpu_shard_stats).  The saved table is the concatenation of the ranks' slices in rank order
 * (kmgpu_shard_slice + the local sketch's kmgpu_download_table).
 * Bigcount (ByteStorage, at most 30 tables): kmgpu_set_use_bigcount on every rank's kmgpu_shard_local, the same value on all ranks
 * (it may change between rounds).  Then kmgpu_shard_apply also marks, in its arena, which touches found their byte at 255 (bit 1
 * of its refusal word tells the senders), and each round gains two steps after kmgpu_shard_count_new:
 *     kmgpu_shard_bigcount_events  every sender reads the marks of its records back and lists its k-mers whose N bytes were all 255
 *                                  before they arrived (ByteStorage::add, storage.hh:606-617): one entry per distinct hash with
 *                                  its number of events, in the order of its first event.  KMGPU_ENOMEM if an owner it sent
 *                                  records to refused the round.  hashes == NULL asks for the number only; the list stays
 *                                  until the next route.  Call it before the barrier that ends the round.
 *     kmgpu_shard_bigcount_apply   every rank applies ALL ranks' lists, concatenated in rank order, to its local sketch's map
 * so that every rank holds the map of one sketch fed the rounds in stream order — same entries, same iteration order
 * (kmgpu_bigcount_export on kmgpu_shard_local).  Query rounds then give counts above 255 from that map. */
typedef struct kmgpu_shard kmgpu_shard_t;
#define KMGPU_SHARD_IPC_HANDLES 5 /* receive arena, demand table, receive offsets, refusal / bigcount word, new-position bitmap */
#define KMGPU_MAX_WORLD 16
int kmgpu_shard_create(int storage, int hash, int ksize, int n_tables, const uint64_t* full_sizes, int device,
                       int rank, int world, uint64_t max_positions_per_route, kmgpu_shard_t** out);
int kmgpu_shard_destroy(kmgpu_shard_t* s);
/* the local sketch holding this rank's slices (table downloads work on it as on any sketch; the counts of k-mers come from
 * query rounds, below) */
kmgpu_t* kmgpu_shard_local(kmgpu_shard_t* s);
int kmgpu_shard_slice(kmgpu_shard_t* s, int table, uint64_t* lo, uint64_t* hi);
/* n_occupied of this rank's slices, this rank's share of n_unique_kmers, bytes of its receive store */
int kmgpu_shard_stats(kmgpu_shard_t* s, uint64_t* n_occupied_local, uint64_t* n_unique_share, uint64_t* store_bytes);
/* peers: CUDA-IPC handles (KMGPU_SHARD_IPC_HANDLES * 64 bytes per rank), or direct pointers when all ranks live in one process */
int kmgpu_shard_ipc_export(kmgpu_shard_t* s, uint8_t* handles);
int kmgpu_shard_ipc_attach(kmgpu_shard_t* s, const uint8_t* all_handles);
int kmgpu_shard_attach_local(kmgpu_shard_t** all, int n);
int kmgpu_shard_route(kmgpu_shard_t* s, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                      uint64_t* n_kmers_out);
int kmgpu_shard_offsets(kmgpu_shard_t* s);
int kmgpu_shard_push(kmgpu_shard_t* s);
int kmgpu_shard_apply(kmgpu_shard_t* s);
int kmgpu_shard_count_new(kmgpu_shard_t* s, uint64_t* n_new_out);
int kmgpu_shard_bigcount_events(kmgpu_shard_t* s, uint64_t* hashes, uint32_t* counts, uint64_t cap, uint64_t* n_out);
int kmgpu_shard_bigcount_apply(kmgpu_shard_t* s, const uint64_t* hashes, const uint32_t* counts, uint64_t n);

/* Query rounds: the counts a single sketch would give the k-mers of every rank's reads (get_count, storage.hh:627-649 / :362-379 /
 * :207-219: the minimum over the N tables, whose bins live on different ranks).  The first three steps are those of an ingest round:
 *     kmgpu_shard_route    kmgpu_shard_offsets    kmgpu_shard_push
 *     kmgpu_shard_lookup   every owner overwrites each record of its arena with the counter it addresses (in place: the answer
 *                          replaces the bin bits, the position stays); tables, n_occupied and n_unique are not touched.  A round
 *                          this owner refused fails here with KMGPU_ENOMEM, like kmgpu_shard_apply.
 *     kmgpu_shard_pull     every sender reads its answered records back from the owners over NVLink and keeps, per position of its
 *                          reads, the minimum over the tables.  KMGPU_ENOMEM (and no counts) if an owner it sent records to refused.
 * again with a barrier (provided by the caller) after each step.  The getters below then work on this rank's reads of the round,
 * as last passed to kmgpu_shard_route (nothing restages the local sketch between the route and them); their layouts and values
 * equal the single-sketch calls named beside them (with bigcount on, a count of 255 is the map's value where the map holds the
 * k-mer).  Before a pull they fail with KMGPU_EINVAL. */
int kmgpu_shard_lookup(kmgpu_shard_t* s);
int kmgpu_shard_pull(kmgpu_shard_t* s);
/* kmgpu_kmer_counts: counts_out holds sum(max(0, len_r - k + 1)) entries */
int kmgpu_shard_kmer_counts(kmgpu_shard_t* s, uint16_t* counts_out, uint64_t* n_kmers_out);
/* kmgpu_read_medians (each output may be NULL) / kmgpu_median_at_least / kmgpu_trim_batch: one entry per read of the route call */
int kmgpu_shard_read_medians(kmgpu_shard_t* s, uint16_t* median_out, float* average_out, float* stddev_out, uint32_t* n_kmers_out);
int kmgpu_shard_median_at_least(kmgpu_shard_t* s, uint32_t cutoff, uint8_t* out);
int kmgpu_shard_trim(kmgpu_shard_t* s, uint32_t abund, int below, uint32_t* trim_pos_out);
/* kmgpu_abundance_distribution for one run of reads of this rank, ACCUMULATED into hist (65536 entries): `tracking` (a BIT shard
 * with the counting shard's hash kind and k) has run an ingest round on the run, up to kmgpu_shard_count_new, and `counts` a query
 * round on the same run; hist[count] += 1 for every k-mer of the run that was new in `tracking`.  Summed over the ranks and runs
 * it equals one kmgpu_abundance_distribution fed the rounds in stream order.  KMGPU_EINVAL when the shards live on different
 * devices, differ in max_positions, hash kind or k, or last routed different reads. */
int kmgpu_shard_abundance_hist(kmgpu_shard_t* counts, kmgpu_shard_t* tracking, uint64_t* hist);

/* ---- measurement -----------------------------------------------------------------------
 * Device time (ms) and launch count of the ingest kernel accumulated since the last reset, measured
 * with CUDA events on the handle's own stream. */
int kmgpu_profile_reset(kmgpu_t* h);
int kmgpu_profile_get(kmgpu_t* h, double* ingest_kernel_ms, uint64_t* ingest_launches, uint64_t* all_launches);
int kmgpu_sync(kmgpu_t* h);
/* Device timer: two CUDA events on the handle's stream bracket whatever the handle executes in between
 * (copies included); stop synchronises and returns the elapsed device time in ms. */
int kmgpu_timer_start(kmgpu_t* h);
int kmgpu_timer_stop(kmgpu_t* h, double* ms);

/* ---- HyperLogLog registers (unique-kmers.py; HLLCounter, src/oxli/hllcounter.cc:262-317) -------------------------------
 * The counter's ingest: for every k-mer of the reads, its canonical Murmur hash (_hash_murmur, kmer_hash.cc:177-198); register
 * index = the hash's low n_counters_log2 bits, value = leading zeros of the remaining bits + 1; register = max(register, value).
 * The registers are HLLCounter::counters (one byte each, 2^n_counters_log2 of them): estimate_cardinality() and its bias
 * tables stay with the caller.  consume: HLLCounter::consume_string over every read (KMGPU_CLEAN: Read::set_clean_seq first, as
 * consume_seqfile does); without KMGPU_CLEAN a byte outside ACGT fails with KMGPU_ENONACGT.
 * merge_registers: HLLCounter::merge (replace == 0: element-wise max) / set_counters (replace != 0). */
typedef struct kmgpu_hll kmgpu_hll_t;
int kmgpu_hll_create(int device, int ksize, int n_counters_log2, kmgpu_hll_t** out);
int kmgpu_hll_destroy(kmgpu_hll_t* c);
int kmgpu_hll_consume(kmgpu_hll_t* c, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags, uint64_t* n_kmers_out);
int kmgpu_hll_get_registers(kmgpu_hll_t* c, uint8_t* out);
int kmgpu_hll_merge_registers(kmgpu_hll_t* c, const uint8_t* in, int replace);

#ifdef __cplusplus
}
#endif
#endif /* KMGPU_H */
