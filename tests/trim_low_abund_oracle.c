/*
 * TEST INFRASTRUCTURE — the serial loop of scripts/trim-low-abund.py:196-271 (Trimmer.pass1 / pass2) with
 * khmer/trimming.py:36-66 (trim_record), read by read over the oracle port's sketch (oracle/khmer_oracle.c: get_kmer_counts,
 * get_median_count, median_at_least, consume_string).  Built and loaded by tests/trim_low_abund_oracle.py; linked against
 * libkhmer_oracle.so.  Per-read outcomes as include/kmgpu.h's KMGPU_TLA_*.
 */
#include <stdint.h>
#include <stdlib.h>

typedef struct ko_sketch ko_sketch;
int64_t ko_get_kmer_counts(const ko_sketch* s, const char* seq, uint64_t len, uint16_t* out, int64_t cap);
int ko_median(const ko_sketch* s, const char* seq, uint64_t len, uint16_t* med, float* avg, float* sd);
int ko_median_at_least(const ko_sketch* s, const char* seq, uint64_t len, unsigned cutoff);
int64_t ko_consume_string(ko_sketch* s, const char* seq, uint64_t len);

enum { TLA_DROP = 0, TLA_SKIP = 1, TLA_SAVE = 2, TLA_TRIM = 3, TLA_KEEP = 4 };

/* Hashtable::trim_on_abundance (src/oxli/hashtable.cc:504-530): the length the read keeps.  No k-mer, a single k-mer or a
 * first k-mer below min_abund: 0; first k-mer below at index i >= 1: k - 1 + i; none: the whole read. */
static uint32_t trim_at(const ko_sketch* s, int k, const char* seq, uint64_t len, unsigned min_abund)
{
    if (len < (uint64_t)k) return 0;
    int64_t n = (int64_t)(len - (uint64_t)k + 1);
    uint16_t* c = malloc(2 * (size_t)n);
    ko_get_kmer_counts(s, seq, len, c, n);
    uint64_t t = len;
    if (n == 1 || c[0] < min_abund) t = 0;
    else
        for (int64_t j = 1; j < n; j++)
            if (c[j] < min_abund) {
                t = (uint64_t)k - 1 + (uint64_t)j;
                break;
            }
    free(c);
    return (uint32_t)t;
}

/* Trimmer.pass1 (trim-low-abund.py:196-238): for each bundle (a read, or a read and the next one when pair_with_next[r] != 0;
 * reads shorter than k are removed by the script's reader: DROP, and take no part in their bundle's coverage), med = the minimum
 * over its reads of get_median_count in the table as it is now.  diginorm != 0 and med >= diginorm: SKIP; else
 * med >= trim_at_coverage: TRIM with trim_pos = trim_on_abundance(read, cutoff); else every read is consumed and SAVEd.
 * Sequences are used as given (the caller cleans them).  Returns the number of k-mers consumed. */
int64_t tla_pass1(ko_sketch* s, int k, const char* seqs, const uint64_t* offsets, uint64_t n_reads, const uint8_t* pair_with_next,
                  unsigned trim_at_coverage, unsigned cutoff, unsigned diginorm, uint8_t* action_out, uint32_t* trim_pos_out)
{
    int64_t total = 0;
    for (uint64_t r = 0; r < n_reads;) {
        uint64_t e = r + 1;
        while (e < n_reads && pair_with_next && pair_with_next[e - 1]) e++;
        unsigned med = 0xFFFFFFFFu;
        int any = 0;
        for (uint64_t q = r; q < e; q++) {
            uint16_t m;
            float a, sd;
            if (ko_median(s, seqs + offsets[q], offsets[q + 1] - offsets[q], &m, &a, &sd) == 0) {
                any = 1;
                if (m < med) med = m;
            }
        }
        const int skip = any && diginorm && med >= diginorm;
        const int trim = any && !skip && med >= trim_at_coverage;
        for (uint64_t q = r; q < e; q++) {
            const char* sq = seqs + offsets[q];
            const uint64_t len = offsets[q + 1] - offsets[q];
            trim_pos_out[q] = 0;
            if (!any || len < (uint64_t)k) action_out[q] = TLA_DROP;
            else if (skip) action_out[q] = TLA_SKIP;
            else if (trim) {
                action_out[q] = TLA_TRIM;
                trim_pos_out[q] = trim_at(s, k, sq, len, cutoff);
            } else
                action_out[q] = TLA_SAVE;
        }
        if (any && !skip && !trim)
            for (uint64_t q = r; q < e; q++) total += ko_consume_string(s, seqs + offsets[q], offsets[q + 1] - offsets[q]);
        r = e;
    }
    return total;
}

/* Trimmer.pass2 (trim-low-abund.py:240-271) over the saved reads: TRIM; with variable coverage, a bundle whose reads all have
 * median_at_least(trim_at_coverage) (ReadBundle.coverages_at_least, khmer/utils.py:178-180) is TRIMmed and any other KEEPs its
 * reads untrimmed.  Reads shorter than k: DROP. */
void tla_pass2(const ko_sketch* s, int k, const char* seqs, const uint64_t* offsets, uint64_t n_reads, const uint8_t* pair_with_next,
               unsigned trim_at_coverage, unsigned cutoff, int variable, uint8_t* action_out, uint32_t* trim_pos_out)
{
    for (uint64_t r = 0; r < n_reads;) {
        uint64_t e = r + 1;
        while (e < n_reads && pair_with_next && pair_with_next[e - 1]) e++;
        int trim = 1;
        if (variable)
            for (uint64_t q = r; q < e; q++)
                if (ko_median_at_least(s, seqs + offsets[q], offsets[q + 1] - offsets[q], trim_at_coverage) == 0) trim = 0;
        for (uint64_t q = r; q < e; q++) {
            const uint64_t len = offsets[q + 1] - offsets[q];
            trim_pos_out[q] = 0;
            if (len < (uint64_t)k) action_out[q] = TLA_DROP;
            else if (trim) {
                action_out[q] = TLA_TRIM;
                trim_pos_out[q] = trim_at(s, k, seqs + offsets[q], len, cutoff);
            } else
                action_out[q] = TLA_KEEP;
        }
        r = e;
    }
}
