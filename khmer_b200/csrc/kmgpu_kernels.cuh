// Kernels of the k-mer ingestion path.  Every kernel walks the 2-bit read stream (or a hash array) in
// CTA tiles of TILE positions; a "position" is a base index of the chunk's concatenated stream and
// doubles as the k-mer's rank in stream order (the order the reference consumes k-mers at one thread).
#pragma once
#include "kmgpu_device.cuh"

namespace kmgpu {

// per-chunk control block (device), zeroed before each chunk
struct Ctrl {
    unsigned long long n_kmers;   // k-mers consumed (valid and passing band/mask)
    unsigned long long n_z0;      // updates that occupied a bin of table 0      -> n_occupied
    unsigned long long n_zbits;   // updates that occupied a bin of any table    -> #keys for resolution
    unsigned long long n_sat;     // updates that found their byte saturated (the chunk has bigcount candidates)
    unsigned long long n_cross;   // updates that moved a byte 254 -> 255 in this chunk
    unsigned long long n_unique;  // result of the first-toucher resolution
    unsigned long long n_events;  // entries appended to a list (bin list, bigcount records, first-touch log)
    unsigned long long non_acgt;  // pack kernel: bytes outside ACGT seen in raw mode
    unsigned long long n_new_t[32];  // newly occupied bins per table
    unsigned long long pass_list_end[64];  // delta path: bin list entries appended by each (table, block) pass
    unsigned long long overflow;  // bucket path: a bucket ran out of room (the chunk is redone by the delta passes);
                                  // grouped path: bit 2g = a super-bucket region of table group g ran out of room,
                                  // bit 2g+1 = a bucket region did (the group is regrouped with exact offsets)
    unsigned long long queue_overflow;  // address-sharded mode: updates that did not fit a receive queue
};

constexpr int F_MAXT = 10;   // most tables the bins and delta paths take (per-table arrays of fixed size); more: grouped path
constexpr uint64_t FILTER_BITS = 1ull << 23;  // per table
constexpr uint64_t FILTER_WORDS = FILTER_BITS / 32;

struct Input {
    const uint64_t* words;   // SRC 0: packed stream of the chunk (+ TILE_PAD_WORDS zero words)
    const uint32_t* offs;    //        read offsets (n_reads + 1), chunk relative
    const uint32_t* tfr;     //        per tile: last read with offs[r] <= tile start (n_tiles + 1 entries)
    uint32_t n_reads;
    const uint64_t* hashes;  // SRC 1: hash array
    uint32_t n_pos;          // stream positions (bases) or number of hashes
    const uint32_t* read_keep;  // optional: one bit per read of the chunk; reads whose bit is clear yield no k-mers
    const uint32_t* valid;      // optional: precomputed bitmap of the positions where a k-mer starts (k_valid_bits); ignores read_keep
};

struct TileSmem {
    uint64_t words[TILE / 32 + TILE_PAD_WORDS];
    uint32_t valid[TILE / 32];
    uint32_t lut[256];
    uint32_t r_lo, r_hi;
    unsigned long long acc[8];
};

// ---- tile staging --------------------------------------------------------------------------------
// Loads the tile's slice of the packed stream into shared memory (coalesced 8-byte loads), finds the
// reads overlapping the tile with two binary searches, and builds the bitmap of positions where a
// k-mer starts (start + k <= end of its read; reads shorter than k yield none, kmer_hash.cc:278-296).
template <int HK, int SRC>
__device__ __forceinline__ void tile_begin(const Input& in, int k, uint32_t t0, TileSmem& sm)
{
    const int tid = threadIdx.x;
    for (int i = tid; i < TILE / 32; i += THREADS) sm.valid[i] = 0;
    if (tid < 8) sm.acc[tid] = 0;
    if (SRC == 1) {
        __syncthreads();
        uint32_t n = in.n_pos - t0 < (uint32_t)TILE ? in.n_pos - t0 : (uint32_t)TILE;
        for (int i = tid; i < TILE / 32; i += THREADS) {
            uint32_t lo = i * 32;
            sm.valid[i] = lo >= n ? 0u : (n - lo >= 32 ? ~0u : ((1u << (n - lo)) - 1));
        }
        __syncthreads();
        return;
    }
    if (HK == MURMUR) fill_lut4(sm.lut, tid, THREADS);
    const uint64_t* src = in.words + (t0 >> 5);
    for (int i = tid; i < TILE / 32 + TILE_PAD_WORDS; i += THREADS) sm.words[i] = __ldg(src + i);
    __syncthreads();
    // reads overlapping the tile come from the per-tile index k_tile_index built for the chunk (a serial
    // binary search here cost more than the tile's useful work)
    const uint32_t r_lo = in.tfr[blockIdx.x];
    uint32_t r_hi = in.tfr[blockIdx.x + 1] + 1;
    if (r_hi > in.n_reads) r_hi = in.n_reads;
    for (uint32_t r = r_lo + tid; r < r_hi; r += THREADS) {
        uint32_t s = in.offs[r], e = in.offs[r + 1];
        if (e - s < (uint32_t)k) continue;
        if (in.read_keep && !((in.read_keep[r >> 5] >> (r & 31)) & 1u)) continue;
        uint32_t first = s > t0 ? s : t0;
        uint32_t last = e - k;  // inclusive
        if (last >= t0 + TILE) last = t0 + TILE - 1;
        if (first > last) continue;
        uint32_t a = first - t0, b = last - t0;
        for (uint32_t wd = a >> 5; wd <= (b >> 5); wd++) {
            uint32_t lo = wd == (a >> 5) ? (a & 31) : 0;
            uint32_t hi = wd == (b >> 5) ? (b & 31) : 31;
            uint32_t m = (hi == 31 ? ~0u : ((1u << (hi + 1)) - 1)) & ~((1u << lo) - 1);
            atomicOr(&sm.valid[wd], m);
        }
    }
    __syncthreads();
}

template <int HK, int SRC>
__device__ __forceinline__ bool tile_valid(const TileSmem& sm, uint32_t lp)
{
    return (sm.valid[lp >> 5] >> (lp & 31)) & 1u;
}

template <int HK, int SRC>
__device__ __forceinline__ uint64_t tile_hash(const Input& in, const TileSmem& sm, int k, uint32_t t0, uint32_t lp)
{
    if (SRC == 1) return in.hashes[t0 + lp];
    if (HK == TWOBIT) return hash_twobit(sm.words, lp, k);
    return hash_murmur(sm.words, sm.lut, lp, k);
}

__device__ __forceinline__ void tile_accumulate(TileSmem& sm, int slot, unsigned long long v)
{
    v = __reduce_add_sync(0xffffffffu, (unsigned)v);  // per-thread values are < 2^32 per tile
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sm.acc[slot], v);
}

// count of a k-mer in an arbitrary sketch: min over tables (Storage::get_count); no bigcount here
__device__ __forceinline__ uint32_t sketch_count(const SketchDev& S, uint64_t h)
{
    uint32_t mn = S.kind == BYTE ? 255u : S.kind == NIBBLE ? 15u : 1u;
    for (int i = 0; i < S.n_tables; i++) {
        uint64_t bin = mod_magic(h, S.sizes[i], S.magic[i]);
        uint32_t c = S.kind == BYTE ? read_byte(S.tables[i], bin)
                   : S.kind == NIBBLE ? read_nibble(S.tables[i], bin) : read_bit(S.tables[i], bin);
        mn = c < mn ? c : mn;
    }
    return mn;
}

__device__ __forceinline__ bool pred_pass(const Pred& P, const SketchDev& M, uint64_t h)
{
    if (P.band_on && !(h >= P.band_lo && h < P.band_hi)) return false;
    if (P.mask_on) {
        uint32_t c = sketch_count(M, h);
        // mask->get_count(kmer) (hashtable.cc:177-178) is Storage::get_count: a saturated ByteStorage count is replaced by
        // the bigcount map's value (storage.hh:640-647)
        if (c == 255u && P.mask_n_big) {
            uint32_t lo = 0, hi = P.mask_n_big;
            while (lo < hi) {
                uint32_t mid = (lo + hi) >> 1;
                if (P.mask_big_keys[mid] < h) lo = mid + 1; else hi = mid;
            }
            if (lo < P.mask_n_big && P.mask_big_keys[lo] == h) c = P.mask_big_vals[lo];
        }
        return P.mask_ge ? c >= P.mask_threshold : c <= P.mask_threshold;
    }
    return true;
}

// tfr[t] = last read r (0 <= r < n_reads) with offs[r] <= t * TILE, for t = 0..n_tiles (inclusive)
__global__ void k_tile_index(const uint32_t* __restrict__ offs, uint32_t n_reads, uint32_t n_tiles, uint32_t* __restrict__ tfr)
{
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    uint64_t start = (uint64_t)t * TILE;
    uint32_t lo = 0, hi = n_reads ? n_reads - 1 : 0;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if ((uint64_t)offs[mid] <= start) lo = mid; else hi = mid - 1;
    }
    tfr[t] = lo;
}

// bitmap of the positions where a k-mer starts (start + k <= end of its read), one thread per read; `out` zeroed before.
// Computed once per staged chunk so that the grouping kernel's CTAs load it instead of rebuilding it from the read offsets
// (a dependent chain of three global loads per tile and table).
__global__ void k_valid_bits(const uint32_t* __restrict__ offs, uint32_t n_reads, int k, uint32_t* __restrict__ out)
{
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const uint32_t s = offs[r], e = offs[r + 1];
    if (e - s < (uint32_t)k) return;
    const uint32_t a = s, b = e - k;   // inclusive
    for (uint32_t wd = a >> 5; wd <= (b >> 5); wd++) {
        const uint32_t lo = wd == (a >> 5) ? (a & 31) : 0;
        const uint32_t hi = wd == (b >> 5) ? (b & 31) : 31;
        const uint32_t m = (hi == 31 ? ~0u : ((1u << (hi + 1)) - 1)) & ~((1u << lo) - 1);
        if (m == ~0u) out[wd] = m;   // a word wholly inside one read is nobody else's
        else atomicOr(&out[wd], m);
    }
}

// ---- bigcount support --------------------------------------------------------------------------------
// k-mers that found all N bytes saturated (ByteStorage::add storage.hh:606-617) are shipped to the host,
// which owns the std::unordered_map and applies them in stream order.
struct Event {
    uint64_t hash;
    uint32_t pos;
    uint32_t info;  // crossmask | allsat_after << 30
};

// ---- queries ---------------------------------------------------------------------------------------
// Storage::get_count per position (min over tables; saturated bytes looked up in the sorted device copy
// of the bigcount map, storage.hh:640-647), optionally also the hash.
template <int KIND, int HK, int SRC>
__global__ void __launch_bounds__(THREADS)
k_counts(SketchDev S, HashCfg H, Input in, const uint64_t* __restrict__ big_keys, const uint16_t* __restrict__ big_vals,
         uint32_t n_big, uint16_t* __restrict__ counts, uint64_t* __restrict__ hashes, const uint32_t* __restrict__ only_bits, int t_lo, int t_hi)
{
    // tables [t_lo, t_hi): all of them in one launch, or one table per launch when every table fits L2 on its own (random loads
    // from an L2-resident table run several times faster than from HBM; the later passes fold into counts[] with min)
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
    for (uint32_t lp = threadIdx.x; lp < TILE && t0 + lp < in.n_pos; lp += THREADS) {
        if (!tile_valid<HK, SRC>(sm, lp)) continue;
        uint32_t p = t0 + lp;
        if (only_bits && !((only_bits[p >> 5] >> (p & 31)) & 1u)) continue;
        uint64_t h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
        if (hashes) hashes[p] = h;
        if (!counts) continue;
        uint32_t mn = t_lo ? (uint32_t)counts[p] : counter_cap<KIND>();
        for (int i0 = t_lo; i0 < t_hi; i0 += 4) {   // four tables at a time: all four loads in flight before the first is used
            uint32_t c[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int i = i0 + j < t_hi ? i0 + j : i0;
                c[j] = read_counter<KIND>(S.tables[i], mod_magic(h, S.sizes[i], S.magic[i]));
            }
#pragma unroll
            for (int j = 0; j < 4; j++) mn = c[j] < mn ? c[j] : mn;
        }
        if (KIND == BYTE && mn == 255u && n_big && t_hi == S.n_tables) {
            uint32_t lo = 0, hi = n_big;
            while (lo < hi) {
                uint32_t mid = (lo + hi) >> 1;
                if (big_keys[mid] < h) lo = mid + 1; else hi = mid;
            }
            if (lo < n_big && big_keys[lo] == h) mn = big_vals[lo];
        }
        counts[p] = (uint16_t)mn;
    }
}

// abundance histogram over the positions marked new in the tracking filter
// (Hashtable::abundance_distribution, src/oxli/hashtable.cc:480-489)
__global__ void k_hist(const uint16_t* __restrict__ counts, const uint32_t* __restrict__ newbits, uint32_t n_pos,
                       unsigned long long* hist)
{
    __shared__ unsigned int sh[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_pos; p += gridDim.x * blockDim.x) {
        if (!((newbits[p >> 5] >> (p & 31)) & 1u)) continue;
        uint32_t c = counts[p];
        if (c < 256) atomicAdd(&sh[c], 1u);
        else atomicAdd(&hist[c], 1ull);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], (unsigned long long)sh[i]);
}

// per-read statistics over the per-position counts: one warp per read.
//   get_median_count (src/oxli/hashtable.cc:299-328): median = sorted[n/2]; mean and population stddev in
//   float with the reference's left-to-right summation order (no FMA contraction);
//   median_at_least (hashtable.cc:333-364): #(count >= cutoff) >= (unsigned)(0.5 + float(n)/2).
__global__ void __launch_bounds__(256)
k_read_stats(const uint16_t* __restrict__ counts, const uint32_t* __restrict__ offs, uint32_t n_reads, int k,
             uint16_t* median, float* average, float* stddev, uint32_t* n_kmers, uint32_t cutoff, uint8_t* at_least)
{
    __shared__ unsigned int hist[8][256];
    __shared__ uint16_t buf[8][256];
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t r = blockIdx.x * 8 + wid;
    if (r >= n_reads) return;
    const uint32_t s = offs[r], e = offs[r + 1];
    const uint32_t n = e - s >= (uint32_t)k ? e - s - k + 1 : 0;
    if (n_kmers && lane == 0) n_kmers[r] = n;
    if (n == 0) {
        if (lane == 0) {
            if (median) median[r] = 0;
            if (average) average[r] = 0.f;
            if (stddev) stddev[r] = 0.f;
            if (at_least) at_least[r] = 2;
        }
        return;
    }
    const uint16_t* c = counts + s;
    if (at_least) {
        unsigned hit = 0;
        for (uint32_t i = lane; i < n; i += 32) hit += c[i] >= cutoff;
        hit = __reduce_add_sync(0xffffffffu, hit);
        unsigned min_req = (unsigned)(0.5 + (double)((float)n / 2));
        if (lane == 0) at_least[r] = hit >= min_req;
    }
    if (!median) return;
    // radix select of rank n/2 over 16-bit values: high byte, then low byte
    const uint32_t rank = n / 2;
    uint32_t prefix = 0, remaining = rank;
    for (int pass = 0; pass < 2; pass++) {
        for (int i = lane; i < 256; i += 32) hist[wid][i] = 0;
        __syncwarp();
        for (uint32_t i = lane; i < n; i += 32) {
            uint32_t v = c[i];
            if (pass == 0) atomicAdd(&hist[wid][v >> 8], 1u);
            else if ((v >> 8) == prefix) atomicAdd(&hist[wid][v & 255], 1u);
        }
        __syncwarp();
        // lane 0 walks the histogram (256 steps, negligible next to the table lookups that fed it)
        uint32_t sel = 0;
        if (lane == 0) {
            uint32_t acc = 0;
            for (int b = 0; b < 256; b++) {
                uint32_t hb = hist[wid][b];
                if (remaining < acc + hb) { sel = b; remaining -= acc; break; }
                acc += hb;
            }
        }
        sel = __shfl_sync(0xffffffffu, sel, 0);
        remaining = __shfl_sync(0xffffffffu, remaining, 0);
        prefix = pass == 0 ? sel : ((prefix << 8) | sel);
        __syncwarp();
    }
    if (lane == 0) median[r] = (uint16_t)prefix;
    // float mean / stddev, strictly sequential like the reference
    float avg = 0.f;
    for (uint32_t base = 0; base < n; base += 256) {
        uint32_t m = n - base < 256 ? n - base : 256;
        for (uint32_t i = lane; i < m; i += 32) buf[wid][i] = c[base + i];
        __syncwarp();
        if (lane == 0)
            for (uint32_t i = 0; i < m; i++) avg = __fadd_rn(avg, (float)buf[wid][i]);
        __syncwarp();
    }
    avg = __shfl_sync(0xffffffffu, avg, 0);
    avg = __fdiv_rn(avg, (float)n);
    float var = 0.f;
    for (uint32_t base = 0; base < n; base += 256) {
        uint32_t m = n - base < 256 ? n - base : 256;
        for (uint32_t i = lane; i < m; i += 32) buf[wid][i] = c[base + i];
        __syncwarp();
        if (lane == 0)
            for (uint32_t i = 0; i < m; i++) {
                float d = __fsub_rn((float)buf[wid][i], avg);
                var = __fadd_rn(var, __fmul_rn(d, d));
            }
        __syncwarp();
    }
    if (lane == 0) {
        var = __fdiv_rn(var, (float)n);
        average[r] = avg;
        stddev[r] = __fsqrt_rn(var);
    }
}

// Hashtable::trim_on_abundance / trim_below_abundance (src/oxli/hashtable.cc:504-560) for a batch, one warp per read, over the
// per-position counts: the length the read keeps.  below == 0: a k-mer is bad when count < abund; below != 0: when count > abund.
// No k-mer, a single k-mer, or a bad first k-mer: 0.  First bad k-mer at index i >= 1: k - 1 + i.  None: the whole read.
__global__ void __launch_bounds__(256)
k_trim_scan(const uint16_t* __restrict__ counts, const uint32_t* __restrict__ offs, uint32_t n_reads, int k, uint32_t abund, int below,
            uint32_t* __restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const uint32_t r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= n_reads) return;
    const uint32_t s = offs[r], e = offs[r + 1], len = e - s;
    const uint32_t n = len >= (uint32_t)k ? len - k + 1 : 0;
    uint32_t first_bad = 0xFFFFFFFFu;
    const uint16_t* c = counts + s;
    for (uint32_t i = lane; i < n; i += 32) {
        const uint32_t v = c[i];
        if (below ? v > abund : v < abund) {
            first_bad = i;
            break;
        }
    }
    first_bad = __reduce_min_sync(0xffffffffu, first_bad);
    if (lane == 0) out[r] = n <= 1 || first_bad == 0 ? 0u : first_bad == 0xFFFFFFFFu ? len : (uint32_t)k - 1 + first_bad;
}

// ---- host feed: ASCII -> 2-bit stream -----------------------------------------------------------------
// One thread per output word (32 bases).  clean != 0: Read::set_clean_seq then twobit_repr
// (read_parsers.cc:53-69, kmer_hash.hh:70-72): A/a 0, T/t 1, C/c 2, G/g 3, anything else 0 ('A').
// clean == 0: twobit_repr alone: 'A' 0, 'T' 1, 'C' 2, anything else 3; bytes outside ACGT are counted so the
// Murmur path (which hashes the letters themselves) can refuse them.
__global__ void k_pack(const uint8_t* __restrict__ ascii, uint32_t n_bases, int clean, uint64_t* __restrict__ words,
                       uint32_t n_words, Ctrl* ctrl)
{
    uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    uint64_t v = 0;
    unsigned bad = 0;
    uint32_t base = w * 32;
    if (base < n_bases) {
        uint32_t m = n_bases - base < 32 ? n_bases - base : 32;
        for (uint32_t j = 0; j < m; j++) {
            uint8_t ch = ascii[base + j];
            uint32_t code;
            if (clean) {
                uint8_t u = ch & 0xDF;  // fold case for letters
                bool letter = (ch >= 'A' && ch <= 'Z') || (ch >= 'a' && ch <= 'z');
                code = !letter ? 0 : u == 'T' ? 1 : u == 'C' ? 2 : u == 'G' ? 3 : 0;
            } else {
                code = ch == 'A' ? 0 : ch == 'T' ? 1 : ch == 'C' ? 2 : 3;
                bad += !(ch == 'A' || ch == 'T' || ch == 'C' || ch == 'G');
            }
            v |= (uint64_t)code << (62 - 2 * j);
        }
    }
    words[w] = v;
    if (bad) atomicAdd(&ctrl->non_acgt, (unsigned long long)bad);
}

// ---- merges -------------------------------------------------------------------------------------------
// dst = dst (+) src over 32-bit words: bytes saturate at 255 (__vaddus4), nibbles at 15, bits OR
// (BitStorage::update_from, src/oxli/storage.cc:63-96, extended to the counting storages).
__device__ __forceinline__ uint32_t merge_word(int kind, uint32_t a, uint32_t b)
{
    if (kind == BYTE) return __vaddus4(a, b);
    if (kind == BIT) return a | b;
    uint32_t lo = __vminu4((a & 0x0F0F0F0Fu) + (b & 0x0F0F0F0Fu), 0x0F0F0F0Fu);
    uint32_t hi = __vminu4(((a >> 4) & 0x0F0F0F0Fu) + ((b >> 4) & 0x0F0F0F0Fu), 0x0F0F0F0Fu);
    return lo | (hi << 4);
}

__global__ void k_merge(int kind, uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, uint64_t n_words)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_words; i += (uint64_t)gridDim.x * blockDim.x)
        dst[i] = merge_word(kind, dst[i], src[i]);
}

// fold word range [w0, w1) of up to 8 peers into dst (peer pointers are NVLink-mapped device memory)
struct PeerPtrs {
    const uint32_t* p[8];
    int n;
};
__global__ void k_merge_peers(int kind, uint32_t* __restrict__ dst, PeerPtrs peers, uint64_t w0, uint64_t w1)
{
    // 16 bytes per thread and peer; the loads from all peers are issued before any is merged (the loop runs over the
    // compile-time bound with a guard so that the pointer array stays in registers / constant space)
    const uint64_t q0 = (w0 + 3) / 4, q1 = w1 / 4;   // whole uint4 groups inside [w0, w1)
    for (uint64_t q = q0 + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; q < q1; q += (uint64_t)gridDim.x * blockDim.x) {
        uint4 v[8];
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (j < peers.n) v[j] = __ldcg(reinterpret_cast<const uint4*>(peers.p[j]) + q);
        uint4 a = reinterpret_cast<uint4*>(dst)[q];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (j >= peers.n) continue;
            a.x = merge_word(kind, a.x, v[j].x);
            a.y = merge_word(kind, a.y, v[j].y);
            a.z = merge_word(kind, a.z, v[j].z);
            a.w = merge_word(kind, a.w, v[j].w);
        }
        reinterpret_cast<uint4*>(dst)[q] = a;
    }
    // ragged head and tail: at most 3 words each
    if (blockIdx.x == 0 && threadIdx.x < 6) {
        const uint64_t head_end = q0 * 4 < w1 ? q0 * 4 : w1, tail_begin = q1 * 4 > head_end ? q1 * 4 : head_end;
        const uint64_t i = threadIdx.x < 3 ? w0 + threadIdx.x : tail_begin + (threadIdx.x - 3);
        if (threadIdx.x < 3 ? i < head_end : i < w1) {
            uint32_t a = dst[i];
#pragma unroll
            for (int j = 0; j < 8; j++)
                if (j < peers.n) a = merge_word(kind, a, __ldcg(peers.p[j] + i));
            dst[i] = a;
        }
    }
}

// number of occupied bins of a table (non-zero bytes / nibbles / set bits) — n_occupied after a merge or upload
__global__ void k_count_occupied(int kind, const uint32_t* __restrict__ t, uint64_t n_words, unsigned long long* out)
{
    unsigned long long cnt = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_words; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t v = t[i];
        if (kind == BIT) cnt += __popc(v);
        else if (kind == BYTE) cnt += __popc(__vcmpne4(v, 0) & 0x01010101u);
        else {
            uint32_t nz = (v | (v >> 1) | (v >> 2) | (v >> 3)) & 0x11111111u;
            cnt += __popc(nz);
        }
    }
    cnt = __reduce_add_sync(0xffffffffu, (unsigned)cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(out, cnt);
}


// =====================================================================================================
// Delta + fold ingestion (byte and nibble storages, tables up to 2^32 bins).
//
// Instead of one compare-and-swap round trip per counter update, the chunk's updates of one table block are
// accumulated with return-less `red.global.add.noftz.f16x2` into a block of half-precision lanes that stays
// L2-resident (2 bytes per bin; profiles/r1_red_ceiling.txt: ~200 G updates/s at <= 50 MB), then one streaming
// kernel folds the block into the byte/nibble table: new = min(cap, old + touches).  A half lane counts
// exactly up to 2048 and then sticks there (2048 + 1 rounds back to 2048), so a lane can neither wrap nor
// carry into its neighbour however hot the bin is, and any touch count >= cap saturates the counter anyway.
// The fold sees, per BIN, the value before the chunk and the number of touches — everything the exactness
// resolutions need (newly occupied bins, bins that saturate inside the chunk) without per-update return values.
// =====================================================================================================
constexpr uint32_t BIN_NONE = 0xFFFFFFFFu;   // position not consumed
constexpr uint64_t BL_NEW = 1ull << 56;      // bin list entry flags: bin went 0 -> occupied in this chunk
constexpr uint64_t BL_CROSS = 1ull << 57;    //                       bin reached the cap in this chunk (bits 48..55: value before)

__device__ __forceinline__ void red_add_half_lane(uint16_t* lanes, uint32_t idx)
{
    // lanes is 4-byte aligned; lane idx&1 of word idx>>1 gets +1.0h
    uint32_t* word = reinterpret_cast<uint32_t*>(lanes) + (idx >> 1);
    uint32_t v = (idx & 1) ? 0x3C000000u : 0x00003C00u;
    asm volatile("red.global.add.noftz.f16x2 [%0], %1;" ::"l"(word), "r"(v) : "memory");
}

// 1. hash every k-mer once and keep its bin in each table: bins[i * stride + pos] (BIN_NONE if not consumed)
// NT > 0: the number of tables is a compile-time constant (table loop unrolled, sizes and magics read as immediate
// constant-bank operands); NT == 0: any number of tables.
template <int HK, int SRC, bool PRED, int NT>
__global__ void __launch_bounds__(THREADS)
k_hashbins(SketchDev S, SketchDev M, HashCfg H, Pred P, Input in, uint32_t* __restrict__ bins, uint64_t stride, Ctrl* ctrl)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
    unsigned n_k = 0;
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        bool consumed = false;
        uint64_t h = 0;
        if (tile_valid<HK, SRC>(sm, lp)) {
            h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
            consumed = !PRED || pred_pass(P, M, h);
        }
        n_k += consumed;
        if (NT > 0) {
#pragma unroll
            for (int i = 0; i < NT; i++) {
                uint32_t b = consumed ? (uint32_t)mod_magic(h, S.sizes[i], S.magic[i]) : BIN_NONE;
                __stcs(&bins[i * stride + t0 + lp], b);
            }
        } else {
            for (int i = 0; i < S.n_tables; i++) {
                uint32_t b = consumed ? (uint32_t)mod_magic(h, S.sizes[i], S.magic[i]) : BIN_NONE;
                __stcs(&bins[i * stride + t0 + lp], b);
            }
        }
    }
    tile_accumulate(sm, 0, n_k);
    __syncthreads();
    if (threadIdx.x == 0 && sm.acc[0]) atomicAdd(&ctrl->n_kmers, sm.acc[0]);
}

// 2. touches of one table block: bins of this table in [lo, hi) -> +1 on their half lane (counting storages)
//    or their bit set in the block's bitmap (BitStorage: OR is idempotent, so a return-less red.or is exact)
template <bool BITS>
__global__ void __launch_bounds__(256)
k_scatter(const uint32_t* __restrict__ bins, uint32_t n_pos, uint32_t lo, uint32_t hi, uint16_t* __restrict__ delta)
{
    const uint32_t i0 = (blockIdx.x * 256u + threadIdx.x) * 8u;
    if (i0 >= n_pos) return;
    uint32_t v[8];
    if (i0 + 8 <= n_pos) {
        uint4 a = __ldcs(reinterpret_cast<const uint4*>(bins + i0));
        uint4 b = __ldcs(reinterpret_cast<const uint4*>(bins + i0 + 4));
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = i0 + j < n_pos ? __ldcs(bins + i0 + j) : BIN_NONE;
    }
    const uint32_t span = hi - lo;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        uint32_t d = v[j] - lo;           // BIN_NONE and bins below lo wrap far above span
        if (d >= span) continue;
        if (BITS) {
            uint32_t* word = reinterpret_cast<uint32_t*>(delta) + (d >> 5);
            asm volatile("red.global.or.b32 [%0], %1;" ::"l"(word), "r"(1u << (d & 31)) : "memory");
        } else {
            red_add_half_lane(delta, d);
        }
    }
}

// 3b. BitStorage fold: 128 bins (4 words) per thread.  new bits = block & ~table (BitStorage::test_and_set_bits,
//     storage.hh:176-195: a k-mer is new iff one of its bits was clear); table |= block; block re-zeroed.
__global__ void __launch_bounds__(256)
k_fold_bits(uint8_t* __restrict__ table, int table_idx, uint32_t lo, uint32_t hi, uint16_t* __restrict__ delta, uint64_t* __restrict__ binlist,
            unsigned long long list_cap, Ctrl* ctrl, int pass)
{
    const uint32_t g = blockIdx.x * 256u + threadIdx.x;   // group of 128 bins
    const uint32_t span = hi - lo;
    unsigned n_new = 0;
    uint4 fresh = make_uint4(0, 0, 0, 0);
    if ((uint64_t)g * 128u < span) {
        uint4* dp = reinterpret_cast<uint4*>(delta) + g;
        uint4 d = *dp;
        if (d.x | d.y | d.z | d.w) {
            *dp = make_uint4(0, 0, 0, 0);
            uint4* tp = reinterpret_cast<uint4*>(table + (lo >> 3)) + g;
            uint4 t = *tp;
            fresh = make_uint4(d.x & ~t.x, d.y & ~t.y, d.z & ~t.z, d.w & ~t.w);
            if (fresh.x | fresh.y | fresh.z | fresh.w) {
                *tp = make_uint4(t.x | d.x, t.y | d.y, t.z | d.z, t.w | d.w);
                n_new = __popc(fresh.x) + __popc(fresh.y) + __popc(fresh.z) + __popc(fresh.w);
            }
        }
    }
    __shared__ unsigned s_cnt[8];
    __shared__ unsigned long long s_base;
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned incl = n_new;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += v;
    }
    if (lane == 31) s_cnt[wid] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned tot = 0;
        for (int w = 0; w < 8; w++) tot += s_cnt[w];
        s_base = tot ? atomicAdd(&ctrl->n_events, (unsigned long long)tot) : 0ull;
        if (tot) {
            if (pass >= 0) atomicAdd(&ctrl->pass_list_end[pass], (unsigned long long)tot);
            atomicAdd(&ctrl->n_zbits, (unsigned long long)tot);
            atomicAdd(&ctrl->n_new_t[table_idx], (unsigned long long)tot);
            if (table_idx == 0) atomicAdd(&ctrl->n_z0, (unsigned long long)tot);
        }
    }
    __syncthreads();
    if (n_new) {
        unsigned long long at = s_base + (incl - n_new);
        for (unsigned w = 0; w < wid; w++) at += s_cnt[w];
        const uint32_t fw[4] = {fresh.x, fresh.y, fresh.z, fresh.w};
        const uint32_t b0 = lo + g * 128u;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t m = fw[q];
            while (m) {
                int bit = __ffs(m) - 1;
                m &= m - 1;
                if (at < list_cap) binlist[at] = BL_NEW | ht_key((uint64_t)(b0 + q * 32 + bit), table_idx);
                at++;
            }
        }
    }
}

// 3. fold the block into the table, 8 bins per thread; zeroes the lanes it consumed.
//    byte: ByteStorage::add's `+1 while < 255` applied `touches` times (storage.hh:599-603);
//    nibble: NibbleStorage::add (storage.hh:345-351), even bin -> high nibble.
template <int KIND>
__global__ void __launch_bounds__(256)
k_fold(uint8_t* __restrict__ table, int table_idx, uint32_t lo, uint32_t hi, uint16_t* __restrict__ delta, uint64_t* __restrict__ binlist,
       unsigned long long list_cap, Ctrl* ctrl, int want_cross, uint8_t* __restrict__ satbits, int pass)
{
    const uint32_t g = blockIdx.x * 256u + threadIdx.x;  // group of 8 bins
    const uint32_t span = hi - lo;
    const uint32_t b0 = lo + g * 8u;
    // per-thread outcome as 8-bit masks over its bins (kept in registers: the list entries are rebuilt from them below)
    unsigned newm = 0, crossm = 0, n_sat = 0;
    uint64_t old64 = 0;
    if (g * 8u < span) {
        // both loads are issued before either is looked at (the table slice streams from HBM, the lanes from L2)
        uint4 d4 = __ldcg(reinterpret_cast<const uint4*>(delta + (size_t)g * 8));
        uint32_t old32 = 0;
        if (KIND == BYTE) old64 = __ldcs(reinterpret_cast<const unsigned long long*>(table + b0));
        else old32 = __ldcs(reinterpret_cast<const uint32_t*>(table + (b0 >> 1)));
        if (d4.x | d4.y | d4.z | d4.w) {
            *reinterpret_cast<uint4*>(delta + (size_t)g * 8) = make_uint4(0, 0, 0, 0);
            const uint32_t dw[4] = {d4.x, d4.y, d4.z, d4.w};
            constexpr uint32_t CAP = KIND == BYTE ? 255u : 15u;
            uint64_t new64 = old64;
            uint32_t new32 = old32;
            unsigned fullm = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                uint32_t hbits = (dw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu;
                if (!hbits) continue;
                uint32_t m = (uint32_t)__half2float(__ushort_as_half((unsigned short)hbits));
                uint32_t s, sh;
                if (KIND == BYTE) {
                    sh = j * 8;
                    s = (uint32_t)(old64 >> sh) & 255u;
                } else {
                    sh = (j >> 1) * 8 + ((j & 1) ? 0 : 4);   // bin b0+j: byte j/2, even bin -> high nibble
                    s = (old32 >> sh) & 15u;
                }
                uint32_t t = s + m;
                uint32_t nv = t > CAP ? CAP : t;
                if (KIND == BYTE) new64 = (new64 & ~(255ull << sh)) | ((uint64_t)nv << sh);
                else new32 = (new32 & ~(15u << sh)) | (nv << sh);
                newm |= (unsigned)(s == 0) << j;
                if (KIND == BYTE) {
                    n_sat += t > CAP;                               // a touch of this chunk found the byte already saturated
                    crossm |= (unsigned)(t >= CAP && s < CAP) << j;  // the byte reached 255 inside this chunk
                    fullm |= (unsigned)(nv == CAP) << j;
                }
            }
            if (KIND == BYTE) {
                *reinterpret_cast<uint64_t*>(table + b0) = new64;
                if (satbits && fullm) {   // one bit per bin "byte is 255": this thread owns the whole byte of the bitmap
                    unsigned m = 0;
#pragma unroll
                    for (int j = 0; j < 8; j++) m |= (unsigned)(((new64 >> (8 * j)) & 255u) == 255u) << j;
                    satbits[b0 >> 3] = (uint8_t)m;
                }
            } else {
                *reinterpret_cast<uint32_t*>(table + (b0 >> 1)) = new32;
            }
        }
    }
    // one list reservation and one set of counter updates per CTA (same-address atomics from every warp of a
    // cold chunk were costing more than the fold itself)
    const unsigned entm = newm | (want_cross ? crossm : 0u);
    const unsigned n_ent = __popc(entm);
    __shared__ unsigned s_cnt[8][4];   // per warp: entries, new, sat, cross
    __shared__ unsigned long long s_base;
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned incl = n_ent;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += v;
    }
    unsigned w_new = __reduce_add_sync(0xffffffffu, (unsigned)__popc(newm));
    unsigned w_sat = __reduce_add_sync(0xffffffffu, n_sat);
    unsigned w_cross = __reduce_add_sync(0xffffffffu, (unsigned)__popc(crossm));
    if (lane == 31) {
        s_cnt[wid][0] = incl;
        s_cnt[wid][1] = w_new;
        s_cnt[wid][2] = w_sat;
        s_cnt[wid][3] = w_cross;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned tot[4] = {0, 0, 0, 0};
        for (int w = 0; w < 8; w++)
            for (int q = 0; q < 4; q++) tot[q] += s_cnt[w][q];
        s_base = 0;
        if (tot[0]) {
            s_base = atomicAdd(&ctrl->n_events, (unsigned long long)tot[0]);
            if (pass >= 0) atomicAdd(&ctrl->pass_list_end[pass], (unsigned long long)tot[0]);
        }
        if (tot[1]) {
            atomicAdd(&ctrl->n_zbits, (unsigned long long)tot[1]);
            atomicAdd(&ctrl->n_new_t[table_idx], (unsigned long long)tot[1]);
            if (table_idx == 0) atomicAdd(&ctrl->n_z0, (unsigned long long)tot[1]);
        }
        if (tot[2]) atomicAdd(&ctrl->n_sat, (unsigned long long)tot[2]);
        if (tot[3]) atomicAdd(&ctrl->n_cross, (unsigned long long)tot[3]);
    }
    __syncthreads();
    if (n_ent) {
        unsigned long long at = s_base + (incl - n_ent);
        for (unsigned w = 0; w < wid; w++) at += s_cnt[w][0];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (!((entm >> j) & 1u)) continue;
            uint64_t entry = ht_key((uint64_t)(b0 + j), table_idx);
            if ((newm >> j) & 1u) entry |= BL_NEW;
            if (KIND == BYTE && want_cross && ((crossm >> j) & 1u)) entry |= BL_CROSS | (((old64 >> (8 * j)) & 255ull) << 48);
            if (at < list_cap) binlist[at] = entry;
            at++;
        }
    }
}

// 4a. hash table of the listed bins carrying `flag` (+ bitmap prefilter); cross entries keep "value before" in vals
__global__ void k_list_register(const uint64_t* __restrict__ binlist, uint64_t n, uint64_t flag, uint64_t* keys, uint32_t* vals,
                                uint64_t mask, uint32_t* filter, int store_before)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = binlist[i];
        if (!(e & flag)) continue;
        uint64_t key = e & 0xFFFFFFFFFFFFull;
        uint64_t s = ht_insert(keys, mask, key);
        if (store_before) vals[s] = (uint32_t)((e >> 48) & 255u);
        if (filter) {
            uint64_t bin = key >> 8;
            int t = (int)(key & 255u);
            atomicOr(&filter[t * FILTER_WORDS + ((bin & (FILTER_BITS - 1)) >> 5)], 1u << (bin & 31));
        }
    }
}

// 4c. per-table stamp tables with packed 8-byte slots (bin << 32 | stamp): one 8-byte load per probe, the stamp
//     lowered with a 64-bit atomicMin (the key half of a slot never changes once claimed).  One table at a
//     time keeps the structure small enough to stay in L2 unless almost every bin of the chunk is new.
constexpr unsigned long long PK_EMPTY = ~0ull;
__device__ __forceinline__ uint64_t pk_slot0(uint32_t bin, uint64_t mask) { return fmix64((uint64_t)bin) & mask; }

__global__ void k_pk_register(const uint64_t* __restrict__ binlist, uint64_t n, int table, unsigned long long* slots, uint64_t mask,
                              uint32_t* filter)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = binlist[i];
        if (!(e & BL_NEW) || (int)(e & 255u) != table) continue;
        uint32_t bin = (uint32_t)((e & 0xFFFFFFFFFFFFull) >> 8);
        unsigned long long fresh = ((unsigned long long)bin << 32) | 0xFFFFFFFFull;
        uint64_t s = pk_slot0(bin, mask);
        while (true) {
            unsigned long long prev = atomicCAS(&slots[s], PK_EMPTY, fresh);
            if (prev == PK_EMPTY || (uint32_t)(prev >> 32) == bin) break;
            s = (s + 1) & mask;
        }
        if (filter) atomicOr(&filter[(bin & (FILTER_BITS - 1)) >> 5], 1u << (bin & 31));
    }
}


// finish one probe whose first slot value `v` has already been loaded
__device__ __forceinline__ void pk_finish(unsigned long long* tb, uint64_t mask, uint64_t s, unsigned long long v, uint32_t bin, uint32_t p)
{
    while (true) {
        if (v == PK_EMPTY) return;
        if ((uint32_t)(v >> 32) == bin) {
            if ((uint32_t)v > p) atomicMin(&tb[s], ((unsigned long long)bin << 32) | p);
            return;
        }
        s = (s + 1) & mask;
        v = __ldcg(&tb[s]);
    }
}

// 4 consecutive positions per thread, their first probes issued together (the kernel is latency-bound otherwise)
__global__ void __launch_bounds__(256)
k_pk_replay(const uint32_t* __restrict__ bins, uint32_t n_pos, uint32_t lo, uint32_t hi, unsigned long long* slots, uint64_t mask,
            const uint32_t* __restrict__ filter)
{
    const uint32_t p0 = (blockIdx.x * 256u + threadIdx.x) * 4u;
    if (p0 >= n_pos) return;
    uint32_t b[4];
    if (p0 + 4 <= n_pos) {
        uint4 q = __ldcs(reinterpret_cast<const uint4*>(bins + p0));
        b[0] = q.x; b[1] = q.y; b[2] = q.z; b[3] = q.w;
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++) b[j] = p0 + j < n_pos ? __ldcs(bins + p0 + j) : BIN_NONE;
    }
    const uint32_t span = hi - lo;
    bool act[4];
    uint64_t s[4];
    unsigned long long v[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        act[j] = b[j] - lo < span;   // BIN_NONE and bins of other blocks fall out
        if (act[j] && filter) act[j] = (__ldg(&filter[(b[j] & (FILTER_BITS - 1)) >> 5]) >> (b[j] & 31)) & 1u;
        s[j] = act[j] ? pk_slot0(b[j], mask) : 0;
    }
#pragma unroll
    for (int j = 0; j < 4; j++) v[j] = act[j] ? __ldcg(&slots[s[j]]) : PK_EMPTY;
#pragma unroll
    for (int j = 0; j < 4; j++)
        if (act[j]) pk_finish(slots, mask, s[j], v[j], b[j], p0 + j);
}

__global__ void k_pk_mark(const unsigned long long* __restrict__ slots, uint64_t n_slots, uint32_t* newbits, Ctrl* ctrl)
{
    unsigned cnt = 0;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < n_slots; s += (uint64_t)gridDim.x * blockDim.x) {
        unsigned long long v = slots[s];
        if (v == PK_EMPTY) continue;
        uint32_t p = (uint32_t)v;
        if (p == 0xFFFFFFFFu) continue;  // registered but never stamped: cannot happen for a touched bin
        uint32_t bit = 1u << (p & 31);
        uint32_t old = atomicOr(&newbits[p >> 5], bit);
        cnt += !(old & bit);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&ctrl->n_unique, (unsigned long long)cnt);
}

// 4d. cold chunks, direct-addressed form: the block's new bins as a bitmap with running ranks (8 bytes per 32 bins:
//     {bits, number of new bins before this word}), so that a toucher finds "is my bin new, and which one is it" with
//     one 8-byte load from a few-MB structure, and lowers minpos[rank] with a return-less red.min.  Against the
//     stamp hash table: no key compare, no probing, 4 instead of 16 bytes of L2 per new bin.
__global__ void k_rank_setbits(const uint64_t* __restrict__ binlist, uint64_t n, uint32_t lo, uint2* rec)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = binlist[i];
        if (!(e & BL_NEW)) continue;
        uint32_t d = (uint32_t)((e & 0xFFFFFFFFFFFFull) >> 8) - lo;
        atomicOr(&rec[d >> 5].x, 1u << (d & 31));
    }
}

// three-step exclusive scan of the words' popcounts: 1024 words per CTA (4 per thread)
__global__ void __launch_bounds__(256) k_rank_sums(const uint2* __restrict__ rec, uint32_t n_words, uint32_t* __restrict__ sums)
{
    const uint32_t w0 = (blockIdx.x * 256u + threadIdx.x) * 4u;
    unsigned c = 0;
#pragma unroll
    for (int j = 0; j < 4; j++)
        if (w0 + j < n_words) c += __popc(rec[w0 + j].x);
    c = __reduce_add_sync(0xffffffffu, c);
    __shared__ unsigned s[8];
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) sums[blockIdx.x] = s[0] + s[1] + s[2] + s[3] + s[4] + s[5] + s[6] + s[7];
}

__global__ void __launch_bounds__(1024) k_rank_scan(uint32_t* sums, uint32_t n)   // one CTA; sums -> exclusive prefix
{
    __shared__ unsigned s_w[32];
    __shared__ unsigned s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        uint32_t i = base + threadIdx.x;
        unsigned v = i < n ? sums[i] : 0, incl = v;
        const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (unsigned)o) incl += t;
        }
        if (lane == 31) s_w[wid] = incl;
        __syncthreads();
        unsigned before = s_carry;
        for (unsigned w = 0; w < wid; w++) before += s_w[w];
        if (i < n) sums[i] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + incl;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) k_rank_prefix(uint2* rec, uint32_t n_words, const uint32_t* __restrict__ sums)
{
    const uint32_t w0 = (blockIdx.x * 256u + threadIdx.x) * 4u;
    unsigned c[4], tot = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        c[j] = w0 + j < n_words ? __popc(rec[w0 + j].x) : 0;
        tot += c[j];
    }
    unsigned incl = tot;
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    __shared__ unsigned s[8];
    if (lane == 31) s[wid] = incl;
    __syncthreads();
    unsigned at = sums[blockIdx.x] + incl - tot;
    for (unsigned w = 0; w < wid; w++) at += s[w];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        if (w0 + j < n_words) rec[w0 + j].y = at;
        at += c[j];
    }
}

// 8 consecutive positions per thread; all record loads are issued before any is used
__global__ void __launch_bounds__(256)
k_rank_replay(const uint32_t* __restrict__ bins, uint32_t n_pos, uint32_t lo, uint32_t hi, const uint2* __restrict__ rec, uint32_t* minpos)
{
    const uint32_t p0 = (blockIdx.x * 256u + threadIdx.x) * 8u;
    if (p0 >= n_pos) return;
    uint32_t v[8];
    if (p0 + 8 <= n_pos) {
        uint4 a = __ldcs(reinterpret_cast<const uint4*>(bins + p0));
        uint4 b = __ldcs(reinterpret_cast<const uint4*>(bins + p0 + 4));
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = p0 + j < n_pos ? __ldcs(bins + p0 + j) : BIN_NONE;
    }
    const uint32_t span = hi - lo;
    uint2 r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        v[j] -= lo;                       // BIN_NONE and bins of other blocks wrap far above span
        r[j] = v[j] < span ? __ldcg(&rec[v[j] >> 5]) : make_uint2(0, 0);
    }
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const uint32_t bit = 1u << (v[j] & 31);
        if (r[j].x & bit) atomicMin(&minpos[r[j].y + __popc(r[j].x & (bit - 1))], p0 + j);
    }
}

__global__ void k_rank_mark(const uint32_t* __restrict__ minpos, uint64_t n, uint32_t* newbits, Ctrl* ctrl)
{
    unsigned cnt = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t p = minpos[i];
        if (p == 0xFFFFFFFFu) continue;
        uint32_t bit = 1u << (p & 31);
        uint32_t old = atomicOr(&newbits[p >> 5], bit);
        cnt += !(old & bit);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&ctrl->n_unique, (unsigned long long)cnt);
}

// fused forms over all tables: table i owns slots [base[i], base[i] + mask[i] + 1) of one buffer
struct PkLayout {
    uint64_t base[F_MAXT];
    uint64_t mask[F_MAXT];   // 0 => table has no new bin in this chunk
    int use_filter;
    uint32_t filter_bits;    // per table, power of two: small enough to sit in L1 when few bins are new
};

__global__ void k_pk_register_all(const uint64_t* __restrict__ binlist, uint64_t n, PkLayout L, unsigned long long* slots, uint32_t* filter)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t e = binlist[i];
        if (!(e & BL_NEW)) continue;
        int t = (int)(e & 255u);
        uint32_t bin = (uint32_t)((e & 0xFFFFFFFFFFFFull) >> 8);
        unsigned long long fresh = ((unsigned long long)bin << 32) | 0xFFFFFFFFull;
        unsigned long long* tb = slots + L.base[t];
        uint64_t s = pk_slot0(bin, L.mask[t]);
        while (true) {
            unsigned long long prev = atomicCAS(&tb[s], PK_EMPTY, fresh);
            if (prev == PK_EMPTY || (uint32_t)(prev >> 32) == bin) break;
            s = (s + 1) & L.mask[t];
        }
        if (L.use_filter) atomicOr(&filter[t * (L.filter_bits >> 5) + ((bin & (L.filter_bits - 1)) >> 5)], 1u << (bin & 31));
    }
}

__global__ void __launch_bounds__(256)
k_pk_replay_all(const uint32_t* __restrict__ bins, uint64_t stride, int n_tables, uint32_t n_pos, PkLayout L, unsigned long long* slots,
                const uint32_t* __restrict__ filter)
{
    uint32_t p = blockIdx.x * 256u + threadIdx.x;
    if (p >= n_pos) return;
    uint32_t b[F_MAXT];
    bool act[F_MAXT];
    // bins of all tables, then all filter words, then all first probes: three rounds of independent loads.  The loops
    // run over the compile-time bound with a guard so that the small arrays live in registers.
#pragma unroll
    for (int t = 0; t < F_MAXT; t++) b[t] = t < n_tables ? __ldcs(&bins[t * stride + p]) : BIN_NONE;
    if (b[0] == BIN_NONE) return;
    const uint32_t fmask = L.filter_bits - 1, fwords = L.filter_bits >> 5;
#pragma unroll
    for (int t = 0; t < F_MAXT; t++) {
        act[t] = t < n_tables && L.mask[t] != 0;
        if (act[t] && L.use_filter) act[t] = (__ldg(&filter[t * fwords + ((b[t] & fmask) >> 5)]) >> (b[t] & 31)) & 1u;
    }
#pragma unroll
    for (int t = 0; t < F_MAXT; t++) {
        if (!act[t]) continue;
        unsigned long long* tb = slots + L.base[t];
        uint64_t s = pk_slot0(b[t], L.mask[t]);
        pk_finish(tb, L.mask[t], s, __ldcg(&tb[s]), b[t], p);
    }
}

// =====================================================================================================
// Bucket path (tables of up to BKT_MAX_BUCKETS x 32 Ki bins): the chunk's updates are first grouped by 32 Ki-bin
// bucket of their table, then one CTA per bucket applies them in SHARED memory and sweeps the result into the
// table.  What the delta passes need 16 sweeps of the bin arrays, ~350 M L2 reductions and a separate
// first-toucher replay for, happens here in two kernels: the per-bin touch counts and the smallest touching
// position (the first toucher in stream order) both live in the CTA's 192 KB of shared memory, so the
// counters, n_occupied, n_unique_kmers (marks in `newbits`) and the saturation bookkeeping all come out of
// the same sweep.  DRAM sees: the bin arrays once, the 8-byte update records once out and once back, the
// table once in and once out.
// =====================================================================================================
struct SatBits {
    const uint8_t* t[F_MAXT];
};

constexpr int BKT_SHIFT = 15;
constexpr uint32_t BKT_BINS = 1u << BKT_SHIFT;   // bins per bucket
constexpr int BKT_MAX_BUCKETS = 6144;            // per table (shared-memory histogram of k_bucketize)
constexpr int BKT_PER = 16;                      // positions per k_bucketize thread (32 with half the threads: measured slower)
constexpr int BKT_TILE = 16384;                  // positions per k_bucketize CTA (smaller tiles: more reservations, shorter runs — measured slower)
constexpr size_t BKT_APPLY_SMEM = (size_t)BKT_BINS * 2 + (size_t)BKT_BINS * 4;
// k_bucketize<T> works on T positions with T/16 threads: sorted records (4 B) + their destinations (4 B) + histogram
// + run offsets (u16 would do; u32 keeps the atomics simple)
constexpr size_t bkt_sort_smem(int tile) { return (size_t)tile * 8 + (size_t)BKT_MAX_BUCKETS * 12; }

struct BucketLayout {
    uint32_t first[F_MAXT + 1];   // table i owns buckets [first[i], first[i+1]) of the record store
    uint32_t cap;                 // records per bucket (<= 65535: a 16-bit lane cannot overflow)
    int n_tables;
};

// 1. group the bins of table blockIdx.y held by T consecutive positions by bucket (counting sort in shared
//    memory), reserve room in each bucket with one atomicAdd per (CTA, bucket), and write the records
//    (position << 15 | bin within bucket) as runs of consecutive addresses.  `bins` and `n_pos` describe one part of the
//    chunk (host input arrives in parts); `pos_base` is the part's first position within the chunk.
template <int T, int PER>
__global__ void __launch_bounds__(T / PER, 1)
k_bucketize(const uint32_t* __restrict__ bins, uint64_t stride, uint32_t n_pos, uint32_t pos_base, BucketLayout L,
            unsigned long long* __restrict__ records, uint32_t* __restrict__ cursors, Ctrl* ctrl)
{
    constexpr int NT = T / PER;              // threads
    constexpr int BPT = (BKT_MAX_BUCKETS + NT - 1) / NT;
    extern __shared__ __align__(16) unsigned char bk_raw[];
    uint2* stage = reinterpret_cast<uint2*>(bk_raw);          // per slot, grouped by bucket: {position in tile << 15 | bin in
                                                              // bucket, bucket << 16 | rank in this CTA's run}
    uint2* run = stage + T;                                   // per bucket: {offset of the run in `stage`, its first index in the bucket}
    uint32_t* hist = reinterpret_cast<uint32_t*>(run + BKT_MAX_BUCKETS);
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_total;
    const int t = blockIdx.y;
    const uint32_t nb = L.first[t + 1] - L.first[t];
    const uint32_t p0 = blockIdx.x * (uint32_t)T;
    const uint32_t tid = threadIdx.x;
    uint32_t bin[PER], rk[PER / 2];
    const uint32_t* src = bins + (size_t)t * stride;
#pragma unroll
    for (int j = 0; j < PER; j++) {
        uint32_t p = p0 + j * NT + tid;
        bin[j] = p < n_pos ? __ldcs(src + p) : BIN_NONE;
    }
    for (uint32_t i = tid; i < nb; i += NT) hist[i] = 0;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PER; j++) {
        uint32_t r = bin[j] != BIN_NONE ? atomicAdd(&hist[bin[j] >> BKT_SHIFT], 1u) : 0u;   // rank inside this CTA's run
        if (j & 1) rk[j >> 1] |= r << 16; else rk[j >> 1] = r;
    }
    __syncthreads();
    // exclusive scan of the bucket counts: BPT consecutive buckets per thread
    uint32_t c[BPT], mine = 0;
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        uint32_t b = tid * BPT + q;
        c[q] = b < nb ? hist[b] : 0;
        mine += c[q];
    }
    uint32_t incl = mine;
    const uint32_t lane = tid & 31, wid = tid >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (uint32_t)o) incl += v;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        uint32_t v = lane < NT / 32 ? s_warp[lane] : 0, w = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t u = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= (uint32_t)o) w += u;
        }
        s_warp[lane] = w - v;
        if (lane == 31) s_total = w;
    }
    __syncthreads();
    // run offsets, and one reservation per non-empty run: the atomics are in flight while the records are placed
    uint32_t at = s_warp[wid] + incl - mine, gbase[BPT];
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        uint32_t b = tid * BPT + q;
        if (b < nb) run[b].x = at;
        gbase[q] = c[q] ? atomicAdd(&cursors[L.first[t] + b], c[q]) : 0u;
        at += c[q];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PER; j++) {
        if (bin[j] == BIN_NONE) continue;
        const uint32_t b = bin[j] >> BKT_SHIFT;
        const uint32_t r = (j & 1) ? rk[j >> 1] >> 16 : rk[j >> 1] & 0xFFFFu;
        stage[run[b].x + r] = make_uint2(((uint32_t)(j * NT + tid) << BKT_SHIFT) | (bin[j] & (BKT_BINS - 1)), (b << 16) | r);
    }
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        uint32_t b = tid * BPT + q;
        if (b < nb) run[b].y = gbase[q];
    }
    __syncthreads();
    const uint32_t total = s_total;
    const size_t base = (size_t)L.first[t] * L.cap;
    bool over = false;
    for (uint32_t s = tid; s < total; s += NT) {
        const uint2 m = stage[s];
        const uint32_t b = m.y >> 16, idx = run[b].y + (m.y & 0xFFFFu);
        if (idx < L.cap)
            records[base + (size_t)b * L.cap + idx] = ((unsigned long long)(pos_base + p0 + (m.x >> BKT_SHIFT)) << BKT_SHIFT) | (m.x & (BKT_BINS - 1));
        else
            over = true;
    }
    if (over) atomicExch(&ctrl->overflow, 1ull);
}

__global__ void k_popc(const uint32_t* __restrict__ words, uint64_t n, unsigned long long* out)
{
    unsigned cnt = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) cnt += __popc(words[i]);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(out, (unsigned long long)cnt);
}

// 2. one CTA per bucket: touch counts (16-bit lanes) and first-toucher positions in shared memory, then the sweep:
//    counter = min(cap, old + touches) (ByteStorage::add storage.hh:599-603, NibbleStorage::add :345-351,
//    BitStorage::test_and_set_bits :176-195), newly occupied bins mark their first toucher in `newbits`
//    (n_unique_kmers = the number of marks, counted by k_popc afterwards).
template <int KIND>
__global__ void __launch_bounds__(1024, 1)
k_apply(SketchDev S, BucketLayout L, const unsigned long long* __restrict__ records, const uint32_t* __restrict__ cursors,
        uint32_t* __restrict__ newbits, uint64_t* __restrict__ binlist, unsigned long long list_cap, Ctrl* ctrl, int want_cross, SatBits sb)
{
    extern __shared__ __align__(16) uint32_t ap_smem[];
    uint32_t* cnt = ap_smem;                    // BKT_BINS / 2 words, two 16-bit lanes each
    uint32_t* minpos = ap_smem + BKT_BINS / 2;  // BKT_BINS words
    if (ctrl->overflow) return;                 // the chunk is redone by the delta passes; leave the tables alone
    const uint32_t n = cursors[blockIdx.x];
    if (n == 0) return;
    int t = 0;
    uint32_t first_t = 0;
    const uint8_t* sat = nullptr;
#pragma unroll
    for (int i = 0; i < F_MAXT; i++)   // compile-time bound: the parameter arrays stay in constant space
        if (i < L.n_tables && blockIdx.x >= L.first[i]) {
            t = i;
            first_t = L.first[i];
            sat = sb.t[i];
        }
    const uint32_t bin0 = (blockIdx.x - first_t) << BKT_SHIFT;
    const uint32_t tid = threadIdx.x;
    const uint64_t size = S.sizes[t];
    uint8_t* table = S.tables[t];
    // the thread's four 8-bin groups of the table are fetched now and used after the records have been counted
    constexpr int GPT = BKT_BINS / 8 / 1024;
    uint64_t oldv[GPT];
#pragma unroll
    for (int q = 0; q < GPT; q++) {
        const uint32_t b0 = bin0 + (q * 1024 + tid) * 8;
        oldv[q] = 0;
        if (b0 < size) {
            if (KIND == BYTE) oldv[q] = __ldcs(reinterpret_cast<const unsigned long long*>(table + b0));
            else if (KIND == NIBBLE) oldv[q] = __ldcs(reinterpret_cast<const uint32_t*>(table + (b0 >> 1)));
            else oldv[q] = __ldcs(table + (b0 >> 3));
        }
    }
    {
        uint4* z = reinterpret_cast<uint4*>(cnt);
        for (uint32_t i = tid; i < BKT_BINS / 8; i += 1024) z[i] = make_uint4(0, 0, 0, 0);
        uint4* f = reinterpret_cast<uint4*>(minpos);
        for (uint32_t i = tid; i < BKT_BINS / 4; i += 1024) f[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
    }
    __syncthreads();
    const unsigned long long* src = records + (size_t)blockIdx.x * L.cap;
    constexpr int RIF = 16;   // records in flight per thread: the loop is latency-bound at one CTA per SM
    for (uint32_t e0 = 0; e0 < n; e0 += RIF * 1024) {
        unsigned long long v[RIF];
#pragma unroll
        for (int j = 0; j < RIF; j++) {
            uint32_t e = e0 + j * 1024 + tid;
            v[j] = e < n ? __ldcs(src + e) : ~0ull;
        }
#pragma unroll
        for (int j = 0; j < RIF; j++) {
            if (v[j] == ~0ull) continue;
            uint32_t lb = (uint32_t)v[j] & (BKT_BINS - 1);
            atomicAdd(&cnt[lb >> 1], (lb & 1) ? 0x10000u : 1u);
            atomicMin(&minpos[lb], (uint32_t)(v[j] >> BKT_SHIFT));
        }
    }
    __syncthreads();
    unsigned n_new = 0, n_sat = 0, n_cross = 0;
#pragma unroll
    for (int q = 0; q < GPT; q++) {
        const uint32_t g = q * 1024 + tid;
        const uint32_t b0 = bin0 + g * 8;
        if (b0 >= size) continue;
        const uint4 c4 = reinterpret_cast<const uint4*>(cnt)[g];
        if (!(c4.x | c4.y | c4.z | c4.w)) continue;
        const uint32_t cw[4] = {c4.x, c4.y, c4.z, c4.w};
        unsigned newm = 0, crossm = 0;
        if (KIND == BYTE) {
            const uint64_t old64 = oldv[q];
            uint64_t new64 = old64;
            unsigned fullm = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                uint32_t m = (cw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu;
                if (!m) continue;
                uint32_t s = (uint32_t)(old64 >> (8 * j)) & 255u, tt = s + m, nv = tt > 255u ? 255u : tt;
                new64 = (new64 & ~(255ull << (8 * j))) | ((uint64_t)nv << (8 * j));
                newm |= (unsigned)(s == 0) << j;
                n_sat += tt > 255u;
                crossm |= (unsigned)(tt >= 255u && s < 255u) << j;
                fullm |= (unsigned)(nv == 255u) << j;
            }
            *reinterpret_cast<uint64_t*>(table + b0) = new64;
            if (want_cross && fullm) {
                unsigned m = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) m |= (unsigned)(((new64 >> (8 * j)) & 255u) == 255u) << j;
                const_cast<uint8_t*>(sat)[b0 >> 3] = (uint8_t)m;
            }
            n_cross += __popc(crossm);
            if (want_cross && crossm) {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if (!((crossm >> j) & 1u)) continue;
                    unsigned long long at = atomicAdd(&ctrl->n_events, 1ull);
                    if (at < list_cap) binlist[at] = BL_CROSS | (((old64 >> (8 * j)) & 255ull) << 48) | ht_key((uint64_t)(b0 + j), t);
                }
            }
        } else if (KIND == NIBBLE) {
            const uint32_t old32 = (uint32_t)oldv[q];
            uint32_t new32 = old32;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                uint32_t m = (cw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu;
                if (!m) continue;
                const uint32_t sh = (j >> 1) * 8 + ((j & 1) ? 0 : 4);   // even bin -> high nibble
                uint32_t s = (old32 >> sh) & 15u, tt = s + m, nv = tt > 15u ? 15u : tt;
                new32 = (new32 & ~(15u << sh)) | (nv << sh);
                newm |= (unsigned)(s == 0) << j;
            }
            *reinterpret_cast<uint32_t*>(table + (b0 >> 1)) = new32;
        } else {
            const unsigned old8 = (unsigned)oldv[q];
            unsigned touched = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) touched |= (unsigned)(((cw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu) != 0) << j;
            newm = touched & ~old8;
            if (newm) table[b0 >> 3] = (uint8_t)(old8 | touched);
        }
        n_new += __popc(newm);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (!((newm >> j) & 1u)) continue;
            const uint32_t p = minpos[g * 8 + j];
            atomicOr(&newbits[p >> 5], 1u << (p & 31));
        }
    }
    // one set of counter updates per CTA
    __shared__ unsigned s_tot[3];
    if (tid < 3) s_tot[tid] = 0;
    __syncthreads();
    n_new = __reduce_add_sync(0xffffffffu, n_new);
    n_sat = __reduce_add_sync(0xffffffffu, n_sat);
    n_cross = __reduce_add_sync(0xffffffffu, n_cross);
    if ((tid & 31) == 0) {
        if (n_new) atomicAdd(&s_tot[0], n_new);
        if (n_sat) atomicAdd(&s_tot[1], n_sat);
        if (n_cross) atomicAdd(&s_tot[2], n_cross);
    }
    __syncthreads();
    if (tid == 0) {
        if (s_tot[0]) {
            atomicAdd(&ctrl->n_zbits, (unsigned long long)s_tot[0]);
            atomicAdd(&ctrl->n_new_t[t], (unsigned long long)s_tot[0]);
            if (t == 0) atomicAdd(&ctrl->n_z0, (unsigned long long)s_tot[0]);
        }
        if (s_tot[1]) atomicAdd(&ctrl->n_sat, (unsigned long long)s_tot[1]);
        if (s_tot[2]) atomicAdd(&ctrl->n_cross, (unsigned long long)s_tot[2]);
    }
}

// chunk-relative 32-bit read offsets from the caller's 64-bit ones, clipped to the chunk [b0, b1)
__global__ void k_clip_offsets(const uint64_t* __restrict__ off64, uint32_t n, uint64_t b0, uint64_t b1, uint32_t* __restrict__ out)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t v = off64[i];
    v = v < b0 ? b0 : (v > b1 ? b1 : v);
    out[i] = (uint32_t)(v - b0);
}

// 5. bigcount scan after the fold.  satbits[t] holds one bit per bin of table t, set iff the byte is 255 (kept by
//    k_fold, rebuilt by k_build_satbits after uploads/merges), 12.5 MB per 1e8-bin table: L2-resident, so nearly
//    every k-mer is dismissed after one cached load.  Reported: k-mers whose N bytes are all 255 now, and — when
//    bins reached 255 inside this chunk — every k-mer touching such a bin (the host needs all their positions).

__global__ void k_build_satbits(const uint8_t* __restrict__ table, uint64_t n_groups, uint8_t* __restrict__ satbits)
{
    for (uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; g < n_groups; g += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t v = *reinterpret_cast<const uint64_t*>(table + g * 8);
        uint32_t m = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) m |= (uint32_t)(((v >> (8 * j)) & 255u) == 255u) << j;
        satbits[g] = (uint8_t)m;
    }
}

// hash of the k-mer at stream position p straight from global memory (rare path: candidates only)
template <int HK, int SRC>
__device__ __forceinline__ uint64_t hash_at(const Input& in, int k, uint32_t p)
{
    if (SRC == 1) return in.hashes[p];
    if (HK == TWOBIT) return hash_twobit(in.words, p, k);
    // Murmur without the shared-memory LUT: rebuild the four-letter words arithmetically
    Murmur F, R;
    F.init();
    R.init();
    bool same = true;
    auto expand = [](uint32_t v, uint64_t& k1, uint64_t& k2) {
        uint64_t w[2] = {0, 0};
        for (int j = 0; j < 16; j++) {
            uint32_t c = (v >> (30 - 2 * j)) & 3u;
            uint64_t ch = c == 0 ? 'A' : c == 1 ? 'T' : c == 2 ? 'C' : 'G';
            w[j >> 3] |= ch << (8 * (j & 7));
        }
        k1 = w[0];
        k2 = w[1];
    };
    int nfull = k >> 4, rem = k & 15;
    for (int b = 0; b < nfull; b++) {
        uint32_t fv = get16(in.words, p + 16 * b);
        uint32_t rv = pair_reverse32(get16(in.words, p + k - 16 * b - 16)) ^ 0x55555555u;
        same &= fv == rv;
        uint64_t k1, k2;
        expand(fv, k1, k2);
        F.block(k1, k2);
        expand(rv, k1, k2);
        R.block(k1, k2);
    }
    if (rem) {
        uint32_t keep = ~0u << (32 - 2 * rem);
        uint32_t fv = get16(in.words, p + 16 * nfull) & keep;
        uint32_t src = get16(in.words, p) >> (32 - 2 * rem);
        uint32_t rv = ((pair_reverse32(src) >> (32 - 2 * rem)) ^ (0x55555555u >> (32 - 2 * rem))) << (32 - 2 * rem);
        same &= fv == rv;
        uint64_t m1 = rem >= 8 ? ~0ull : ((1ull << (8 * rem)) - 1);
        uint64_t m2 = rem > 8 ? ((1ull << (8 * (rem - 8))) - 1) : 0;
        uint64_t k1, k2;
        expand(fv, k1, k2);
        F.tail(k1 & m1, k2 & m2, rem);
        expand(rv, k1, k2);
        R.tail(k1 & m1, k2 & m2, rem);
    }
    uint64_t h = F.finish((uint64_t)k);
    return same ? h : h ^ R.finish((uint64_t)k);
}

template <int HK, int SRC>
__global__ void __launch_bounds__(256)
k_bigscan(int n_tables, HashCfg H, Input in, const uint32_t* __restrict__ bins, uint64_t stride, SatBits sat,
          const uint64_t* __restrict__ keys, uint64_t mask, int have_cross, Event* out, unsigned long long cap, Ctrl* ctrl, uint32_t pos_base)
{
    const uint32_t p = blockIdx.x * 256u + threadIdx.x;   // position inside this part of the chunk (`bins` points at the part)
    if (p >= in.n_pos) return;
    uint32_t b[F_MAXT];
#pragma unroll
    for (int i = 0; i < F_MAXT; i++) b[i] = i < n_tables ? __ldcs(&bins[i * stride + p]) : BIN_NONE;
    if (b[0] == BIN_NONE) return;
    uint32_t satmask = 0;
#pragma unroll
    for (int i = 0; i < F_MAXT; i++) {
        if (i >= n_tables) continue;
        uint32_t bit = (__ldg(&sat.t[i][b[i] >> 3]) >> (b[i] & 7)) & 1u;
        satmask |= bit << i;
    }
    if (!have_cross && satmask != (1u << n_tables) - 1u) return;   // a byte below 255 and no crossing bins to report
    uint32_t cross = 0;
    if (have_cross) {
#pragma unroll
        for (int i = 0; i < F_MAXT; i++)
            if (i < n_tables && (satmask >> i & 1u) && ht_find(keys, mask, ht_key(b[i], i)) != ~0ull) cross |= 1u << i;
    }
    const uint32_t allsat = satmask == (1u << n_tables) - 1u;
    if (!cross && !allsat) return;
    Event e;
    e.hash = hash_at<HK, SRC>(in, H.k, p);
    e.pos = pos_base + p;
    e.info = cross | (allsat << 30);
    unsigned long long at = atomicAdd(&ctrl->n_events, 1ull);
    if (at < cap) out[at] = e;
}

// 6. bigcount events resolved on the device (delta path).
//    For a bin that reached 255 inside the chunk with value s before it, the saturating touch is its
//    need = 255 - s -th touch in stream order; T = that touch's position is found for all such bins at once by a
//    radix select over the positions of the reported touches (one counting pass per position bit).  A k-mer whose N
//    bytes are all 255 after the chunk is a bigcount event iff it comes after T in every such bin it touches.  Events
//    are aggregated per k-mer hash (count, first position) so the host applies one map update per distinct k-mer.
struct SelState {          // per slot of the crossing-bin hash table
    uint32_t* need;        // remaining rank to find (starts at 255 - before)
    uint32_t* prefix;      // bits of T decided so far
    uint32_t* cnt;         // scratch: touches matching the prefix with the current bit clear
};

// slot of every (record, crossing table) pair, computed once
__global__ void k_sel_slots(const Event* __restrict__ recs, uint64_t n_rec, SketchDev S, const uint64_t* __restrict__ keys, uint64_t mask,
                            uint32_t* __restrict__ rec_slot)
{
    uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    Event e = recs[r];
    uint32_t cross = e.info & 0x3FFFFFFFu;
    for (int i = 0; i < S.n_tables; i++) {
        uint32_t sl = 0xFFFFFFFFu;
        if (cross >> i & 1u) sl = (uint32_t)ht_find(keys, mask, ht_key(mod_magic(e.hash, S.sizes[i], S.magic[i]), i));
        rec_slot[r * S.n_tables + i] = sl;
    }
}

__global__ void k_sel_init(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ before, uint64_t n_slots, SelState st)
{
    uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (s >= n_slots) return;
    st.need[s] = keys[s] == HT_EMPTY ? 0u : 255u - before[s];
    st.prefix[s] = 0;
    st.cnt[s] = 0;
}

__global__ void k_sel_count(const Event* __restrict__ recs, uint64_t n_rec, int n_tables, const uint32_t* __restrict__ rec_slot, int bit,
                            SelState st)
{
    uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    uint32_t pos = recs[r].pos;
    if ((pos >> bit) & 1u) return;
    for (int i = 0; i < n_tables; i++) {
        uint32_t sl = rec_slot[r * n_tables + i];
        if (sl == 0xFFFFFFFFu) continue;
        // same bits above `bit` as the prefix decided so far
        if (bit == 31 || (pos >> (bit + 1)) == (st.prefix[sl] >> (bit + 1))) atomicAdd(&st.cnt[sl], 1u);
    }
}

__global__ void k_sel_update(uint64_t n_slots, int bit, SelState st)
{
    uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (s >= n_slots) return;
    uint32_t need = st.need[s];
    if (need) {
        uint32_t c = st.cnt[s];
        if (c < need) {            // the need-th smallest position has this bit set
            st.need[s] = need - c;
            st.prefix[s] |= 1u << bit;
        }
    }
    st.cnt[s] = 0;
}

// events hash table keyed by k-mer hash: count of events, first position
struct EvTable {
    unsigned long long* keys;   // HT_EMPTY = free
    uint32_t* count;
    uint32_t* first;
    uint64_t mask;
};

__global__ void k_ev_decide(const Event* __restrict__ recs, uint64_t n_rec, int n_tables, const uint32_t* __restrict__ rec_slot,
                            const uint32_t* __restrict__ T, int have_cross, EvTable ev, Ctrl* ctrl)
{
    uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    Event e = recs[r];
    if (!(e.info >> 30 & 1u)) return;   // some byte of this k-mer is still below 255
    if (have_cross) {
        for (int i = 0; i < n_tables; i++) {
            uint32_t sl = rec_slot[r * n_tables + i];
            if (sl != 0xFFFFFFFFu && !(e.pos > T[sl])) return;   // arrived before (or as) the saturating touch
        }
    }
    uint64_t s = fmix64(e.hash) & ev.mask;
    while (true) {
        unsigned long long prev = atomicCAS(&ev.keys[s], (unsigned long long)HT_EMPTY, (unsigned long long)e.hash);
        if (prev == HT_EMPTY) atomicAdd(&ctrl->n_unique, 1ull);   // distinct k-mers with events (n_unique is free here)
        if (prev == HT_EMPTY || prev == e.hash) break;
        s = (s + 1) & ev.mask;
    }
    atomicAdd(&ev.count[s], 1u);
    atomicMin(&ev.first[s], e.pos);
}

struct EvOut {
    uint64_t hash;
    uint32_t count;
    uint32_t first;
};

__global__ void k_ev_compact(EvTable ev, EvOut* out, Ctrl* ctrl)
{
    uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (s > ev.mask) return;
    unsigned long long k = ev.keys[s];
    if (k == HT_EMPTY) return;
    unsigned long long at = atomicAdd(&ctrl->n_events, 1ull);
    EvOut o;
    o.hash = k;
    o.count = ev.count[s];
    o.first = ev.first[s];
    out[at] = o;
}

// 7. address-sharded sketches: route every bin of one table to the rank that owns it.  Per CTA the bins are
//    counted per owner in shared memory, one remote atomicAdd per owner reserves a run in that owner's receive
//    queue (NVLink peer memory), then the slice-relative bins are written into the runs.
struct RouteDst {
    uint32_t* queue[8];              // receive queue of this table on every rank
    unsigned long long* cursor[8];   // its fill cursor (same rank's memory)
    int world;
};

__global__ void __launch_bounds__(256)
k_route(const uint32_t* __restrict__ bins, uint32_t n_pos, uint32_t slice, RouteDst dst, unsigned long long cap, Ctrl* ctrl)
{
    __shared__ unsigned cnt[8];
    __shared__ unsigned long long base[8];
    if (threadIdx.x < 8) cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t i0 = (blockIdx.x * 256u + threadIdx.x) * 8u;
    uint32_t v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = i0 + j < n_pos ? __ldcs(bins + i0 + j) : BIN_NONE;
    uint32_t own[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        own[j] = v[j] == BIN_NONE ? 0xFFu : v[j] / slice;
        if (own[j] != 0xFFu) atomicAdd(&cnt[own[j]], 1u);
    }
    __syncthreads();
    if (threadIdx.x < (unsigned)dst.world) {
        unsigned c = cnt[threadIdx.x];
        base[threadIdx.x] = c ? atomicAdd(dst.cursor[threadIdx.x], (unsigned long long)c) : 0ull;
        cnt[threadIdx.x] = 0;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; j++) {
        if (own[j] == 0xFFu) continue;
        unsigned long long at = base[own[j]] + atomicAdd(&cnt[own[j]], 1u);
        if (at < cap) dst.queue[own[j]][at] = v[j] - own[j] * slice;
        else atomicAdd(&ctrl->non_acgt, 1ull);   // overflow of a receive queue (reported by apply)
    }
}

}  // namespace kmgpu
