// Device-side building blocks: 2-bit stream access, the two hash functions, modulo by an
// arbitrary table size, and the three counter reads.  sm_100a only.
#pragma once
#include <cstdint>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace kmgpu {

constexpr int MAX_TABLES = 32;  // NibbleStorage's own limit (include/oxli/storage.hh:278-280)
constexpr int TILE = 4096;      // stream positions (bases) per CTA tile
constexpr int THREADS = 256;
constexpr int MAX_K = 255;      // WordLength is unsigned char (include/oxli/oxli.hh)
constexpr int TILE_PAD_WORDS = (MAX_K + 64 + 31) / 32 + 2;  // extra 64-bit words staged past a tile

enum { BYTE = 0, NIBBLE = 1, BIT = 2 };
enum { TWOBIT = 0, MURMUR = 1 };

struct SketchDev {
    uint8_t* tables[MAX_TABLES];
    uint64_t sizes[MAX_TABLES];
    uint64_t magic[MAX_TABLES];  // floor((2^64 - 1) / size)
    int n_tables;
    int kind;
};

struct HashCfg {
    int kind;
    int k;
};

struct Pred {  // band and mask predicates; both off in the plain path
    int band_on;
    uint64_t band_lo, band_hi;
    int mask_on;
    uint32_t mask_threshold;
    int mask_ge;  // consume_masked: consume iff count >= threshold, else iff count <= threshold
    const uint64_t* mask_big_keys;  // sorted device copy of the mask sketch's bigcount map (ByteStorage with bigcount)
    const uint16_t* mask_big_vals;
    uint32_t mask_n_big;
};

// ------------------------------------------------------------------------------------------------
// h % d for an arbitrary 64-bit d without a hardware divide: q' = mulhi(h, floor((2^64-1)/d)) is
// floor(h/d) or one less, so a single conditional subtract finishes it.  Valid for 1 <= d < 2^63.
// Replaces the `khash % _tablesizes[i]` of every storage (storage.hh:177,321-333,577).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t mod_magic(uint64_t h, uint64_t d, uint64_t m)
{
    uint64_t q = __umul64hi(h, m);
    uint64_t r = h - q * d;
    return r >= d ? r - d : r;
}

// ------------------------------------------------------------------------------------------------
// 2-bit stream: 64-bit words, 32 bases per word, first base in the top two bits.
// ------------------------------------------------------------------------------------------------
// 32 bases starting at stream position p, left-aligned (first base in bits 63..62)
__device__ __forceinline__ uint64_t get32(const uint64_t* __restrict__ w, uint32_t p)
{
    uint32_t i = p >> 5, s = (p & 31) * 2;
    uint64_t hi = w[i], lo = w[i + 1];
    return s ? (hi << s) | (lo >> (64 - s)) : hi;
}
// 16 bases starting at p, left-aligned in 32 bits
__device__ __forceinline__ uint32_t get16(const uint64_t* __restrict__ w, uint32_t p) { return (uint32_t)(get32(w, p) >> 32); }

// reverse the order of the 2-bit groups of a word
__device__ __forceinline__ uint64_t pair_reverse64(uint64_t x)
{
    x = __brevll(x);
    return ((x & 0xAAAAAAAAAAAAAAAAull) >> 1) | ((x & 0x5555555555555555ull) << 1);
}
__device__ __forceinline__ uint32_t pair_reverse32(uint32_t x)
{
    x = __brev(x);
    return ((x & 0xAAAAAAAAu) >> 1) | ((x & 0x55555555u) << 1);
}

// _hash (src/oxli/kmer_hash.cc:65-95) + uniqify_rc (kmer_hash.hh:92-96): the forward hash of the k-mer at
// stream position p is simply its 2k bits of the stream; the reverse hash is the complement (code ^ 1:
// A0<->T1, C2<->G3) of the groups in reverse order.  Equals what KmerIterator's rolling update
// (kmer_hash.cc:310-343) yields for every window.
__device__ __forceinline__ uint64_t hash_twobit(const uint64_t* __restrict__ w, uint32_t p, int k)
{
    uint64_t f = get32(w, p) >> (64 - 2 * k);
    uint64_t mask = k == 32 ? ~0ull : ((1ull << (2 * k)) - 1);
    uint64_t r = (pair_reverse64(f) >> (64 - 2 * k)) ^ (0x5555555555555555ull & mask);
    return f < r ? f : r;
}

// ------------------------------------------------------------------------------------------------
// MurmurHash3_x64_128 (third-party/smhasher/MurmurHash3.cc:56-144) streamed over 16-base blocks that are
// expanded from the 2-bit stream to the ASCII the reference hashes.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
__device__ __forceinline__ uint64_t fmix64(uint64_t v)
{
    v ^= v >> 33;
    v *= 0xff51afd7ed558ccdull;
    v ^= v >> 33;
    v *= 0xc4ceb9fe1a85ec53ull;
    v ^= v >> 33;
    return v;
}

struct Murmur {
    uint64_t h1, h2;
    __device__ __forceinline__ void init() { h1 = 0; h2 = 0; }  // seed 0 (kmer_hash.cc:181)
    __device__ __forceinline__ void block(uint64_t k1, uint64_t k2)
    {
        const uint64_t c1 = 0x87c37b91114253d5ull, c2 = 0x4cf5ad432745937full;
        k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
        h1 = rotl64(h1, 27); h1 += h2; h1 = h1 * 5 + 0x52dce729;
        k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
        h2 = rotl64(h2, 31); h2 += h1; h2 = h2 * 5 + 0x38495ab5;
    }
    // tail of nb (1..15) bytes, already masked to nb bytes
    __device__ __forceinline__ void tail(uint64_t k1, uint64_t k2, int nb)
    {
        const uint64_t c1 = 0x87c37b91114253d5ull, c2 = 0x4cf5ad432745937full;
        if (nb > 8) { k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2; }
        k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
    }
    __device__ __forceinline__ uint64_t finish(uint64_t len)
    {
        h1 ^= len; h2 ^= len;
        h1 += h2; h2 += h1;
        h1 = fmix64(h1); h2 = fmix64(h2);
        h1 += h2;
        return h1;  // khmer keeps out[0] only
    }
};

// lut4[b] = the four ASCII letters of the four bases in byte b (first base = top two bits of b) with the
// first letter in the lowest byte.  Filled once per CTA into shared memory.
__device__ __forceinline__ void fill_lut4(uint32_t* lut, int tid, int nthreads)
{
    for (int b = tid; b < 256; b += nthreads) {
        uint32_t v = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            uint32_t c = (b >> (6 - 2 * j)) & 3;
            uint32_t ch = c == 0 ? 'A' : c == 1 ? 'T' : c == 2 ? 'C' : 'G';
            v |= ch << (8 * j);
        }
        lut[b] = v;
    }
}

// expand 16 left-aligned bases (32 bits) to the two little-endian 8-letter words Murmur reads
__device__ __forceinline__ void expand16(const uint32_t* __restrict__ lut, uint32_t v, uint64_t& k1, uint64_t& k2)
{
    k1 = (uint64_t)lut[v >> 24] | ((uint64_t)lut[(v >> 16) & 255] << 32);
    k2 = (uint64_t)lut[(v >> 8) & 255] | ((uint64_t)lut[v & 255] << 32);
}

// _hash_murmur (src/oxli/kmer_hash.cc:177-198): h = Murmur(kmer)[0], r = Murmur(revcomp)[0]; h ^ r, or h
// alone for a k-mer equal to its reverse complement.
__device__ __forceinline__ uint64_t hash_murmur(const uint64_t* __restrict__ w, const uint32_t* __restrict__ lut,
                                                uint32_t p, int k)
{
    Murmur F, R;
    F.init();
    R.init();
    bool same = true;
    int nfull = k >> 4, rem = k & 15;
    for (int b = 0; b < nfull; b++) {
        uint32_t fv = get16(w, p + 16 * b);
        // reverse-complement letters 16b..16b+15 come from k-mer bases k-16b-16 .. k-16b-1 reversed
        uint32_t rv = pair_reverse32(get16(w, p + k - 16 * b - 16)) ^ 0x55555555u;
        same &= fv == rv;
        uint64_t k1, k2;
        expand16(lut, fv, k1, k2);
        F.block(k1, k2);
        expand16(lut, rv, k1, k2);
        R.block(k1, k2);
    }
    if (rem) {
        uint32_t keep = ~0u << (32 - 2 * rem);
        uint32_t fv = get16(w, p + 16 * nfull) & keep;
        uint32_t src = get16(w, p) >> (32 - 2 * rem);  // first `rem` bases, right-aligned
        uint32_t rv = ((pair_reverse32(src) >> (32 - 2 * rem)) ^ (0x55555555u >> (32 - 2 * rem))) << (32 - 2 * rem);
        same &= fv == rv;
        uint64_t m1 = rem >= 8 ? ~0ull : ((1ull << (8 * rem)) - 1);
        uint64_t m2 = rem > 8 ? ((1ull << (8 * (rem - 8))) - 1) : 0;
        uint64_t k1, k2;
        expand16(lut, fv, k1, k2);
        F.tail(k1 & m1, k2 & m2, rem);
        expand16(lut, rv, k1, k2);
        R.tail(k1 & m1, k2 & m2, rem);
    }
    uint64_t h = F.finish((uint64_t)k);
    if (same) return h;
    return h ^ R.finish((uint64_t)k);
}

// ------------------------------------------------------------------------------------------------
// Counter reads.
// ------------------------------------------------------------------------------------------------
// ByteStorage: one byte per bin.
__device__ __forceinline__ uint32_t read_byte(const uint8_t* table, uint64_t bin) { return __ldcg(table + bin); }

// NibbleStorage: even bin -> high nibble (storage.hh:259-272).
__device__ __forceinline__ uint32_t read_nibble(const uint8_t* table, uint64_t bin)
{
    return (__ldcg(table + (bin >> 1)) >> ((bin & 1) ? 0 : 4)) & 15u;
}

// BitStorage: bit (bin % 8) of byte bin / 8 (storage.hh:176-184).
__device__ __forceinline__ uint32_t read_bit(const uint8_t* table, uint64_t bin)
{
    return (__ldcg(table + (bin >> 3)) >> (bin & 7)) & 1u;
}

template <int KIND>
__device__ __forceinline__ uint32_t read_counter(const uint8_t* t, uint64_t bin)
{
    if (KIND == BYTE) return read_byte(t, bin);
    if (KIND == NIBBLE) return read_nibble(t, bin);
    return read_bit(t, bin);
}
template <int KIND>
__device__ __forceinline__ uint32_t counter_cap()
{
    return KIND == BYTE ? 255u : KIND == NIBBLE ? 15u : 1u;
}

// ------------------------------------------------------------------------------------------------
// open-addressing table keyed by (bin, table) used by the exact "first toucher" resolution
// ------------------------------------------------------------------------------------------------
constexpr uint64_t HT_EMPTY = ~0ull;
__device__ __forceinline__ uint64_t ht_key(uint64_t bin, int table) { return (bin << 8) | (uint64_t)table; }
__device__ __forceinline__ uint64_t ht_slot0(uint64_t key, uint64_t mask) { return fmix64(key) & mask; }

__device__ __forceinline__ uint64_t ht_insert(uint64_t* keys, uint64_t mask, uint64_t key)
{
    uint64_t s = ht_slot0(key, mask);
    while (true) {
        unsigned long long prev = atomicCAS(reinterpret_cast<unsigned long long*>(keys + s), (unsigned long long)HT_EMPTY,
                                            (unsigned long long)key);
        if (prev == HT_EMPTY || prev == key) return s;
        s = (s + 1) & mask;
    }
}
// returns slot or ~0
__device__ __forceinline__ uint64_t ht_find(const uint64_t* keys, uint64_t mask, uint64_t key)
{
    uint64_t s = ht_slot0(key, mask);
    while (true) {
        uint64_t kk = __ldcg(keys + s);
        if (kk == key) return s;
        if (kk == HT_EMPTY) return ~0ull;
        s = (s + 1) & mask;
    }
}

}  // namespace kmgpu
