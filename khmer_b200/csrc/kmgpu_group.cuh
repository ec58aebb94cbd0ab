// Grouped ingestion, second generation (the headline path).
//
// A chunk's counter updates are grouped by 32 Ki-bin BUCKET of their table and every bucket is then applied by one CTA
// in shared memory (touch counts, first touchers, the table slice itself), exactly like the first bucket path — but:
//
//   * hashing is fused into the grouping kernel: k_part walks the 2-bit read stream, hashes, reduces modulo the table
//     size and sorts the records of its tile by bucket in shared memory; the bins[N][n_pos] array (37 B per k-mer of
//     DRAM traffic) and the k_hashbins launch are gone;
//   * tables of any size: a table with more than PART_MAXP buckets is grouped in two levels — first by SUPER-BUCKET
//     (2^27 bins = 4096 buckets), then each super-bucket's records by bucket; bins are 64-bit throughout;
//   * a bucket that receives more records than its home region holds does not fail the chunk: the grouping is redone
//     once with exact (CSR) offsets taken from the demand the first run counted, and k_apply clamps its 16-bit touch
//     lanes between rounds of 32 Ki records, so any load is exact;
//   * k_apply moves its table slice with bulk asynchronous copies (cp.async.bulk + mbarrier: global -> shared before the
//     records are counted, shared -> global after the sweep) and keeps it in shared memory, which also tells every
//     record for free whether its bin was empty before the chunk — only those records pay the first-toucher atomicMin;
//   * sparse regimes (a few hundred records per bucket: tables far larger than a chunk) use k_apply_sparse, whose cost
//     is proportional to the records, not to the bucket.
//
// Reference semantics: Storage::add for the three storages (include/oxli/storage.hh:571-624, :320-359, :172-199) applied
// to the k-mer stream of Hashtable::consume_string (src/oxli/hashtable.cc:280-294) in stream order.
#pragma once
#include "kmgpu_kernels.cuh"

namespace kmgpu {

constexpr int G_MAXT = MAX_TABLES;                       // tables per sketch on this path
constexpr int SB_SHIFT_MAX = 12;                         // at most 4096 buckets (2^27 bins) per super-bucket (two-level grouping)
constexpr int PART_MAXP = 6144;                          // partitions one k_part CTA can sort into (shared-memory histogram)

struct GroupLayout {
    uint32_t first[G_MAXT + 1];      // table i owns buckets [first[i], first[i+1])
    uint32_t first_sb[G_MAXT + 1];   // two-level: table i owns super-buckets [first_sb[i], first_sb[i+1])
    uint32_t cap;                    // home region of a bucket, in records (uniform layout)
    uint32_t cap1;                   // home region of a super-bucket
    int n_tables;
    int two_level;
    int sb_shift;                    // log2(buckets per super-bucket): chosen so that both levels sort into about sqrt(buckets)
                                     // partitions (runs stay long at both levels); records of level 1 carry 15 + sb_shift bin bits
};

struct SatBitsG {
    uint8_t* t[G_MAXT];
};

// a record store: region of partition p = [off ? off[p] : p * cap, + (off ? off[p+1] - off[p] : cap))
struct Store {
    unsigned long long* rec;
    const unsigned long long* off;   // exact (CSR) offsets of partitions p0 .. (indexed p - p0), or nullptr for the uniform layout
    uint32_t* cursor;                // records written to (demanded of) every partition (indexed by p)
    uint32_t cap;
    uint32_t p0;                     // first partition held (tables are grouped in turns when memory is short)
    __device__ __forceinline__ unsigned long long base(uint32_t p) const { return off ? off[p - p0] : (unsigned long long)(p - p0) * cap; }
    __device__ __forceinline__ uint32_t room(uint32_t p) const { return off ? (uint32_t)(off[p - p0 + 1] - off[p - p0]) : cap; }
};

constexpr int MAX_WORLD = 16;   // ranks of an address-sharded sketch

// ---- bulk asynchronous copies + mbarrier (sm_90+ PTX; SASS: UBLKCP / SYNCS) -------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "KM_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra KM_DONE_%=;\n"
        "bra KM_WAIT_%=;\n"
        "KM_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_read()
{
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// =====================================================================================================================
// 1. k_part: sort the records of one tile by partition in shared memory and append each partition's run to its region.
//
//   MODE 0  stream -> buckets            partition = bin >> 15            record = position << 15 | bin & 0x7FFF
//   MODE 1  stream -> super-buckets      partition = bin >> 27            record = position << 27 | bin & 0x7FFFFFF
//   MODE 2  super-bucket -> its buckets  partition = (rec >> 15) & 0xFFF  record = position << 15 | bin & 0x7FFF
//   (address-sharded sketches group with MODE 1 over the FULL tables and send whole super-bucket runs to their owners,
//   section 8; writing every CTA's short runs straight into peer memory — one remote atomicAdd per (CTA, partition) — was
//   measured 3x slower over NVLink than the exchange of whole runs)
//
//   SRC 0: the k-mers are hashed here from the 2-bit stream (TwoBit);  SRC 1: 64-bit hashes precomputed by k_hash64
//   (Murmur: hashing 2 x k letters per table would dominate) or supplied by the caller (kmgpu_add_hashes).
//   grid = (tiles, tables) for MODE 0/1, (tiles of the largest super-bucket, super-buckets) for MODE 2.
// =====================================================================================================================
struct PartArgs {
    SketchDev S;          // full table sizes and magics
    HashCfg H;
    Input in;             // MODE 0/1: the part of the chunk being grouped
    uint32_t pos_base;    // its first position within the chunk
    int have_valid;       // SRC 1: 0 = every position of `in` is a k-mer (caller-supplied hashes), 1 = validity from the read offsets
    int table0;           // MODE 0/1: first table of this launch (blockIdx.y is relative to it); MODE 2: first super-bucket
    uint32_t tiles_per_src;   // MODE 2: blockIdx.x = (super-bucket - table0) * tiles_per_src + tile
    int count_kmers;      // MODE 0/1: table 0's CTAs add the k-mers they consumed to ctrl->n_kmers (off in a regrouping run)
    GroupLayout L;
    Store dst;            // MODE 0/2: bucket store; MODE 1: super-bucket store
    Store src;            // MODE 2: super-bucket store
    Ctrl* ctrl;
    unsigned long long ovf_bit;   // set in ctrl->overflow when a destination region runs out of room
};

template <int T>
struct PartTile {
    uint64_t words[T / 32 + TILE_PAD_WORDS];
    uint32_t valid[T / 32];
};

// WIDE: run bases kept in 32 bits (super-buckets; regions with exact offsets, which may hold more than 65535 records)
// pcap: partitions the instantiation can sort into (BPT per thread): the histogram and the run bases take that many words each
__host__ __device__ constexpr int part_cap(int bpt, int nthr) { return bpt * nthr < PART_MAXP ? bpt * nthr : PART_MAXP; }
__host__ __device__ constexpr size_t part_smem(int T, bool wide, int pcap)
{
    return (size_t)T * 8 + (size_t)pcap * 4 * (wide ? 2 : 1) + (size_t)(T / 32 + TILE_PAD_WORDS) * 8 + (size_t)(T / 32) * 4 + 16;
}

// stage the tile's stream words and the bitmap of valid k-mer starts (cf. tile_begin, for tiles of T positions)
template <int T, int NTHR, int SRC>
__device__ __forceinline__ void part_tile_begin(const Input& in, int k, uint32_t t0, int have_valid, PartTile<T>& sm)
{
    const int tid = threadIdx.x;
    const bool pre = in.valid != nullptr && in.read_keep == nullptr && !(SRC == 1 && !have_valid);
    if (pre) {
        // the bitmap was computed when the chunk was staged: one more independent load next to the stream words
        const uint32_t vw = (in.n_pos + 31) >> 5, v0 = t0 >> 5;
        for (int i = tid; i < T / 32; i += NTHR) sm.valid[i] = v0 + i < vw ? __ldg(in.valid + v0 + i) : 0u;
    } else {
        for (int i = tid; i < T / 32; i += NTHR) sm.valid[i] = 0;
    }
    if (SRC == 0) {
        const uint32_t total_words = ((in.n_pos + TILE - 1) / TILE) * (TILE / 32) + TILE_PAD_WORDS;
        const uint32_t w0 = t0 >> 5;
        for (int i = tid; i < T / 32 + TILE_PAD_WORDS; i += NTHR) sm.words[i] = w0 + i < total_words ? __ldg(in.words + w0 + i) : 0ull;
    }
    __syncthreads();
    if (pre) return;
    if (SRC == 1 && !have_valid) {
        const uint32_t n = in.n_pos - t0 < (uint32_t)T ? in.n_pos - t0 : (uint32_t)T;
        for (int i = tid; i < T / 32; i += NTHR) {
            uint32_t lo = i * 32;
            sm.valid[i] = lo >= n ? 0u : (n - lo >= 32 ? ~0u : ((1u << (n - lo)) - 1));
        }
        __syncthreads();
        return;
    }
    const uint32_t n_tiles4k = (in.n_pos + TILE - 1) / TILE;
    const uint32_t tb = t0 / TILE;
    const uint32_t te = tb + T / TILE < n_tiles4k ? tb + T / TILE : n_tiles4k;
    const uint32_t r_lo = in.tfr[tb];
    uint32_t r_hi = in.tfr[te] + 1;
    if (r_hi > in.n_reads) r_hi = in.n_reads;
    for (uint32_t r = r_lo + tid; r < r_hi; r += NTHR) {
        uint32_t s = in.offs[r], e = in.offs[r + 1];
        if (e - s < (uint32_t)k) continue;
        if (in.read_keep && !((in.read_keep[r >> 5] >> (r & 31)) & 1u)) continue;
        uint32_t first = s > t0 ? s : t0;
        uint32_t last = e - k;  // inclusive
        if (last >= t0 + T) last = t0 + T - 1;
        if (first > last || last < t0) continue;
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

// BPT: consecutive partitions per thread in the scan; the launch picks the smallest instantiation with BPT * NTHR >= the
// number of partitions, so that every thread has a share (and no registers are held for partitions that do not exist)
template <int T, int NTHR, int MODE, int SRC, bool PRED, bool WIDEP, int BPT>
__global__ void __launch_bounds__(NTHR, (2 * part_smem(T, MODE == 1 || WIDEP, part_cap(BPT, NTHR)) <= 220 * 1024 && NTHR <= 512) ? 2 : 1)
k_part(const __grid_constant__ PartArgs A, const __grid_constant__ SketchDev M, const __grid_constant__ Pred P)
{
    constexpr bool WIDE = MODE == 1 || WIDEP;
    constexpr int PER = T / NTHR;
    constexpr bool SBMODE = MODE == 1;                         // partitions are super-buckets
    const int SB_SHIFT = A.L.sb_shift, SB_BIN_SHIFT = BKT_SHIFT + SB_SHIFT;
    const int PB = SBMODE ? SB_BIN_SHIFT : BKT_SHIFT;          // payload bits of the records written
    extern __shared__ __align__(16) unsigned char pt_raw[];
    uint2* stage = reinterpret_cast<uint2*>(pt_raw);                          // T slots, grouped by partition
    constexpr int PCAP = part_cap(BPT, NTHR);
    uint32_t* hist = reinterpret_cast<uint32_t*>(stage + T);                  // PCAP: count, then run start | cursor base << 16
    uint32_t* gb32 = hist + PCAP;                                             // WIDE only: 32-bit cursor bases
    PartTile<T>& tile = *reinterpret_cast<PartTile<T>*>(hist + PCAP * (WIDE ? 2 : 1));
    __shared__ uint32_t s_warp[32];
    const uint32_t tid = threadIdx.x;
    const uint32_t p0 = (MODE == 2 ? blockIdx.x % A.tiles_per_src : blockIdx.x) * (uint32_t)T;

    // which partitions this CTA sorts into
    int t;                 // table
    uint32_t np;           // number of partitions
    uint32_t cur0;         // index of partition 0 in dst.cursor / dst regions
    uint32_t n_src = 0;    // MODE 2: records of the source super-bucket
    const unsigned long long* srec = nullptr;
    if (MODE == 2) {
        const uint32_t sb = (uint32_t)A.table0 + blockIdx.x / A.tiles_per_src;
        t = 0;
#pragma unroll 1
        for (int i = 1; i < A.L.n_tables; i++)
            if (sb >= A.L.first_sb[i]) t = i;
        const uint32_t sbi = sb - A.L.first_sb[t];
        const uint32_t nb_t = A.L.first[t + 1] - A.L.first[t];
        np = nb_t - (sbi << SB_SHIFT);
        if (np > (1u << SB_SHIFT)) np = 1u << SB_SHIFT;
        cur0 = A.L.first[t] + (sbi << SB_SHIFT);
        n_src = A.src.cursor[sb];
        const uint32_t room = A.src.room(sb);
        if (n_src > room) n_src = room;   // the super-bucket overflowed: ctrl->overflow is set, the chunk is regrouped
        if (p0 >= n_src) return;
        srec = A.src.rec + A.src.base(sb);
    } else {
        t = A.table0 + blockIdx.y;
        if (MODE == 0) {
            np = A.L.first[t + 1] - A.L.first[t];
            cur0 = A.L.first[t];
        } else {
            np = A.L.first_sb[t + 1] - A.L.first_sb[t];
            cur0 = A.L.first_sb[t];
        }
        if (p0 >= A.in.n_pos) return;
    }

    // ---- phase 1: keys, ranks within this CTA's runs (one shared-memory atomic per record) --------------------------
    uint32_t key[PER];              // MODE 0/2: partition << 15 | payload (15 bits);  MODE 1: payload (27 bits)
    uint32_t pid1[(PER + 1) / 2];   // MODE 1: partitions, two per word
    uint32_t rk[(PER + 1) / 2];     // ranks, two per word
    constexpr uint32_t NONE = 0xFFFFFFFFu;
    for (uint32_t i = tid; i < np; i += NTHR) hist[i] = 0;
    unsigned n_k = 0;
    if (MODE == 2) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < PER; j++) {
            const uint32_t e = p0 + j * NTHR + tid;
            key[j] = NONE;
            if (e < n_src) key[j] = (uint32_t)__ldcs(srec + e) & ((1u << SB_BIN_SHIFT) - 1);   // partition << 15 | bin in bucket
        }
    } else {
        part_tile_begin<T, NTHR, SRC>(A.in, A.H.k, p0, A.have_valid, tile);   // ends with __syncthreads()
        const uint64_t size = A.S.sizes[t], magic = A.S.magic[t];
#pragma unroll
        for (int j = 0; j < PER; j++) {
            const uint32_t lp = j * NTHR + tid;
            key[j] = NONE;
            if (SBMODE) {
                if (j & 1) pid1[j >> 1] |= 0xFFFF0000u; else pid1[j >> 1] = 0xFFFFu;
            }
            if (p0 + lp < A.in.n_pos && ((tile.valid[lp >> 5] >> (lp & 31)) & 1u)) {
                const uint64_t h = SRC == 1 ? __ldcs(A.in.hashes + p0 + lp) : hash_twobit(tile.words, lp, A.H.k);
                if (!PRED || pred_pass(P, M, h)) {
                    uint64_t bin = mod_magic(h, size, magic);
                    n_k++;
                    if (SBMODE) {
                        const uint32_t pid = (uint32_t)(bin >> SB_BIN_SHIFT);
                        key[j] = (uint32_t)bin & ((1u << SB_BIN_SHIFT) - 1);
                        if (j & 1) pid1[j >> 1] = (pid1[j >> 1] & 0xFFFFu) | (pid << 16); else pid1[j >> 1] = (pid1[j >> 1] & 0xFFFF0000u) | pid;
                    } else {
                        key[j] = (uint32_t)bin;   // MODE 0 tables have at most PART_MAXP << 15 < 2^28 bins
                    }
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < PER; j++) {
        uint32_t r = 0;
        if (key[j] != NONE) {
            const uint32_t pid = SBMODE ? ((j & 1) ? pid1[j >> 1] >> 16 : pid1[j >> 1] & 0xFFFFu) : key[j] >> BKT_SHIFT;
            r = atomicAdd(&hist[pid], 1u);
        }
        if (j & 1) rk[j >> 1] |= r << 16; else rk[j >> 1] = r;
    }
    if (MODE != 2 && t == 0 && A.count_kmers) {   // the k-mers of the chunk are counted once, by the CTAs of table 0
        n_k = __reduce_add_sync(0xffffffffu, n_k);
        if ((tid & 31) == 0 && n_k) atomicAdd(&A.ctrl->n_kmers, (unsigned long long)n_k);
    }
    __syncthreads();

    // ---- phase 2: exclusive scan of the partition counts (BPT consecutive partitions per thread), reservations -------
    uint32_t c[BPT], mine = 0;
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        const uint32_t b = tid * BPT + q;
        c[q] = b < np ? hist[b] : 0;
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
    // every warp adds up the totals of the warps before it itself (NTHR / 32 broadcast reads): no second barrier
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < NTHR / 32; w++) {
        const uint32_t v = s_warp[w];
        before += (uint32_t)w < wid ? v : 0u;
        total += v;
    }
    uint32_t at = before + incl - mine, gbase[BPT];
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        const uint32_t b = tid * BPT + q;
        if (b < np) hist[b] = at;   // run start (the count has been read by its only reader, this thread)
        gbase[q] = c[q] ? atomicAdd(&A.dst.cursor[cur0 + b], c[q]) : 0u;   // in flight while the records are placed
        at += c[q];
    }
    __syncthreads();

    // ---- phase 3: place the records in partition order -----------------------------------------------------------------
#pragma unroll
    for (int j = 0; j < PER; j++) {
        if (key[j] == NONE) continue;
        const uint32_t pid = SBMODE ? ((j & 1) ? pid1[j >> 1] >> 16 : pid1[j >> 1] & 0xFFFFu) : key[j] >> BKT_SHIFT;
        const uint32_t r = (j & 1) ? rk[j >> 1] >> 16 : rk[j >> 1] & 0xFFFFu;
        const uint32_t slot = (hist[pid] & 0xFFFFu) + r;
        if (MODE == 2) {
            // the position travels with the record: fetch it again (L1/L2 hit) rather than hold 16 more registers
            const unsigned long long v = __ldcs(srec + p0 + j * NTHR + tid);
            stage[slot] = make_uint2((uint32_t)(v >> SB_BIN_SHIFT), key[j]);
        } else if (SBMODE) {
            stage[slot] = make_uint2(key[j], (pid << 14) | (uint32_t)(j * NTHR + tid));
        } else {
            stage[slot] = make_uint2(key[j] & (BKT_BINS - 1), (pid << 14) | (uint32_t)(j * NTHR + tid));
        }
    }
    // run start (low half) and cursor base: the low half is not changed by this store, so a placement still reading
    // hist[pid] & 0xFFFF sees the same value before and after it
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        const uint32_t b = tid * BPT + q;
        if (b < np) {
            if (WIDE) gb32[b] = gbase[q];
            else hist[b] = (hist[b] & 0xFFFFu) | (gbase[q] << 16);   // uniform regions hold <= 65535 records; a base past 2^16
                                                                     // belongs to a region that has already been reported full
        }
    }
    __syncthreads();

    // ---- phase 4: runs of consecutive records leave for their regions ---------------------------------------------------
    bool over = false;
    for (uint32_t s = tid; s < total; s += NTHR) {
        const uint2 m = stage[s];
        const uint32_t pid = MODE == 2 ? m.y >> BKT_SHIFT : m.y >> 14;
        const uint32_t hv = hist[pid];
        const uint32_t idx = (WIDE ? gb32[pid] : hv >> 16) + (s - (hv & 0xFFFFu));
        unsigned long long rec;
        if (MODE == 2) rec = ((unsigned long long)m.x << BKT_SHIFT) | (m.y & (BKT_BINS - 1));
        else rec = ((unsigned long long)(A.pos_base + p0 + (m.y & 0x3FFFu)) << PB) | m.x;
        if (idx < A.dst.room(cur0 + pid)) A.dst.rec[A.dst.base(cur0 + pid) + idx] = rec;
        else over = true;
    }
    if (over) atomicOr(&A.ctrl->overflow, A.ovf_bit);
}

// 64-bit hashes of every position (Murmur): one pass, then k_part<SRC 1> per table
template <int HK>
__global__ void __launch_bounds__(THREADS)
k_hash64(HashCfg H, Input in, uint64_t* __restrict__ out)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, 0>(in, H.k, t0, sm);
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        if (tile_valid<HK, 0>(sm, lp)) __stcs(&out[t0 + lp], tile_hash<HK, 0>(in, sm, H.k, t0, lp));
    }
}

// exclusive scan of the demanded counts into exact offsets (regrouping run): off[p] for p in [0, n], single CTA
__global__ void __launch_bounds__(1024) k_exact_offsets(const uint32_t* __restrict__ cnt, uint32_t n, unsigned long long* __restrict__ off)
{
    __shared__ unsigned long long s_w[32];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        // regions start on even record indices (16-byte alignment of every run's first record is not required, but an
        // even start keeps 16-byte loads of whole regions possible)
        unsigned long long v = i < n ? (((unsigned long long)cnt[i] + 1) & ~1ull) : 0, incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (uint32_t)o) incl += u;
        }
        if (lane == 31) s_w[wid] = incl;
        __syncthreads();
        unsigned long long before = s_carry;
        for (uint32_t w = 0; w < wid; w++) before += s_w[w];
        if (i < n) off[i] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) off[n] = s_carry;
}

// buckets whose demand exceeds `thresh` records (regrouping run of a sparse plan): list[0 .. *count)
__global__ void k_big_buckets(const uint32_t* __restrict__ cursor, uint32_t b_lo, uint32_t n, uint32_t thresh, uint32_t* __restrict__ list, uint32_t list_cap,
                              unsigned int* count)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || cursor[b_lo + i] <= thresh) return;
    const uint32_t at = atomicAdd(count, 1u);
    if (at < list_cap) list[at] = b_lo + i;
}

// =====================================================================================================================
// 2. k_apply2: one CTA per bucket.  Shared memory: 16-bit touch lanes (64 KB), first-toucher positions (128 KB), the
//    bucket's slice of the table (32 / 16 / 4 KB).
// =====================================================================================================================
template <int KIND>
__host__ __device__ constexpr uint32_t slice_bytes_full() { return KIND == BYTE ? BKT_BINS : KIND == NIBBLE ? BKT_BINS / 2 : BKT_BINS / 8; }
// SPLIT: CTAs per bucket.  Each takes 1/SPLIT of the bucket's bins (and reads all of its records, keeping its own): lightly loaded
// buckets, whose cost is the set-up and the sweep of the shared-memory arrays rather than the records, then run 2-3 CTAs per SM.
template <int KIND, int SPLIT>
constexpr size_t apply2_smem() { return ((size_t)BKT_BINS * 2 + (size_t)BKT_BINS * 4 + slice_bytes_full<KIND>()) / SPLIT + 64; }

template <int KIND, int SPLIT>
__global__ void __launch_bounds__(1024 / SPLIT, SPLIT == 4 ? 3 : SPLIT)
k_apply2(const __grid_constant__ SketchDev S, const __grid_constant__ GroupLayout L, Store st, uint32_t bucket0, uint32_t* __restrict__ newbits,
         uint64_t* __restrict__ binlist, unsigned long long list_cap, Ctrl* ctrl, int want_cross, const __grid_constant__ SatBitsG sb,
         unsigned long long ovf_mask, uint32_t* __restrict__ newmask, const uint32_t* __restrict__ bucket_list)
{
    extern __shared__ __align__(128) unsigned char ap_raw[];
    constexpr uint32_t SUB_BINS = BKT_BINS / SPLIT, NTHR = 1024 / SPLIT, SUB_BYTES = slice_bytes_full<KIND>() / SPLIT;
    uint32_t* cnt = reinterpret_cast<uint32_t*>(ap_raw);                       // SUB_BINS / 2 words, two 16-bit lanes each
    uint32_t* minpos = cnt + SUB_BINS / 2;                                     // SUB_BINS words
    uint8_t* slice = reinterpret_cast<uint8_t*>(minpos + SUB_BINS);
    uint64_t* bar = reinterpret_cast<uint64_t*>(slice + SUB_BYTES);
    if (ctrl->overflow & ovf_mask) return;      // a region of this table group ran out of room: the group is regrouped with exact offsets
    // bucket_list: the launch covers only the listed buckets (the heavily loaded ones of a regrouping run whose other buckets
    // go through k_apply_sparse)
    const uint32_t b = bucket_list ? bucket_list[blockIdx.x / SPLIT] : bucket0 + blockIdx.x / SPLIT;
    const uint32_t sub = blockIdx.x % SPLIT;
    const uint32_t tid = threadIdx.x;
    const uint32_t n = st.cursor[b];
    if (n == 0) return;
    int t = 0;
#pragma unroll 1
    for (int i = 1; i < L.n_tables; i++)
        if (b >= L.first[i]) t = i;
    const uint64_t bin0 = ((uint64_t)(b - L.first[t]) << BKT_SHIFT) + (uint64_t)sub * SUB_BINS;
    const uint64_t size = S.sizes[t];
    if (bin0 >= size) return;   // a part of the table's last bucket that lies past its end
    int changed = 0;
    uint8_t* table = S.tables[t];
    // bytes of the table this bucket covers, rounded up to the 16-byte granule of bulk copies (tables are allocated in
    // whole granules; bytes past the last bin are written back as they were read)
    const uint64_t tbytes = KIND == BYTE ? size : KIND == NIBBLE ? size / 2 + 1 : size / 8 + 1;
    const uint64_t byte0 = KIND == BYTE ? bin0 : KIND == NIBBLE ? bin0 >> 1 : bin0 >> 3;
    uint32_t sbytes = (uint32_t)(tbytes - byte0 < SUB_BYTES ? tbytes - byte0 : SUB_BYTES);
    sbytes = (sbytes + 15u) & ~15u;
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(bar, sbytes);
        bulk_g2s(slice, table + byte0, sbytes, bar);
    }
    {
        uint4* f = reinterpret_cast<uint4*>(minpos);
        for (uint32_t i = tid; i < SUB_BINS / 4; i += NTHR) f[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
    }
    // the slice is first needed by the sweep: its load hides behind the record loop
    constexpr int GPT = SUB_BINS / 8 / NTHR;
    if (KIND != BIT) {
#pragma unroll
        for (int q = 0; q < GPT; q++) reinterpret_cast<uint4*>(cnt)[q * NTHR + tid] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    const unsigned long long* src = st.rec + st.base(b);
    constexpr int RIF = 16;   // records in flight per thread
    constexpr uint32_t ITER_REC = RIF * NTHR, CLAMP_EVERY = 32768u / ITER_REC;
    for (uint32_t e0 = 0; e0 < n; e0 += ITER_REC) {
        // four records per thread in flight at a time (a lightly loaded bucket ends after the first group: no predicated-off
        // copies of the loop body for records that do not exist)
#pragma unroll
        for (int jj = 0; jj < RIF; jj += 4) {
            if (e0 + (uint32_t)jj * NTHR >= n) break;
            unsigned long long v[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t e = e0 + (uint32_t)(jj + j) * NTHR + tid;
                // the parts of a bucket run side by side and read the same records: the first reader brings them into L2 for the others
                v[j] = e < n ? (SPLIT == 1 ? __ldcs(src + e) : __ldg(src + e)) : ~0ull;
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                if (v[j] == ~0ull) continue;
                uint32_t lb = (uint32_t)v[j] & (BKT_BINS - 1);
                if (SPLIT > 1) {
                    if (lb / SUB_BINS != sub) continue;
                    lb &= SUB_BINS - 1;
                }
                // both updates leave at once, nothing waits for a result (the sweep ignores positions of bins that were occupied)
                if (KIND != BIT) atomicAdd(&cnt[lb >> 1], (lb & 1) ? 0x10000u : 1u);
                atomicMin(&minpos[lb], (uint32_t)(v[j] >> BKT_SHIFT));
            }
        }
        // More records than a 16-bit lane can count: clamp every lane after each 32 Ki records to a value the next round cannot
        // push into the neighbouring lane — any value >= the counter's cap saturates it just the same.
        if (KIND != BIT && n > 65535u && (e0 / ITER_REC) % CLAMP_EVERY == CLAMP_EVERY - 1) {
            const uint32_t lim = 0x7FFFu;
            __syncthreads();
            for (uint32_t i = tid; i < SUB_BINS / 2; i += NTHR) {
                const uint32_t w = cnt[i];
                const uint32_t lo = w & 0xFFFFu, hi = w >> 16;
                cnt[i] = (lo > lim ? lim : lo) | ((hi > lim ? lim : hi) << 16);
            }
            __syncthreads();
        }
    }
    __syncthreads();
    mbar_wait(bar, 0);
    unsigned n_new = 0, n_sat = 0, n_cross = 0;
#pragma unroll
    for (int q = 0; q < GPT; q++) {
        const uint32_t g = q * NTHR + tid;
        const uint64_t b0 = bin0 + (uint64_t)g * 8;
        unsigned newm = 0;
        if (KIND == BIT) {
            const uint4 m0 = reinterpret_cast<const uint4*>(minpos)[g * 2], m1 = reinterpret_cast<const uint4*>(minpos)[g * 2 + 1];
            const uint32_t mp[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
#pragma unroll
            for (int j = 0; j < 8; j++) newm |= (unsigned)(mp[j] != ~0u) << j;   // touched bins ...
            newm &= ~(unsigned)slice[g];                                         // ... that were clear
            if (!newm) continue;
            changed = 1;
            slice[g] = (uint8_t)(slice[g] | newm);
            n_new += __popc(newm);
#pragma unroll
            for (int j = 0; j < 8; j++)
                if ((newm >> j) & 1u) {
                    atomicOr(&newbits[mp[j] >> 5], 1u << (mp[j] & 31));
                    if (newmask) atomicOr(&newmask[mp[j]], 1u << t);   // first-touch log: which tables made the position new
                }
            continue;
        }
        const uint4 c4 = reinterpret_cast<const uint4*>(cnt)[g];
        if (!(c4.x | c4.y | c4.z | c4.w)) continue;
        const uint32_t cw[4] = {c4.x, c4.y, c4.z, c4.w};
        unsigned crossm = 0;
        changed = 1;
        if (KIND == BYTE) {
            const uint64_t old64 = *reinterpret_cast<const uint64_t*>(slice + (size_t)g * 8);
            uint64_t new64 = old64;
            unsigned fullm = 0;
            // only the lanes that were touched (in a lightly loaded bucket one or two of the eight): a loop over the set bits
            // of a mask instead of eight predicated copies of the update
            unsigned nz = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) nz |= (unsigned)(((cw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu) != 0) << j;
            auto bump = [&](int j, uint32_t m) {
                uint32_t s = (uint32_t)(old64 >> (8 * j)) & 255u, tt = s + m, nv = tt > 255u ? 255u : tt;
                new64 = (new64 & ~(255ull << (8 * j))) | ((uint64_t)nv << (8 * j));
                newm |= (unsigned)(s == 0) << j;
                n_sat += tt > 255u;
                crossm |= (unsigned)(tt >= 255u && s < 255u) << j;
                fullm |= (unsigned)(nv == 255u) << j;
            };
            if (__popc(nz) > 3) {   // a well-filled group: the unrolled form (constant shifts)
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const uint32_t m = (cw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu;
                    if (m) bump(j, m);
                }
            } else {
                while (nz) {
                    const int j = __ffs(nz) - 1;
                    nz &= nz - 1;
                    const uint32_t wj = j < 2 ? c4.x : j < 4 ? c4.y : j < 6 ? c4.z : c4.w;   // (selects: no dynamically indexed array)
                    bump(j, (wj >> ((j & 1) * 16)) & 0xFFFFu);
                }
            }
            *reinterpret_cast<uint64_t*>(slice + (size_t)g * 8) = new64;
            if (want_cross && fullm) {
                unsigned m = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) m |= (unsigned)(((new64 >> (8 * j)) & 255u) == 255u) << j;
                sb.t[t][b0 >> 3] = (uint8_t)m;
            }
            n_cross += __popc(crossm);
            if (want_cross && crossm) {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if (!((crossm >> j) & 1u)) continue;
                    unsigned long long at = atomicAdd(&ctrl->n_events, 1ull);
                    if (at < list_cap) binlist[at] = BL_CROSS | (((old64 >> (8 * j)) & 255ull) << 48) | ht_key(b0 + j, t);
                }
            }
        } else {
            const uint32_t old32 = *reinterpret_cast<const uint32_t*>(slice + (size_t)g * 4);
            uint32_t new32 = old32;
            unsigned nz = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) nz |= (unsigned)(((cw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu) != 0) << j;
            auto bump = [&](int j, uint32_t m) {
                const uint32_t sh = (j >> 1) * 8 + ((j & 1) ? 0 : 4);   // even bin -> high nibble
                uint32_t s = (old32 >> sh) & 15u, tt = s + m, nv = tt > 15u ? 15u : tt;
                new32 = (new32 & ~(15u << sh)) | (nv << sh);
                newm |= (unsigned)(s == 0) << j;
            };
            if (__popc(nz) > 3) {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const uint32_t m = (cw[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu;
                    if (m) bump(j, m);
                }
            } else {
                while (nz) {
                    const int j = __ffs(nz) - 1;
                    nz &= nz - 1;
                    const uint32_t wj = j < 2 ? c4.x : j < 4 ? c4.y : j < 6 ? c4.z : c4.w;
                    bump(j, (wj >> ((j & 1) * 16)) & 0xFFFFu);
                }
            }
            *reinterpret_cast<uint32_t*>(slice + (size_t)g * 4) = new32;
        }
        n_new += __popc(newm);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (!((newm >> j) & 1u)) continue;
            const uint32_t p = minpos[g * 8 + j];
            atomicOr(&newbits[p >> 5], 1u << (p & 31));
            if (newmask) atomicOr(&newmask[p], 1u << t);
        }
    }
    // the slice goes back in one bulk copy (generic-proxy writes made visible to the async proxy first)
    fence_proxy_async();
    __shared__ unsigned s_tot[3];
    if (tid < 3) s_tot[tid] = 0;
    changed = __syncthreads_or(changed);
    if (tid == 0 && changed) {   // a bucket whose touches changed nothing (a warm Bloom filter) writes nothing
        bulk_s2g(table + byte0, slice, sbytes);
        bulk_commit_wait_read();
    }
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
        if (s_tot[0]) atomicAdd(&ctrl->n_new_t[t], (unsigned long long)s_tot[0]);   // the host sums these (any table / table 0)
        if (s_tot[1]) atomicAdd(&ctrl->n_sat, (unsigned long long)s_tot[1]);
        if (s_tot[2]) atomicAdd(&ctrl->n_cross, (unsigned long long)s_tot[2]);
    }
}

// =====================================================================================================================
// 3. k_apply_sparse: buckets that receive few records (tables far larger than a chunk).  The records of a bucket are
//    aggregated per bin in a small shared-memory hash table (slots = power of two >= 2 n), then every distinct bin is
//    updated in place with a compare-and-swap on its 32-bit word — DRAM sees only the sectors that are touched.
//    One CTA of 128 threads per bucket; shared memory 12 bytes per slot.
// =====================================================================================================================
constexpr uint32_t SPARSE_MAX_RECORDS = 4096;   // per bucket (8192 slots = 96 KB)

template <int KIND>
__global__ void __launch_bounds__(128)
k_apply_sparse(const __grid_constant__ SketchDev S, const __grid_constant__ GroupLayout L, Store st, uint32_t bucket0, uint32_t* __restrict__ newbits,
               uint64_t* __restrict__ binlist, unsigned long long list_cap, Ctrl* ctrl, int want_cross, const __grid_constant__ SatBitsG sb,
               unsigned long long ovf_mask, uint32_t* __restrict__ newmask, uint32_t max_n)
{
    extern __shared__ __align__(16) uint32_t sp_raw[];
    if (ctrl->overflow & ovf_mask) return;
    const uint32_t b = bucket0 + blockIdx.x;
    const uint32_t n = st.cursor[b];
    if (n == 0) return;
    // more than the region holds: reported by k_part; more than max_n (regrouping runs): the bucket is on k_apply2's list
    if (n > st.room(b) || n > max_n) return;
    uint32_t slots = 64;
    while (slots < 2 * n) slots <<= 1;
    uint32_t* hk = sp_raw;            // bin in bucket + 1, 0 = free
    uint32_t* hc = hk + slots;        // touches
    uint32_t* hp = hc + slots;        // smallest touching position
    int t = 0;
#pragma unroll 1
    for (int i = 1; i < L.n_tables; i++)
        if (b >= L.first[i]) t = i;
    const uint64_t bin0 = (uint64_t)(b - L.first[t]) << BKT_SHIFT;
    uint8_t* table = S.tables[t];
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < slots; i += 128) {
        hk[i] = 0;
        hc[i] = 0;
        hp[i] = ~0u;
    }
    __syncthreads();
    const unsigned long long* src = st.rec + st.base(b);
    const uint32_t mask = slots - 1;
    for (uint32_t e = tid; e < n; e += 128) {
        const unsigned long long v = __ldcs(src + e);
        const uint32_t lb = (uint32_t)v & (BKT_BINS - 1), key = lb + 1;
        uint32_t s = (lb * 0x9E3779B1u) >> 7 & mask;
        while (true) {
            const uint32_t prev = atomicCAS(&hk[s], 0u, key);
            if (prev == 0u || prev == key) break;
            s = (s + 1) & mask;
        }
        atomicAdd(&hc[s], 1u);
        atomicMin(&hp[s], (uint32_t)(v >> BKT_SHIFT));
    }
    __syncthreads();
    unsigned n_new = 0, n_sat = 0, n_cross = 0;
    // every distinct bin: read its word, compare-and-swap the new value in.  Four slots per thread and round, all loads issued
    // before the first is used and all first swaps before the first is checked: the two DRAM round trips of an update overlap
    // with those of the thread's other slots instead of queueing behind them.
    constexpr int U = 4;
    constexpr uint32_t CAP = KIND == BYTE ? 255u : KIND == NIBBLE ? 15u : 1u;
    for (uint32_t s0 = 0; s0 < slots; s0 += 128 * U) {
        uint32_t* word[U];
        uint32_t sh[U], cur[U], m[U], before[U], pos[U];
        uint64_t bin[U];
        bool act[U];
#pragma unroll
        for (int j = 0; j < U; j++) {
            const uint32_t sl = s0 + j * 128 + tid;
            act[j] = sl < slots && hk[sl] != 0;
            word[j] = nullptr;
            sh[j] = cur[j] = m[j] = before[j] = pos[j] = 0;
            bin[j] = 0;
            if (!act[j]) continue;
            bin[j] = bin0 + (hk[sl] - 1);
            m[j] = hc[sl];
            pos[j] = hp[sl];
            if (KIND == BIT) {
                word[j] = reinterpret_cast<uint32_t*>(table) + (bin[j] >> 5);
                sh[j] = (uint32_t)(bin[j] & 31);
            } else if (KIND == BYTE) {
                word[j] = reinterpret_cast<uint32_t*>(table + (bin[j] & ~3ull));
                sh[j] = (uint32_t)(bin[j] & 3) * 8;
            } else {
                const uint64_t byte = bin[j] >> 1;
                word[j] = reinterpret_cast<uint32_t*>(table + (byte & ~3ull));
                sh[j] = (uint32_t)(byte & 3) * 8 + ((bin[j] & 1) ? 0 : 4);
            }
            if (KIND != BIT) cur[j] = __ldcg(word[j]);
        }
        if (KIND == BIT) {
#pragma unroll
            for (int j = 0; j < U; j++)
                if (act[j]) before[j] = (atomicOr(word[j], 1u << sh[j]) >> sh[j]) & 1u;
        } else {
            uint32_t seen[U];
            bool pend[U];
#pragma unroll
            for (int j = 0; j < U; j++) {
                pend[j] = false;
                seen[j] = 0;
                if (!act[j]) continue;
                before[j] = (cur[j] >> sh[j]) & CAP;
                const uint32_t tt = before[j] + m[j], nv = tt > CAP ? CAP : tt;
                if (nv == before[j]) continue;
                seen[j] = atomicCAS(word[j], cur[j], (cur[j] & ~(CAP << sh[j])) | (nv << sh[j]));
                pend[j] = true;
            }
#pragma unroll
            for (int j = 0; j < U; j++) {
                if (!pend[j] || seen[j] == cur[j]) continue;
                uint32_t c = seen[j];   // somebody else changed the word in between (a neighbouring bin): the usual loop
                while (true) {
                    before[j] = (c >> sh[j]) & CAP;
                    const uint32_t tt = before[j] + m[j], nv = tt > CAP ? CAP : tt;
                    if (nv == before[j]) break;
                    const uint32_t sn = atomicCAS(word[j], c, (c & ~(CAP << sh[j])) | (nv << sh[j]));
                    if (sn == c) break;
                    c = sn;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < U; j++) {
            if (!act[j]) continue;
            if (KIND == BYTE) {
                const uint32_t tt = before[j] + m[j];
                n_sat += tt > 255u;
                if (tt >= 255u && before[j] < 255u) {
                    n_cross++;
                    if (want_cross) {
                        unsigned long long at = atomicAdd(&ctrl->n_events, 1ull);
                        if (at < list_cap) binlist[at] = BL_CROSS | ((unsigned long long)before[j] << 48) | ht_key(bin[j], t);
                    }
                }
                if (want_cross && tt >= 255u) atomicOr(reinterpret_cast<uint32_t*>(sb.t[t]) + (bin[j] >> 5), 1u << (bin[j] & 31));
            }
            if (before[j] == 0) {
                n_new++;
                atomicOr(&newbits[pos[j] >> 5], 1u << (pos[j] & 31));
                if (newmask) atomicOr(&newmask[pos[j]], 1u << t);
            }
        }
    }
    // one update of the chunk's counters per CTA (millions of CTAs adding to the same few words would queue at their L2 slice);
    // the host derives "bins newly occupied in any table / in table 0" from the per-table counts
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
        if (s_tot[0]) atomicAdd(&ctrl->n_new_t[t], (unsigned long long)s_tot[0]);
        if (s_tot[1]) atomicAdd(&ctrl->n_sat, (unsigned long long)s_tot[1]);
        if (s_tot[2]) atomicAdd(&ctrl->n_cross, (unsigned long long)s_tot[2]);
    }
}

// =====================================================================================================================
// 4. bigcount scan for this path (no bins[] array): re-hash the stream, probe the saturation bitmaps (one bit per bin,
//    kept by k_apply2 / k_apply_sparse).  Reports the same events as k_bigscan.
// =====================================================================================================================
template <int HK, int SRC>
__global__ void __launch_bounds__(THREADS)
k_bigscan2(const __grid_constant__ SketchDev S, HashCfg H, Input in, const __grid_constant__ SatBitsG sat, const uint64_t* __restrict__ keys,
           uint64_t mask, int have_cross, Event* out, unsigned long long cap, Ctrl* ctrl, uint32_t pos_base, const __grid_constant__ SketchDev M,
           const __grid_constant__ Pred P, int pred)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
    const int nt = S.n_tables;
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        if (!tile_valid<HK, SRC>(sm, lp)) continue;
        const uint64_t h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
        if (pred && !pred_pass(P, M, h)) continue;
        bool allsat = true;
        uint32_t cross = 0;
        for (int i = 0; i < nt; i++) {
            const uint64_t bin = mod_magic(h, S.sizes[i], S.magic[i]);
            const bool s = (__ldg(&sat.t[i][bin >> 3]) >> (bin & 7)) & 1u;
            allsat &= s;
            if (!s && !have_cross) break;
            if (s && have_cross && ht_find(keys, mask, ht_key(bin, i)) != ~0ull) cross |= 1u << i;
        }
        if (!cross && !allsat) continue;
        Event e;
        e.hash = h;
        e.pos = pos_base + t0 + lp;
        e.info = cross | ((uint32_t)allsat << 30);
        unsigned long long at = atomicAdd(&ctrl->n_events, 1ull);
        if (at < cap) out[at] = e;
    }
}

}  // namespace kmgpu

namespace kmgpu {

// =====================================================================================================================
// 5. Digital normalization (scripts/normalize-by-median.py:155-179, khmer/utils.py:178-180, Hashtable::median_at_least
//    src/oxli/hashtable.cc:333-364).  The reference keeps a read bundle iff one of its reads has a median count below
//    the cutoff in the table AS IT IS when the bundle arrives, and consumes it at once — a serial dependency.  Counts
//    only grow, so for a window of reads: a bundle at or above the cutoff at the window's start is discarded for good;
//    a candidate still below the cutoff after EVERY candidate of the window has been added (the overlay below) is kept
//    for good; the few in between are resolved on the device in rounds (k_norm_resolve) from exact per-bin data.
// =====================================================================================================================

// overlay: (table, bin) -> touches by the window's candidate reads (open addressing, keys as ht_key)
template <int HK, int SRC>
__global__ void __launch_bounds__(THREADS)
k_norm_overlay_add(const __grid_constant__ SketchDev S, HashCfg H, Input in, uint64_t* keys, uint32_t* vals, uint64_t mask)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        if (!tile_valid<HK, SRC>(sm, lp)) continue;
        const uint64_t h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
        for (int i = 0; i < S.n_tables; i++) {
            const uint64_t s = ht_insert(keys, mask, ht_key(mod_magic(h, S.sizes[i], S.magic[i]), i));
            atomicAdd(&vals[s], 1u);
        }
    }
}

// counts of the candidates' k-mers as if every candidate of the window had been consumed: min over tables of
// min(cap, counter + overlay) (Storage::get_count; a saturated ByteStorage count compares >= any cutoff <= 255)
template <int KIND, int HK, int SRC>
__global__ void __launch_bounds__(THREADS)
k_norm_counts_overlay(const __grid_constant__ SketchDev S, HashCfg H, Input in, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                      uint64_t mask, uint16_t* __restrict__ counts)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        if (!tile_valid<HK, SRC>(sm, lp)) continue;
        const uint64_t h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
        uint32_t mn = counter_cap<KIND>();
        for (int i = 0; i < S.n_tables; i++) {
            const uint64_t bin = mod_magic(h, S.sizes[i], S.magic[i]);
            uint32_t c = read_counter<KIND>(S.tables[i], bin);
            const uint64_t s = ht_find(keys, mask, ht_key(bin, i));
            if (s != ~0ull) c += vals[s];
            mn = c < mn ? c : mn;
        }
        counts[t0 + lp] = (uint16_t)mn;
    }
}

// per position of an in-between read (upos[j] = chunk position): for every table, the counter of its bin at the window's start
// and the slot of (table, bin) in the set the next kernels probe
template <int KIND, int HK>
__global__ void __launch_bounds__(256)
k_norm_gather(const __grid_constant__ SketchDev S, HashCfg H, Input in, const uint32_t* __restrict__ upos, uint32_t n_up, uint32_t* __restrict__ out_slot,
              uint16_t* __restrict__ out_c0, uint64_t* keys2, uint64_t mask2)
{
    const uint32_t j = blockIdx.x * 256u + threadIdx.x;
    if (j >= n_up) return;
    const uint64_t h = hash_at<HK, 0>(in, H.k, upos[j]);
    for (int i = 0; i < S.n_tables; i++) {
        const uint64_t bin = mod_magic(h, S.sizes[i], S.magic[i]);
        out_c0[(size_t)j * S.n_tables + i] = (uint16_t)read_counter<KIND>(S.tables[i], bin);
        out_slot[(size_t)j * S.n_tables + i] = (uint32_t)ht_insert(keys2, mask2, ht_key(bin, i));
    }
}

// touches of the registered (table, bin) pairs by the window's candidate reads (in.read_keep), as one list per pair.
// PASS 0 counts them (cnt[slot]); k_norm_hit_offsets gives every pair its range; PASS 1 writes (position, read) into the range
// (fill[slot] ends at the range's end).
template <int HK, int SRC, int PASS>
__global__ void __launch_bounds__(THREADS)
k_norm_hits(const __grid_constant__ SketchDev S, HashCfg H, Input in, const uint64_t* __restrict__ keys2, uint64_t mask2, uint32_t* cnt_or_fill,
            uint2* __restrict__ hits)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        if (!tile_valid<HK, SRC>(sm, lp)) continue;
        const uint64_t h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
        uint32_t read = ~0u;
        for (int i = 0; i < S.n_tables; i++) {
            const uint64_t sl = ht_find(keys2, mask2, ht_key(mod_magic(h, S.sizes[i], S.magic[i]), i));
            if (sl == ~0ull) continue;
            const uint32_t at = atomicAdd(&cnt_or_fill[sl], 1u);
            if (PASS == 1) {
                if (read == ~0u) {   // the read this position belongs to: last r with offs[r] <= position
                    uint32_t lo = in.tfr[blockIdx.x], hi = in.tfr[blockIdx.x + 1];
                    const uint32_t p = t0 + lp;
                    while (lo < hi) {
                        const uint32_t mid = (lo + hi + 1) >> 1;
                        if (in.offs[mid] <= p) lo = mid; else hi = mid - 1;
                    }
                    read = lo;
                }
                hits[at] = make_uint2(t0 + lp, read);
            }
        }
    }
}

__global__ void k_norm_hit_offsets(const uint32_t* __restrict__ cnt, uint32_t* __restrict__ fill, uint64_t n_slots, unsigned long long* total)
{
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < n_slots; s += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t c = cnt[s];
        if (c) fill[s] = (uint32_t)atomicAdd(total, (unsigned long long)c);
    }
}

// One round of the in-between resolution, one warp per in-between bundle.  state[read]: 0 discarded, 1 kept, 2 undecided.
// The reference's decision for a bundle depends on the bundles kept BEFORE it; counts only grow with every kept read, so with
// lo = (kept so far) and hi = (kept or undecided) every count is bracketed: below the cutoff even under hi => kept; at or
// above it already under lo => discarded.  The first undecided bundle of the stream always decides (lo = hi before it), every
// round decides at least that one; rounds repeat until none is left.  Reading a state another warp has just decided only
// tightens the bracket.
struct NormResolve {
    const uint32_t* ub_first;   // [n_ub + 1] first in-between read (index into ur_*) of every in-between bundle
    const uint32_t* ub_start;   // [n_ub]     chunk position where the bundle starts: only touches before it count
    const uint32_t* ur_first;   // [n_ur + 1] first entry of every in-between read in slot[] / c0[] (entries = its k-mers)
    const uint32_t* ur_read;    // [n_ur]     read number within the window
    const uint32_t* slot;       // [entries x N]
    const uint16_t* c0;         // [entries x N]
    const uint32_t* cnt;        // per slot: number of hits; they end at fill[slot]
    const uint32_t* fill;
    const uint2* hits;
    uint8_t* state;
    int n_tables;
    uint32_t cutoff, cap;
};

__global__ void __launch_bounds__(256)
k_norm_resolve(const __grid_constant__ NormResolve R, uint32_t n_ub, unsigned int* n_left)
{
    const int lane = threadIdx.x & 31;
    const uint32_t b = blockIdx.x * 8u + (threadIdx.x >> 5);
    if (b >= n_ub) return;
    const uint32_t q0 = R.ub_first[b], q1 = R.ub_first[b + 1];
    volatile uint8_t* state = R.state;
    if (state[R.ur_read[q0]] != 2) return;
    const uint32_t bstart = R.ub_start[b];
    bool kept = false, all_above = true;
    for (uint32_t q = q0; q < q1; q++) {
        const uint32_t e0 = R.ur_first[q], nk = R.ur_first[q + 1] - e0;
        unsigned ge_lo = 0, ge_hi = 0;
        for (uint32_t i = lane; i < nk; i += 32) {
            uint32_t mn_lo = R.cap, mn_hi = R.cap;
            for (int t = 0; t < R.n_tables; t++) {
                const size_t at = (size_t)(e0 + i) * R.n_tables + t;
                const uint32_t sl = R.slot[at];
                uint32_t v_lo = R.c0[at], v_hi = v_lo;
                const uint32_t end = R.fill[sl], beg = end - R.cnt[sl];
                for (uint32_t x = beg; x < end; x++) {
                    const uint2 hit = R.hits[x];
                    if (hit.x >= bstart) continue;
                    const uint32_t st = state[hit.y];
                    v_lo += st == 1;
                    v_hi += st >= 1;
                }
                mn_lo = v_lo < mn_lo ? v_lo : mn_lo;
                mn_hi = v_hi < mn_hi ? v_hi : mn_hi;
            }
            ge_lo += mn_lo >= R.cutoff;
            ge_hi += mn_hi >= R.cutoff;
        }
        ge_lo = __reduce_add_sync(0xffffffffu, ge_lo);
        ge_hi = __reduce_add_sync(0xffffffffu, ge_hi);
        const unsigned req = (unsigned)(0.5 + (double)((float)nk / 2));   // Hashtable::median_at_least (hashtable.cc:337)
        kept |= ge_hi < req;
        all_above &= !(ge_lo < req);
    }
    if (!kept && !all_above) {
        if (lane == 0) atomicAdd(n_left, 1u);
        return;
    }
    const uint8_t v = kept ? 1 : 0;
    for (uint32_t q = q0 + lane; q < q1; q += 32) state[R.ur_read[q]] = v;
}

// keep bits of a window from the per-read states (1 = kept)
__global__ void k_norm_keep_bits(const uint8_t* __restrict__ state, uint32_t n_reads, uint32_t* __restrict__ bits)
{
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w * 32u >= n_reads) return;
    uint32_t m = 0;
    for (uint32_t j = 0; j < 32 && w * 32u + j < n_reads; j++) m |= (uint32_t)(state[w * 32u + j] == 1) << j;
    bits[w] = m;
}

}  // namespace kmgpu

namespace kmgpu {

// =====================================================================================================================
// 6. First-touch log (replicated sketches, SURVEY.md §8e): n_unique_kmers and abundance_distribution count a k-mer
//    occurrence iff one of its bins was empty when it arrived IN STREAM ORDER.  With one replica per rank and the ranks'
//    read shards taken in rank order, an occurrence on rank r is globally new iff, for some table, it was the first
//    toucher of an empty bin locally AND no rank below r touched that bin.  Every rank therefore logs, per chunk, one
//    entry per newly occupied bin: (table, bin), position, chunk — and, for abundance_distribution, the k-mer's count.
//    At merge time (before any table is modified) rank r drops the entries whose bin is occupied on a lower rank and
//    counts the distinct positions that are left.
// =====================================================================================================================
struct FtEntry {
    uint64_t key;      // ht_key(bin, table)
    uint32_t pos;      // position within its chunk
    uint16_t chunk;    // chunk number within the epoch (mod 2^16: (chunk, pos) pairs only need to be distinct per position)
    uint16_t count;    // abundance_distribution: the k-mer's count in the counting sketch
};

// entries of one chunk: for every position marked new, one entry per table whose bin it occupied (newmask[p])
template <int HK, int SRC>
__global__ void __launch_bounds__(THREADS)
k_ft_emit(const __grid_constant__ SketchDev S, HashCfg H, Input in, const uint32_t* __restrict__ newbits, const uint32_t* __restrict__ newmask,
          uint32_t pos_base, uint32_t chunk, const uint16_t* __restrict__ counts, FtEntry* __restrict__ out, unsigned long long cap,
          unsigned long long* cursor)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        if (!tile_valid<HK, SRC>(sm, lp)) continue;
        const uint32_t p = pos_base + t0 + lp;
        if (!((newbits[p >> 5] >> (p & 31)) & 1u)) continue;
        uint32_t m = newmask[p];
        if (!m) continue;
        const uint64_t h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
        const uint16_t c = counts ? counts[p] : (uint16_t)0;
        while (m) {
            const int t = __ffs(m) - 1;
            m &= m - 1;
            FtEntry e;
            e.key = ht_key(mod_magic(h, S.sizes[t], S.magic[t]), t);
            e.pos = p;
            e.chunk = (uint16_t)chunk;
            e.count = c;
            const unsigned long long at = atomicAdd(cursor, 1ull);
            if (at < cap) out[at] = e;
        }
    }
}

struct LowerRanks {
    const uint8_t* tables[MAX_WORLD][G_MAXT];   // the tables of the ranks below this one (peer memory)
    int n;
};

// entries whose bin no lower rank occupies survive; the distinct (chunk, position) pairs among the survivors are the
// globally new k-mer occurrences of this rank: counted, and histogrammed by their count
template <int KIND>
__global__ void __launch_bounds__(256)
k_ft_resolve(const FtEntry* __restrict__ ent, unsigned long long n, const LowerRanks* __restrict__ lower, unsigned long long* seen, uint64_t mask,
             unsigned long long* n_new, unsigned long long* hist)
{
    for (unsigned long long i = blockIdx.x * 256ull + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * 256ull) {
        const FtEntry e = ent[i];
        const int t = (int)(e.key & 255u);
        const uint64_t bin = e.key >> 8;
        bool alive = true;
        for (int q = 0; q < lower->n && alive; q++) alive = read_counter<KIND>(lower->tables[q][t], bin) == 0;
        if (!alive) continue;
        const unsigned long long id = ((unsigned long long)e.chunk << 32) | e.pos;
        uint64_t s = fmix64(id) & mask;
        while (true) {
            const unsigned long long prev = atomicCAS(&seen[s], ~0ull, id);
            if (prev == ~0ull) {
                atomicAdd(n_new, 1ull);
                if (hist) atomicAdd(&hist[e.count], 1ull);
                break;
            }
            if (prev == id) break;
            s = (s + 1) & mask;
        }
    }
}

}  // namespace kmgpu

namespace kmgpu {

// =====================================================================================================================
// 7. HyperLogLog registers (HLLCounter::add, src/oxli/hllcounter.cc:262-298; unique-kmers.py): for every k-mer, its
//    canonical Murmur hash (_hash_murmur, kmer_hash.cc:177-198); register = low p bits, value = leading zeros of the
//    remaining 64 - p bits + 1 (64 - p + 1 when they are all zero); registers[index] = max(registers[index], value).
//    Registers are 32-bit words on the device (atomicMax), bytes at the ABI.  After the first few thousand k-mers almost
//    no k-mer raises its register: the plain load in front of the atomic is what the kernel mostly does.
// =====================================================================================================================
template <int HK, int SRC>
__global__ void __launch_bounds__(THREADS)
k_hll(HashCfg H, Input in, int p, uint32_t* __restrict__ regs)
{
    __shared__ TileSmem sm;
    const uint32_t t0 = blockIdx.x * TILE;
    tile_begin<HK, SRC>(in, H.k, t0, sm);
    const uint64_t mask = (1ull << p) - 1;
#pragma unroll 1
    for (uint32_t lp = threadIdx.x; lp < TILE; lp += THREADS) {
        if (t0 + lp >= in.n_pos) break;
        if (!tile_valid<HK, SRC>(sm, lp)) continue;
        const uint64_t h = tile_hash<HK, SRC>(in, sm, H.k, t0, lp);
        const uint64_t rest = h >> p;
        const uint32_t v = (uint32_t)(rest ? __clzll((long long)rest) : 64) - (uint32_t)p + 1u;
        uint32_t* r = regs + (h & mask);
        if (*r < v) atomicMax(r, v);
    }
}

__global__ void k_hll_bytes(const uint32_t* __restrict__ regs, uint32_t n, uint8_t* __restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint8_t)regs[i];
}

__global__ void k_hll_max_bytes(uint32_t* __restrict__ regs, uint32_t n, const uint8_t* __restrict__ in, int replace)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) regs[i] = replace ? (uint32_t)in[i] : max(regs[i], (uint32_t)in[i]);
}

}  // namespace kmgpu

namespace kmgpu {

// =====================================================================================================================
// 8. Address-sharded sketches (SURVEY.md §8e, config C5): the k-mer exchange.  Every rank groups its own counter updates by
//    super-bucket of the FULL tables (k_part MODE 1; a rank's slice is a whole number of super-buckets, so "owner" is a
//    division of the super-bucket index), tells every owner how many records it holds for each of the owner's super-buckets
//    (k_shard_post), the owner lays its receive arena out exactly (k_shard_scan, k_shard_sb: per super-bucket, per sender),
//    and every sender then writes its runs — contiguous, hundreds of KB each — straight into the owner's HBM over NVLink
//    peer memory (k_shard_push).  No per-record remote atomics, no staging on the receiving side, no NCCL.
// =====================================================================================================================
struct ShardGeom {
    uint32_t first_sb[G_MAXT + 1];      // full-table layout: table i owns global super-buckets [first_sb[i], first_sb[i+1])
    uint32_t sb_per_rank[G_MAXT];       // super-buckets of table i held by every rank (the last ranks may hold fewer or none)
    uint32_t local_first[G_MAXT + 1];   // a rank's local numbering: table i starts at local_first[i] (= prefix sums of sb_per_rank)
    int n_tables, world, rank;
};

struct ShardPeers {
    uint32_t* demand[MAX_WORLD];                 // [local super-bucket * world + sender]
    const unsigned long long* recv_off[MAX_WORLD];   // same indexing (+1): where that sender's run starts in the owner's arena
    unsigned long long* rec[MAX_WORLD];          // the owner's arena
    const unsigned long long* flags[MAX_WORLD];  // bit 0: the owner's arena cannot hold this round
};

__device__ __forceinline__ void shard_owner(const ShardGeom& G, uint32_t g, int* owner, uint32_t* local)
{
    int t = 0;
#pragma unroll 1
    for (int i = 1; i < G.n_tables; i++)
        if (g >= G.first_sb[i]) t = i;
    const uint32_t sb = g - G.first_sb[t];
    const uint32_t q = sb / G.sb_per_rank[t];
    *owner = (int)q;
    *local = G.local_first[t] + (sb - q * G.sb_per_rank[t]);
}

// my record counts per global super-bucket -> the owners' demand tables
__global__ void k_shard_post(const __grid_constant__ ShardGeom G, const uint32_t* __restrict__ count, uint32_t n_sb_total, const __grid_constant__ ShardPeers P)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_sb_total) return;
    int q;
    uint32_t j;
    shard_owner(G, g, &q, &j);
    P.demand[q][(size_t)j * G.world + G.rank] = count[g];
}

// exclusive scan (no padding between entries): off[i] for i in [0, n], single CTA
__global__ void __launch_bounds__(1024) k_shard_scan(const uint32_t* __restrict__ cnt, uint32_t n, unsigned long long* __restrict__ off)
{
    __shared__ unsigned long long s_w[32];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        unsigned long long v = i < n ? cnt[i] : 0, incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (uint32_t)o) incl += u;
        }
        if (lane == 31) s_w[wid] = incl;
        __syncthreads();
        unsigned long long before = s_carry;
        for (uint32_t w = 0; w < wid; w++) before += s_w[w];
        if (i < n) off[i] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) off[n] = s_carry;
}

// per local super-bucket: where its records start (all senders' runs are adjacent) and how many there are; the largest count
__global__ void k_shard_sb(const unsigned long long* __restrict__ recv_off, uint32_t n_sb_local, int world, unsigned long long* __restrict__ sb_off,
                           uint32_t* __restrict__ sb_cnt, unsigned int* max_cnt)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j > n_sb_local) return;
    const unsigned long long a = recv_off[(size_t)j * world];
    sb_off[j] = a;
    if (j < n_sb_local) {
        const uint32_t c = (uint32_t)(recv_off[(size_t)(j + 1) * world] - a);
        sb_cnt[j] = c;
        atomicMax(max_cnt, c);
    }
}

// my runs go to their owners: grid (global super-buckets, PUSH_Y); plain coalesced 8-byte stores into peer memory
__global__ void __launch_bounds__(256)
k_shard_push(const __grid_constant__ ShardGeom G, Store src, const __grid_constant__ ShardPeers P)
{
    const uint32_t g = blockIdx.x;
    uint32_t c = src.cursor[g];
    if (c == 0) return;
    const uint32_t room = src.room(g);
    if (c > room) c = room;   // cannot happen after the exact regrouping run; the owner's count would then disagree and refuse
    int q;
    uint32_t j;
    shard_owner(G, g, &q, &j);
    if (*P.flags[q] & 1ull) return;
    const unsigned long long* from = src.rec + src.base(g);
    unsigned long long* to = P.rec[q] + P.recv_off[q][(size_t)j * G.world + G.rank];
    for (uint32_t e = blockIdx.y * 256u + threadIdx.x; e < c; e += gridDim.y * 256u) to[e] = __ldcs(from + e);
}

// ---- query rounds: route, offsets and push as above, then the owner answers every record in place and the sender reads
//      its answers back.  An answered record keeps its position bits; its low 15 + s bits hold the counter.
// owner: grid (local super-buckets, Y); the records of super-bucket j are arena[sb_off[j] .. + sb_cnt[j])
template <int KIND>
__global__ void __launch_bounds__(256)
k_shard_lookup(const __grid_constant__ ShardGeom G, const __grid_constant__ SketchDev S, unsigned long long* __restrict__ arena,
               const unsigned long long* __restrict__ sb_off, const uint32_t* __restrict__ sb_cnt, int sb_bin_shift)
{
    const uint32_t j = blockIdx.x;
    const uint32_t c = sb_cnt[j];
    if (c == 0) return;
    int t = 0;
#pragma unroll 1
    for (int i = 1; i < G.n_tables; i++)
        if (j >= G.local_first[i]) t = i;
    const unsigned long long mask = (1ull << sb_bin_shift) - 1;
    const uint64_t bin0 = (uint64_t)(j - G.local_first[t]) << sb_bin_shift;
    const uint8_t* tab = S.tables[t];
    unsigned long long* rec = arena + sb_off[j];
    const uint32_t step = gridDim.y * 256u;
    for (uint32_t e0 = blockIdx.y * 256u + threadIdx.x; e0 < c; e0 += 4 * step) {   // four random table loads in flight per thread
        unsigned long long r[4];
        uint32_t v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) r[u] = e0 + u * step < c ? rec[e0 + u * step] : 0ull;
#pragma unroll
        for (int u = 0; u < 4; u++) v[u] = e0 + u * step < c ? read_counter<KIND>(tab, bin0 | (r[u] & mask)) : 0u;
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (e0 + u * step < c) rec[e0 + u * step] = (r[u] & ~mask) | v[u];
    }
}

// sender: grid (global super-buckets, Y), the runs the push wrote; answers land in one byte plane per table (plain stores: every
// (table, position) has exactly one record).  A run whose owner refused the round sets *refused and is not read.
__global__ void __launch_bounds__(256)
k_shard_pull(const __grid_constant__ ShardGeom G, Store src, const __grid_constant__ ShardPeers P, int sb_bin_shift, uint32_t pos_base,
             uint64_t plane_stride, uint8_t* __restrict__ planes, unsigned long long* refused)
{
    const uint32_t g = blockIdx.x;
    uint32_t c = src.cursor[g];
    if (c == 0) return;
    const uint32_t room = src.room(g);
    if (c > room) c = room;
    int q;
    uint32_t j;
    shard_owner(G, g, &q, &j);
    if (*P.flags[q] & 1ull) {
        if (blockIdx.y == 0 && threadIdx.x == 0) atomicOr(refused, 1ull);
        return;
    }
    int t = 0;
#pragma unroll 1
    for (int i = 1; i < G.n_tables; i++)
        if (g >= G.first_sb[i]) t = i;
    const unsigned long long* from = P.rec[q] + P.recv_off[q][(size_t)j * G.world + G.rank];
    uint8_t* plane = planes + (size_t)t * plane_stride;
    const unsigned long long mask = (1ull << sb_bin_shift) - 1;
    for (uint32_t e = blockIdx.y * 256u + threadIdx.x; e < c; e += gridDim.y * 256u) {
        const unsigned long long r = __ldcs(from + e);
        plane[(uint32_t)(r >> sb_bin_shift) - pos_base] = (uint8_t)(r & mask);
    }
}

// count per position = min over the tables' planes (get_count, storage.hh:627-649 / :362-379 / :207-219, without bigcount)
__global__ void k_shard_fold(const uint8_t* __restrict__ planes, int n_tables, uint64_t plane_stride, uint32_t n_pos, uint16_t* __restrict__ counts)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_pos; p += gridDim.x * blockDim.x) {
        uint32_t m = planes[p];
        for (int t = 1; t < n_tables; t++) m = min(m, (uint32_t)planes[(size_t)t * plane_stride + p]);
        counts[p] = (uint16_t)m;
    }
}

}  // namespace kmgpu

