// C ABI (include/kmgpu.h) + host orchestration of the kernels in kmgpu_kernels.cuh.
//
// One handle = one sketch resident in HBM.  Reads are processed in chunks of at most CHUNK_BASES stream
// positions; per chunk: H2D (ASCII or packed) -> k_pack -> one of the bins, delta or grouped paths (choose_path)
// -> [only when bytes saturated] bigcount events to the host map.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <functional>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/kmgpu.h"
#include "kmgpu_kernels.cuh"
#include "kmgpu_group.cuh"

using namespace kmgpu;

// ------------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t _e = (call);                                                                          \
        if (_e != cudaSuccess) {                                                                          \
            int _c = (_e == cudaErrorMemoryAllocation) ? KMGPU_ENOMEM                                      \
                     : (_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver) ? KMGPU_ENODEV      \
                                                                                      : KMGPU_ECUDA;      \
            return fail(_c, "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__,       \
                        cudaGetErrorString(_e));                                                          \
        }                                                                                                 \
    } while (0)

#define CKR(call)                  \
    do {                           \
        int _r = (call);           \
        if (_r != KMGPU_OK) return _r; \
    } while (0)

static uint64_t env_u64(const char* name, uint64_t dflt)
{
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    return strtoull(v, nullptr, 10);
}

// stream positions per chunk (multiple of TILE).  Bounded so positions fit 32 bits.
static uint64_t chunk_bases()
{
    static uint64_t c = [] {
        uint64_t v = env_u64("KMGPU_CHUNK_BASES", 152000000ull);   // ~0.85 ms of every chunk does not depend on its size
        v = std::max<uint64_t>(TILE, std::min<uint64_t>(v, 1ull << 31));
        return (v / TILE) * TILE;
    }();
    return c;
}

// ------------------------------------------------------------------------------------------------------
// growable device / pinned buffers
// ------------------------------------------------------------------------------------------------------
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    int ensure(size_t n)
    {
        if (n <= cap) return KMGPU_OK;
        if (p) cudaFree(p);
        p = nullptr;
        size_t want = std::max<size_t>(n, cap + cap / 2);
        cap = 0;   // a failed allocation leaves an empty buffer, not a stale capacity
        cudaError_t e = cudaMalloc(&p, want * sizeof(T));
        if (e == cudaErrorMemoryAllocation && want > n) {   // no room for the growth margin: take exactly what is needed
            cudaGetLastError();
            want = n;
            e = cudaMalloc(&p, want * sizeof(T));
        }
        if (e != cudaSuccess) p = nullptr;
        CK(e);
        cap = want;
        return KMGPU_OK;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

template <class T>
struct PinBuf {
    T* p = nullptr;
    size_t cap = 0;
    int ensure(size_t n)
    {
        if (n <= cap) return KMGPU_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        size_t want = std::max<size_t>(n, cap + cap / 2);
        cap = 0;
        CK(cudaMallocHost(&p, want * sizeof(T)));
        cap = want;
        return KMGPU_OK;
    }
    void release()
    {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// a chunk of reads staged on the device
struct ChunkDev {
    const uint64_t* words = nullptr;
    const uint32_t* offs = nullptr;
    const uint32_t* tfr = nullptr;
    const uint32_t* valid = nullptr;   // bitmap of k-mer starts (k_valid_bits)
    uint32_t n_reads = 0;
    uint32_t n_pos = 0;
};

struct kmgpu_batch {
    int device = 0;
    int ksize = 0;
    uint64_t n_reads = 0, n_bases = 0, bytes = 0;
    struct Piece {
        uint64_t* words;
        uint32_t* offs;
        uint32_t* tfr;
        uint32_t n_reads, n_pos;
        uint32_t* valid;
    };
    std::vector<Piece> pieces;
};

struct Peer {
    uint8_t* tables[MAX_TABLES];
};

struct kmgpu_sketch {
    int device = 0;
    int kind = 0, hash = 0, k = 0, nt = 0;
    uint64_t sizes[MAX_TABLES];
    uint64_t nbytes[MAX_TABLES];
    uint64_t alloc_bytes[MAX_TABLES];
    SketchDev dev;
    uint64_t n_occupied = 0, n_unique = 0;
    bool use_bigcount = false;
    std::unordered_map<uint64_t, uint16_t> big;  // same container as the reference (storage.hh:50)
    bool big_dirty = true;
    DevBuf<uint64_t> big_keys;
    DevBuf<uint16_t> big_vals;
    uint32_t n_big_dev = 0;

    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, tev0 = nullptr, tev1 = nullptr;
    std::mutex mu;

    // staging of read chunks: two slots so that the upload + packing of chunk i+1 (copy stream) overlaps the
    // ingestion of chunk i (main stream)
    static constexpr int MAX_PARTS = 16;           // parts of a chunk of host input (each staged in its own slot)
    static constexpr int N_STAGE = 2 * MAX_PARTS;   // two sets: the next chunk is uploaded while this one is ingested
    struct Stage {
        DevBuf<uint8_t> ascii;
        DevBuf<uint64_t> words;
        DevBuf<uint32_t> offs;
        DevBuf<uint64_t> offs64;
        DevBuf<uint32_t> tfr;
        DevBuf<uint32_t> valid;
        PinBuf<uint32_t> h_offs;
        PinBuf<uint64_t> h_offs64;
        cudaEvent_t ready = nullptr;
    } stage[N_STAGE];
    cudaStream_t copy_stream = nullptr;
    Ctrl* d_ctrl_copy = nullptr;
    Ctrl* h_ctrl_copy = nullptr;  // pinned
    // workspace
    DevBuf<uint32_t> d_newbits;
    DevBuf<uint32_t> d_filter;
    DevBuf<uint32_t> d_rank;
    DevBuf<unsigned long long> d_records;   // bucket path: update records, bucket-major
    DevBuf<uint32_t> d_cursors;
    DevBuf<unsigned long long> d_rec1;      // grouped path, two-level: records by super-bucket
    DevBuf<uint32_t> d_cur1;
    DevBuf<unsigned long long> d_off1, d_off2;   // exact region offsets of a regrouping run
    DevBuf<uint64_t> d_hash64;              // Murmur: 64-bit hash of every position of the chunk
    DevBuf<uint32_t> d_readbits;            // one bit per read of a window (normalization: candidates / kept)
    DevBuf<uint32_t> d_upos;                // normalization: positions of the in-between reads' k-mers + bundle / read index arrays
    DevBuf<uint32_t> d_nslot, d_ncnt, d_nfill;   // normalization: in-between resolution (k_norm_resolve)
    DevBuf<uint2> d_nhits;
    DevBuf<uint8_t> d_nstate;
    uint64_t n_norm_rounds = 0;
    DevBuf<uint16_t> d_uc0;
    uint64_t n_norm_unsure = 0;
    // first-touch log (replicated sketches: exact n_unique_kmers / abundance_distribution across ranks)
    bool ft_on = false, ft_defer = false;
    DevBuf<uint32_t> d_newmask;
    std::vector<std::pair<void*, uint64_t>> ft_segs;   // one segment of FtEntry per chunk
    uint64_t ft_pending = 0, ft_epoch_unique = 0;
    uint32_t ft_chunk = 0;
    uint64_t n_regroups = 0;
    double group_boost1 = 1.0, group_boost2 = 1.0;   // grouped path: slack factors learnt from regions that overflowed
    DevBuf<uint32_t> d_biglist;                      // regrouping run: heavily loaded buckets
    uint64_t chunk_cap = 0;                 // positions per chunk (sketch_chunk_bases)
    bool bucket_attr_set = false;
    DevBuf<uint32_t> d_bins;
    DevBuf<uint16_t> d_delta;
    size_t delta_zeroed = 0;
    DevBuf<uint64_t> d_binlist;
    DevBuf<uint32_t> d_sel;      // radix-select state (need / prefix / cnt per crossing-bin slot) + record slots
    DevBuf<uint32_t> d_recslot;
    DevBuf<unsigned long long> d_evkeys;
    DevBuf<uint32_t> d_evvals;
    DevBuf<EvOut> d_evout;
    PinBuf<EvOut> h_evout;
    DevBuf<uint8_t> d_satbits[MAX_TABLES];   // delta path + bigcount: bitmap of saturated bytes per table
    bool satbits_valid = false;
    DevBuf<uint64_t> d_htkeys;
    DevBuf<uint32_t> d_htvals;
    DevBuf<Event> d_events;
    DevBuf<uint16_t> d_counts;
    DevBuf<uint16_t> d_ocounts;             // normalization: counts under the overlay (d_counts keeps the window's start)
    DevBuf<uint64_t> d_hashes;
    DevBuf<uint64_t> d_hashin;
    DevBuf<uint16_t> d_stat_med;
    DevBuf<float> d_stat_f;
    DevBuf<uint32_t> d_stat_n;
    DevBuf<uint8_t> d_stat_b;
    DevBuf<unsigned long long> d_hist;
    Ctrl* d_ctrl = nullptr;
    Ctrl* h_ctrl = nullptr;  // pinned

    // profile
    double ingest_ms = 0;
    uint64_t ingest_launches = 0, all_launches = 0;

    // peers (multi-GPU)
    int rank = 0, world = 1;
    std::vector<Peer> peers;
    bool peers_ipc = false;
};

static int set_device(int dev) { CK(cudaSetDevice(dev)); return KMGPU_OK; }

// ------------------------------------------------------------------------------------------------------
// kernel dispatch
// ------------------------------------------------------------------------------------------------------
static Input make_input(const ChunkDev& c)
{
    Input in;
    in.words = c.words;
    in.offs = c.offs;
    in.tfr = c.tfr;
    in.n_reads = c.n_reads;
    in.hashes = nullptr;
    in.n_pos = c.n_pos;
    in.read_keep = nullptr;
    in.valid = c.valid;
    return in;
}
static Input make_hash_input(const uint64_t* d_hashes, uint32_t n)
{
    Input in;
    in.words = nullptr;
    in.offs = nullptr;
    in.tfr = nullptr;
    in.n_reads = 0;
    in.hashes = d_hashes;
    in.n_pos = n;
    in.read_keep = nullptr;
    in.valid = nullptr;
    return in;
}

static inline unsigned n_tiles(uint32_t n_pos) { return (n_pos + TILE - 1) / TILE; }

static void launch_counts(int src, const SketchDev& S, HashCfg H, const Input& in, const uint64_t* bk, const uint16_t* bv,
                          uint32_t nb, uint16_t* counts, uint64_t* hashes, const uint32_t* only_bits, cudaStream_t st)
{
    unsigned g = n_tiles(in.n_pos);
#define LC(KIND, T0, T1)                                                                                                  \
    do {                                                                                                                  \
        if (src == 1) k_counts<KIND, TWOBIT, 1><<<g, THREADS, 0, st>>>(S, H, in, bk, bv, nb, counts, hashes, only_bits, T0, T1);   \
        else if (H.kind == TWOBIT) k_counts<KIND, TWOBIT, 0><<<g, THREADS, 0, st>>>(S, H, in, bk, bv, nb, counts, hashes, only_bits, T0, T1); \
        else k_counts<KIND, MURMUR, 0><<<g, THREADS, 0, st>>>(S, H, in, bk, bv, nb, counts, hashes, only_bits, T0, T1);            \
    } while (0)
    // One table per launch when every table fits L2 by itself and the batch is large enough to re-use it (2-bit hashes are cheap
    // to recompute; a 400 MB sketch read through 100 MB at a time turns HBM-random loads into L2 hits).  KMGPU_COUNT_PASSES=0: off.
    static const bool passes_on = env_u64("KMGPU_COUNT_PASSES", 1) != 0;
    static const uint64_t count_pass_max = env_u64("KMGPU_COUNT_PASS_MAX_MB", 110) * 1000000ull;
    static const uint64_t count_pass_min_pos = env_u64("KMGPU_COUNT_PASS_MIN_POS", 1u << 22);   // tests: 1
    bool passes = passes_on && counts && !only_bits && S.n_tables > 1 && in.n_pos >= count_pass_min_pos && (src == 1 || H.kind == TWOBIT);
    for (int i = 0; passes && i < S.n_tables; i++) {
        const uint64_t bytes = S.kind == BYTE ? S.sizes[i] : S.kind == NIBBLE ? S.sizes[i] / 2 : S.sizes[i] / 8;
        if (bytes > count_pass_max) passes = false;
    }
    for (int t0 = 0; t0 < S.n_tables; t0 += passes ? 1 : S.n_tables) {
        const int t1 = passes ? t0 + 1 : S.n_tables;
        if (S.kind == BYTE) LC(BYTE, t0, t1);
        else if (S.kind == NIBBLE) LC(NIBBLE, t0, t1);
        else LC(BIT, t0, t1);
    }
#undef LC
}

// ------------------------------------------------------------------------------------------------------
// lifetime
// ------------------------------------------------------------------------------------------------------
extern "C" const char* kmgpu_last_error(void) { return g_err.c_str(); }
extern "C" int kmgpu_abi_version(void) { return KMGPU_ABI_VERSION; }

extern "C" int kmgpu_device_count(int* n)
{
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        *n = 0;
        return fail(KMGPU_ENODEV, "no CUDA device: %s", cudaGetErrorString(e));
    }
    *n = c;
    return KMGPU_OK;
}

extern "C" int kmgpu_alloc_pinned(size_t nbytes, void** out)
{
    if (!out) return fail(KMGPU_EINVAL, "out is NULL");
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return fail(KMGPU_ENODEV, "no CUDA device");
    CK(cudaMallocHost(out, nbytes ? nbytes : 1));
    return KMGPU_OK;
}
extern "C" int kmgpu_free_pinned(void* p)
{
    if (p) CK(cudaFreeHost(p));
    return KMGPU_OK;
}

static uint64_t table_nbytes(int kind, uint64_t size)
{
    // ByteStorage: size; NibbleStorage: size/2+1; BitStorage: size/8+1 (storage.hh:505-507, :290, :118)
    return kind == BYTE ? size : kind == NIBBLE ? size / 2 + 1 : size / 8 + 1;
}

static void refresh_dev(kmgpu_sketch* h)
{
    h->dev.n_tables = h->nt;
    h->dev.kind = h->kind;
    for (int i = 0; i < h->nt; i++) {
        h->dev.sizes[i] = h->sizes[i];
        h->dev.magic[i] = ~0ull / h->sizes[i];
    }
}

extern "C" int kmgpu_create(int storage, int hash, int ksize, int n_tables, const uint64_t* sizes, int device, kmgpu_t** out)
{
    if (!out) return fail(KMGPU_EINVAL, "out is NULL");
    *out = nullptr;
    if (storage < 0 || storage > 2) return fail(KMGPU_EINVAL, "bad storage kind %d", storage);
    if (hash < 0 || hash > 1) return fail(KMGPU_EINVAL, "bad hash kind %d", hash);
    if (ksize < 1 || ksize > MAX_K) return fail(KMGPU_EINVAL, "ksize %d out of range", ksize);
    if (hash == KMGPU_TWOBIT && ksize > 32)
        return fail(KMGPU_EINVAL, "Supplied kmer string doesn't match the underlying k-size.");  // kmer_hash.cc:70-72
    if (n_tables < 1 || n_tables > MAX_TABLES)
        return fail(KMGPU_EUNSUPPORTED, "n_tables %d not supported (1..%d)", n_tables, MAX_TABLES);
    for (int i = 0; i < n_tables; i++)
        if (sizes[i] == 0 || sizes[i] >= (1ull << 55)) return fail(KMGPU_EINVAL, "table size %llu out of range", (unsigned long long)sizes[i]);
    int ndev = 0;
    CKR(kmgpu_device_count(&ndev));
    if (ndev == 0) return fail(KMGPU_ENODEV, "no CUDA device");
    if (device < 0 || device >= ndev) return fail(KMGPU_EINVAL, "device %d out of range (%d devices)", device, ndev);
    CKR(set_device(device));
    kmgpu_sketch* h = new kmgpu_sketch();
    h->device = device;
    h->kind = storage;
    h->hash = hash;
    h->k = ksize;
    h->nt = n_tables;
    memset(&h->dev, 0, sizeof h->dev);
    for (int i = 0; i < n_tables; i++) {
        h->sizes[i] = sizes[i];
        h->nbytes[i] = table_nbytes(storage, sizes[i]);
        h->alloc_bytes[i] = (h->nbytes[i] + 15) & ~15ull;
        cudaError_t e = cudaMalloc(&h->dev.tables[i], h->alloc_bytes[i]);
        if (e == cudaSuccess) e = cudaMemset(h->dev.tables[i], 0, h->alloc_bytes[i]);
        if (e != cudaSuccess) {
            const unsigned long long want = h->alloc_bytes[i];
            cudaGetLastError();
            for (int j = 0; j <= i; j++)
                if (h->dev.tables[j]) cudaFree(h->dev.tables[j]);
            delete h;
            return fail(e == cudaErrorMemoryAllocation ? KMGPU_ENOMEM : KMGPU_ECUDA, "table %d (%llu bytes): %s", i, want, cudaGetErrorString(e));
        }
    }
    refresh_dev(h);
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&h->tev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->tev1);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_ctrl, sizeof(Ctrl));
    if (e == cudaSuccess) e = cudaMallocHost(&h->h_ctrl, sizeof(Ctrl));
    if (e == cudaSuccess) {   // the copy stream's small kernels (pack, offsets) must not queue behind the ingest grids
        int lo_prio = 0, hi_prio = 0;
        cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio);
        e = cudaStreamCreateWithPriority(&h->copy_stream, cudaStreamNonBlocking, hi_prio);
    }
    if (e == cudaSuccess) e = cudaMalloc(&h->d_ctrl_copy, sizeof(Ctrl));
    if (e == cudaSuccess) e = cudaMallocHost(&h->h_ctrl_copy, sizeof(Ctrl));
    for (int sl = 0; sl < kmgpu_sketch::N_STAGE && e == cudaSuccess; sl++) e = cudaEventCreateWithFlags(&h->stage[sl].ready, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        kmgpu_destroy(h);
        return fail(KMGPU_ECUDA, "handle setup: %s", cudaGetErrorString(e));
    }
    *out = h;
    return KMGPU_OK;
}

extern "C" int kmgpu_ipc_detach(kmgpu_t* h);

extern "C" int kmgpu_destroy(kmgpu_t* h)
{
    if (!h) return KMGPU_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    kmgpu_ipc_detach(h);
    for (int i = 0; i < h->nt; i++)
        if (h->dev.tables[i]) cudaFree(h->dev.tables[i]);
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    for (int sl = 0; sl < kmgpu_sketch::N_STAGE; sl++) {
        h->stage[sl].ascii.release(); h->stage[sl].words.release(); h->stage[sl].offs.release(); h->stage[sl].offs64.release(); h->stage[sl].tfr.release(); h->stage[sl].valid.release();
        h->stage[sl].h_offs.release(); h->stage[sl].h_offs64.release();
        if (h->stage[sl].ready) cudaEventDestroy(h->stage[sl].ready);
    }
    if (h->d_ctrl_copy) cudaFree(h->d_ctrl_copy);
    if (h->h_ctrl_copy) cudaFreeHost(h->h_ctrl_copy);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    h->d_newbits.release(); h->d_filter.release(); h->d_rank.release(); h->d_records.release(); h->d_cursors.release(); h->d_rec1.release(); h->d_cur1.release(); h->d_off1.release(); h->d_off2.release(); h->d_hash64.release(); h->d_newmask.release(); for (auto& sg : h->ft_segs) cudaFree(sg.first); h->ft_segs.clear(); h->d_readbits.release(); h->d_upos.release(); h->d_uc0.release(); h->d_nslot.release(); h->d_ncnt.release(); h->d_nfill.release(); h->d_nhits.release(); h->d_nstate.release(); h->d_biglist.release(); h->d_bins.release(); h->d_delta.release(); h->d_binlist.release(); h->d_sel.release(); h->d_recslot.release();
    h->d_evkeys.release(); h->d_evvals.release(); h->d_evout.release(); h->h_evout.release();
    for (int i = 0; i < MAX_TABLES; i++) h->d_satbits[i].release();
    h->d_htkeys.release(); h->d_htvals.release(); h->d_events.release(); h->d_counts.release(); h->d_hashes.release();
    h->d_hashin.release(); h->d_stat_med.release(); h->d_stat_f.release(); h->d_stat_n.release(); h->d_stat_b.release();
    h->d_hist.release(); h->big_keys.release(); h->big_vals.release();
    if (h->d_ctrl) cudaFree(h->d_ctrl);
    if (h->h_ctrl) cudaFreeHost(h->h_ctrl);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->tev0) cudaEventDestroy(h->tev0);
    if (h->tev1) cudaEventDestroy(h->tev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return KMGPU_OK;
}

extern "C" int kmgpu_set_use_bigcount(kmgpu_t* h, int on)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (h->kind != KMGPU_BYTE) return fail(KMGPU_EUNSUPPORTED, "bigcount is not supported for this storage.");  // storage.cc:52-54
    std::lock_guard<std::mutex> g(h->mu);
    h->use_bigcount = on != 0;
    h->satbits_valid = false;
    return KMGPU_OK;
}
extern "C" int kmgpu_get_use_bigcount(kmgpu_t* h, int* on)
{
    if (!h || !on) return fail(KMGPU_EINVAL, "null argument");
    *on = h->use_bigcount ? 1 : 0;
    return KMGPU_OK;
}

extern "C" int kmgpu_stats(kmgpu_t* h, uint64_t* n_occupied, uint64_t* n_unique)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (n_occupied) *n_occupied = h->n_occupied;
    if (n_unique) *n_unique = h->n_unique;
    return KMGPU_OK;
}
extern "C" int kmgpu_set_stats(kmgpu_t* h, uint64_t n_occupied, uint64_t n_unique)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    h->n_occupied = n_occupied;
    h->n_unique = n_unique;
    return KMGPU_OK;
}
extern "C" int kmgpu_shape(kmgpu_t* h, int* storage, int* hash, int* ksize, int* n_tables, uint64_t* sizes)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (storage) *storage = h->kind;
    if (hash) *hash = h->hash;
    if (ksize) *ksize = h->k;
    if (n_tables) *n_tables = h->nt;
    if (sizes) for (int i = 0; i < h->nt; i++) sizes[i] = h->sizes[i];
    return KMGPU_OK;
}
extern "C" int kmgpu_set_ksize(kmgpu_t* h, int ksize)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (ksize < 1 || ksize > MAX_K || (h->hash == KMGPU_TWOBIT && ksize > 32)) return fail(KMGPU_EINVAL, "ksize %d out of range", ksize);
    std::lock_guard<std::mutex> g(h->mu);
    h->k = ksize;
    return KMGPU_OK;
}

extern "C" int kmgpu_table_nbytes(kmgpu_t* h, int table, uint64_t* nbytes)
{
    if (!h || table < 0 || table >= h->nt) return fail(KMGPU_EINVAL, "bad table index");
    *nbytes = h->nbytes[table];
    return KMGPU_OK;
}
extern "C" int kmgpu_download_table(kmgpu_t* h, int table, uint8_t* dst, uint64_t offset, uint64_t nbytes)
{
    if (!h || table < 0 || table >= h->nt) return fail(KMGPU_EINVAL, "bad table index");
    if (offset > h->nbytes[table] || nbytes > h->nbytes[table] - offset) return fail(KMGPU_EINVAL, "range past end of table");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(dst, h->dev.tables[table] + offset, nbytes, cudaMemcpyDeviceToHost));
    return KMGPU_OK;
}
extern "C" int kmgpu_upload_table(kmgpu_t* h, int table, const uint8_t* src, uint64_t offset, uint64_t nbytes)
{
    if (!h || table < 0 || table >= h->nt) return fail(KMGPU_EINVAL, "bad table index");
    if (offset > h->nbytes[table] || nbytes > h->nbytes[table] - offset) return fail(KMGPU_EINVAL, "range past end of table");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->dev.tables[table] + offset, src, nbytes, cudaMemcpyHostToDevice));
    h->satbits_valid = false;
    return KMGPU_OK;
}

extern "C" int kmgpu_sync(kmgpu_t* h)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    CKR(set_device(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return KMGPU_OK;
}
extern "C" int kmgpu_reset(kmgpu_t* h)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    for (int i = 0; i < h->nt; i++) CK(cudaMemsetAsync(h->dev.tables[i], 0, h->alloc_bytes[i], h->stream));
    h->n_occupied = 0;
    h->n_unique = 0;
    h->big.clear();
    h->big_dirty = true;
    h->satbits_valid = false;
    if (h->ft_on) {   // a new epoch of the first-touch log
        CK(cudaStreamSynchronize(h->stream));
        for (auto& sg : h->ft_segs) cudaFree(sg.first);
        h->ft_segs.clear();
        h->ft_pending = 0;
        h->ft_epoch_unique = 0;
        h->ft_chunk = 0;
    }
    return KMGPU_OK;
}
extern "C" int kmgpu_timer_start(kmgpu_t* h)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    CK(cudaEventRecord(h->tev0, h->stream));
    return KMGPU_OK;
}
extern "C" int kmgpu_timer_stop(kmgpu_t* h, double* ms)
{
    if (!h || !ms) return fail(KMGPU_EINVAL, "null argument");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    CK(cudaEventRecord(h->tev1, h->stream));
    CK(cudaEventSynchronize(h->tev1));
    float f = 0;
    CK(cudaEventElapsedTime(&f, h->tev0, h->tev1));
    *ms = f;
    return KMGPU_OK;
}
extern "C" int kmgpu_profile_reset(kmgpu_t* h)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    h->ingest_ms = 0;
    h->ingest_launches = 0;
    h->all_launches = 0;
    return KMGPU_OK;
}
extern "C" int kmgpu_profile_get(kmgpu_t* h, double* ms, uint64_t* launches, uint64_t* all_launches)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (ms) *ms = h->ingest_ms;
    if (launches) *launches = h->ingest_launches;
    if (all_launches) *all_launches = h->all_launches;
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// bigcount map
// ------------------------------------------------------------------------------------------------------
extern "C" int kmgpu_bigcount_size(kmgpu_t* h, uint64_t* n)
{
    if (!h || !n) return fail(KMGPU_EINVAL, "null argument");
    std::lock_guard<std::mutex> g(h->mu);
    *n = h->big.size();
    return KMGPU_OK;
}
extern "C" int kmgpu_bigcount_export(kmgpu_t* h, uint64_t* hashes, uint16_t* counts, uint64_t cap)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    uint64_t i = 0;
    for (auto it = h->big.begin(); it != h->big.end() && i < cap; ++it, ++i) {  // writer order, storage.cc:623-632
        hashes[i] = it->first;
        counts[i] = it->second;
    }
    return KMGPU_OK;
}
extern "C" int kmgpu_bigcount_import(kmgpu_t* h, const uint64_t* hashes, const uint16_t* counts, uint64_t n)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (n) h->big.clear();  // reader clears only when the file holds entries (storage.cc:369-379)
    for (uint64_t i = 0; i < n; i++) h->big[hashes[i]] = counts[i];
    h->big_dirty = true;
    return KMGPU_OK;
}

static int sync_big_to_device(kmgpu_sketch* h)
{
    if (!h->big_dirty) return KMGPU_OK;
    std::vector<std::pair<uint64_t, uint16_t>> v(h->big.begin(), h->big.end());
    std::sort(v.begin(), v.end());
    std::vector<uint64_t> kk(v.size());
    std::vector<uint16_t> vv(v.size());
    for (size_t i = 0; i < v.size(); i++) { kk[i] = v[i].first; vv[i] = v[i].second; }
    CKR(h->big_keys.ensure(std::max<size_t>(1, v.size())));
    CKR(h->big_vals.ensure(std::max<size_t>(1, v.size())));
    if (!v.empty()) {
        CK(cudaMemcpyAsync(h->big_keys.p, kk.data(), 8 * v.size(), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->big_vals.p, vv.data(), 2 * v.size(), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    h->n_big_dev = (uint32_t)v.size();
    h->big_dirty = false;
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// chunk processing
// ------------------------------------------------------------------------------------------------------
static uint64_t pow2_at_least(uint64_t n)
{
    uint64_t p = 1024;
    while (p < n) p <<= 1;
    return p;
}

static int read_ctrl(kmgpu_sketch* h)
{
    CK(cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return KMGPU_OK;
}

struct ChunkResult {
    uint64_t n_kmers = 0, n_new = 0;
    bool have_newbits = false;
};

// ------------------------------------------------------------------------------------------------------
// delta + fold ingestion (see kmgpu_kernels.cuh): byte / nibble storages with every table <= 2^32 - 2 bins
// ------------------------------------------------------------------------------------------------------
struct DeltaPass {
    int table;
    uint32_t lo, hi;
};

// bins per delta block: 2 bytes per bin for the counting storages (half lanes), 1 bit per bin for BitStorage
static uint64_t delta_block_bins(int kind)
{
    uint64_t b = env_u64("KMGPU_DELTA_BLOCK_BINS", 0);  // test hook
    if (!b) {
        uint64_t bytes = env_u64("KMGPU_DELTA_BLOCK_MB", 50) * 1000000ull;
        b = kind == BIT ? bytes * 8 : bytes / 2;
    }
    const uint64_t gran = kind == BIT ? 128 : 8;
    b = (b / gran) * gran;
    return b < gran ? gran : b;
}

static bool plan_delta(const kmgpu_sketch* h, std::vector<DeltaPass>& out)
{
    out.clear();
    const uint64_t block = delta_block_bins(h->kind);
    const uint64_t gran = h->kind == BIT ? 128 : 8;
    for (int i = 0; i < h->nt; i++) {
        if (h->sizes[i] > 0xFFFFFFFEull - 128) return false;
        uint64_t r = (h->sizes[i] + block - 1) / block;
        uint64_t per = (((h->sizes[i] + r - 1) / r + gran - 1) / gran) * gran;
        for (uint64_t j = 0; j * per < h->sizes[i]; j++)
            out.push_back(DeltaPass{i, (uint32_t)(j * per), (uint32_t)std::min<uint64_t>(h->sizes[i], (j + 1) * per)});
    }
    if (out.size() > env_u64("KMGPU_DELTA_MAX_PASSES", 64)) {
        out.clear();
        return false;
    }
    return true;
}

template <int HK, int SRC>
static void launch_hashbins(bool pred, unsigned g, cudaStream_t st, const SketchDev& S, const SketchDev& M, HashCfg H, const Pred& P,
                            const Input& in, uint32_t* bins, uint64_t stride, Ctrl* ctrl)
{
    if (pred) k_hashbins<HK, SRC, true, 0><<<g, THREADS, 0, st>>>(S, M, H, P, in, bins, stride, ctrl);
    else if (S.n_tables == 4) k_hashbins<HK, SRC, false, 4><<<g, THREADS, 0, st>>>(S, M, H, P, in, bins, stride, ctrl);   // khmer's default N
    else k_hashbins<HK, SRC, false, 0><<<g, THREADS, 0, st>>>(S, M, H, P, in, bins, stride, ctrl);
}

// ByteStorage::add tail (storage.hh:606-617) applied `count` times to one k-mer
static inline void big_events(kmgpu_sketch* h, uint64_t hash, uint32_t count)
{
    uint16_t& v = h->big[hash];
    uint32_t base = v == 0 ? 255u : v;
    uint32_t nv = base + count;
    v = (uint16_t)(nv > 65535u ? 65535u : nv);
    h->big_dirty = true;
}

// A chunk may arrive in parts (host input: one staged range each, uploaded while the previous part is hashed): part j holds
// positions [pos_off, pos_off + in.n_pos) of the chunk; the main stream waits for `ready` before it touches the part.
struct Part {
    Input in;
    uint32_t pos_off;
    cudaEvent_t ready;
};

// `rehash`: the chunk has no bins[] array (grouped path): candidates are found by hashing the stream again (k_bigscan2)
static int resolve_bigcount_delta(kmgpu_sketch* h, int src, HashCfg H, const std::vector<Part>& parts, uint32_t n_pos, uint64_t stride, uint64_t n_list,
                                  uint64_t n_cross, bool rehash = false, const Pred* P = nullptr, bool pred = false, const SketchDev* MS = nullptr)
{
    cudaStream_t st = h->stream;
    // the small workspaces start at a size that rarely has to grow: a regrowth is a cudaFree + cudaMalloc, i.e. a device
    // synchronisation plus milliseconds of driver time in the middle of the stream
    constexpr uint64_t WS_MIN = 1ull << 20;
    static const bool dbg = env_u64("KMGPU_DEBUG", 0) != 0;
    const auto t_begin = std::chrono::steady_clock::now();
    auto lap = [&](const char* what, uint64_t n) {
        if (!dbg) return;
        cudaStreamSynchronize(st);
        fprintf(stderr, "[kmgpu] bigcount %s: n=%llu t=%.3f ms\n", what, (unsigned long long)n,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count());
    };
    lap("begin (n_cross)", n_cross);
    uint64_t slots = 1024;
    if (n_cross) {
        slots = pow2_at_least(2 * n_cross);
        CKR(h->d_htkeys.ensure(std::max<uint64_t>(slots, WS_MIN)));
        CKR(h->d_htvals.ensure(std::max<uint64_t>(slots, WS_MIN)));
        CK(cudaMemsetAsync(h->d_htkeys.p, 0xFF, slots * 8, st));
        unsigned gl = (unsigned)std::min<uint64_t>((n_list + 255) / 256, 148 * 8);
        k_list_register<<<gl, 256, 0, st>>>(h->d_binlist.p, n_list, BL_CROSS, h->d_htkeys.p, h->d_htvals.p, slots - 1, nullptr, 1);
        h->all_launches += 1;
    }
    // 1. candidates and touches of crossing bins
    uint64_t cap = n_pos;
    CKR(h->d_events.ensure(cap));
    CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
    if (rehash) {
        SatBitsG sg;
        memset(&sg, 0, sizeof sg);
        for (int i = 0; i < h->nt; i++) sg.t[i] = h->d_satbits[i].p;
        Pred P0;
        memset(&P0, 0, sizeof P0);
        const Pred& PP = P ? *P : P0;
        const SketchDev& MM = MS ? *MS : h->dev;
        for (const Part& pt : parts) {
            const Input& in = pt.in;
            if (in.n_pos == 0) continue;
            const unsigned gt = n_tiles(in.n_pos);
            if (src == 1) k_bigscan2<TWOBIT, 1><<<gt, THREADS, 0, st>>>(h->dev, H, in, sg, h->d_htkeys.p, slots - 1, n_cross ? 1 : 0, h->d_events.p,
                                                                       (unsigned long long)cap, h->d_ctrl, pt.pos_off, MM, PP, pred ? 1 : 0);
            else if (H.kind == TWOBIT) k_bigscan2<TWOBIT, 0><<<gt, THREADS, 0, st>>>(h->dev, H, in, sg, h->d_htkeys.p, slots - 1, n_cross ? 1 : 0, h->d_events.p,
                                                                                   (unsigned long long)cap, h->d_ctrl, pt.pos_off, MM, PP, pred ? 1 : 0);
            else k_bigscan2<MURMUR, 0><<<gt, THREADS, 0, st>>>(h->dev, H, in, sg, h->d_htkeys.p, slots - 1, n_cross ? 1 : 0, h->d_events.p,
                                                             (unsigned long long)cap, h->d_ctrl, pt.pos_off, MM, PP, pred ? 1 : 0);
            h->all_launches += 1;
        }
    }
    SatBits sb;
    memset(&sb, 0, sizeof sb);
    for (int i = 0; i < h->nt && i < F_MAXT; i++) sb.t[i] = h->d_satbits[i].p;
    for (size_t pi = 0; pi < parts.size(); pi++) {
        const Part& pt = parts[pi];
        Input in = pt.in;
        if (in.n_pos == 0 || rehash) continue;
        // a part's last k-1 positions are the next part's first ones (their bins[] entries are the next part's by now): scan its own only
        if (pi + 1 < parts.size()) in.n_pos = std::min<uint32_t>(in.n_pos, parts[pi + 1].pos_off - pt.pos_off);
        const uint32_t* bins = h->d_bins.p + pt.pos_off;
        unsigned gb = (in.n_pos + 255) / 256;
        if (src == 1) k_bigscan<TWOBIT, 1><<<gb, 256, 0, st>>>(h->nt, H, in, bins, stride, sb, h->d_htkeys.p, slots - 1, n_cross ? 1 : 0,
                                                                h->d_events.p, (unsigned long long)cap, h->d_ctrl, pt.pos_off);
        else if (H.kind == TWOBIT) k_bigscan<TWOBIT, 0><<<gb, 256, 0, st>>>(h->nt, H, in, bins, stride, sb, h->d_htkeys.p, slots - 1,
                                                                            n_cross ? 1 : 0, h->d_events.p, (unsigned long long)cap, h->d_ctrl, pt.pos_off);
        else k_bigscan<MURMUR, 0><<<gb, 256, 0, st>>>(h->nt, H, in, bins, stride, sb, h->d_htkeys.p, slots - 1, n_cross ? 1 : 0,
                                                      h->d_events.p, (unsigned long long)cap, h->d_ctrl, pt.pos_off);
        h->all_launches += 1;
    }
    CK(cudaGetLastError());
    CKR(read_ctrl(h));
    const uint64_t n_rec = h->h_ctrl->n_events;
    lap("scan done (n_rec)", n_rec);
    if (n_rec > cap) return fail(KMGPU_ECUDA, "internal: bigcount scan overflow");
    if (n_rec == 0) return KMGPU_OK;
    const unsigned gr = (unsigned)((n_rec + 255) / 256);
    // 2. stream position of the saturating touch of every crossing bin (radix select over the reported touches)
    uint32_t* Tarr = nullptr;
    if (n_cross) {
        CKR(h->d_sel.ensure(std::max<uint64_t>(3 * slots, WS_MIN)));
        CKR(h->d_recslot.ensure(std::max<uint64_t>(n_rec * h->nt, 4 * WS_MIN)));
        SelState ss{h->d_sel.p, h->d_sel.p + slots, h->d_sel.p + 2 * slots};
        const unsigned gsl = (unsigned)((slots + 255) / 256);
        k_sel_slots<<<gr, 256, 0, st>>>(h->d_events.p, n_rec, h->dev, h->d_htkeys.p, slots - 1, h->d_recslot.p);
        k_sel_init<<<gsl, 256, 0, st>>>(h->d_htkeys.p, h->d_htvals.p, slots, ss);
        int top = 0;
        while (top < 31 && (1ull << (top + 1)) <= (uint64_t)n_pos) top++;
        for (int bit = top; bit >= 0; bit--) {
            k_sel_count<<<gr, 256, 0, st>>>(h->d_events.p, n_rec, h->nt, h->d_recslot.p, bit, ss);
            k_sel_update<<<gsl, 256, 0, st>>>(slots, bit, ss);
        }
        h->all_launches += 2 + 2 * (top + 1);
        Tarr = ss.prefix;
    }
    // 3. decide and aggregate per k-mer
    uint64_t evslots = pow2_at_least(2 * n_rec);
    CKR(h->d_evkeys.ensure(std::max<uint64_t>(evslots, WS_MIN)));
    CKR(h->d_evvals.ensure(std::max<uint64_t>(2 * evslots, 2 * WS_MIN)));
    CK(cudaMemsetAsync(h->d_evkeys.p, 0xFF, evslots * 8, st));
    CK(cudaMemsetAsync(h->d_evvals.p, 0, evslots * 4, st));
    CK(cudaMemsetAsync(h->d_evvals.p + evslots, 0xFF, evslots * 4, st));
    CK(cudaMemsetAsync(&h->d_ctrl->n_unique, 0, sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
    EvTable ev{h->d_evkeys.p, h->d_evvals.p, h->d_evvals.p + evslots, evslots - 1};
    k_ev_decide<<<gr, 256, 0, st>>>(h->d_events.p, n_rec, h->nt, h->d_recslot.p, Tarr, n_cross ? 1 : 0, ev, h->d_ctrl);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CKR(read_ctrl(h));
    const uint64_t n_distinct = h->h_ctrl->n_unique;
    lap("decided (n_distinct)", n_distinct);
    if (n_distinct == 0) return KMGPU_OK;
    CKR(h->d_evout.ensure(std::max<uint64_t>(n_distinct, WS_MIN / 4)));
    CKR(h->h_evout.ensure(std::max<uint64_t>(n_distinct, WS_MIN / 4)));
    k_ev_compact<<<(unsigned)((evslots + 255) / 256), 256, 0, st>>>(ev, h->d_evout.p, h->d_ctrl);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_evout.p, h->d_evout.p, n_distinct * sizeof(EvOut), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    // 4. one map update per distinct k-mer, new keys inserted in the order of their first event (stream order)
    std::vector<EvOut> evs(h->h_evout.p, h->h_evout.p + n_distinct);
    std::sort(evs.begin(), evs.end(), [](const EvOut& a, const EvOut& b) { return a.first < b.first; });
    for (const EvOut& e : evs) big_events(h, e.hash, e.count);
    return KMGPU_OK;
}

// Bucket path eligibility for a chunk of n_pos positions: every table within BKT_MAX_BUCKETS buckets, and the expected
// bucket load (+25% + 2048 of slack) within what a 16-bit touch lane can count.  Skewed input that overflows a bucket
// anyway is caught on the device and the chunk falls back to the delta passes.
static bool plan_buckets(const kmgpu_sketch* h, uint32_t n_pos, BucketLayout* L)
{
    if (!env_u64("KMGPU_BUCKETS", 1)) return false;
    memset(L, 0, sizeof *L);
    L->n_tables = h->nt;
    uint64_t cap = 0, total = 0;
    for (int i = 0; i < h->nt; i++) {
        if (h->sizes[i] > 0xFFFFFFFEull - 128) return false;
        uint64_t nb = (h->sizes[i] + BKT_BINS - 1) / BKT_BINS;
        if (nb > (uint64_t)BKT_MAX_BUCKETS) return false;
        L->first[i] = (uint32_t)total;
        total += nb;
        uint64_t expect = nb == 1 ? n_pos : (uint64_t)((double)n_pos * BKT_BINS / (double)h->sizes[i]) + 1;
        cap = std::max(cap, expect + expect / 4 + 2048);
    }
    L->first[h->nt] = (uint32_t)total;
    cap = std::min<uint64_t>(cap, (uint64_t)n_pos);
    if (uint64_t forced = env_u64("KMGPU_BUCKET_CAP", 0)) cap = forced;   // tests: provoke the overflow fallback
    if (cap > 65535 || cap == 0) return false;
    L->cap = (uint32_t)cap;
    return true;
}

template <int KIND>
static void launch_apply(unsigned g, cudaStream_t st, const SketchDev& S, const BucketLayout& L, const unsigned long long* rec, const uint32_t* cur,
                         uint32_t* newbits, uint64_t* binlist, unsigned long long list_cap, Ctrl* ctrl, int want_cross, const SatBits& sb)
{
    k_apply<KIND><<<g, 1024, BKT_APPLY_SMEM, st>>>(S, L, rec, cur, newbits, binlist, list_cap, ctrl, want_cross, sb);
}

// `between` (optional) runs on the host after the chunk's kernels have been queued and before the host waits for
// them: the caller uses it to prepare and upload the next chunk while this one is being ingested.
typedef std::function<int()> Between;

#include "kmgpu_group_host.inc"

static int ingest_chunk_delta(kmgpu_sketch* h, const std::vector<DeltaPass>& passes, int src, HashCfg H, const std::vector<Part>& parts, const Pred& P,
                              bool pred, const SketchDev* M, ChunkResult* res, const Between& between)
{
    cudaStream_t st = h->stream;
    uint32_t n_pos = 0;
    for (const Part& pt : parts) n_pos = std::max(n_pos, pt.pos_off + pt.in.n_pos);
    const uint64_t stride = ((uint64_t)n_pos + 7) & ~7ull;
    CKR(h->d_bins.ensure((size_t)h->nt * stride));
    uint64_t total_bins = 0, max_span = 0;
    for (int i = 0; i < h->nt; i++) total_bins += h->sizes[i];
    for (const DeltaPass& p : passes) max_span = std::max<uint64_t>(max_span, p.hi - p.lo);
    const uint64_t list_cap = std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)h->nt * n_pos, total_bins));
    CKR(h->d_binlist.ensure(list_cap));
    // block storage in 2-byte units: one half lane per bin, or one bit per bin for BitStorage
    size_t need_lanes = h->kind == BIT ? ((max_span + 127) / 128) * 8 + 8 : ((max_span + 7) & ~7ull) + 8;
    if (h->d_delta.cap < need_lanes) h->delta_zeroed = 0;
    CKR(h->d_delta.ensure(need_lanes));
    if (h->delta_zeroed < h->d_delta.cap) {  // the fold keeps the block zeroed from then on
        CK(cudaMemsetAsync(h->d_delta.p, 0, h->d_delta.cap * 2, st));
        h->delta_zeroed = h->d_delta.cap;
    }
    CK(cudaMemsetAsync(h->d_ctrl, 0, sizeof(Ctrl), st));
    CK(cudaEventRecord(h->ev0, st));
    const int want_cross = h->kind == BYTE && h->use_bigcount;
    if (want_cross && !h->satbits_valid) {
        for (int i = 0; i < h->nt; i++) {
            uint64_t groups = (h->sizes[i] + 7) / 8;
            CKR(h->d_satbits[i].ensure(groups));
            k_build_satbits<<<(unsigned)std::min<uint64_t>((groups + 255) / 256, 148 * 16), 256, 0, st>>>(h->dev.tables[i], groups, h->d_satbits[i].p);
            h->all_launches += 1;
        }
        h->satbits_valid = true;
    }
    bool kmers_counted = false;
    BucketLayout BL;
    bool use_buckets = plan_buckets(h, n_pos, &BL);
    if (use_buckets) {
        // bucket path: group the updates by 32 Ki-bin bucket, apply each bucket in shared memory (counters, n_occupied,
        // first touchers -> newbits / n_unique, saturation bookkeeping in one sweep)
        if (!h->bucket_attr_set) {
            CK(cudaFuncSetAttribute(k_bucketize<BKT_TILE, BKT_PER>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bkt_sort_smem(BKT_TILE)));
            CK(cudaFuncSetAttribute(k_apply<BYTE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BKT_APPLY_SMEM));
            CK(cudaFuncSetAttribute(k_apply<NIBBLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BKT_APPLY_SMEM));
            CK(cudaFuncSetAttribute(k_apply<BIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BKT_APPLY_SMEM));
            h->bucket_attr_set = true;
        }
        const uint32_t n_buckets = BL.first[h->nt];
        if (h->d_records.ensure((size_t)n_buckets * BL.cap) != KMGPU_OK) {   // no room for the record store: delta passes
            cudaGetLastError();
            use_buckets = false;
        }
    }
    if (use_buckets) {
        const uint32_t n_buckets = BL.first[h->nt];
        CKR(h->d_cursors.ensure(n_buckets));
        const size_t nb_words = (n_pos + 31) / 32;
        CKR(h->d_newbits.ensure(nb_words));
        CK(cudaMemsetAsync(h->d_cursors.p, 0, (size_t)n_buckets * 4, st));
        CK(cudaMemsetAsync(h->d_newbits.p, 0, nb_words * 4, st));
    }
    // hash every part as soon as it has arrived; on the bucket path its records follow at once
    for (const Part& pt : parts) {
        const Input& in = pt.in;
        if (pt.ready) CK(cudaStreamWaitEvent(st, pt.ready, 0));
        if (in.n_pos == 0) continue;
        uint32_t* bins = h->d_bins.p + pt.pos_off;
        const unsigned g = n_tiles(in.n_pos);
        const SketchDev& MS = M ? *M : h->dev;
        if (src == 1) launch_hashbins<TWOBIT, 1>(pred, g, st, h->dev, MS, H, P, in, bins, stride, h->d_ctrl);
        else if (H.kind == TWOBIT) launch_hashbins<TWOBIT, 0>(pred, g, st, h->dev, MS, H, P, in, bins, stride, h->d_ctrl);
        else launch_hashbins<MURMUR, 0>(pred, g, st, h->dev, MS, H, P, in, bins, stride, h->d_ctrl);
        if (use_buckets)
            k_bucketize<BKT_TILE, BKT_PER><<<dim3((in.n_pos + BKT_TILE - 1) / BKT_TILE, h->nt), BKT_TILE / BKT_PER, bkt_sort_smem(BKT_TILE), st>>>(
                bins, stride, in.n_pos, pt.pos_off, BL, h->d_records.p, h->d_cursors.p, h->d_ctrl);
        h->ingest_launches += use_buckets ? 2 : 1;
        h->all_launches += use_buckets ? 2 : 1;
    }
    if (use_buckets) {
        const uint32_t n_buckets = BL.first[h->nt];
        const size_t nb_words = (n_pos + 31) / 32;
        SatBits sb;
        memset(&sb, 0, sizeof sb);
        if (want_cross)
            for (int i = 0; i < h->nt; i++) sb.t[i] = h->d_satbits[i].p;
        if (h->kind == BYTE) launch_apply<BYTE>(n_buckets, st, h->dev, BL, h->d_records.p, h->d_cursors.p, h->d_newbits.p, h->d_binlist.p, list_cap, h->d_ctrl, want_cross, sb);
        else if (h->kind == NIBBLE) launch_apply<NIBBLE>(n_buckets, st, h->dev, BL, h->d_records.p, h->d_cursors.p, h->d_newbits.p, h->d_binlist.p, list_cap, h->d_ctrl, 0, sb);
        else launch_apply<BIT>(n_buckets, st, h->dev, BL, h->d_records.p, h->d_cursors.p, h->d_newbits.p, h->d_binlist.p, list_cap, h->d_ctrl, 0, sb);
        k_popc<<<(unsigned)std::min<size_t>((nb_words + 255) / 256, 148 * 8), 256, 0, st>>>(h->d_newbits.p, nb_words, &h->d_ctrl->n_unique);
        CK(cudaEventRecord(h->ev1, st));
        CK(cudaGetLastError());
        if (between) CKR(between());
        CKR(read_ctrl(h));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        h->ingest_ms += ms;
        h->ingest_launches += 2;
        h->all_launches += 2;
        Ctrl c = *h->h_ctrl;
        res->n_kmers += c.n_kmers;
        kmers_counted = true;
        if (!c.overflow) {
            if (c.n_events > list_cap) return fail(KMGPU_ECUDA, "internal: bin list overflow");
            h->n_occupied += c.n_z0;
            if (c.n_zbits) {
                h->n_unique += c.n_unique;
                res->n_new += c.n_unique;
                res->have_newbits = true;
            }
            if (want_cross && c.n_sat) CKR(resolve_bigcount_delta(h, src, H, parts, n_pos, stride, c.n_events, c.n_cross));
            return KMGPU_OK;
        }
        // a bucket overflowed (heavily repeated k-mers): nothing was applied; redo the chunk with the delta passes
        if (env_u64("KMGPU_DEBUG", 0)) fprintf(stderr, "[kmgpu] bucket overflow (cap %u, %u positions): chunk redone by the delta passes\n", BL.cap, n_pos);
        CK(cudaMemsetAsync(h->d_ctrl, 0, sizeof(Ctrl), st));
        CK(cudaEventRecord(h->ev0, st));
    }
    const Between none;
    const Between& between2 = kmers_counted ? none : between;   // the hook has already run
    const unsigned gs = (n_pos + 2047) / 2048;
    for (const DeltaPass& p : passes) {
        const int pass_id = passes.size() <= 64 ? (int)(&p - passes.data()) : -1;   // per-pass entry counts for the cold resolution
        if (h->kind == BIT) {
            k_scatter<true><<<gs, 256, 0, st>>>(h->d_bins.p + (size_t)p.table * stride, n_pos, p.lo, p.hi, h->d_delta.p);
            unsigned gb = (unsigned)(((uint64_t)(p.hi - p.lo) + 128 * 256 - 1) / (128 * 256));
            k_fold_bits<<<gb, 256, 0, st>>>(h->dev.tables[p.table], p.table, p.lo, p.hi, h->d_delta.p, h->d_binlist.p, list_cap, h->d_ctrl, pass_id);
            continue;
        }
        k_scatter<false><<<gs, 256, 0, st>>>(h->d_bins.p + (size_t)p.table * stride, n_pos, p.lo, p.hi, h->d_delta.p);
        unsigned gf = (unsigned)(((uint64_t)(p.hi - p.lo) + 2047) / 2048);
        if (h->kind == BYTE)
            k_fold<BYTE><<<gf, 256, 0, st>>>(h->dev.tables[p.table], p.table, p.lo, p.hi, h->d_delta.p, h->d_binlist.p, list_cap, h->d_ctrl, want_cross,
                                             want_cross ? h->d_satbits[p.table].p : nullptr, pass_id);
        else
            k_fold<NIBBLE><<<gf, 256, 0, st>>>(h->dev.tables[p.table], p.table, p.lo, p.hi, h->d_delta.p, h->d_binlist.p, list_cap, h->d_ctrl, 0, nullptr, pass_id);
    }
    CK(cudaEventRecord(h->ev1, st));
    CK(cudaGetLastError());
    if (between2) CKR(between2());
    CKR(read_ctrl(h));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->ingest_ms += ms;
    h->ingest_launches += 2 * passes.size();
    h->all_launches += 2 * passes.size();
    Ctrl c = *h->h_ctrl;
    if (c.n_events > list_cap) return fail(KMGPU_ECUDA, "internal: bin list overflow");
    if (!kmers_counted) res->n_kmers += c.n_kmers;
    h->n_occupied += c.n_z0;
    const uint64_t n_list = c.n_events;
    if (c.n_zbits) {
        // first-toucher stamps: per-table sub-tables of packed 8-byte slots in one buffer, bitmap prefilter
        size_t nb_words = (n_pos + 31) / 32;
        CKR(h->d_newbits.ensure(nb_words));
        CK(cudaMemsetAsync(h->d_newbits.p, 0, nb_words * 4, st));
        CK(cudaMemsetAsync(&h->d_ctrl->n_unique, 0, sizeof(unsigned long long), st));
        const uint64_t cold_min = env_u64("KMGPU_COLD_MIN_NEW", 8ull << 20);
        if (passes.size() <= 64 && c.n_zbits >= cold_min) {
            // cold chunk (most bins new): resolve one (table, block) at a time, so that the block's stamp table
            // (a few tens of MB) stays in L2 while every position of the chunk probes it
            unsigned long long* sl = reinterpret_cast<unsigned long long*>(h->d_htkeys.p);
            uint64_t seg0 = 0;
            for (size_t pi = 0; pi < passes.size(); pi++) {
                uint64_t seg1 = seg0 + c.pass_list_end[pi];   // entries the fold of pass pi appended (passes run in order)
                if (seg1 > seg0) {
                    const DeltaPass& p = passes[pi];
                    const uint32_t span = p.hi - p.lo;
                    if (span <= (1u << 26) && env_u64("KMGPU_COLD_RANK", 1)) {
                        // direct-addressed form: ranked bitmap of the block's new bins + one min-position per new bin
                        const uint32_t n_words = (span + 31) / 32;
                        const unsigned gw = (n_words + 1023) / 1024;
                        const uint64_t n_ent = seg1 - seg0;
                        CKR(h->d_rank.ensure((size_t)n_words * 2 + gw));
                        CKR(h->d_htkeys.ensure((n_ent + 1) / 2));
                        uint2* rec = reinterpret_cast<uint2*>(h->d_rank.p);
                        uint32_t* sums = h->d_rank.p + (size_t)n_words * 2;
                        uint32_t* minpos = reinterpret_cast<uint32_t*>(h->d_htkeys.p);
                        CK(cudaMemsetAsync(rec, 0, (size_t)n_words * 8, st));
                        CK(cudaMemsetAsync(minpos, 0xFF, n_ent * 4, st));
                        unsigned gl = (unsigned)std::min<uint64_t>((n_ent + 255) / 256, 148 * 8);
                        k_rank_setbits<<<gl, 256, 0, st>>>(h->d_binlist.p + seg0, n_ent, p.lo, rec);
                        k_rank_sums<<<gw, 256, 0, st>>>(rec, n_words, sums);
                        k_rank_scan<<<1, 1024, 0, st>>>(sums, gw);
                        k_rank_prefix<<<gw, 256, 0, st>>>(rec, n_words, sums);
                        k_rank_replay<<<(n_pos + 2047) / 2048, 256, 0, st>>>(h->d_bins.p + (size_t)p.table * stride, n_pos, p.lo, p.hi, rec, minpos);
                        k_rank_mark<<<gl, 256, 0, st>>>(minpos, n_ent, h->d_newbits.p, h->d_ctrl);
                        h->all_launches += 6;
                        seg0 = seg1;
                        continue;
                    }
                    uint64_t slots = pow2_at_least(2 * (seg1 - seg0));
                    CKR(h->d_htkeys.ensure(slots));
                    sl = reinterpret_cast<unsigned long long*>(h->d_htkeys.p);
                    CK(cudaMemsetAsync(sl, 0xFF, slots * 8, st));
                    unsigned gl = (unsigned)std::min<uint64_t>((seg1 - seg0 + 255) / 256, 148 * 8);
                    k_pk_register<<<gl, 256, 0, st>>>(h->d_binlist.p + seg0, seg1 - seg0, p.table, sl, slots - 1, nullptr);
                    k_pk_replay<<<(n_pos + 1023) / 1024, 256, 0, st>>>(h->d_bins.p + (size_t)p.table * stride, n_pos, p.lo, p.hi, sl,
                                                                    slots - 1, nullptr);
                    unsigned gm = (unsigned)std::min<uint64_t>((slots + 255) / 256, 148 * 8);
                    k_pk_mark<<<gm, 256, 0, st>>>(sl, slots, h->d_newbits.p, h->d_ctrl);
                    h->all_launches += 3;
                }
                seg0 = seg1;
            }
        } else {
        PkLayout L;
        memset(&L, 0, sizeof L);
        uint64_t total_slots = 0;
        for (int i = 0; i < h->nt; i++) {
            if (!c.n_new_t[i]) continue;
            uint64_t sl = pow2_at_least(2 * c.n_new_t[i]);
            L.base[i] = total_slots;
            L.mask[i] = sl - 1;
            total_slots += sl;
        }
        L.use_filter = c.n_zbits < (uint64_t)h->nt * FILTER_BITS / 4;
        {   // bitmap of ~32 bits per new bin, between 32 Kbit (4 KB, L1-resident) and FILTER_BITS per table
            uint64_t mx = 0;
            for (int i = 0; i < h->nt; i++) mx = std::max<uint64_t>(mx, c.n_new_t[i]);
            uint64_t fb = 1u << 15;
            while (fb < 32 * mx && fb < FILTER_BITS) fb <<= 1;
            L.filter_bits = (uint32_t)fb;
        }
        CKR(h->d_htkeys.ensure(total_slots));
        CK(cudaMemsetAsync(h->d_htkeys.p, 0xFF, total_slots * 8, st));
        if (L.use_filter) {
            CKR(h->d_filter.ensure((size_t)h->nt * FILTER_WORDS));
            CK(cudaMemsetAsync(h->d_filter.p, 0, (size_t)h->nt * (L.filter_bits >> 5) * 4, st));
        }
        unsigned long long* sl = reinterpret_cast<unsigned long long*>(h->d_htkeys.p);
        unsigned gl = (unsigned)std::min<uint64_t>((n_list + 255) / 256, 148 * 8);
        k_pk_register_all<<<gl, 256, 0, st>>>(h->d_binlist.p, n_list, L, sl, h->d_filter.p);
        k_pk_replay_all<<<(n_pos + 255) / 256, 256, 0, st>>>(h->d_bins.p, stride, h->nt, n_pos, L, sl, h->d_filter.p);
        unsigned gm = (unsigned)std::min<uint64_t>((total_slots + 255) / 256, 148 * 8);
        k_pk_mark<<<gm, 256, 0, st>>>(sl, total_slots, h->d_newbits.p, h->d_ctrl);
        h->all_launches += 3;
        }
        CK(cudaGetLastError());
        CKR(read_ctrl(h));
        h->n_unique += h->h_ctrl->n_unique;
        res->n_new += h->h_ctrl->n_unique;
        res->have_newbits = true;
    }
    if (want_cross && c.n_sat) CKR(resolve_bigcount_delta(h, src, H, parts, n_pos, stride, n_list, c.n_cross));
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// path of a chunk
// ------------------------------------------------------------------------------------------------------
// Bins: k_hashbins + k_bucketize + k_apply (ingest_chunk_delta; a bucket that overflows sends the chunk through the delta passes)
// Delta: k_hashbins + k_scatter + k_fold per table block (ingest_chunk_delta)
// Grouped: k_part + k_apply2 / k_apply_sparse (ingest_chunk_grouped)
enum class Path { Choose, Unsupported, Bins, Delta, Grouped };

constexpr size_t PREFER_DELTA_MAX_BLOCKS = 12;

// The path of a chunk of n_pos positions; G (optional) receives the grouped layout.  `first_touch`: the sketch keeps a first-touch
// log, which only the grouped path writes.
static Path choose_path(const kmgpu_sketch* h, uint32_t n_pos, bool first_touch, GroupPlan* G = nullptr)
{
    GroupPlan own;
    if (!G) G = &own;
    if (h->nt > F_MAXT || first_touch) return plan_group(h, n_pos, G) ? Path::Grouped : Path::Unsupported;
    std::vector<DeltaPass> dp;
    const bool delta = plan_delta(h, dp);
    BucketLayout BL;
    const bool bins = delta && plan_buckets(h, n_pos, &BL);
    const uint64_t min_buckets = env_u64("KMGPU_GROUP_MIN_BUCKETS", 1024);
    // tests steer small shapes onto the grouped path
    const bool hooked = !env_u64("KMGPU_PREFER_BINS", 1) || env_u64("KMGPU_FORCE_TWO_LEVEL", 0) || min_buckets == 0;
    // Shapes the bins path can take (every table within 6144 buckets, <= 65535 records per bucket and chunk) stay with it: hashing
    // once per position into the bins[] array and grouping with k_bucketize measures faster there than the fused kernel
    // (profiles/r2_grouping_variants.txt), at the price of 37 B per k-mer more DRAM traffic
    if (!hooked && bins) return Path::Bins;
    // ... and shapes the delta + fold passes cover in a dozen L2-sized blocks (config C2's Bloom filter: 18.3 against 10.1
    // G k-mers/s) measure faster there than through two grouping levels; with more blocks (SmallCountgraph at 4 x 4e8: 16
    // blocks, 9.1 against 10.7) the grouped path wins
    if (!hooked && delta && dp.size() <= PREFER_DELTA_MAX_BLOCKS) return Path::Delta;
    const bool grouped = plan_group(h, n_pos, G);
    if (grouped && G->n_buckets >= min_buckets) return Path::Grouped;
    if (delta) return bins ? Path::Bins : Path::Delta;   // a handful of buckets cannot fill the machine
    return grouped ? Path::Grouped : Path::Unsupported;
}

// Ingest one chunk into sketch `h` (hash config may come from another sketch: abundance tracking).  `path`: the caller's
// choice; by default it is chosen here for the chunk's extent.
static int ingest_chunk(kmgpu_sketch* h, int src, HashCfg H, const std::vector<Part>& parts, const Pred& P, bool pred, const SketchDev* M,
                        ChunkResult* res, const Between& between = Between(), Path path = Path::Choose)
{
    uint32_t n_pos = 0;
    for (const Part& pt : parts) n_pos = std::max(n_pos, pt.pos_off + pt.in.n_pos);
    if (n_pos == 0) return between ? between() : KMGPU_OK;
    GroupPlan G;   // the regions are sized for this chunk's positions
    if (path == Path::Choose) path = choose_path(h, n_pos, h->ft_on, &G);
    else if (path == Path::Grouped && !plan_group(h, n_pos, &G)) return fail(KMGPU_ECUDA, "internal: grouped plan changed between chunks");
    static const bool dbg = env_u64("KMGPU_DEBUG", 0) != 0;
    if (path == Path::Grouped) {
        if (dbg)
            fprintf(stderr, "[kmgpu] chunk: path=grouped delta_blocks=0 levels=%d sb_shift=%d apply=%s n_pos=%u\n", G.L.two_level ? 2 : 1,
                    G.L.two_level ? (int)G.L.sb_shift : 0, G.sparse ? "sparse" : G.split == 4 ? "split4" : G.split == 2 ? "split2" : "dense", n_pos);
        return ingest_chunk_grouped(h, G, src, H, parts, P, pred, M, res, between);
    }
    std::vector<DeltaPass> dp;
    if (path == Path::Unsupported || !plan_delta(h, dp))
        return fail(KMGPU_EUNSUPPORTED, "no ingestion path can take this sketch (%d tables; more than %d need the grouped path)", h->nt, F_MAXT);
    if (dbg) {
        BucketLayout BL;   // ingest_chunk_delta takes the bins path whenever the buckets can be planned
        const bool bins = plan_buckets(h, n_pos, &BL);
        fprintf(stderr, "[kmgpu] chunk: path=%s delta_blocks=%zu levels=0 sb_shift=0 apply=- n_pos=%u\n", bins ? "bins" : "delta", bins ? (size_t)0 : dp.size(),
                n_pos);
    }
    return ingest_chunk_delta(h, dp, src, H, parts, P, pred, M, res, between);
}

// Positions per chunk for this sketch.  A chunk costs one pass over every bucket of the sketch; where the two-level grouped path is
// taken (tables of billions of bins) that pass is what dominates, so chunks grow to what half of the free device memory holds in
// record stores (two levels of 8-byte records with their slack, plus hashes and bitmaps).  The first-touch log, which takes every
// chunk onto the grouped path, does not change the chunk size.
static uint64_t sketch_chunk_bases(kmgpu_sketch* h)
{
    if (getenv("KMGPU_CHUNK_BASES")) return chunk_bases();
    if (h->chunk_cap) return h->chunk_cap;
    uint64_t cap = chunk_bases();
    GroupPlan G;
    if (choose_path(h, (uint32_t)cap, false, &G) == Path::Grouped && G.L.two_level) {
        size_t fr = 0, tot = 0;
        if (cudaMemGetInfo(&fr, &tot) == cudaSuccess) {
            const uint64_t per_pos = (uint64_t)h->nt * 21 + 16;
            uint64_t p = std::min<uint64_t>((fr / 2) / per_pos, 1ull << 30);
            cap = std::max<uint64_t>(cap, (p / TILE) * TILE);
        }
        cudaGetLastError();
    }
    h->chunk_cap = cap;
    return cap;
}

// ------------------------------------------------------------------------------------------------------
// equal-sized chunks (multiples of 32 bases) of at most `cap` bases covering [0, total): starts[i] .. starts[i+1]
static void balanced_chunks(uint64_t total, uint64_t cap, std::vector<uint64_t>& starts)
{
    starts.assign(1, 0);
    if (total == 0) return;
    const uint64_t n = (total + cap - 1) / cap;
    uint64_t size = (((total + n - 1) / n) + 31) & ~31ull;
    if (size > cap) size = cap;
    for (uint64_t b = size; b < total; b += size) starts.push_back(b);
    starts.push_back(total);
}

// staging reads: split [seqs, offsets] into chunks of <= chunk_bases() positions, cutting at read
// boundaries where possible; a read longer than a chunk continues in the next chunk with k-1 bases of
// overlap, which yields exactly the same k-mer stream.
// ------------------------------------------------------------------------------------------------------
struct ChunkPlan {
    uint64_t base0, base1;          // range of the concatenated buffer
    std::vector<uint32_t> offs;     // chunk-relative read offsets (n+1)
};

static void plan_chunks(const uint64_t* offsets, uint64_t n_reads, int k, uint64_t cap, std::vector<ChunkPlan>& out)
{
    uint64_t r = 0;
    uint64_t carry_start = 0;  // start (absolute base) of the current piece of read r
    bool in_piece = false;
    while (r < n_reads) {
        ChunkPlan c;
        c.base0 = in_piece ? carry_start : offsets[r];
        c.offs.push_back(0);
        uint64_t used = 0;
        while (r < n_reads) {
            uint64_t s = in_piece ? carry_start : offsets[r];
            uint64_t e = offsets[r + 1];
            uint64_t len = e - s;
            if (used + len <= cap && c.offs.size() <= cap / 4 + 1) {
                used += len;
                c.offs.push_back((uint32_t)used);
                r++;
                in_piece = false;
                continue;
            }
            if (used == 0) {
                // a single read longer than the chunk: take cap bases, continue k-1 before the cut
                uint64_t cut = s + cap;
                used = cap;
                c.offs.push_back((uint32_t)used);
                carry_start = cut - (uint64_t)(k - 1);
                in_piece = true;
            }
            break;
        }
        c.base1 = c.base0 + used;
        out.push_back(std::move(c));
    }
}

// upload chunk (ASCII -> device -> 2-bit) into staging slot `slot` on stream `st`
static int stage_chunk(kmgpu_sketch* h, const char* seqs, const ChunkPlan& c, uint32_t flags, ChunkDev* out, bool need_acgt_check,
                       int slot = 0, cudaStream_t st = nullptr)
{
    if (!st) st = h->stream;
    kmgpu_sketch::Stage& S = h->stage[slot];
    uint32_t n_pos = (uint32_t)(c.base1 - c.base0);
    uint32_t n_reads = (uint32_t)c.offs.size() - 1;
    size_t n_words = (size_t)n_tiles(n_pos) * (TILE / 32) + TILE_PAD_WORDS;
    CKR(S.ascii.ensure(std::max<size_t>(n_pos, 1)));
    CKR(S.words.ensure(n_words));
    CKR(S.offs.ensure(n_reads + 1));
    CKR(S.h_offs.ensure(n_reads + 1));
    memcpy(S.h_offs.p, c.offs.data(), (n_reads + 1) * sizeof(uint32_t));
    if (n_pos) CK(cudaMemcpyAsync(S.ascii.p, seqs + c.base0, n_pos, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(S.offs.p, S.h_offs.p, (n_reads + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    if (need_acgt_check) CK(cudaMemsetAsync(h->d_ctrl_copy, 0, sizeof(Ctrl), st));
    k_pack<<<(unsigned)((n_words + 255) / 256), 256, 0, st>>>(S.ascii.p, n_pos, (flags & KMGPU_CLEAN) ? 1 : 0, S.words.p,
                                                             (uint32_t)n_words, h->d_ctrl_copy);
    CKR(S.tfr.ensure(n_tiles(n_pos) + 1));
    k_tile_index<<<(n_tiles(n_pos) + 1 + 255) / 256, 256, 0, st>>>(S.offs.p, n_reads, n_tiles(n_pos), S.tfr.p);
    CKR(S.valid.ensure((size_t)n_pos / 32 + 2));
    CK(cudaMemsetAsync(S.valid.p, 0, ((size_t)n_pos / 32 + 2) * 4, st));
    if (n_reads) k_valid_bits<<<(n_reads + 255) / 256, 256, 0, st>>>(S.offs.p, n_reads, h->k, S.valid.p);
    h->all_launches += 3;
    CK(cudaGetLastError());
    if (need_acgt_check) {
        CK(cudaMemcpyAsync(h->h_ctrl_copy, h->d_ctrl_copy, sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (h->h_ctrl_copy->non_acgt)
            return fail(KMGPU_ENONACGT, "sequence holds %llu bytes outside ACGT; the Murmur hash of uncleaned sequences is not computed on the device",
                        (unsigned long long)h->h_ctrl_copy->non_acgt);
    }
    out->words = S.words.p;
    out->offs = S.offs.p;
    out->tfr = S.tfr.p;
    out->valid = S.valid.p;
    out->n_reads = n_reads;
    out->n_pos = n_pos;
    return KMGPU_OK;
}

static int make_pred(kmgpu_sketch* h, const kmgpu_band_t* band, const kmgpu_mask_t* mask, Pred* P, bool* pred, const SketchDev** M)
{
    memset(P, 0, sizeof *P);
    *pred = false;
    *M = nullptr;
    if (band) {
        P->band_on = 1;
        P->band_lo = band->lo;
        P->band_hi = band->hi;
        *pred = true;
    }
    if (mask) {
        kmgpu_sketch* m = mask->mask;
        if (!m) return fail(KMGPU_EINVAL, "mask sketch is NULL");
        if (m->device != h->device) return fail(KMGPU_EINVAL, "mask sketch lives on another device");
        P->mask_on = 1;
        P->mask_threshold = mask->threshold;
        P->mask_ge = mask->consume_masked ? 1 : 0;
        *M = &m->dev;
        *pred = true;
        if (m != h) {
            // whatever the mask sketch still has queued (a reset, an ingest) must have landed before this stream reads its
            // tables; its bigcount map goes along as a sorted device copy (mask->get_count, hashtable.cc:177-178)
            std::lock_guard<std::mutex> gm(m->mu);
            CK(cudaStreamSynchronize(m->stream));
            if (m->kind == BYTE && m->use_bigcount && !m->big.empty()) {
                CKR(sync_big_to_device(m));
                P->mask_big_keys = m->big_keys.p;
                P->mask_big_vals = m->big_vals.p;
                P->mask_n_big = m->n_big_dev;
            }
        }
    }
    return KMGPU_OK;
}

static bool needs_acgt_check(const kmgpu_sketch* h, uint32_t flags) { return h->hash == KMGPU_MURMUR && !(flags & KMGPU_CLEAN); }

// upload the base range [b0, b1) of the caller's buffer with the reads overlapping it; offsets are clipped and
// rebased on the device, so the host does O(log n_reads) work per chunk
// `packed` != nullptr: the caller's buffer is the 2-bit stream itself (32 bases per word, b0 a multiple of 32): the words covering
// [b0, b1) are uploaded as they are (a quarter of the bytes, no packing kernel)
static int stage_range(kmgpu_sketch* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint64_t b0, uint64_t b1,
                       uint32_t flags, ChunkDev* out, bool need_acgt_check, int slot, cudaStream_t st, const uint64_t* packed = nullptr,
                       uint64_t packed_words = 0)
{
    kmgpu_sketch::Stage& S = h->stage[slot];
    // r_lo = last read starting at or before b0; r_hi = first index whose offset is >= b1
    uint64_t r_lo = (uint64_t)(std::upper_bound(offsets, offsets + n_reads + 1, b0) - offsets);
    r_lo = r_lo ? r_lo - 1 : 0;
    if (r_lo >= n_reads) r_lo = n_reads - 1;
    uint64_t r_hi = (uint64_t)(std::lower_bound(offsets + r_lo, offsets + n_reads + 1, b1) - offsets);
    if (r_hi > n_reads) r_hi = n_reads;
    if (r_hi <= r_lo) r_hi = r_lo + 1;
    uint32_t n_pos = (uint32_t)(b1 - b0);
    uint32_t nr = (uint32_t)(r_hi - r_lo);
    size_t n_words = (size_t)n_tiles(n_pos) * (TILE / 32) + TILE_PAD_WORDS;
    if (!packed) CKR(S.ascii.ensure(std::max<size_t>(n_pos, 1)));
    CKR(S.words.ensure(n_words));
    CKR(S.offs.ensure(nr + 1));
    CKR(S.offs64.ensure(nr + 1));
    CKR(S.tfr.ensure(n_tiles(n_pos) + 1));
    if (packed) {
        const uint64_t w0 = b0 / 32, w1 = std::min<uint64_t>(packed_words, w0 + n_words);
        if (w1 - w0 < n_words) CK(cudaMemsetAsync(S.words.p + (w1 - w0), 0, (n_words - (w1 - w0)) * 8, st));
        if (w1 > w0) CK(cudaMemcpyAsync(S.words.p, packed + w0, (w1 - w0) * 8, cudaMemcpyHostToDevice, st));
    } else if (n_pos) {
        CK(cudaMemcpyAsync(S.ascii.p, seqs + b0, n_pos, cudaMemcpyHostToDevice, st));
    }
    // the caller's offsets may be pageable: a copy from pageable memory would block this thread until everything queued
    // before it on the stream (the sequence bytes just above) has gone over the bus; go through a pinned slice instead
    {
        cudaPointerAttributes pa;
        const bool pinned = cudaPointerGetAttributes(&pa, offsets) == cudaSuccess && pa.type == cudaMemoryTypeHost;
        cudaGetLastError();
        const uint64_t* src = offsets + r_lo;
        if (!pinned) {
            CKR(S.h_offs64.ensure(nr + 1));
            memcpy(S.h_offs64.p, src, (size_t)(nr + 1) * 8);
            src = S.h_offs64.p;
        }
        CK(cudaMemcpyAsync(S.offs64.p, src, (size_t)(nr + 1) * 8, cudaMemcpyHostToDevice, st));
    }
    k_clip_offsets<<<(nr + 1 + 255) / 256, 256, 0, st>>>(S.offs64.p, nr + 1, b0, b1, S.offs.p);
    if (packed) need_acgt_check = false;
    if (need_acgt_check) CK(cudaMemsetAsync(h->d_ctrl_copy, 0, sizeof(Ctrl), st));
    if (!packed)
        k_pack<<<(unsigned)((n_words + 255) / 256), 256, 0, st>>>(S.ascii.p, n_pos, (flags & KMGPU_CLEAN) ? 1 : 0, S.words.p,
                                                                 (uint32_t)n_words, h->d_ctrl_copy);
    k_tile_index<<<(n_tiles(n_pos) + 1 + 255) / 256, 256, 0, st>>>(S.offs.p, nr, n_tiles(n_pos), S.tfr.p);
    CKR(S.valid.ensure((size_t)n_pos / 32 + 2));
    CK(cudaMemsetAsync(S.valid.p, 0, ((size_t)n_pos / 32 + 2) * 4, st));
    k_valid_bits<<<(nr + 255) / 256, 256, 0, st>>>(S.offs.p, nr, h->k, S.valid.p);
    h->all_launches += packed ? 3 : 4;
    CK(cudaGetLastError());
    if (need_acgt_check) {
        CK(cudaMemcpyAsync(h->h_ctrl_copy, h->d_ctrl_copy, sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (h->h_ctrl_copy->non_acgt)
            return fail(KMGPU_ENONACGT, "sequence holds %llu bytes outside ACGT; the Murmur hash of uncleaned sequences is not computed on the device",
                        (unsigned long long)h->h_ctrl_copy->non_acgt);
    }
    out->words = S.words.p;
    out->offs = S.offs.p;
    out->tfr = S.tfr.p;
    out->valid = S.valid.p;
    out->n_reads = nr;
    out->n_pos = n_pos;
    return KMGPU_OK;
}

// host input, ASCII (seqs) or 2-bit packed (packed, packed_words): chunked, uploaded in parts on the copy stream, ingested
// newbits_out (optional): one bit per base of [offsets[0], offsets[n_reads]), set iff the k-mer starting there was new
// (Storage::add / test_and_set_bits returned true for it in stream order); n_new_out: their number
static int consume_host(kmgpu_t* h, const char* seqs, const uint64_t* packed, uint64_t packed_words, const uint64_t* offsets, uint64_t n_reads,
                        uint32_t flags, const kmgpu_band_t* band, const kmgpu_mask_t* mask, uint64_t* n_kmers_out, uint32_t* newbits_out = nullptr,
                        uint64_t* n_new_out = nullptr)
{
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    Pred P;
    bool pred;
    const SketchDev* M;
    CKR(make_pred(h, band, mask, &P, &pred, &M));
    HashCfg H{h->hash, h->k};
    ChunkResult res;
    // Chunk i covers bases [first + i*cap, first + i*cap + cap + k-1) of the caller's buffer with the reads clipped to
    // it: a clipped piece inside the k-1 overlap is shorter than k and yields nothing, the piece that continues past it
    // starts exactly at the first k-mer the previous chunk could not hold — the k-mer stream is unchanged.
    // Chunk i+1 is uploaded and packed on the copy stream while chunk i is ingested on the main stream.
    const uint64_t first = offsets[0], last = offsets[n_reads];
    const bool chk = needs_acgt_check(h, flags);
    if (last <= first) return KMGPU_OK;
    {
        // Sketches on the bucket path take host input in PARTS: a chunk (the unit that pays one sweep of the sketch) is as
        // large as for device-resident input, but it is uploaded, packed, hashed and bucketized part by part, so that only
        // the first part's trip over PCIe is exposed.  All of a chunk's copies are queued on the copy stream at once (one
        // staging slot per part, two sets of slots: the next chunk's parts are queued while this chunk is being applied).
        const uint64_t total = last - first, cap = sketch_chunk_bases(h);
        const uint64_t n_chunks = (total + cap - 1) / cap;
        const uint64_t per_chunk = (((total + n_chunks - 1) / n_chunks) + 31) & ~31ull;
        // parts start on word boundaries of the stream (packed input is uploaded word-wise)
        const uint64_t part_cap = (std::max<uint64_t>(std::min<uint64_t>(env_u64("KMGPU_PART_BASES", 24ull << 20), per_chunk),
                                                      (per_chunk + kmgpu_sketch::MAX_PARTS - 1) / kmgpu_sketch::MAX_PARTS) + 31) & ~31ull;
        const uint64_t worst_pos = per_chunk + (uint64_t)kmgpu_sketch::MAX_PARTS * h->k;
        // the path is kept for every chunk of the call: a short last chunk that the bins path could take stays grouped
        const Path path = worst_pos < (1ull << 31) ? choose_path(h, (uint32_t)worst_pos, h->ft_on) : Path::Unsupported;
        if (env_u64("KMGPU_PARTS", 1) && total > part_cap && (path == Path::Bins || path == Path::Grouped)) {
            struct Staged { std::vector<Part> parts; };
            Staged set[2];
            auto stage_chunk_parts = [&](uint64_t ci, Staged* out) -> int {
                out->parts.clear();
                const uint64_t c0 = first + ci * per_chunk, c1 = std::min(last, c0 + per_chunk);
                if (c0 >= last) return KMGPU_OK;   // rounding per_chunk up to 32 can leave nothing for the last chunk
                std::vector<uint64_t> cuts;   // equal parts (a short, growing first part was measured: no gain)
                for (uint64_t b = c0; b < c1; b += part_cap) cuts.push_back(b);
                cuts.push_back(c1);
                uint32_t pos = 0;
                int slot = (int)(ci & 1) * kmgpu_sketch::MAX_PARTS;
                for (size_t pi = 0; pi + 1 < cuts.size(); pi++, slot++) {
                    const uint64_t b0 = cuts[pi];
                    const uint64_t b1 = std::min(last, cuts[pi + 1] + (uint64_t)(h->k - 1));
                    ChunkDev cd;
                    CKR(stage_range(h, seqs, offsets, n_reads, b0, b1, flags, &cd, chk, slot, h->copy_stream, packed, packed_words));
                    CK(cudaEventRecord(h->stage[slot].ready, h->copy_stream));
                    out->parts.push_back(Part{make_input(cd), pos, h->stage[slot].ready});
                    // a position is the base's offset within the chunk: the k-1 positions a part shares with the next one hold
                    // no k-mer start in this part (the reads are clipped to it), they are the next part's first positions
                    pos = (uint32_t)(cuts[pi + 1] - c0);
                }
                return KMGPU_OK;
            };
            CKR(stage_chunk_parts(0, &set[0]));
            for (uint64_t ci = 0; ci < n_chunks; ci++) {
                if (set[ci & 1].parts.empty()) break;
                const Between next = [&]() -> int { return ci + 1 < n_chunks ? stage_chunk_parts(ci + 1, &set[(ci + 1) & 1]) : KMGPU_OK; };
                ChunkResult cr;
                CKR(ingest_chunk(h, 0, H, set[ci & 1].parts, P, pred, M, &cr, next, path));
                res.n_kmers += cr.n_kmers;
                res.n_new += cr.n_new;
                if (newbits_out && cr.have_newbits) {
                    // chunk ci starts on a word of the output (per_chunk is a multiple of 32); its k-1 bases of overlap hold no k-mer start
                    const uint64_t c0 = ci * per_chunk, c1 = std::min(last - first, c0 + per_chunk);
                    CK(cudaMemcpy(newbits_out + c0 / 32, h->d_newbits.p, ((c1 - c0 + 31) / 32) * 4, cudaMemcpyDeviceToHost));
                }
            }
            if (n_kmers_out) *n_kmers_out = res.n_kmers;
            if (n_new_out) *n_new_out = res.n_new;
            return KMGPU_OK;
        }
    }
    // Every chunk pays one sweep of the whole sketch (the folds) plus the fixed part of the resolutions, so there are
    // as few chunks as the cap allows; nothing can start before chunk 0 has crossed PCIe, so chunk 0 is the short one
    // (half of the others when the cap leaves that freedom) and the copy of chunk i+1 hides behind the ingest of chunk i.
    std::vector<uint64_t> starts(1, 0);
    if (packed || newbits_out) {
        balanced_chunks(last - first, sketch_chunk_bases(h), starts);   // packed input / per-base result bits: chunks cut on word boundaries
    } else {
        // one chunk more than a device-resident batch would get as soon as that leaves chunk 0 at most half of the others
        const uint64_t total = last - first, cap = sketch_chunk_bases(h), n = (2 * total + cap + 2 * cap - 1) / (2 * cap);
        bool ramp = false;
        if (n >= 2 && 2 * total <= (n + 1) * cap) {
            // sizes 1 : 2 : ... : n — the copy of every chunk still hides behind the ingest of the one before it (PCIe
            // moves a base about twice as fast as the kernels consume it) and chunk 0 is as short as that allows
            const uint64_t unit = ((2 * total / (n * (n + 1))) + 31) & ~31ull;
            const uint64_t head = unit * (n * (n - 1) / 2);   // everything but the last chunk
            if (unit && head < total && total - head <= cap && (n - 1) * unit <= cap) {
                uint64_t b = 0;
                for (uint64_t i = 1; i < n; i++) {
                    b += i * unit;
                    starts.push_back(b);
                }
                ramp = true;
            }
        }
        if (!ramp && n >= 2) {
            uint64_t c0 = std::max<uint64_t>(total > (n - 1) * cap ? total - (n - 1) * cap : 0, total / (2 * n - 1));
            uint64_t c = (((total - c0) + (n - 2)) / (n - 1) + 31) & ~31ull;
            c = std::min(c, cap);
            c0 = total - (n - 1) * c;   // > 0: (n-1)*c < total since c0 was at least total/(2n-1) before rounding
            if ((int64_t)c0 <= 0) c0 = 1;
            for (uint64_t b = c0; b < total; b += c) starts.push_back(b);
        }
        starts.push_back(total);
    }
    const uint64_t n_chunks = starts.size() - 1;
    auto range = [&](uint64_t i, uint64_t* b0, uint64_t* b1) {
        *b0 = first + starts[i];
        *b1 = std::min(last, first + starts[i + 1] + (uint64_t)(h->k - 1));
    };
    ChunkDev cd[2];
    uint64_t b0, b1;
    range(0, &b0, &b1);
    CKR(stage_range(h, seqs, offsets, n_reads, b0, b1, flags, &cd[0], chk, 0, h->copy_stream, packed, packed_words));
    CK(cudaEventRecord(h->stage[0].ready, h->copy_stream));
    for (uint64_t i = 0; i < n_chunks; i++) {
        CK(cudaStreamWaitEvent(h->stream, h->stage[i & 1].ready, 0));
        ChunkResult cr;
        CKR(ingest_chunk(h, 0, H, {Part{make_input(cd[i & 1]), 0u, nullptr}}, P, pred, M, &cr, [&]() -> int {
            if (i + 1 < n_chunks) {
                int ns = (int)((i + 1) & 1);
                uint64_t c0, c1;
                range(i + 1, &c0, &c1);
                CKR(stage_range(h, seqs, offsets, n_reads, c0, c1, flags, &cd[ns], chk, ns, h->copy_stream, packed, packed_words));
                CK(cudaEventRecord(h->stage[ns].ready, h->copy_stream));
            }
            return KMGPU_OK;
        }));
        res.n_kmers += cr.n_kmers;
        res.n_new += cr.n_new;
        if (newbits_out && cr.have_newbits)
            CK(cudaMemcpy(newbits_out + starts[i] / 32, h->d_newbits.p, ((starts[i + 1] - starts[i] + 31) / 32) * 4, cudaMemcpyDeviceToHost));
    }
    if (n_kmers_out) *n_kmers_out = res.n_kmers;
    if (n_new_out) *n_new_out = res.n_new;
    return KMGPU_OK;
}

extern "C" int kmgpu_consume_reads(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                   const kmgpu_band_t* band, const kmgpu_mask_t* mask, uint64_t* n_kmers_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n_kmers_out) *n_kmers_out = 0;
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets) return fail(KMGPU_EINVAL, "null input");
    return consume_host(h, seqs, nullptr, 0, offsets, n_reads, flags, band, mask, n_kmers_out);
}

// consume + per-k-mer "was new" bits, for consumers that act on them in stream order (tagging: Hashgraph::consume_sequence_and_tag,
// src/oxli/hashgraph.cc:200-271, tests the bool of store->test_and_set_bits for every k-mer)
extern "C" int kmgpu_consume_reads_new(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags, uint32_t* newbits_out,
                                       uint64_t* n_kmers_out, uint64_t* n_new_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n_kmers_out) *n_kmers_out = 0;
    if (n_new_out) *n_new_out = 0;
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets || !newbits_out) return fail(KMGPU_EINVAL, "null argument");
    memset(newbits_out, 0, ((offsets[n_reads] - offsets[0] + 31) / 32) * 4);
    return consume_host(h, seqs, nullptr, 0, offsets, n_reads, flags, nullptr, nullptr, n_kmers_out, newbits_out, n_new_out);
}

extern "C" int kmgpu_consume_packed(kmgpu_t* h, const uint64_t* words, uint64_t n_words, const uint64_t* offsets, uint64_t n_reads,
                                    const kmgpu_band_t* band, const kmgpu_mask_t* mask, uint64_t* n_kmers_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n_kmers_out) *n_kmers_out = 0;
    if (n_reads == 0) return KMGPU_OK;
    if (!words || !offsets) return fail(KMGPU_EINVAL, "null input");
    if (n_words * 32 < offsets[n_reads]) return fail(KMGPU_EINVAL, "packed buffer shorter than offsets[n_reads]");
    if (offsets[0] % 32) return fail(KMGPU_EINVAL, "offsets[0] of a packed buffer must be a multiple of 32 bases");
    // same pipeline as ASCII input (chunks uploaded in parts on the copy stream while the previous part is grouped), a quarter of the bytes
    return consume_host(h, nullptr, words, n_words, offsets, n_reads, 0, band, mask, n_kmers_out);
}

// ------------------------------------------------------------------------------------------------------
// device-resident batches
// ------------------------------------------------------------------------------------------------------
extern "C" int kmgpu_batch_create(int device, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags, int ksize,
                                  kmgpu_batch_t** out)
{
    if (!out) return fail(KMGPU_EINVAL, "out is NULL");
    *out = nullptr;
    if (ksize < 1 || ksize > MAX_K) return fail(KMGPU_EINVAL, "ksize out of range");
    if (n_reads && (!seqs || !offsets)) return fail(KMGPU_EINVAL, "null input");
    CKR(set_device(device));
    kmgpu_batch* b = new kmgpu_batch();
    b->device = device;
    b->ksize = ksize;
    b->n_reads = n_reads;
    b->n_bases = n_reads ? offsets[n_reads] - offsets[0] : 0;
    std::vector<ChunkPlan> plan;
    if (n_reads) {
        // equal pieces (every piece costs one sweep of the sketch when it is consumed); cut at read boundaries
        const uint64_t cap = chunk_bases(), n = (b->n_bases + cap - 1) / cap;
        uint64_t piece = n ? (((b->n_bases + n - 1) / n + 65536 + TILE - 1) / TILE) * TILE : cap;
        plan_chunks(offsets, n_reads, ksize, std::min(cap, piece), plan);
    }
    uint8_t* d_ascii = nullptr;
    Ctrl* d_ctrl = nullptr;
    size_t ascii_cap = 0;
    int rc = KMGPU_OK;
    auto bail = [&](cudaError_t e) {
        rc = fail(e == cudaErrorMemoryAllocation ? KMGPU_ENOMEM : KMGPU_ECUDA, "batch upload: %s", cudaGetErrorString(e));
    };
    cudaError_t e = cudaMalloc(&d_ctrl, sizeof(Ctrl));
    if (e != cudaSuccess) bail(e);
    for (size_t ci = 0; rc == KMGPU_OK && ci < plan.size(); ci++) {
        const ChunkPlan& c = plan[ci];
        uint32_t n_pos = (uint32_t)(c.base1 - c.base0);
        uint32_t nr = (uint32_t)c.offs.size() - 1;
        size_t nw = (size_t)n_tiles(n_pos) * (TILE / 32) + TILE_PAD_WORDS;
        if (n_pos > ascii_cap) {
            if (d_ascii) cudaFree(d_ascii);
            d_ascii = nullptr;
            if ((e = cudaMalloc(&d_ascii, n_pos)) != cudaSuccess) { bail(e); break; }
            ascii_cap = n_pos;
        }
        kmgpu_batch::Piece p{nullptr, nullptr, nullptr, nr, n_pos, nullptr};
        if ((e = cudaMalloc(&p.words, nw * 8)) != cudaSuccess) { bail(e); break; }
        if ((e = cudaMalloc(&p.offs, (nr + 1) * 4)) != cudaSuccess) { cudaFree(p.words); bail(e); break; }
        if ((e = cudaMalloc(&p.tfr, (n_tiles(n_pos) + 1) * 4)) != cudaSuccess) { cudaFree(p.words); cudaFree(p.offs); bail(e); break; }
        if ((e = cudaMalloc(&p.valid, ((size_t)n_pos / 32 + 2) * 4)) != cudaSuccess) { cudaFree(p.words); cudaFree(p.offs); cudaFree(p.tfr); bail(e); break; }
        b->pieces.push_back(p);
        b->bytes += nw * 8 + (nr + 1) * 4 + (n_tiles(n_pos) + 1) * 4;
        if (n_pos && (e = cudaMemcpy(d_ascii, seqs + c.base0, n_pos, cudaMemcpyHostToDevice)) != cudaSuccess) { bail(e); break; }
        if ((e = cudaMemcpy(p.offs, c.offs.data(), (nr + 1) * 4, cudaMemcpyHostToDevice)) != cudaSuccess) { bail(e); break; }
        cudaMemset(d_ctrl, 0, sizeof(Ctrl));
        k_pack<<<(unsigned)((nw + 255) / 256), 256>>>(d_ascii, n_pos, (flags & KMGPU_CLEAN) ? 1 : 0, p.words, (uint32_t)nw, d_ctrl);
        k_tile_index<<<(n_tiles(n_pos) + 1 + 255) / 256, 256>>>(p.offs, nr, n_tiles(n_pos), p.tfr);
        cudaMemset(p.valid, 0, ((size_t)n_pos / 32 + 2) * 4);
        if (nr) k_valid_bits<<<(nr + 255) / 256, 256>>>(p.offs, nr, ksize, p.valid);
        if ((e = cudaDeviceSynchronize()) != cudaSuccess) { bail(e); break; }
    }
    if (d_ascii) cudaFree(d_ascii);
    if (d_ctrl) cudaFree(d_ctrl);
    if (rc != KMGPU_OK) {
        kmgpu_batch_destroy(b);
        return rc;
    }
    *out = b;
    return KMGPU_OK;
}

extern "C" int kmgpu_batch_destroy(kmgpu_batch_t* b)
{
    if (!b) return KMGPU_OK;
    cudaSetDevice(b->device);
    for (auto& p : b->pieces) {
        if (p.words) cudaFree(p.words);
        if (p.offs) cudaFree(p.offs);
        if (p.tfr) cudaFree(p.tfr);
        if (p.valid) cudaFree(p.valid);
    }
    delete b;
    return KMGPU_OK;
}

extern "C" int kmgpu_batch_info(const kmgpu_batch_t* b, uint64_t* n_reads, uint64_t* n_bases, uint64_t* device_bytes)
{
    if (!b) return fail(KMGPU_EINVAL, "null batch");
    if (n_reads) *n_reads = b->n_reads;
    if (n_bases) *n_bases = b->n_bases;
    if (device_bytes) *device_bytes = b->bytes;
    return KMGPU_OK;
}

extern "C" int kmgpu_consume_batch(kmgpu_t* h, const kmgpu_batch_t* b, const kmgpu_band_t* band, const kmgpu_mask_t* mask,
                                   uint64_t* n_kmers_out)
{
    if (!h || !b) return fail(KMGPU_EINVAL, "null argument");
    if (n_kmers_out) *n_kmers_out = 0;
    if (b->device != h->device) return fail(KMGPU_EINVAL, "batch lives on another device");
    if (b->ksize != h->k) return fail(KMGPU_EINVAL, "batch was cut for k=%d, sketch has k=%d", b->ksize, h->k);
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    Pred P;
    bool pred;
    const SketchDev* M;
    CKR(make_pred(h, band, mask, &P, &pred, &M));
    HashCfg H{h->hash, h->k};
    ChunkResult res;
    const uint64_t cap = sketch_chunk_bases(h);
    for (size_t i = 0; i < b->pieces.size();) {
        // a sketch that prefers larger chunks (two-level grouped path) takes several pieces of the batch as the parts of one chunk
        std::vector<Part> parts;
        uint64_t pos = 0;
        size_t j = i;
        while (j < b->pieces.size() && (j == i || pos + b->pieces[j].n_pos <= cap)) {
            const auto& p = b->pieces[j];
            ChunkDev cd;
            cd.words = p.words;
            cd.offs = p.offs;
            cd.tfr = p.tfr;
            cd.valid = p.valid;
            cd.n_reads = p.n_reads;
            cd.n_pos = p.n_pos;
            parts.push_back(Part{make_input(cd), (uint32_t)pos, nullptr});
            pos += p.n_pos;
            j++;
        }
        if (parts.size() > 1 && pos < (1ull << 31) && choose_path(h, (uint32_t)pos, h->ft_on) == Path::Grouped) {
            CKR(ingest_chunk(h, 0, H, parts, P, pred, M, &res));
        } else {
            for (const Part& pt : parts) CKR(ingest_chunk(h, 0, H, {Part{pt.in, 0u, nullptr}}, P, pred, M, &res));
        }
        i = j;
    }
    if (n_kmers_out) *n_kmers_out = res.n_kmers;
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// hashed k-mers
// ------------------------------------------------------------------------------------------------------
extern "C" int kmgpu_add_hashes(kmgpu_t* h, const uint64_t* hashes, uint64_t n, uint8_t* is_new_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n == 0) return KMGPU_OK;
    if (!hashes) return fail(KMGPU_EINVAL, "null input");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    HashCfg H{h->hash, h->k};
    Pred P;
    memset(&P, 0, sizeof P);
    const uint64_t cap = chunk_bases();
    std::vector<uint32_t> bits;
    for (uint64_t i0 = 0; i0 < n; i0 += cap) {
        uint32_t m = (uint32_t)std::min<uint64_t>(cap, n - i0);
        CKR(h->d_hashin.ensure(m));
        CK(cudaMemcpyAsync(h->d_hashin.p, hashes + i0, 8ull * m, cudaMemcpyHostToDevice, h->stream));
        ChunkResult res;
        CKR(ingest_chunk(h, 1, H, {Part{make_hash_input(h->d_hashin.p, m), 0u, nullptr}}, P, false, nullptr, &res));
        if (is_new_out) {
            if (res.have_newbits) {
                bits.resize((m + 31) / 32);
                CK(cudaMemcpy(bits.data(), h->d_newbits.p, bits.size() * 4, cudaMemcpyDeviceToHost));
                for (uint32_t j = 0; j < m; j++) is_new_out[i0 + j] = (bits[j >> 5] >> (j & 31)) & 1u;
            } else {
                memset(is_new_out + i0, 0, m);
            }
        }
    }
    return KMGPU_OK;
}

extern "C" int kmgpu_get_counts(kmgpu_t* h, const uint64_t* hashes, uint64_t n, uint16_t* counts_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n == 0) return KMGPU_OK;
    if (!hashes || !counts_out) return fail(KMGPU_EINVAL, "null argument");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    if (h->kind == BYTE && h->use_bigcount) CKR(sync_big_to_device(h));
    uint32_t nb = (h->kind == BYTE && h->use_bigcount) ? h->n_big_dev : 0;
    HashCfg H{h->hash, h->k};
    const uint64_t cap = chunk_bases();
    for (uint64_t i0 = 0; i0 < n; i0 += cap) {
        uint32_t m = (uint32_t)std::min<uint64_t>(cap, n - i0);
        CKR(h->d_hashin.ensure(m));
        CKR(h->d_counts.ensure(m));
        CK(cudaMemcpyAsync(h->d_hashin.p, hashes + i0, 8ull * m, cudaMemcpyHostToDevice, h->stream));
        launch_counts(1, h->dev, H, make_hash_input(h->d_hashin.p, m), h->big_keys.p, h->big_vals.p, nb, h->d_counts.p, nullptr, nullptr,
                      h->stream);
        h->all_launches += 1;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(counts_out + i0, h->d_counts.p, 2ull * m, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// per-k-mer and per-read queries over sequences
// ------------------------------------------------------------------------------------------------------
// the values of every read's k-mers, read after read, from an array over a chunk's positions (read j starts at offs[j]);
// returns how many were written
template <typename T>
static uint64_t compact_kmers(const T* per_pos, const uint32_t* offs, size_t n_reads, int k, T* out)
{
    uint64_t w = 0;
    for (size_t j = 0; j < n_reads; j++) {
        const uint32_t s = offs[j], e = offs[j + 1];
        if (e - s < (uint32_t)k) continue;
        const uint32_t n = e - s - k + 1;
        memcpy(out + w, per_pos + s, sizeof(T) * n);
        w += n;
    }
    return w;
}

static int per_kmer_query(kmgpu_sketch* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                          uint16_t* counts_out, uint64_t* hashes_out, uint64_t* n_kmers_out)
{
    if (n_kmers_out) *n_kmers_out = 0;
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets) return fail(KMGPU_EINVAL, "null input");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    bool want_c = counts_out != nullptr;
    if (want_c && h->kind == BYTE && h->use_bigcount) CKR(sync_big_to_device(h));
    uint32_t nb = (h->kind == BYTE && h->use_bigcount) ? h->n_big_dev : 0;
    HashCfg H{h->hash, h->k};
    std::vector<ChunkPlan> plan;
    plan_chunks(offsets, n_reads, h->k, chunk_bases(), plan);
    std::vector<uint16_t> hc;
    std::vector<uint64_t> hh;
    uint64_t w = 0;
    for (const ChunkPlan& c : plan) {
        ChunkDev cd;
        CKR(stage_chunk(h, seqs, c, flags, &cd, needs_acgt_check(h, flags)));
        if (cd.n_pos == 0) continue;
        if (want_c) CKR(h->d_counts.ensure(cd.n_pos));
        if (hashes_out) CKR(h->d_hashes.ensure(cd.n_pos));
        launch_counts(0, h->dev, H, make_input(cd), h->big_keys.p, h->big_vals.p, nb, want_c ? h->d_counts.p : nullptr,
                      hashes_out ? h->d_hashes.p : nullptr, nullptr, h->stream);
        h->all_launches += 1;
        CK(cudaGetLastError());
        if (want_c) {
            hc.resize(cd.n_pos);
            CK(cudaMemcpyAsync(hc.data(), h->d_counts.p, 2ull * cd.n_pos, cudaMemcpyDeviceToHost, h->stream));
        }
        if (hashes_out) {
            hh.resize(cd.n_pos);
            CK(cudaMemcpyAsync(hh.data(), h->d_hashes.p, 8ull * cd.n_pos, cudaMemcpyDeviceToHost, h->stream));
        }
        CK(cudaStreamSynchronize(h->stream));
        const size_t nr = c.offs.size() - 1;
        uint64_t n = 0;
        if (want_c) n = compact_kmers(hc.data(), c.offs.data(), nr, h->k, counts_out + w);
        if (hashes_out) n = compact_kmers(hh.data(), c.offs.data(), nr, h->k, hashes_out + w);
        w += n;
    }
    if (n_kmers_out) *n_kmers_out = w;
    return KMGPU_OK;
}

extern "C" int kmgpu_kmer_counts(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                 uint16_t* counts_out, uint64_t* n_kmers_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (!counts_out && n_reads) return fail(KMGPU_EINVAL, "null output");
    return per_kmer_query(h, seqs, offsets, n_reads, flags, counts_out, nullptr, n_kmers_out);
}

extern "C" int kmgpu_kmer_hashes(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                 uint64_t* hashes_out, uint64_t* n_kmers_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (!hashes_out && n_reads) return fail(KMGPU_EINVAL, "null output");
    return per_kmer_query(h, seqs, offsets, n_reads, flags, nullptr, hashes_out, n_kmers_out);
}

// one staged chunk of whole reads with its counts per position: one warp per read (median / mean / stddev, or median_at_least),
// results written from read r0 on
static int read_stats_counts(kmgpu_sketch* h, const uint16_t* counts, const ChunkDev& cd, uint64_t r0, uint16_t* median_out,
                             float* average_out, float* stddev_out, uint32_t* n_kmers_out, bool at_least, uint32_t cutoff,
                             uint8_t* at_least_out)
{
    cudaStream_t st = h->stream;
    uint32_t nr = cd.n_reads;
    CKR(h->d_stat_med.ensure(nr));
    CKR(h->d_stat_f.ensure(2ull * nr));
    CKR(h->d_stat_n.ensure(nr));
    CKR(h->d_stat_b.ensure(nr));
    bool want_med = !at_least;
    k_read_stats<<<(nr + 7) / 8, 256, 0, st>>>(counts, cd.offs, nr, h->k, want_med ? h->d_stat_med.p : nullptr,
                                              want_med ? h->d_stat_f.p : nullptr, want_med ? h->d_stat_f.p + nr : nullptr,
                                              h->d_stat_n.p, cutoff, at_least ? h->d_stat_b.p : nullptr);
    h->all_launches += 1;
    CK(cudaGetLastError());
    if (want_med) {
        if (median_out) CK(cudaMemcpyAsync(median_out + r0, h->d_stat_med.p, 2ull * nr, cudaMemcpyDeviceToHost, st));
        if (average_out) CK(cudaMemcpyAsync(average_out + r0, h->d_stat_f.p, 4ull * nr, cudaMemcpyDeviceToHost, st));
        if (stddev_out) CK(cudaMemcpyAsync(stddev_out + r0, h->d_stat_f.p + nr, 4ull * nr, cudaMemcpyDeviceToHost, st));
    } else {
        CK(cudaMemcpyAsync(at_least_out + r0, h->d_stat_b.p, nr, cudaMemcpyDeviceToHost, st));
    }
    if (n_kmers_out) CK(cudaMemcpyAsync(n_kmers_out + r0, h->d_stat_n.p, 4ull * nr, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return KMGPU_OK;
}

// one staged chunk of whole reads: counts per position, then read_stats_counts
static int read_stats_chunk(kmgpu_sketch* h, const ChunkDev& cd, uint64_t r0, uint32_t nb, uint16_t* median_out, float* average_out,
                            float* stddev_out, uint32_t* n_kmers_out, bool at_least, uint32_t cutoff, uint8_t* at_least_out)
{
    HashCfg H{h->hash, h->k};
    CKR(h->d_counts.ensure(std::max<uint32_t>(cd.n_pos, 1)));
    if (cd.n_pos) {
        launch_counts(0, h->dev, H, make_input(cd), h->big_keys.p, h->big_vals.p, nb, h->d_counts.p, nullptr, nullptr, h->stream);
        h->all_launches += 1;
    }
    return read_stats_counts(h, h->d_counts.p, cd, r0, median_out, average_out, stddev_out, n_kmers_out, at_least, cutoff, at_least_out);
}

// the same for trim_on_abundance / trim_below_abundance: the length every read keeps
static int trim_counts(kmgpu_sketch* h, const uint16_t* counts, const ChunkDev& cd, uint64_t r0, uint32_t abund, int below,
                       uint32_t* trim_pos_out)
{
    cudaStream_t st = h->stream;
    const uint32_t nr = cd.n_reads;
    CKR(h->d_stat_n.ensure(nr));
    k_trim_scan<<<(nr + 7) / 8, 256, 0, st>>>(counts, cd.offs, nr, h->k, abund, below, h->d_stat_n.p);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(trim_pos_out + r0, h->d_stat_n.p, 4ull * nr, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return KMGPU_OK;
}

static int per_read_query(kmgpu_sketch* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                          uint16_t* median_out, float* average_out, float* stddev_out, uint32_t* n_kmers_out, bool at_least,
                          uint32_t cutoff, uint8_t* at_least_out)
{
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets) return fail(KMGPU_EINVAL, "null input");
    for (uint64_t r = 0; r < n_reads; r++)
        if (offsets[r + 1] - offsets[r] > chunk_bases())
            return fail(KMGPU_EUNSUPPORTED, "read %llu is longer than a device chunk (%llu bases); per-read statistics need whole reads",
                        (unsigned long long)r, (unsigned long long)chunk_bases());
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    if (h->kind == BYTE && h->use_bigcount) CKR(sync_big_to_device(h));
    uint32_t nb = (h->kind == BYTE && h->use_bigcount) ? h->n_big_dev : 0;
    std::vector<ChunkPlan> plan;
    plan_chunks(offsets, n_reads, h->k, chunk_bases(), plan);
    uint64_t r0 = 0;
    for (const ChunkPlan& c : plan) {
        ChunkDev cd;
        CKR(stage_chunk(h, seqs, c, flags, &cd, needs_acgt_check(h, flags)));
        CKR(read_stats_chunk(h, cd, r0, nb, median_out, average_out, stddev_out, n_kmers_out, at_least, cutoff, at_least_out));
        r0 += cd.n_reads;
    }
    return KMGPU_OK;
}

extern "C" int kmgpu_batch_read_medians(kmgpu_t* h, const kmgpu_batch_t* b, uint16_t* median_out, float* average_out, float* stddev_out,
                                        uint32_t* n_kmers_out)
{
    if (!h || !b) return fail(KMGPU_EINVAL, "null argument");
    if (b->device != h->device) return fail(KMGPU_EINVAL, "batch lives on another device");
    if (b->ksize != h->k) return fail(KMGPU_EINVAL, "batch was cut for k=%d, sketch has k=%d", b->ksize, h->k);
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    if (h->kind == BYTE && h->use_bigcount) CKR(sync_big_to_device(h));
    uint32_t nb = (h->kind == BYTE && h->use_bigcount) ? h->n_big_dev : 0;
    uint64_t r0 = 0;
    for (const auto& p : b->pieces) r0 += p.n_reads;
    if (r0 != b->n_reads) return fail(KMGPU_EUNSUPPORTED, "the batch holds a read longer than a device chunk; per-read statistics need whole reads");
    r0 = 0;
    for (const auto& p : b->pieces) {
        ChunkDev cd;
        cd.words = p.words;
        cd.offs = p.offs;
        cd.tfr = p.tfr;
        cd.valid = p.valid;
        cd.n_reads = p.n_reads;
        cd.n_pos = p.n_pos;
        CKR(read_stats_chunk(h, cd, r0, nb, median_out, average_out, stddev_out, n_kmers_out, false, 0, nullptr));
        r0 += p.n_reads;
    }
    return KMGPU_OK;
}

extern "C" int kmgpu_read_medians(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                  uint16_t* median_out, float* average_out, float* stddev_out, uint32_t* n_kmers_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    return per_read_query(h, seqs, offsets, n_reads, flags, median_out, average_out, stddev_out, n_kmers_out, false, 0, nullptr);
}

extern "C" int kmgpu_median_at_least(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                     uint32_t cutoff, uint8_t* out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (!out && n_reads) return fail(KMGPU_EINVAL, "null output");
    return per_read_query(h, seqs, offsets, n_reads, flags, nullptr, nullptr, nullptr, nullptr, true, cutoff, out);
}

extern "C" int kmgpu_trim_batch(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags, uint32_t abund, int below,
                                uint32_t* trim_pos_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets || !trim_pos_out) return fail(KMGPU_EINVAL, "null argument");
    for (uint64_t r = 0; r < n_reads; r++)
        if (offsets[r + 1] - offsets[r] > chunk_bases())
            return fail(KMGPU_EUNSUPPORTED, "read %llu is longer than a device chunk", (unsigned long long)r);
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    if (h->kind == BYTE && h->use_bigcount) CKR(sync_big_to_device(h));
    const uint32_t nb = (h->kind == BYTE && h->use_bigcount) ? h->n_big_dev : 0;
    const HashCfg H{h->hash, h->k};
    std::vector<ChunkPlan> plan;
    plan_chunks(offsets, n_reads, h->k, chunk_bases(), plan);
    uint64_t r0 = 0;
    for (const ChunkPlan& c : plan) {
        ChunkDev cd;
        CKR(stage_chunk(h, seqs, c, flags, &cd, needs_acgt_check(h, flags)));
        CKR(h->d_counts.ensure(std::max<uint32_t>(cd.n_pos, 1)));
        if (cd.n_pos) launch_counts(0, h->dev, H, make_input(cd), h->big_keys.p, h->big_vals.p, nb, h->d_counts.p, nullptr, nullptr, h->stream);
        h->all_launches += 1;
        CKR(trim_counts(h, h->d_counts.p, cd, r0, abund, below, trim_pos_out));
        r0 += cd.n_reads;
    }
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// abundance distribution
// ------------------------------------------------------------------------------------------------------
extern "C" int kmgpu_abundance_distribution(kmgpu_t* counts, kmgpu_t* tracking, const char* seqs, const uint64_t* offsets,
                                            uint64_t n_reads, uint32_t flags, uint64_t* hist)
{
    if (!counts || !tracking || !hist) return fail(KMGPU_EINVAL, "null argument");
    if (counts == tracking) return fail(KMGPU_EINVAL, "tracking sketch must differ from the counting sketch");
    if (counts->device != tracking->device) return fail(KMGPU_EINVAL, "sketches live on different devices");
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets) return fail(KMGPU_EINVAL, "null input");
    kmgpu_sketch* a = counts < tracking ? counts : tracking;
    kmgpu_sketch* b = counts < tracking ? tracking : counts;
    std::lock_guard<std::mutex> ga(a->mu);
    std::lock_guard<std::mutex> gb(b->mu);
    CKR(set_device(counts->device));
    CK(cudaStreamSynchronize(counts->stream));
    if (counts->kind == BYTE && counts->use_bigcount) CKR(sync_big_to_device(counts));
    uint32_t nb = (counts->kind == BYTE && counts->use_bigcount) ? counts->n_big_dev : 0;
    kmgpu_sketch* t = tracking;
    cudaStream_t st = t->stream;
    HashCfg H{counts->hash, counts->k};  // k-mers are hashed by the counting table (hashtable.cc:478-480)
    Pred P;
    memset(&P, 0, sizeof P);
    CKR(t->d_hist.ensure(65536));
    CK(cudaMemsetAsync(t->d_hist.p, 0, 65536 * 8, st));
    std::vector<ChunkPlan> plan;
    plan_chunks(offsets, n_reads, counts->k, chunk_bases(), plan);
    bool acgt = counts->hash == KMGPU_MURMUR && !(flags & KMGPU_CLEAN);
    for (const ChunkPlan& c : plan) {
        ChunkDev cd;
        CKR(stage_chunk(t, seqs, c, flags, &cd, acgt));
        if (cd.n_pos == 0) continue;
        ChunkResult res;
        Input in = make_input(cd);
        const std::vector<Part> one(1, Part{in, 0u, nullptr});
        t->ft_defer = t->ft_on;   // first-touch log: the entries of this chunk carry the k-mers' counts, known below
        int rc = ingest_chunk(t, 0, H, one, P, false, nullptr, &res);
        t->ft_defer = false;
        CKR(rc);
        if (!res.have_newbits || res.n_new == 0) {
            if (t->ft_on) CKR(ft_emit(t, 0, H, one, nullptr));
            continue;
        }
        CKR(t->d_counts.ensure(cd.n_pos));
        launch_counts(0, counts->dev, H, in, counts->big_keys.p, counts->big_vals.p, nb, t->d_counts.p, nullptr, t->d_newbits.p, st);
        k_hist<<<148 * 4, 256, 0, st>>>(t->d_counts.p, t->d_newbits.p, cd.n_pos, t->d_hist.p);
        t->all_launches += 2;
        CK(cudaGetLastError());
        if (t->ft_on) CKR(ft_emit(t, 0, H, one, t->d_counts.p));
    }
    std::vector<unsigned long long> hh(65536);
    CK(cudaMemcpyAsync(hh.data(), t->d_hist.p, 65536 * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < 65536; i++) hist[i] += hh[i];
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// digital normalization
// ------------------------------------------------------------------------------------------------------
// KMGPU_DEBUG: wall clock per phase of normalize_batch / trim_low_abund_pass1 (every phase ends in a synchronisation)
struct NormClock {
    const bool dbg = env_u64("KMGPU_DEBUG", 0) != 0;
    // stage + first test, overlay test, in-between resolution, ingest of the kept reads, host loops;
    // 5..8: parts of the in-between resolution; 9: refinement of trim-low-abund's pass 1
    double t[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    double mark = dbg ? now() : 0;
    static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
    void lap(int i)
    {
        if (!dbg) return;
        const double x = now();
        t[i] += x - mark;
        mark = x;
    }
};

// one bit per read -> d_readbits
static int upload_read_bits(kmgpu_sketch* h, const std::vector<uint8_t>& flag, uint32_t nr)
{
    std::vector<uint32_t> bits((nr + 31) / 32, 0u);
    for (uint32_t r = 0; r < nr; r++)
        if (flag[r]) bits[r >> 5] |= 1u << (r & 31);
    CKR(h->d_readbits.ensure(bits.size()));
    CK(cudaMemcpyAsync(h->d_readbits.p, bits.data(), bits.size() * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // `bits` goes
    return KMGPU_OK;
}

// end of the bundle that starts at read r of a window (pw: the window's pair flags, or null)
static uint32_t bundle_end(const uint8_t* pw, uint32_t nr, uint32_t r)
{
    uint32_t e = r + 1;
    while (e < nr && pw && pw[e - 1]) e++;
    return e;
}

// A window of whole bundles, at most W reads and max_bases bases, from read r0 on; staged on the device.
static int stage_window(kmgpu_sketch* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                        const uint8_t* pair_with_next, uint64_t r0, uint64_t W, ChunkPlan& c, ChunkDev& cd, uint64_t* r1_out)
{
    const uint64_t max_bases = chunk_bases() / 2;
    uint64_t r1 = r0;
    while (r1 < n_reads && r1 - r0 < W && offsets[r1 + 1] - offsets[r0] <= max_bases) r1++;
    if (r1 == r0) r1 = r0 + 1;
    while (r1 < n_reads && pair_with_next && pair_with_next[r1 - 1]) r1++;   // do not cut a pair
    const uint32_t nr = (uint32_t)(r1 - r0);
    c.base0 = offsets[r0];
    c.base1 = offsets[r1];
    c.offs.resize(nr + 1);
    for (uint32_t r = 0; r <= nr; r++) c.offs[r] = (uint32_t)(offsets[r0 + r] - offsets[r0]);
    *r1_out = r1;
    return stage_chunk(h, seqs, c, flags, &cd, needs_acgt_check(h, flags));
}

// Steps 1-3 of digital normalization for one staged window with k-mers (cd.n_pos > 0): keep[r] = 1 iff read r's bundle is kept,
// i.e. consumed in stream order.  h->d_counts keeps step 1's counts (the table at the window's start).  *any_cand: some bundle
// was a candidate (steps 2-3 ran); *n_unsure: in-between reads.  *too_large: the in-between lists would pass 32 bits (refused).
// `fl`: room to reserve for the lists from the start (large calls).
static int norm_window_decide(kmgpu_sketch* h, const ChunkPlan& c, const ChunkDev& cd, const uint8_t* pw, uint32_t cutoff, size_t fl,
                              NormClock& clk, std::vector<uint8_t>& keep, bool* any_cand, uint64_t* n_unsure_out, bool* too_large)
{
    cudaStream_t st = h->stream;
    const HashCfg H{h->hash, h->k};
    const int N = h->nt;
    const uint32_t cap_c = h->kind == BYTE ? 255u : h->kind == NIBBLE ? 15u : 1u;
    const uint32_t nr = cd.n_reads;
    *any_cand = false;
    *n_unsure_out = 0;
    *too_large = false;
    keep.assign(nr, 0);
    Input in = make_input(cd);
    // 1. median_at_least of every read in the table as it is at the window's start
    if (h->kind == BYTE && h->use_bigcount) CKR(sync_big_to_device(h));
    const uint32_t nb = (h->kind == BYTE && h->use_bigcount) ? h->n_big_dev : 0;
    CKR(h->d_counts.ensure(cd.n_pos));
    CKR(h->d_stat_n.ensure(nr));
    CKR(h->d_stat_b.ensure(nr));
    launch_counts(0, h->dev, H, in, h->big_keys.p, h->big_vals.p, nb, h->d_counts.p, nullptr, nullptr, st);
    k_read_stats<<<(nr + 7) / 8, 256, 0, st>>>(h->d_counts.p, cd.offs, nr, h->k, nullptr, nullptr, nullptr, h->d_stat_n.p, cutoff, h->d_stat_b.p);
    h->all_launches += 2;
    CK(cudaGetLastError());
    std::vector<uint8_t> al1(nr), al2;
    CK(cudaMemcpyAsync(al1.data(), h->d_stat_b.p, nr, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    clk.lap(0);
    // candidates: bundles with a read below the cutoff (a read without k-mers never makes its bundle a candidate)
    std::vector<uint8_t> cand(nr, 0);
    uint64_t cand_bases = 0, n_cand = 0;
    for (uint32_t r = 0; r < nr;) {
        const uint32_t e = bundle_end(pw, nr, r);
        bool below = false;
        for (uint32_t q = r; q < e; q++) below |= al1[q] == 0;
        if (below)
            for (uint32_t q = r; q < e; q++) {
                cand[q] = 1;
                cand_bases += c.offs[q + 1] - c.offs[q];
                n_cand++;
            }
        r = e;
    }
    if (!n_cand) return KMGPU_OK;
    *any_cand = true;
    // 2. the same test with every candidate of the window added on top (overlay): still below => kept for good.  The overlay's
    //    counts go to their own buffer.
    CKR(upload_read_bits(h, cand, nr));
    const uint64_t slots = pow2_at_least(2 * cand_bases * (uint64_t)N);
    CKR(h->d_htkeys.ensure(slots));
    CKR(h->d_htvals.ensure(slots));
    CKR(h->d_ocounts.ensure(cd.n_pos));
    CK(cudaMemsetAsync(h->d_htkeys.p, 0xFF, slots * 8, st));
    CK(cudaMemsetAsync(h->d_htvals.p, 0, slots * 4, st));
    in.read_keep = h->d_readbits.p;
    const unsigned gt = n_tiles(cd.n_pos);
    if (H.kind == TWOBIT) k_norm_overlay_add<TWOBIT, 0><<<gt, THREADS, 0, st>>>(h->dev, H, in, h->d_htkeys.p, h->d_htvals.p, slots - 1);
    else k_norm_overlay_add<MURMUR, 0><<<gt, THREADS, 0, st>>>(h->dev, H, in, h->d_htkeys.p, h->d_htvals.p, slots - 1);
#define NORM_COUNTS(KIND)                                                                                                                  \
    do {                                                                                                                                   \
        if (H.kind == TWOBIT) k_norm_counts_overlay<KIND, TWOBIT, 0><<<gt, THREADS, 0, st>>>(h->dev, H, in, h->d_htkeys.p, h->d_htvals.p, slots - 1, h->d_ocounts.p); \
        else k_norm_counts_overlay<KIND, MURMUR, 0><<<gt, THREADS, 0, st>>>(h->dev, H, in, h->d_htkeys.p, h->d_htvals.p, slots - 1, h->d_ocounts.p);                 \
    } while (0)
    if (h->kind == BYTE) NORM_COUNTS(BYTE);
    else if (h->kind == NIBBLE) NORM_COUNTS(NIBBLE);
    else NORM_COUNTS(BIT);
#undef NORM_COUNTS
    k_read_stats<<<(nr + 7) / 8, 256, 0, st>>>(h->d_ocounts.p, cd.offs, nr, h->k, nullptr, nullptr, nullptr, h->d_stat_n.p, cutoff, h->d_stat_b.p);
    h->all_launches += 3;
    CK(cudaGetLastError());
    al2.resize(nr);
    CK(cudaMemcpyAsync(al2.data(), h->d_stat_b.p, nr, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    clk.lap(1);
    std::vector<uint8_t> sure(nr, 0), unsure(nr, 0);
    uint64_t n_unsure = 0, up_total = 0;
    for (uint32_t r = 0; r < nr;) {
        const uint32_t e = bundle_end(pw, nr, r);
        if (cand[r]) {
            bool below = false;
            for (uint32_t q = r; q < e; q++) below |= al2[q] == 0;
            for (uint32_t q = r; q < e; q++) {
                (below ? sure : unsure)[q] = 1;
                if (!below) {
                    n_unsure++;
                    const uint32_t len = c.offs[q + 1] - c.offs[q];
                    if (len >= (uint32_t)h->k) up_total += len - h->k + 1;
                }
            }
        }
        r = e;
    }
    keep = sure;
    *n_unsure_out = n_unsure;
    if (n_unsure) {
        // 3. in-between bundles: the state each of them meets is the window's start + the candidates kept before it.
        //    Gather, for every k-mer of theirs, the counters at the window's start and the touches of its bins by the
        //    window's candidates (position, read); then decide in rounds on the device (k_norm_resolve).
        h->n_norm_unsure += n_unsure;
        std::vector<uint32_t> upos, meta_ub, meta_start, meta_ur, meta_read;
        upos.reserve(up_total);
        meta_ur.push_back(0);
        for (uint32_t r = 0; r < nr;) {
            const uint32_t e = bundle_end(pw, nr, r);
            if (unsure[r]) {
                meta_ub.push_back((uint32_t)meta_read.size());
                meta_start.push_back(c.offs[r]);
                for (uint32_t q = r; q < e; q++) {
                    const uint32_t s0 = c.offs[q], len = c.offs[q + 1] - s0;
                    for (uint32_t i = 0; i + h->k <= len; i++) upos.push_back(s0 + i);
                    meta_read.push_back(q);
                    meta_ur.push_back((uint32_t)upos.size());
                }
            }
            r = e;
        }
        meta_ub.push_back((uint32_t)meta_read.size());
        const uint32_t n_up = (uint32_t)upos.size(), n_ub = (uint32_t)meta_start.size();
        std::vector<uint8_t> state(nr, 0);
        for (uint32_t r = 0; r < nr; r++) state[r] = sure[r] ? 1 : unsure[r] ? 2 : 0;
        double t_sub = clk.dbg ? NormClock::now() : 0;
        auto sub = [&](int i) {
            if (!clk.dbg) return;
            const double t = NormClock::now();
            clk.t[i] += t - t_sub;
            t_sub = t;
        };
        sub(5);   // host: the lists of the in-between bundles
        if (n_up) {
            const uint64_t slots2 = pow2_at_least(2 * (uint64_t)n_up * N);
            if (slots2 > (1ull << 32)) {
                *too_large = true;
                return fail(KMGPU_EUNSUPPORTED, "normalize_batch: window too large");
            }
            // one upload: upos | ub_first | ub_start | ur_first | ur_read
            std::vector<uint32_t> pack;
            pack.reserve((size_t)n_up + meta_ub.size() + meta_start.size() + meta_ur.size() + meta_read.size());
            pack.insert(pack.end(), upos.begin(), upos.end());
            const size_t o_ub = pack.size();
            pack.insert(pack.end(), meta_ub.begin(), meta_ub.end());
            const size_t o_st = pack.size();
            pack.insert(pack.end(), meta_start.begin(), meta_start.end());
            const size_t o_ur = pack.size();
            pack.insert(pack.end(), meta_ur.begin(), meta_ur.end());
            const size_t o_rd = pack.size();
            pack.insert(pack.end(), meta_read.begin(), meta_read.end());
            // large calls: room for a typical window's in-between reads from the start (growing these buffers window
            // by window costs a cudaFree + cudaMalloc each time, milliseconds apiece on some hosts)
            CKR(h->d_upos.ensure(std::max(pack.size(), fl + fl / 8)));
            CKR(h->d_nslot.ensure(std::max((size_t)n_up, fl) * N));
            CKR(h->d_uc0.ensure(std::max((size_t)n_up, fl) * N));
            CKR(h->d_evkeys.ensure(std::max<uint64_t>(slots2, pow2_at_least(2 * (uint64_t)fl * N))));
            CKR(h->d_ncnt.ensure(std::max<uint64_t>(slots2, pow2_at_least(2 * (uint64_t)fl * N))));
            CKR(h->d_nfill.ensure(std::max<uint64_t>(slots2, pow2_at_least(2 * (uint64_t)fl * N))));
            CKR(h->d_nstate.ensure(std::max<size_t>(nr, fl ? (size_t)1 << 17 : 0)));
            CK(cudaMemcpyAsync(h->d_upos.p, pack.data(), pack.size() * 4, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(h->d_nstate.p, state.data(), nr, cudaMemcpyHostToDevice, st));
            CK(cudaMemsetAsync(h->d_evkeys.p, 0xFF, slots2 * 8, st));
            CK(cudaMemsetAsync(h->d_ncnt.p, 0, slots2 * 4, st));
            CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
            uint64_t* keys2 = reinterpret_cast<uint64_t*>(h->d_evkeys.p);
            Input in0 = make_input(cd);
#define NORM_GATHER(KIND)                                                                                                                                    \
    do {                                                                                                                                                     \
        if (H.kind == TWOBIT) k_norm_gather<KIND, TWOBIT><<<(n_up + 255) / 256, 256, 0, st>>>(h->dev, H, in0, h->d_upos.p, n_up, h->d_nslot.p, h->d_uc0.p, keys2, slots2 - 1); \
        else k_norm_gather<KIND, MURMUR><<<(n_up + 255) / 256, 256, 0, st>>>(h->dev, H, in0, h->d_upos.p, n_up, h->d_nslot.p, h->d_uc0.p, keys2, slots2 - 1);               \
    } while (0)
            if (h->kind == BYTE) NORM_GATHER(BYTE);
            else if (h->kind == NIBBLE) NORM_GATHER(NIBBLE);
            else NORM_GATHER(BIT);
#undef NORM_GATHER
            Input inc = make_input(cd);
            inc.read_keep = h->d_readbits.p;   // still the candidates' bits (uploaded for the overlay)
            if (H.kind == TWOBIT) k_norm_hits<TWOBIT, 0, 0><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_ncnt.p, nullptr);
            else k_norm_hits<MURMUR, 0, 0><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_ncnt.p, nullptr);
            k_norm_hit_offsets<<<148 * 8, 256, 0, st>>>(h->d_ncnt.p, h->d_nfill.p, slots2, &h->d_ctrl->n_events);
            h->all_launches += 3;
            CK(cudaGetLastError());
            CKR(read_ctrl(h));   // synchronises: the host vectors above may go
            sub(6);   // uploads, gather, counting pass of the hits
            const uint64_t n_hits = h->h_ctrl->n_events;
            if (n_hits >= (1ull << 32)) {
                *too_large = true;
                return fail(KMGPU_EUNSUPPORTED, "normalize_batch: window too large");
            }
            CKR(h->d_nhits.ensure(std::max<uint64_t>(std::max<uint64_t>(n_hits, 1), 8 * (uint64_t)fl)));
            if (H.kind == TWOBIT) k_norm_hits<TWOBIT, 0, 1><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_nfill.p, h->d_nhits.p);
            else k_norm_hits<MURMUR, 0, 1><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_nfill.p, h->d_nhits.p);
            h->all_launches += 1;
            NormResolve R;
            R.ub_first = h->d_upos.p + o_ub;
            R.ub_start = h->d_upos.p + o_st;
            R.ur_first = h->d_upos.p + o_ur;
            R.ur_read = h->d_upos.p + o_rd;
            R.slot = h->d_nslot.p;
            R.c0 = h->d_uc0.p;
            R.cnt = h->d_ncnt.p;
            R.fill = h->d_nfill.p;
            R.hits = h->d_nhits.p;
            R.state = h->d_nstate.p;
            R.n_tables = N;
            R.cutoff = cutoff;
            R.cap = cap_c;
            unsigned int* n_left = reinterpret_cast<unsigned int*>(&h->d_ctrl->n_events);
            if (clk.dbg) CK(cudaStreamSynchronize(st));
            sub(7);   // fill pass of the hits
            for (uint64_t round = 0;; round++) {
                // two rounds per look at the counter (a round is a few microseconds, the look a round trip)
                CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
                k_norm_resolve<<<(n_ub + 7) / 8, 256, 0, st>>>(R, n_ub, n_left);
                CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
                k_norm_resolve<<<(n_ub + 7) / 8, 256, 0, st>>>(R, n_ub, n_left);
                h->all_launches += 2;
                h->n_norm_rounds += 2;
                CK(cudaGetLastError());
                CKR(read_ctrl(h));
                if (h->h_ctrl->n_events == 0) break;
                if (round > n_ub) return fail(KMGPU_ECUDA, "normalize_batch: the in-between resolution does not converge");
            }
            CK(cudaMemcpyAsync(state.data(), h->d_nstate.p, nr, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            sub(8);   // rounds
        } else {
            // in-between bundles without a single k-mer cannot be "below": never kept (they were no candidates at all)
            for (uint32_t r = 0; r < nr; r++)
                if (state[r] == 2) state[r] = 0;
        }
        for (uint32_t r = 0; r < nr; r++) keep[r] = state[r] == 1;
    }
    clk.lap(2);
    return KMGPU_OK;
}

// 4. the kept reads of a window are consumed in stream order (one ordinary ingest with a read mask); adds the k-mers consumed
static int norm_window_ingest(kmgpu_sketch* h, const ChunkDev& cd, const std::vector<uint8_t>& keep, uint64_t* n_kmers)
{
    const uint32_t nr = cd.n_reads;
    uint64_t nk_reads = 0;
    for (uint32_t r = 0; r < nr; r++) nk_reads += keep[r];
    if (!nk_reads) return KMGPU_OK;
    CKR(upload_read_bits(h, keep, nr));
    Input ink = make_input(cd);
    ink.read_keep = h->d_readbits.p;
    ChunkResult res;
    Pred P0;
    memset(&P0, 0, sizeof P0);
    CKR(ingest_chunk(h, 0, HashCfg{h->hash, h->k}, {Part{ink, 0u, nullptr}}, P0, false, nullptr, &res));
    *n_kmers += res.n_kmers;
    return KMGPU_OK;
}

extern "C" int kmgpu_normalize_batch(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                     const uint8_t* pair_with_next, uint32_t cutoff, uint8_t* keep_out, uint64_t* n_kept_out,
                                     uint64_t* n_kmers_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n_kept_out) *n_kept_out = 0;
    if (n_kmers_out) *n_kmers_out = 0;
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets || !keep_out) return fail(KMGPU_EINVAL, "null argument");
    if (h->kind == BYTE && h->use_bigcount && cutoff > 255)
        return fail(KMGPU_EUNSUPPORTED, "normalize_batch: cutoffs above 255 on a bigcount table are not supported");
    for (uint64_t r = 0; r < n_reads; r++)
        if (offsets[r + 1] - offsets[r] > chunk_bases() / 4)
            return fail(KMGPU_EUNSUPPORTED, "read %llu is too long for a normalization window", (unsigned long long)r);
    if (pair_with_next && pair_with_next[n_reads - 1]) return fail(KMGPU_EINVAL, "the last read cannot be paired with a next one");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    // reads per window: fixed by KMGPU_NORM_WINDOW, else adapted so that only a small share of a window's bundles is "in between"
    // (their number grows with the coverage a window adds; they are resolved one by one on the host)
    const uint64_t W_fixed = env_u64("KMGPU_NORM_WINDOW", 0);
    uint64_t W = W_fixed ? std::max<uint64_t>(2, W_fixed) : 32768;
    uint64_t n_windows = 0;
    const uint64_t unsure0 = h->n_norm_unsure, rounds0 = h->n_norm_rounds;
    NormClock clk;
    const size_t fl = n_reads >= 100000 ? ((size_t)1 << 21) : 0;
    uint64_t kept_total = 0, kmers_total = 0;
    std::vector<uint8_t> keep;
    for (uint64_t r0 = 0; r0 < n_reads;) {
        ChunkPlan c;
        ChunkDev cd;
        uint64_t r1;
        CKR(stage_window(h, seqs, offsets, n_reads, flags, pair_with_next, r0, W, c, cd, &r1));
        const uint32_t nr = (uint32_t)(r1 - r0);
        n_windows++;
        keep.assign(nr, 0);
        if (cd.n_pos) {
            bool any_cand, too_large;
            uint64_t n_unsure;
            CKR(norm_window_decide(h, c, cd, pair_with_next ? pair_with_next + r0 : nullptr, cutoff, fl, clk, keep, &any_cand, &n_unsure,
                                   &too_large));
            if (any_cand) {
                if (!W_fixed) {
                    // a window costs ~1 ms of launches and round trips whatever its size; the in-between bundles (their number grows
                    // with the square of the window) cost a few rounds of k_norm_resolve over their k-mers
                    if (n_unsure > 8192) W = std::max<uint64_t>(2048, W / 2);
                    else if (n_unsure < 2048) W = std::min<uint64_t>(1u << 17, W * 2);
                }
                CKR(norm_window_ingest(h, cd, keep, &kmers_total));
                for (uint32_t r = 0; r < nr; r++) kept_total += keep[r];
                clk.lap(3);
            }
        }
        memcpy(keep_out + r0, keep.data(), nr);
        clk.lap(4);
        r0 = r1;
    }
    if (n_kept_out) *n_kept_out = kept_total;
    if (n_kmers_out) *n_kmers_out = kmers_total;
    if (clk.dbg)
        fprintf(stderr, "[kmgpu] normalize_batch: %llu reads in %llu windows (last %llu reads), %llu in-between reads, %llu resolve rounds; "
                        "seconds: first test %.3f, overlay test %.3f, in-between %.3f (lists %.3f, gather + count %.3f, fill %.3f, rounds %.3f), ingest %.3f, other %.3f\n",
                (unsigned long long)n_reads, (unsigned long long)n_windows, (unsigned long long)W,
                (unsigned long long)(h->n_norm_unsure - unsure0), (unsigned long long)(h->n_norm_rounds - rounds0), clk.t[0], clk.t[1], clk.t[2],
                clk.t[5], clk.t[6], clk.t[7], clk.t[8], clk.t[3], clk.t[4]);
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// trim-low-abund (scripts/trim-low-abund.py:196-271, khmer/trimming.py:36-66)
// ------------------------------------------------------------------------------------------------------
extern "C" int kmgpu_trim_low_abund_pass1(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                          const uint8_t* pair_with_next, uint32_t trim_at_coverage, uint32_t cutoff,
                                          uint32_t diginorm_coverage, uint8_t* action_out, uint32_t* trim_pos_out, uint64_t* n_kmers_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n_kmers_out) *n_kmers_out = 0;
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets || !action_out || !trim_pos_out) return fail(KMGPU_EINVAL, "null argument");
    const uint32_t Z = trim_at_coverage, C = cutoff, D = diginorm_coverage;
    if (h->kind == BYTE && h->use_bigcount && (Z > 255 || C > 255 || D > 255))
        return fail(KMGPU_EUNSUPPORTED, "trim_low_abund_pass1: coverages and cutoffs above 255 on a bigcount table are not supported");
    for (uint64_t r = 0; r < n_reads; r++)
        if (offsets[r + 1] - offsets[r] > chunk_bases() / 4)
            return fail(KMGPU_EUNSUPPORTED, "read %llu is too long for a trimming window", (unsigned long long)r);
    if (pair_with_next && pair_with_next[n_reads - 1]) return fail(KMGPU_EINVAL, "the last read cannot be paired with a next one");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    const HashCfg H{h->hash, h->k};
    const int N = h->nt;
    const uint32_t cap_c = h->kind == BYTE ? 255u : h->kind == NIBBLE ? 15u : 1u;
    // a bundle is consumed iff some read of it has median_at_least(min(Z, D)) false: normalization's keep rule.  The others are
    // skipped (med >= D) or trimmed (Z <= med < D); with D <= Z all of them are skipped.  Their judgement compares counts with C
    // (trim) and D (the skip test when Z < D): counts at or above R = the larger of the two need no refinement.
    const uint32_t cut = D ? std::min(Z, D) : Z;
    const bool judge = !(D && D <= Z);
    const bool test_d = D && Z < D;
    const uint32_t R = test_d ? std::max(C, D) : C;
    const uint64_t W_fixed = env_u64("KMGPU_NORM_WINDOW", 0);
    uint64_t W = W_fixed ? std::max<uint64_t>(2, W_fixed) : 32768;
    uint64_t n_windows = 0, n_refined = 0;
    NormClock clk;
    const size_t fl = n_reads >= 100000 ? ((size_t)1 << 21) : 0;
    uint64_t kmers_total = 0;
    std::vector<uint8_t> keep, al;
    std::vector<uint32_t> bstart;
    for (uint64_t r0 = 0; r0 < n_reads;) {
        ChunkPlan c;
        ChunkDev cd;
        uint64_t r1;
        CKR(stage_window(h, seqs, offsets, n_reads, flags, pair_with_next, r0, W, c, cd, &r1));
        const uint32_t nr = (uint32_t)(r1 - r0);
        const uint8_t* pw = pair_with_next ? pair_with_next + r0 : nullptr;
        uint8_t* act = action_out + r0;
        uint32_t* tpos = trim_pos_out + r0;
        n_windows++;
        keep.assign(nr, 0);
        bool too_large = false;
        if (cd.n_pos) {
            bool any_cand;
            uint64_t n_unsure;
            const int rc = norm_window_decide(h, c, cd, pw, cut, fl, clk, keep, &any_cand, &n_unsure, &too_large);
            if (rc != KMGPU_OK && !too_large) return rc;
            if (!too_large && any_cand && !W_fixed) {
                if (n_unsure > 8192) W = std::max<uint64_t>(2048, W / 2);
                else if (n_unsure < 2048) W = std::min<uint64_t>(1u << 17, W * 2);
            }
        }
        // reads that were not consumed: their judgement.  Positions to refine: those of such reads whose window-start count is
        // below R, when a consumed bundle may come before them.
        uint64_t n_cons = 0, cap_up = 0;
        bool any_judged = false;
        bstart.assign(nr, ~0u);
        for (uint32_t r = 0; r < nr && !too_large;) {
            const uint32_t e = bundle_end(pw, nr, r);
            for (uint32_t q = r; q < e; q++) {
                const uint32_t len = c.offs[q + 1] - c.offs[q];
                if (keep[q]) n_cons++;
                else if (len >= (uint32_t)h->k) {
                    bstart[q] = c.offs[r];
                    cap_up += len - h->k + 1;
                    any_judged = true;
                }
            }
            r = e;
        }
        if (!too_large && judge && any_judged) {
            if (n_cons && R) {
                CKR(upload_read_bits(h, keep, nr));
                CKR(h->d_upos.ensure(2 * cap_up));
                CKR(h->d_nstate.ensure(4ull * nr));
                uint32_t* d_bstart = reinterpret_cast<uint32_t*>(h->d_nstate.p);
                CK(cudaMemcpyAsync(d_bstart, bstart.data(), 4ull * nr, cudaMemcpyHostToDevice, st));
                CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
                k_tla_refine_list<<<(nr + 7) / 8, 256, 0, st>>>(h->d_counts.p, cd.offs, nr, h->k, d_bstart, R, h->d_upos.p, h->d_upos.p + cap_up,
                                                               &h->d_ctrl->n_events);
                h->all_launches += 1;
                CK(cudaGetLastError());
                CKR(read_ctrl(h));
                const uint64_t n_up = h->h_ctrl->n_events;
                const uint64_t slots2 = pow2_at_least(2 * n_up * N);
                if (slots2 > (1ull << 32)) too_large = true;
                if (n_up && !too_large) {
                    n_refined += n_up;
                    CKR(h->d_nslot.ensure(n_up * N));
                    CKR(h->d_uc0.ensure(n_up * N));
                    CKR(h->d_evkeys.ensure(slots2));
                    CKR(h->d_ncnt.ensure(slots2));
                    CKR(h->d_nfill.ensure(slots2));
                    CK(cudaMemsetAsync(h->d_evkeys.p, 0xFF, slots2 * 8, st));
                    CK(cudaMemsetAsync(h->d_ncnt.p, 0, slots2 * 4, st));
                    CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
                    uint64_t* keys2 = reinterpret_cast<uint64_t*>(h->d_evkeys.p);
                    const Input in0 = make_input(cd);
                    const uint32_t nu = (uint32_t)n_up;
#define TLA_GATHER(KIND)                                                                                                                                    \
    do {                                                                                                                                                    \
        if (H.kind == TWOBIT) k_norm_gather<KIND, TWOBIT><<<(nu + 255) / 256, 256, 0, st>>>(h->dev, H, in0, h->d_upos.p, nu, h->d_nslot.p, h->d_uc0.p, keys2, slots2 - 1); \
        else k_norm_gather<KIND, MURMUR><<<(nu + 255) / 256, 256, 0, st>>>(h->dev, H, in0, h->d_upos.p, nu, h->d_nslot.p, h->d_uc0.p, keys2, slots2 - 1);               \
    } while (0)
                    if (h->kind == BYTE) TLA_GATHER(BYTE);
                    else if (h->kind == NIBBLE) TLA_GATHER(NIBBLE);
                    else TLA_GATHER(BIT);
#undef TLA_GATHER
                    Input inc = make_input(cd);
                    inc.read_keep = h->d_readbits.p;   // the consumed reads
                    const unsigned gt = n_tiles(cd.n_pos);
                    if (H.kind == TWOBIT) k_norm_hits<TWOBIT, 0, 0><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_ncnt.p, nullptr);
                    else k_norm_hits<MURMUR, 0, 0><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_ncnt.p, nullptr);
                    k_norm_hit_offsets<<<148 * 8, 256, 0, st>>>(h->d_ncnt.p, h->d_nfill.p, slots2, &h->d_ctrl->n_events);
                    h->all_launches += 3;
                    CK(cudaGetLastError());
                    CKR(read_ctrl(h));
                    const uint64_t n_hits = h->h_ctrl->n_events;
                    if (n_hits >= (1ull << 32)) too_large = true;
                    if (!too_large) {
                        CKR(h->d_nhits.ensure(std::max<uint64_t>(n_hits, 1)));
                        if (H.kind == TWOBIT) k_norm_hits<TWOBIT, 0, 1><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_nfill.p, h->d_nhits.p);
                        else k_norm_hits<MURMUR, 0, 1><<<gt, THREADS, 0, st>>>(h->dev, H, inc, keys2, slots2 - 1, h->d_nfill.p, h->d_nhits.p);
                        k_tla_refine<<<(nu + 255) / 256, 256, 0, st>>>(h->d_upos.p, h->d_upos.p + cap_up, nu, h->d_nslot.p, h->d_uc0.p, h->d_ncnt.p,
                                                                      h->d_nfill.p, h->d_nhits.p, N, R, cap_c, h->d_counts.p);
                        h->all_launches += 2;
                        CK(cudaGetLastError());
                    }
                }
            }
            if (!too_large) {
                // d_counts: every judged read's counts as its bundle meets the table (exact below R)
                if (test_d) {
                    al.resize(nr);
                    CKR(read_stats_counts(h, h->d_counts.p, cd, 0, nullptr, nullptr, nullptr, nullptr, true, D, al.data()));
                }
                CKR(trim_counts(h, h->d_counts.p, cd, 0, C, 0, tpos));
                clk.lap(9);
            }
        }
        if (too_large) {
            // the refinement's lists would pass 32 bits: the same reads in smaller windows (the table has not changed)
            if (nr < 2) return fail(KMGPU_EUNSUPPORTED, "trim_low_abund_pass1: a window of one bundle is too large");
            W = std::max<uint64_t>(1, nr / 2);
            continue;
        }
        for (uint32_t r = 0; r < nr;) {
            const uint32_t e = bundle_end(pw, nr, r);
            bool skip = !judge;
            if (test_d) {
                skip = true;
                for (uint32_t q = r; q < e; q++)
                    if (!keep[q] && bstart[q] != ~0u && al[q] == 0) skip = false;
            }
            for (uint32_t q = r; q < e; q++) {
                const bool kmers = c.offs[q + 1] - c.offs[q] >= (uint32_t)h->k;
                act[q] = !kmers ? KMGPU_TLA_DROP : keep[q] ? KMGPU_TLA_SAVE : skip ? KMGPU_TLA_SKIP : KMGPU_TLA_TRIM;
                if (act[q] != KMGPU_TLA_TRIM) tpos[q] = 0;
            }
            r = e;
        }
        CKR(norm_window_ingest(h, cd, keep, &kmers_total));
        clk.lap(3);
        r0 = r1;
    }
    if (n_kmers_out) *n_kmers_out = kmers_total;
    if (clk.dbg)
        fprintf(stderr, "[kmgpu] trim_low_abund_pass1: %llu reads in %llu windows (last %llu reads), %llu refined positions; "
                        "seconds: first test %.3f, overlay test %.3f, in-between %.3f, refinement + judgement %.3f, ingest %.3f, other %.3f\n",
                (unsigned long long)n_reads, (unsigned long long)n_windows, (unsigned long long)W, (unsigned long long)n_refined,
                clk.t[0], clk.t[1], clk.t[2], clk.t[9], clk.t[3], clk.t[4]);
    return KMGPU_OK;
}

extern "C" int kmgpu_trim_low_abund_pass2(kmgpu_t* h, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                          const uint8_t* pair_with_next, uint32_t trim_at_coverage, uint32_t cutoff, int variable_coverage,
                                          uint8_t* action_out, uint32_t* trim_pos_out)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets || !action_out || !trim_pos_out) return fail(KMGPU_EINVAL, "null argument");
    for (uint64_t r = 0; r < n_reads; r++)
        if (offsets[r + 1] - offsets[r] > chunk_bases())
            return fail(KMGPU_EUNSUPPORTED, "read %llu is longer than a device chunk", (unsigned long long)r);
    if (pair_with_next && pair_with_next[n_reads - 1]) return fail(KMGPU_EINVAL, "the last read cannot be paired with a next one");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    if (h->kind == BYTE && h->use_bigcount) CKR(sync_big_to_device(h));
    const uint32_t nb = (h->kind == BYTE && h->use_bigcount) ? h->n_big_dev : 0;
    const HashCfg H{h->hash, h->k};
    // one count per k-mer: median_at_least (variable coverage) and the trim scan read the same counts
    std::vector<uint8_t> al(variable_coverage ? n_reads : 0);
    std::vector<ChunkPlan> plan;
    plan_chunks(offsets, n_reads, h->k, chunk_bases(), plan);
    uint64_t r0 = 0;
    for (const ChunkPlan& c : plan) {
        ChunkDev cd;
        CKR(stage_chunk(h, seqs, c, flags, &cd, needs_acgt_check(h, flags)));
        if (variable_coverage) {
            CKR(read_stats_chunk(h, cd, r0, nb, nullptr, nullptr, nullptr, nullptr, true, trim_at_coverage, al.data()));
        } else {
            CKR(h->d_counts.ensure(std::max<uint32_t>(cd.n_pos, 1)));
            if (cd.n_pos) launch_counts(0, h->dev, H, make_input(cd), h->big_keys.p, h->big_vals.p, nb, h->d_counts.p, nullptr, nullptr, h->stream);
            h->all_launches += 1;
        }
        CKR(trim_counts(h, h->d_counts.p, cd, r0, cutoff, 0, trim_pos_out));
        r0 += cd.n_reads;
    }
    // bundles: ReadBundle.coverages_at_least (khmer/utils.py:178-180) over the reads with k-mers
    for (uint64_t r = 0; r < n_reads;) {
        uint64_t e = r + 1;
        while (e < n_reads && pair_with_next && pair_with_next[e - 1]) e++;
        bool trim = true;
        if (variable_coverage)
            for (uint64_t q = r; q < e; q++) trim &= al[q] != 0;
        for (uint64_t q = r; q < e; q++) {
            const bool kmers = offsets[q + 1] - offsets[q] >= (uint64_t)h->k;
            action_out[q] = !kmers ? KMGPU_TLA_DROP : trim ? KMGPU_TLA_TRIM : KMGPU_TLA_KEEP;
            if (action_out[q] != KMGPU_TLA_TRIM) trim_pos_out[q] = 0;
        }
        r = e;
    }
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// merges
// ------------------------------------------------------------------------------------------------------
static int recount_occupied_locked(kmgpu_sketch* h)
{
    h->satbits_valid = false;  // callers have just rewritten table words (merge / reduce / gather)
    cudaStream_t st = h->stream;
    CK(cudaMemsetAsync(&h->d_ctrl->n_z0, 0, sizeof(unsigned long long), st));
    uint64_t nw = h->alloc_bytes[0] / 4;
    unsigned g = (unsigned)std::min<uint64_t>((nw + 255) / 256, 148 * 16);
    k_count_occupied<<<g, 256, 0, st>>>(h->kind, reinterpret_cast<const uint32_t*>(h->dev.tables[0]), nw, &h->d_ctrl->n_z0);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CKR(read_ctrl(h));
    h->n_occupied = h->h_ctrl->n_z0;
    return KMGPU_OK;
}

extern "C" int kmgpu_recount_occupied(kmgpu_t* h)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    return recount_occupied_locked(h);
}

static bool same_shape(const kmgpu_sketch* a, const kmgpu_sketch* b)
{
    if (a->kind != b->kind || a->nt != b->nt) return false;
    for (int i = 0; i < a->nt; i++)
        if (a->sizes[i] != b->sizes[i]) return false;
    return true;
}

extern "C" int kmgpu_merge(kmgpu_t* dst, kmgpu_t* src)
{
    if (!dst || !src) return fail(KMGPU_EINVAL, "null handle");
    if (dst == src) return fail(KMGPU_EINVAL, "cannot merge a sketch into itself");
    if (!same_shape(dst, src)) return fail(KMGPU_ESHAPE, "both nodegraphs must have same table sizes");  // storage.cc:65-67
    kmgpu_sketch* a = dst < src ? dst : src;
    kmgpu_sketch* b = dst < src ? src : dst;
    std::lock_guard<std::mutex> ga(a->mu);
    std::lock_guard<std::mutex> gb(b->mu);
    if (dst->device != src->device) {
        int can = 0;
        CK(cudaDeviceCanAccessPeer(&can, dst->device, src->device));
        if (!can) return fail(KMGPU_EUNSUPPORTED, "devices %d and %d have no peer access", dst->device, src->device);
        CKR(set_device(dst->device));
        cudaError_t e = cudaDeviceEnablePeerAccess(src->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
        cudaGetLastError();
    }
    CKR(set_device(src->device));
    CK(cudaStreamSynchronize(src->stream));
    CKR(set_device(dst->device));
    for (int i = 0; i < dst->nt; i++) {
        uint64_t nw = dst->alloc_bytes[i] / 4;
        unsigned g = (unsigned)std::min<uint64_t>((nw + 255) / 256, 148 * 16);
        k_merge<<<g, 256, 0, dst->stream>>>(dst->kind, reinterpret_cast<uint32_t*>(dst->dev.tables[i]),
                                            reinterpret_cast<const uint32_t*>(src->dev.tables[i]), nw);
        dst->all_launches += 1;
    }
    CK(cudaGetLastError());
    return recount_occupied_locked(dst);
}

// ------------------------------------------------------------------------------------------------------
// multi-GPU: replicated sketches folded over NVLink peer memory
// ------------------------------------------------------------------------------------------------------
extern "C" int kmgpu_ipc_export(kmgpu_t* h, uint8_t* handles)
{
    if (!h || !handles) return fail(KMGPU_EINVAL, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == KMGPU_IPC_HANDLE_BYTES, "IPC handle size");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    for (int i = 0; i < h->nt; i++) {
        cudaIpcMemHandle_t mh;
        CK(cudaIpcGetMemHandle(&mh, h->dev.tables[i]));
        memcpy(handles + (size_t)i * KMGPU_IPC_HANDLE_BYTES, &mh, KMGPU_IPC_HANDLE_BYTES);
    }
    return KMGPU_OK;
}

extern "C" int kmgpu_ipc_attach(kmgpu_t* h, int rank, int world, const uint8_t* all_handles)
{
    if (!h || !all_handles) return fail(KMGPU_EINVAL, "null argument");
    if (world < 1 || world > MAX_WORLD || rank < 0 || rank >= world) return fail(KMGPU_EINVAL, "bad rank/world %d/%d", rank, world);
    kmgpu_ipc_detach(h);
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    h->rank = rank;
    h->world = world;
    h->peers.assign(world, Peer());
    for (int q = 0; q < world; q++) {
        for (int i = 0; i < h->nt; i++) {
            if (q == rank) {
                h->peers[q].tables[i] = h->dev.tables[i];
                continue;
            }
            cudaIpcMemHandle_t mh;
            memcpy(&mh, all_handles + ((size_t)q * h->nt + i) * KMGPU_IPC_HANDLE_BYTES, KMGPU_IPC_HANDLE_BYTES);
            void* p = nullptr;
            CK(cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess));
            h->peers[q].tables[i] = (uint8_t*)p;
        }
    }
    h->peers_ipc = true;
    return KMGPU_OK;
}

extern "C" int kmgpu_ipc_detach(kmgpu_t* h)
{
    if (!h) return KMGPU_OK;
    std::lock_guard<std::mutex> g(h->mu);
    if (h->peers_ipc) {
        cudaSetDevice(h->device);
        for (int q = 0; q < (int)h->peers.size(); q++) {
            if (q == h->rank) continue;
            for (int i = 0; i < h->nt; i++)
                if (h->peers[q].tables[i]) cudaIpcCloseMemHandle(h->peers[q].tables[i]);
        }
    }
    h->peers.clear();
    h->peers_ipc = false;
    h->rank = 0;
    h->world = 1;
    return KMGPU_OK;
}

static void slice_words(uint64_t n_words, int world, int r, uint64_t* w0, uint64_t* w1)
{
    uint64_t per = (n_words + world - 1) / world;
    per = (per + 3) & ~3ull;  // 16-byte granules
    *w0 = std::min<uint64_t>(n_words, per * r);
    *w1 = std::min<uint64_t>(n_words, per * (r + 1));
}

extern "C" int kmgpu_slice_range(uint64_t n_words, int world, int rank, uint64_t* w0, uint64_t* w1)
{
    if (world < 1 || rank < 0 || rank >= world || !w0 || !w1) return fail(KMGPU_EINVAL, "bad rank/world %d/%d", rank, world);
    slice_words(n_words, world, rank, w0, w1);
    return KMGPU_OK;
}

// rank r folds word slice r of every peer's tables into its own copy
static int reduce_scatter_locked(kmgpu_sketch* h)
{
    CKR(set_device(h->device));
    for (int i = 0; i < h->nt; i++) {
        uint64_t nw = h->alloc_bytes[i] / 4, w0, w1;
        slice_words(nw, h->world, h->rank, &w0, &w1);
        if (w1 <= w0) continue;
        PeerPtrs pp;
        pp.n = 0;
        for (int q = 0; q < h->world; q++) {   // eight peers per pass
            if (q != h->rank) pp.p[pp.n++] = reinterpret_cast<const uint32_t*>(h->peers[q].tables[i]);
            if (pp.n == 8 || (q == h->world - 1 && pp.n)) {
                unsigned g = (unsigned)std::min<uint64_t>((w1 - w0 + 255) / 256, 148 * 16);
                k_merge_peers<<<g, 256, 0, h->stream>>>(h->kind, reinterpret_cast<uint32_t*>(h->dev.tables[i]), pp, w0, w1);
                h->all_launches += 1;
                pp.n = 0;
            }
        }
    }
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return KMGPU_OK;
}

// rank r pulls every other slice from its owner
static int all_gather_locked(kmgpu_sketch* h)
{
    CKR(set_device(h->device));
    for (int i = 0; i < h->nt; i++) {
        uint64_t nw = h->alloc_bytes[i] / 4;
        for (int q = 0; q < h->world; q++) {
            if (q == h->rank) continue;
            uint64_t w0, w1;
            slice_words(nw, h->world, q, &w0, &w1);
            if (w1 <= w0) continue;
            CK(cudaMemcpyAsync(h->dev.tables[i] + w0 * 4, h->peers[q].tables[i] + w0 * 4, (w1 - w0) * 4, cudaMemcpyDefault, h->stream));
        }
    }
    CK(cudaStreamSynchronize(h->stream));
    return recount_occupied_locked(h);
}

extern "C" int kmgpu_reduce_scatter_peers(kmgpu_t* h)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->peers.empty()) return fail(KMGPU_EINVAL, "no peers attached");
    if (h->kind == BYTE && h->use_bigcount)
        return fail(KMGPU_EUNSUPPORTED, "replicas cannot be merged with bigcount on: which replica saw a counter's 255th touch is not "
                                        "recoverable (turn bigcount off, or shard the sketch by address)");
    return reduce_scatter_locked(h);
}

extern "C" int kmgpu_all_gather_peers(kmgpu_t* h)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->peers.empty()) return fail(KMGPU_EINVAL, "no peers attached");
    return all_gather_locked(h);
}

extern "C" int kmgpu_first_touch_resolve(kmgpu_t* h, uint64_t* n_new_out, uint64_t* n_local_out, uint64_t* hist);

// single-process peers: direct pointers, peer access enabled pairwise; rank r = reps[r]
extern "C" int kmgpu_attach_replicas(kmgpu_t** reps, int n)
{
    if (!reps || n < 1 || n > MAX_WORLD) return fail(KMGPU_EINVAL, "bad replica list");
    for (int r = 1; r < n; r++)
        if (!same_shape(reps[0], reps[r])) return fail(KMGPU_ESHAPE, "replicas must have the same shape");
    for (int a = 0; a < n; a++) {
        CKR(set_device(reps[a]->device));
        for (int b = 0; b < n; b++) {
            if (reps[b]->device == reps[a]->device) continue;
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, reps[a]->device, reps[b]->device));
            if (!can) return fail(KMGPU_EUNSUPPORTED, "devices %d and %d have no peer access", reps[a]->device, reps[b]->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(reps[b]->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
            cudaGetLastError();
        }
    }
    for (int r = 0; r < n; r++) {
        kmgpu_ipc_detach(reps[r]);
        std::lock_guard<std::mutex> g(reps[r]->mu);
        CKR(set_device(reps[r]->device));
        CK(cudaStreamSynchronize(reps[r]->stream));
        reps[r]->rank = r;
        reps[r]->world = n;
        reps[r]->peers.assign(n, Peer());
        for (int q = 0; q < n; q++)
            for (int i = 0; i < reps[r]->nt; i++) reps[r]->peers[q].tables[i] = reps[q]->dev.tables[i];
        reps[r]->peers_ipc = false;
    }
    return KMGPU_OK;
}

extern "C" int kmgpu_reduce_replicas(kmgpu_t** reps, int n)
{
    if (!reps || n < 1 || n > MAX_WORLD) return fail(KMGPU_EINVAL, "bad replica list");
    if (n == 1) return KMGPU_OK;
    CKR(kmgpu_attach_replicas(reps, n));
    // exact n_unique_kmers across the replicas (first-touch logs on): resolved before any table changes
    bool ft = true;
    for (int r = 0; r < n; r++) ft = ft && reps[r]->ft_on;
    uint64_t unique_total = 0;
    if (ft) {
        unique_total = reps[0]->n_unique - reps[0]->ft_epoch_unique;   // the common state the epoch started from
        for (int r = 0; r < n; r++) {
            uint64_t n_new = 0;
            CKR(kmgpu_first_touch_resolve(reps[r], &n_new, nullptr, nullptr));
            unique_total += n_new;
        }
    }
    for (int r = 0; r < n; r++) {
        std::lock_guard<std::mutex> g(reps[r]->mu);
        if (reps[r]->kind == BYTE && reps[r]->use_bigcount)
            return fail(KMGPU_EUNSUPPORTED, "replicas cannot be merged with bigcount on: which replica saw a counter's 255th touch is not "
                                            "recoverable (turn bigcount off, or shard the sketch by address)");
        CKR(reduce_scatter_locked(reps[r]));
    }
    for (int r = 0; r < n; r++) {
        std::lock_guard<std::mutex> g(reps[r]->mu);
        CKR(all_gather_locked(reps[r]));
    }
    for (int r = 0; r < n; r++) {
        std::lock_guard<std::mutex> g(reps[r]->mu);
        reps[r]->peers.clear();
        reps[r]->rank = 0;
        reps[r]->world = 1;
        if (ft) reps[r]->n_unique = unique_total;
    }
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// multi-GPU, replicated: exact n_unique_kmers / abundance_distribution across ranks (first-touch log, kmgpu_group.cuh §6)
// ------------------------------------------------------------------------------------------------------
static void ft_clear(kmgpu_sketch* h)
{
    for (auto& sg : h->ft_segs) cudaFree(sg.first);
    h->ft_segs.clear();
    h->ft_pending = 0;
    h->ft_epoch_unique = 0;
    h->ft_chunk = 0;
}

extern "C" int kmgpu_first_touch_log(kmgpu_t* h, int on)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    CK(cudaStreamSynchronize(h->stream));
    ft_clear(h);
    h->ft_on = on != 0;
    h->ft_defer = false;
    return KMGPU_OK;
}

// Rank r of an attached replica group (kmgpu_ipc_attach / kmgpu_reduce_replicas): how many k-mer occurrences logged since the
// log was switched on (or last resolved) are new in the stream order "rank 0's reads, then rank 1's, ..." — to be called on
// every rank after all ranks have finished ingesting and BEFORE any table is merged.  hist (nullable, 65536 entries) is
// accumulated with the counts the entries carry (abundance_distribution).  The log is emptied.
extern "C" int kmgpu_first_touch_resolve(kmgpu_t* h, uint64_t* n_new_out, uint64_t* n_local_out, uint64_t* hist)
{
    if (!h) return fail(KMGPU_EINVAL, "null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (!h->ft_on) return fail(KMGPU_EINVAL, "the first-touch log of this sketch is off");
    if (h->world > 1 && h->peers.empty()) return fail(KMGPU_EINVAL, "no peers attached");
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    uint64_t total = 0;
    for (auto& sg : h->ft_segs) total += sg.second;
    if (n_local_out) *n_local_out = h->ft_epoch_unique;
    uint64_t n_new = 0;
    if (total) {
        LowerRanks lr;
        memset(&lr, 0, sizeof lr);
        lr.n = h->world > 1 ? h->rank : 0;
        for (int q = 0; q < lr.n; q++)
            for (int i = 0; i < h->nt; i++) lr.tables[q][i] = h->peers[q].tables[i];
        LowerRanks* d_lr = nullptr;
        CK(cudaMalloc(&d_lr, sizeof lr));
        CK(cudaMemcpyAsync(d_lr, &lr, sizeof lr, cudaMemcpyHostToDevice, st));
        const uint64_t slots = pow2_at_least(2 * std::max<uint64_t>(h->ft_epoch_unique, 1));
        CKR(h->d_evkeys.ensure(slots));
        CK(cudaMemsetAsync(h->d_evkeys.p, 0xFF, slots * 8, st));
        CK(cudaMemsetAsync(&h->d_ctrl->n_unique, 0, sizeof(unsigned long long), st));
        unsigned long long* d_hist = nullptr;
        if (hist) {
            CKR(h->d_hist.ensure(65536));
            CK(cudaMemsetAsync(h->d_hist.p, 0, 65536 * 8, st));
            d_hist = h->d_hist.p;
        }
        for (auto& sg : h->ft_segs) {
            const unsigned gsz = (unsigned)std::min<uint64_t>((sg.second + 255) / 256, 148 * 16);
            const FtEntry* ent = (const FtEntry*)sg.first;
            if (h->kind == BYTE) k_ft_resolve<BYTE><<<gsz, 256, 0, st>>>(ent, sg.second, d_lr, h->d_evkeys.p, slots - 1, &h->d_ctrl->n_unique, d_hist);
            else if (h->kind == NIBBLE) k_ft_resolve<NIBBLE><<<gsz, 256, 0, st>>>(ent, sg.second, d_lr, h->d_evkeys.p, slots - 1, &h->d_ctrl->n_unique, d_hist);
            else k_ft_resolve<BIT><<<gsz, 256, 0, st>>>(ent, sg.second, d_lr, h->d_evkeys.p, slots - 1, &h->d_ctrl->n_unique, d_hist);
            h->all_launches += 1;
        }
        CK(cudaGetLastError());
        int rc = read_ctrl(h);
        cudaFree(d_lr);
        CKR(rc);
        n_new = h->h_ctrl->n_unique;
        if (hist) {
            std::vector<unsigned long long> hh(65536);
            CK(cudaMemcpy(hh.data(), h->d_hist.p, 65536 * 8, cudaMemcpyDeviceToHost));
            for (int i = 0; i < 65536; i++) hist[i] += hh[i];
        }
    }
    if (n_new_out) *n_new_out = n_new;
    ft_clear(h);
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// multi-GPU: address-sharded sketches (k-mer all-to-all over NVLink peer memory, see include/kmgpu.h)
//
// Rank r holds a whole number of super-buckets of every table as an ordinary local sketch.  A round:
//   route   every rank hashes its own reads and groups the counter updates by super-bucket of the FULL tables (k_part MODE 1,
//           local; regions that overflow are regrouped exactly like any chunk), then posts its per-super-bucket counts to the
//           owners (k_shard_post, a few KB over NVLink)
//   offsets every owner lays out its receive arena exactly: per super-bucket, the senders' runs side by side (k_shard_scan)
//   push    every sender writes its runs into the owners' arenas (k_shard_push: contiguous 8-byte stores into peer memory)
//   apply   every owner groups what it received by bucket and applies it in shared memory (k_part MODE 2 + k_apply2 / _sparse)
//   count   positions are global (rank * max_positions + position), so "first toucher of a bin" is decided across ranks;
//           every rank ORs the owners' new-position bitmaps for ITS positions — n_unique_kmers is exact
// with a barrier after each step.
// ------------------------------------------------------------------------------------------------------
struct kmgpu_shard {
    kmgpu_sketch* local = nullptr;
    int rank = 0, world = 1, nt = 0;
    uint64_t full_sizes[MAX_TABLES];
    uint64_t slice[MAX_TABLES];
    SketchDev full;   // full-table sizes and magics: what the k-mers are hashed against
    GroupPlan GF;     // layout of the full tables (route): super-buckets only
    GroupPlan G;      // layout of one rank's slices (the same on every rank): apply
    ShardGeom geom;
    uint64_t max_positions = 0;
    uint64_t arena = 0;                    // records the receive arena holds
    uint32_t n_sb_local = 0;               // super-buckets per rank, all tables
    // receive side (peers write / read these)
    unsigned long long* rec1 = nullptr;    // arena
    uint32_t* demand = nullptr;            // [local super-bucket * world + sender]
    unsigned long long* recv_off = nullptr;
    unsigned long long* flags = nullptr;   // bit 0: this round does not fit the arena; bit 1: the arena holds bigcount answers
    uint32_t* newbits = nullptr;           // one bit per global position of a round: marked new by this owner
    struct PeerQ {
        unsigned long long* rec1;
        uint32_t* demand;
        unsigned long long* recv_off;
        unsigned long long* flags;
        uint32_t* newbits;
    } peers[MAX_WORLD];
    // owner side
    DevBuf<unsigned long long> sb_off;
    DevBuf<uint32_t> sb_cnt;
    uint32_t max_cnt = 0;
    uint64_t received = 0;
    bool refused = false;
    // sender side
    DevBuf<unsigned long long> rec_s, off_s;
    DevBuf<uint32_t> cur_s;
    bool exact_s = false;
    bool attached = false, ipc = false;
    uint64_t n_unique = 0;   // k-mers of this rank's reads that were new
    // the reads of the last route call: they stay staged in slot 0 of the local sketch (nothing else stages there between a
    // route and the getters of its round); offs covers every read of the call, n_pos its bases
    ChunkDev q;
    DevBuf<uint32_t> q_offs;   // those offsets when staging dropped empty reads at either end of the range
    DevBuf<uint8_t> planes;    // pull: the answers, one byte per (table, position), planes of max_positions bytes
    bool pulled = false;       // the last route was answered (kmgpu_shard_pull): the local sketch's d_counts hold its counts
    bool counted = false;      // the last route was ingested up to kmgpu_shard_count_new: its d_newbits hold the new positions
    // bigcount (ingest rounds): the owner's (position, crossing-bin slot) pairs, and this rank's events of the last round
    DevBuf<uint2> sel_pairs;
    std::vector<EvOut> big_ev;
    bool big_ev_ready = false;
};

extern "C" int kmgpu_shard_destroy(kmgpu_shard_t* s);

extern "C" int kmgpu_shard_create(int storage, int hash, int ksize, int n_tables, const uint64_t* full_sizes, int device, int rank, int world,
                                  uint64_t max_positions, kmgpu_shard_t** out)
{
    if (!out) return fail(KMGPU_EINVAL, "out is NULL");
    *out = nullptr;
    if (world < 1 || world > MAX_WORLD || rank < 0 || rank >= world) return fail(KMGPU_EINVAL, "bad rank/world %d/%d (at most %d ranks)", rank, world, MAX_WORLD);
    if (n_tables < 1 || n_tables > MAX_TABLES) return fail(KMGPU_EUNSUPPORTED, "n_tables %d not supported", n_tables);
    if (max_positions == 0) max_positions = 8ull << 20;
    max_positions = ((max_positions + 127) / 128) * 128;   // every rank's range of the new-position bitmaps starts on 16 bytes
    if (max_positions > chunk_bases() || (uint64_t)world * max_positions >= (1ull << 32))
        return fail(KMGPU_EINVAL, "max_positions %llu too large (positions of a round are 32-bit across all ranks)", (unsigned long long)max_positions);
    for (int i = 0; i < n_tables; i++)
        if (full_sizes[i] == 0 || full_sizes[i] >= (1ull << 55)) return fail(KMGPU_EINVAL, "table size %llu out of range", (unsigned long long)full_sizes[i]);
    kmgpu_shard* s = new kmgpu_shard();
    s->rank = rank;
    s->world = world;
    s->nt = n_tables;
    s->max_positions = max_positions;
    memset(&s->full, 0, sizeof s->full);
    memset(s->peers, 0, sizeof s->peers);
    memset(&s->geom, 0, sizeof s->geom);
    {
        // layout of the FULL tables: super-buckets of 2^(15 + shift) bins, at most PART_MAXP of them per table (one grouping pass)
        kmgpu_sketch full_shape;
        full_shape.nt = n_tables;
        full_shape.kind = storage;
        for (int i = 0; i < n_tables; i++) full_shape.sizes[i] = full_sizes[i];
        if (!plan_group(&full_shape, (uint32_t)max_positions, &s->GF, true) || !s->GF.L.two_level) {
            delete s;
            return fail(KMGPU_EUNSUPPORTED, "tables of this size cannot be grouped");
        }
    }
    const int shift = s->GF.L.sb_shift;
    uint64_t local_sizes[MAX_TABLES], nominal[MAX_TABLES];
    s->geom.n_tables = n_tables;
    s->geom.world = world;
    s->geom.rank = rank;
    for (int i = 0; i < n_tables; i++) {
        s->full_sizes[i] = full_sizes[i];
        const uint32_t nsb = s->GF.L.first_sb[i + 1] - s->GF.L.first_sb[i];
        const uint32_t per = (nsb + world - 1) / world;
        s->geom.first_sb[i] = s->GF.L.first_sb[i];
        s->geom.sb_per_rank[i] = per;
        s->geom.local_first[i] = s->n_sb_local;
        s->n_sb_local += per;
        s->slice[i] = (uint64_t)per << (BKT_SHIFT + shift);   // a whole number of super-buckets: the owner of a record is a division
        uint64_t lo = std::min<uint64_t>(full_sizes[i], s->slice[i] * rank), hi = std::min<uint64_t>(full_sizes[i], s->slice[i] * (rank + 1));
        local_sizes[i] = std::max<uint64_t>(hi - lo, 1);  // a rank past the end of a table keeps a dummy bin
        nominal[i] = s->slice[i];
        s->full.sizes[i] = full_sizes[i];
        s->full.magic[i] = ~0ull / full_sizes[i];
    }
    s->geom.first_sb[n_tables] = s->GF.L.first_sb[n_tables];
    s->geom.local_first[n_tables] = s->n_sb_local;
    s->full.n_tables = n_tables;
    s->full.kind = storage;
    int rc = kmgpu_create(storage, hash, ksize, n_tables, local_sizes, device, &s->local);
    if (rc != KMGPU_OK) {
        delete s;
        return rc;
    }
    {
        // one layout for every rank: buckets and super-buckets of the NOMINAL slice, with the full tables' super-bucket size
        kmgpu_sketch nominal_shape;
        nominal_shape.nt = n_tables;
        nominal_shape.kind = storage;
        for (int i = 0; i < n_tables; i++) nominal_shape.sizes[i] = nominal[i];
        const bool ok = plan_group(&nominal_shape, (uint32_t)max_positions, &s->G, true, PART_MAXP, (uint64_t)world * max_positions, shift);
        if (!ok || !s->G.L.two_level || s->G.n_sb != s->n_sb_local) {
            kmgpu_shard_destroy(s);
            return fail(KMGPU_EUNSUPPORTED, "slices of this size cannot be grouped");
        }
    }
    // the arena: what all ranks together send an owner in a full round is (its share of the bins) x world x max_positions records
    // on average; half as much again for owners whose bins are hit more often than others' (a round that still does not fit is
    // refused, see kmgpu_shard_offsets)
    {
        double share = 0;   // the part of every table this rank owns, summed over the tables (N / world when the slices are even)
        for (int i = 0; i < n_tables; i++) {
            const uint64_t lo = std::min<uint64_t>(full_sizes[i], s->slice[i] * rank), hi = std::min<uint64_t>(full_sizes[i], s->slice[i] * (rank + 1));
            share += (double)(hi - lo) / (double)full_sizes[i];
        }
        s->arena = (uint64_t)(1.5 * share * (double)world * (double)max_positions) + 4096;
    }
    if (uint64_t f = env_u64("KMGPU_SHARD_ARENA", 0)) s->arena = f;   // tests
    const size_t nb_words = (size_t)world * max_positions / 32;
    const size_t n_dem = (size_t)s->n_sb_local * world;
    cudaError_t e = cudaMalloc(&s->rec1, s->arena * 8);
    if (e == cudaSuccess) e = cudaMalloc(&s->demand, n_dem * 4);
    if (e == cudaSuccess) e = cudaMemset(s->demand, 0, n_dem * 4);
    if (e == cudaSuccess) e = cudaMalloc(&s->recv_off, (n_dem + 1) * 8);
    if (e == cudaSuccess) e = cudaMemset(s->recv_off, 0, (n_dem + 1) * 8);
    if (e == cudaSuccess) e = cudaMalloc(&s->flags, 8);
    if (e == cudaSuccess) e = cudaMemset(s->flags, 0, 8);
    if (e == cudaSuccess) e = cudaMalloc(&s->newbits, nb_words * 4);
    if (e == cudaSuccess) e = cudaMemset(s->newbits, 0, nb_words * 4);
    if (e != cudaSuccess) {
        cudaGetLastError();
        kmgpu_shard_destroy(s);
        return fail(e == cudaErrorMemoryAllocation ? KMGPU_ENOMEM : KMGPU_ECUDA, "shard stores: %s", cudaGetErrorString(e));
    }
    *out = s;
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_destroy(kmgpu_shard_t* s)
{
    if (!s) return KMGPU_OK;
    if (s->local) cudaSetDevice(s->local->device);
    if (s->ipc)
        for (int q = 0; q < s->world; q++) {
            if (q == s->rank) continue;
            if (s->peers[q].rec1) cudaIpcCloseMemHandle(s->peers[q].rec1);
            if (s->peers[q].demand) cudaIpcCloseMemHandle(s->peers[q].demand);
            if (s->peers[q].recv_off) cudaIpcCloseMemHandle(s->peers[q].recv_off);
            if (s->peers[q].flags) cudaIpcCloseMemHandle(s->peers[q].flags);
            if (s->peers[q].newbits) cudaIpcCloseMemHandle(s->peers[q].newbits);
        }
    if (s->rec1) cudaFree(s->rec1);
    if (s->demand) cudaFree(s->demand);
    if (s->recv_off) cudaFree(s->recv_off);
    if (s->flags) cudaFree(s->flags);
    if (s->newbits) cudaFree(s->newbits);
    s->q_offs.release();
    s->planes.release();
    s->sb_off.release();
    s->sb_cnt.release();
    s->sel_pairs.release();
    s->rec_s.release();
    s->off_s.release();
    s->cur_s.release();
    if (s->local) kmgpu_destroy(s->local);
    delete s;
    return KMGPU_OK;
}

extern "C" kmgpu_t* kmgpu_shard_local(kmgpu_shard_t* s) { return s ? s->local : nullptr; }

extern "C" int kmgpu_shard_slice(kmgpu_shard_t* s, int table, uint64_t* lo, uint64_t* hi)
{
    if (!s || table < 0 || table >= s->nt) return fail(KMGPU_EINVAL, "bad table index");
    if (lo) *lo = std::min<uint64_t>(s->full_sizes[table], s->slice[table] * s->rank);
    if (hi) *hi = std::min<uint64_t>(s->full_sizes[table], s->slice[table] * (s->rank + 1));
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_stats(kmgpu_shard_t* s, uint64_t* n_occupied_local, uint64_t* n_unique_share, uint64_t* store_bytes)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    if (n_occupied_local) *n_occupied_local = s->local->n_occupied;
    if (n_unique_share) *n_unique_share = s->n_unique;
    if (store_bytes) *store_bytes = s->arena * 8;
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_ipc_export(kmgpu_shard_t* s, uint8_t* handles)
{
    if (!s || !handles) return fail(KMGPU_EINVAL, "null argument");
    CKR(set_device(s->local->device));
    void* ptrs[KMGPU_SHARD_IPC_HANDLES] = {s->rec1, s->demand, s->recv_off, s->flags, s->newbits};
    for (int i = 0; i < KMGPU_SHARD_IPC_HANDLES; i++) {
        cudaIpcMemHandle_t mh;
        CK(cudaIpcGetMemHandle(&mh, ptrs[i]));
        memcpy(handles + (size_t)i * KMGPU_IPC_HANDLE_BYTES, &mh, KMGPU_IPC_HANDLE_BYTES);
    }
    return KMGPU_OK;
}

static void shard_set_peer(kmgpu_shard* s, int q, void* const* ptrs)
{
    s->peers[q].rec1 = (unsigned long long*)ptrs[0];
    s->peers[q].demand = (uint32_t*)ptrs[1];
    s->peers[q].recv_off = (unsigned long long*)ptrs[2];
    s->peers[q].flags = (unsigned long long*)ptrs[3];
    s->peers[q].newbits = (uint32_t*)ptrs[4];
}

extern "C" int kmgpu_shard_ipc_attach(kmgpu_shard_t* s, const uint8_t* all)
{
    if (!s || !all) return fail(KMGPU_EINVAL, "null argument");
    CKR(set_device(s->local->device));
    for (int q = 0; q < s->world; q++) {
        void* ptrs[KMGPU_SHARD_IPC_HANDLES] = {s->rec1, s->demand, s->recv_off, s->flags, s->newbits};
        if (q != s->rank)
            for (int i = 0; i < KMGPU_SHARD_IPC_HANDLES; i++) {
                cudaIpcMemHandle_t mh;
                memcpy(&mh, all + ((size_t)q * KMGPU_SHARD_IPC_HANDLES + i) * KMGPU_IPC_HANDLE_BYTES, KMGPU_IPC_HANDLE_BYTES);
                CK(cudaIpcOpenMemHandle(&ptrs[i], mh, cudaIpcMemLazyEnablePeerAccess));
            }
        shard_set_peer(s, q, ptrs);
    }
    s->attached = true;
    s->ipc = true;
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_attach_local(kmgpu_shard_t** all, int n)
{
    if (!all || n < 1 || n > MAX_WORLD) return fail(KMGPU_EINVAL, "bad shard list");
    for (int a = 0; a < n; a++) {
        if (!all[a] || all[a]->world != n || all[a]->rank != a) return fail(KMGPU_EINVAL, "shard %d is not rank %d of %d", a, a, n);
        CKR(set_device(all[a]->local->device));
        for (int b = 0; b < n; b++) {
            if (all[b]->local->device != all[a]->local->device) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, all[a]->local->device, all[b]->local->device));
                if (!can) return fail(KMGPU_EUNSUPPORTED, "devices %d and %d have no peer access", all[a]->local->device, all[b]->local->device);
                cudaError_t e = cudaDeviceEnablePeerAccess(all[b]->local->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
                cudaGetLastError();
            }
            void* ptrs[KMGPU_SHARD_IPC_HANDLES] = {all[b]->rec1, all[b]->demand, all[b]->recv_off, all[b]->flags, all[b]->newbits};
            shard_set_peer(all[a], b, ptrs);
        }
        all[a]->attached = true;
        all[a]->ipc = false;
    }
    return KMGPU_OK;
}

static void shard_peers(const kmgpu_shard* s, ShardPeers* P)
{
    memset(P, 0, sizeof *P);
    for (int q = 0; q < s->world; q++) {
        P->demand[q] = s->peers[q].demand;
        P->recv_off[q] = s->peers[q].recv_off;
        P->rec[q] = s->peers[q].rec1;
        P->flags[q] = s->peers[q].flags;
    }
}

// route: group my reads' counter updates by super-bucket of the full tables (locally), post the counts to the owners.
// n_reads == 0: a rank without reads in this round still posts (zero) counts.
extern "C" int kmgpu_shard_route(kmgpu_shard_t* s, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags,
                                 uint64_t* n_kmers_out)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    if (n_kmers_out) *n_kmers_out = 0;
    if (!s->attached) return fail(KMGPU_EINVAL, "peers are not attached");
    if (n_reads && (!seqs || !offsets)) return fail(KMGPU_EINVAL, "null input");
    kmgpu_sketch* h = s->local;
    const uint64_t first = n_reads ? offsets[0] : 0, last = n_reads ? offsets[n_reads] : 0;
    if (last - first > s->max_positions)
        return fail(KMGPU_EINVAL, "%llu bases in one route call; this shard was created for at most %llu", (unsigned long long)(last - first),
                    (unsigned long long)s->max_positions);
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    const GroupLayout& LF = s->GF.L;
    const uint32_t n_sb = s->GF.n_sb;
    CKR(s->cur_s.ensure(n_sb));
    CK(cudaMemsetAsync(s->cur_s.p, 0, (size_t)n_sb * 4, st));
    CK(cudaMemsetAsync(h->d_ctrl, 0, sizeof(Ctrl), st));
    s->exact_s = false;
    s->q = ChunkDev{};
    s->pulled = s->counted = s->big_ev_ready = false;
    uint64_t n_kmers = 0;
    if (last > first) {
        ChunkDev cd;
        CKR(stage_range(h, seqs, offsets, n_reads, first, last, flags, &cd, needs_acgt_check(h, flags), 0, st));
        s->q = cd;
        Input in = make_input(cd);
        CK(cudaEventRecord(h->ev0, st));
        const HashCfg H{h->hash, h->k};
        int srck = 0;
        if (H.kind == MURMUR) {
            CKR(h->d_hash64.ensure(in.n_pos));
            k_hash64<MURMUR><<<n_tiles(in.n_pos), THREADS, 0, st>>>(H, in, h->d_hash64.p);
            in.hashes = h->d_hash64.p;
            srck = 1;
            h->all_launches += 1;
        }
        if (!try_ensure(s->rec_s, std::max<uint64_t>((uint64_t)n_sb * LF.cap1, 2))) return fail(KMGPU_ENOMEM, "no room for the sender's record store");
        PartArgs A;
        memset(&A, 0, sizeof A);
        A.S = s->full;
        A.H = H;
        A.in = in;
        A.pos_base = (uint32_t)((uint64_t)s->rank * s->max_positions);
        A.have_valid = 1;
        A.table0 = 0;
        A.count_kmers = 1;
        A.L = LF;
        A.ctrl = h->d_ctrl;
        A.dst = Store{s->rec_s.p, nullptr, s->cur_s.p, LF.cap1, 0};
        A.ovf_bit = 1ull;
        Pred P0;
        memset(&P0, 0, sizeof P0);
        uint32_t np = 0;
        for (int t = 0; t < s->nt; t++) np = std::max(np, LF.first_sb[t + 1] - LF.first_sb[t]);
        const dim3 grid((in.n_pos + 8191) / 8192, s->nt);
        CKR(launch_part(1, srck, false, 8192, true, np, grid, st, A, s->full, P0));
        h->all_launches += 1;
        CK(cudaGetLastError());
        CKR(read_ctrl(h));
        n_kmers = h->h_ctrl->n_kmers;
        if (h->h_ctrl->overflow) {
            // a super-bucket region ran out of room (heavily repeated k-mers): the cursors hold the exact demand, regroup into
            // exact regions
            CKR(s->off_s.ensure((size_t)n_sb + 1));
            k_exact_offsets<<<1, 1024, 0, st>>>(s->cur_s.p, n_sb, s->off_s.p);
            unsigned long long total = 0;
            CK(cudaMemcpyAsync(&total, s->off_s.p + n_sb, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (!try_ensure(s->rec_s, std::max<size_t>((size_t)total, 2))) return fail(KMGPU_ENOMEM, "no room for the sender's record store");
            CK(cudaMemsetAsync(s->cur_s.p, 0, (size_t)n_sb * 4, st));
            CK(cudaMemsetAsync(&h->d_ctrl->overflow, 0, sizeof(unsigned long long), st));
            A.dst = Store{s->rec_s.p, s->off_s.p, s->cur_s.p, 0, 0};
            A.count_kmers = 0;
            A.ovf_bit = 1ull << 63;
            CKR(launch_part(1, srck, false, 8192, true, np, grid, st, A, s->full, P0));
            h->all_launches += 2;
            h->n_regroups++;
            s->exact_s = true;
            CK(cudaGetLastError());
            CKR(read_ctrl(h));
            if (h->h_ctrl->overflow) return fail(KMGPU_ECUDA, "internal: regrouping run overflowed");
        }
        CK(cudaEventRecord(h->ev1, st));
    }
    if (s->q.n_reads != n_reads) {
        // the staged range leaves out empty reads at its ends (or there was nothing to stage): the per-read getters of a query
        // round need the offsets of every read
        std::vector<uint32_t> o(n_reads + 1);
        for (uint64_t r = 0; r <= n_reads; r++) o[r] = (uint32_t)(offsets[r] - first);
        CKR(s->q_offs.ensure(n_reads + 1));
        CK(cudaMemcpyAsync(s->q_offs.p, o.data(), (n_reads + 1) * 4, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
        s->q.offs = s->q_offs.p;
        s->q.n_reads = (uint32_t)n_reads;
    }
    ShardPeers PP;
    shard_peers(s, &PP);
    k_shard_post<<<(n_sb + 255) / 256, 256, 0, st>>>(s->geom, s->cur_s.p, n_sb, PP);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    if (last > first) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        h->ingest_ms += ms;
    }
    if (n_kmers_out) *n_kmers_out = n_kmers;
    return KMGPU_OK;
}

// offsets (owner): exact layout of what this round sends me; a round larger than the arena is refused (flag read by the senders)
extern "C" int kmgpu_shard_offsets(kmgpu_shard_t* s)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    const uint32_t n_dem = s->n_sb_local * (uint32_t)s->world;
    CKR(s->sb_off.ensure((size_t)s->n_sb_local + 1));
    CKR(s->sb_cnt.ensure(std::max<uint32_t>(s->n_sb_local, 1)));
    unsigned int* mx = reinterpret_cast<unsigned int*>(&h->d_ctrl->n_events);
    CK(cudaMemsetAsync(&h->d_ctrl->n_events, 0, sizeof(unsigned long long), st));
    k_shard_scan<<<1, 1024, 0, st>>>(s->demand, n_dem, s->recv_off);
    k_shard_sb<<<(s->n_sb_local + 256) / 256, 256, 0, st>>>(s->recv_off, s->n_sb_local, s->world, s->sb_off.p, s->sb_cnt.p, mx);
    h->all_launches += 2;
    CK(cudaGetLastError());
    unsigned long long total = 0;
    CK(cudaMemcpyAsync(&total, s->recv_off + n_dem, 8, cudaMemcpyDeviceToHost, st));
    CKR(read_ctrl(h));
    s->max_cnt = (uint32_t)h->h_ctrl->n_events;
    s->received = total;
    s->refused = total > s->arena;
    const unsigned long long fl = s->refused ? 1ull : 0ull;
    CK(cudaMemcpyAsync(s->flags, &fl, 8, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    return KMGPU_OK;
}

// push (sender): my runs into the owners' arenas
extern "C" int kmgpu_shard_push(kmgpu_shard_t* s)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    if (!s->rec_s.p) return KMGPU_OK;   // nothing was ever routed
    ShardPeers PP;
    shard_peers(s, &PP);
    const Store src = s->exact_s ? Store{s->rec_s.p, s->off_s.p, s->cur_s.p, 0, 0} : Store{s->rec_s.p, nullptr, s->cur_s.p, s->GF.L.cap1, 0};
    CK(cudaEventRecord(h->ev0, st));
    k_shard_push<<<dim3(s->GF.n_sb, 8), 256, 0, st>>>(s->geom, src, PP);
    h->all_launches += 1;
    CK(cudaEventRecord(h->ev1, st));
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->ingest_ms += ms;
    return KMGPU_OK;
}

// bigcount (owner, after the apply): every record of my arena is answered with "its byte was 255 before it arrived" (k_shard_satmark),
// and bit 1 of my flags tells the senders to read the answers.  A bin that crossed 255 in this round was saturated for the touches
// after its (255 - before)-th in global position order: that touch's position T is found by a radix select over the records of
// the crossing bins.
static int shard_satmark(kmgpu_shard* s, uint64_t n_list, uint64_t n_cross, uint32_t n_pos_all)
{
    kmgpu_sketch* h = s->local;
    cudaStream_t st = h->stream;
    constexpr uint64_t WS_MIN = 1ull << 20;
    const int sbb = BKT_SHIFT + s->GF.L.sb_shift;
    const dim3 grid(s->n_sb_local, 8);
    uint64_t slots = 1024;
    const uint32_t* T = nullptr;
    if (n_cross) {
        slots = pow2_at_least(2 * n_cross);
        CKR(h->d_htkeys.ensure(std::max<uint64_t>(slots, WS_MIN)));
        CKR(h->d_htvals.ensure(std::max<uint64_t>(slots, WS_MIN)));
        CK(cudaMemsetAsync(h->d_htkeys.p, 0xFF, slots * 8, st));
        k_list_register<<<(unsigned)std::min<uint64_t>((n_list + 255) / 256, 148 * 8), 256, 0, st>>>(h->d_binlist.p, n_list, BL_CROSS, h->d_htkeys.p,
                                                                                                  h->d_htvals.p, slots - 1, nullptr, 1);
        h->all_launches += 1;
        // the touches of the crossing bins; the buffer grows (and the pass runs again) when they do not fit
        unsigned long long* n_pairs = &h->d_ctrl->n_events;
        uint64_t n = 0;
        for (int pass = 0; pass < 2; pass++) {
            CKR(s->sel_pairs.ensure(std::max<uint64_t>(n, WS_MIN)));
            CK(cudaMemsetAsync(n_pairs, 0, sizeof(unsigned long long), st));
            k_shard_sel_pairs<<<grid, 256, 0, st>>>(s->geom, s->rec1, s->sb_off.p, s->sb_cnt.p, sbb, h->d_htkeys.p, slots - 1, s->sel_pairs.p,
                                                    (unsigned long long)s->sel_pairs.cap, n_pairs);
            h->all_launches += 1;
            CK(cudaGetLastError());
            CKR(read_ctrl(h));
            n = h->h_ctrl->n_events;
            if (n <= s->sel_pairs.cap) break;
        }
        if (n > s->sel_pairs.cap) return fail(KMGPU_ECUDA, "internal: crossing-bin touches overflowed");
        CKR(h->d_sel.ensure(std::max<uint64_t>(3 * slots, WS_MIN)));
        SelState ss{h->d_sel.p, h->d_sel.p + slots, h->d_sel.p + 2 * slots};
        const unsigned gsl = (unsigned)((slots + 255) / 256), gp = (unsigned)std::max<uint64_t>((n + 255) / 256, 1);
        k_sel_init<<<gsl, 256, 0, st>>>(h->d_htkeys.p, h->d_htvals.p, slots, ss);
        int top = 0;
        while (top < 31 && (1ull << (top + 1)) <= (uint64_t)n_pos_all) top++;
        for (int bit = top; bit >= 0; bit--) {
            k_sel_count_pairs<<<gp, 256, 0, st>>>(s->sel_pairs.p, n, bit, ss);
            k_sel_update<<<gsl, 256, 0, st>>>(slots, bit, ss);
        }
        h->all_launches += 1 + 2 * (top + 1);
        T = ss.prefix;
    }
    k_shard_satmark<<<grid, 256, 0, st>>>(s->geom, h->dev, s->rec1, s->sb_off.p, s->sb_cnt.p, sbb, h->d_htkeys.p, slots - 1, T, n_cross ? 1 : 0);
    h->all_launches += 1;
    CK(cudaGetLastError());
    const unsigned long long fl = 2ull;
    CK(cudaMemcpyAsync(s->flags, &fl, 8, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_apply(kmgpu_shard_t* s)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    const int want_cross = h->kind == BYTE && h->use_bigcount;
    if (want_cross && h->nt > 30) return fail(KMGPU_EUNSUPPORTED, "bigcount is supported for up to 30 tables");
    cudaStream_t st = h->stream;
    const size_t n_dem = (size_t)s->n_sb_local * s->world;
    if (s->refused) {
        // the refusal flag stays up: with bigcount on, the senders read it in kmgpu_shard_bigcount_events (kmgpu_shard_offsets
        // writes it anew every round)
        s->refused = false;
        CK(cudaMemsetAsync(s->demand, 0, n_dem * 4, st));
        CK(cudaStreamSynchronize(st));
        return fail(KMGPU_ENOMEM, "rank %d was sent %llu records in one round, its arena holds %llu (this rank owns far more than its share of the "
                                  "k-mers): the round was not applied; create the shards with a smaller max_positions_per_route",
                    s->rank, (unsigned long long)s->received, (unsigned long long)s->arena);
    }
    GroupPlan G = s->G;
    G.L.cap1 = std::max<uint32_t>(s->max_cnt, 2);   // the level-2 pass covers the fullest super-bucket
    const uint32_t n_pos_all = (uint32_t)((uint64_t)s->world * s->max_positions);
    CKR(h->d_cursors.ensure(G.n_buckets));
    if (!try_ensure(h->d_records, std::max<uint64_t>((uint64_t)G.n_buckets * G.L.cap, 2)))
        return fail(KMGPU_ENOMEM, "no room for the bucket store of a sharded round");
    // bigcount: one crossing-list entry per bin that reaches 255 in this round, at most one per record received
    uint64_t list_cap = 1;
    if (want_cross) {
        uint64_t bins = 0;
        for (int i = 0; i < h->nt; i++) bins += h->sizes[i];
        list_cap = std::max<uint64_t>(1, std::min<uint64_t>(s->received, bins));
    }
    CKR(h->d_binlist.ensure(list_cap));
    CK(cudaMemsetAsync(s->newbits, 0, (size_t)n_pos_all / 8, st));
    CK(cudaMemsetAsync(h->d_ctrl, 0, sizeof(Ctrl), st));
    CK(cudaEventRecord(h->ev0, st));
    const GroupTurn tn{0, h->nt, 0, G.n_buckets, 0, G.n_sb};
    const Store s1{s->rec1, s->sb_off.p, s->sb_cnt.p, 0, 0};
    SatBitsG sb;
    memset(&sb, 0, sizeof sb);
    Pred P0;
    memset(&P0, 0, sizeof P0);
    const HashCfg H{h->hash, h->k};
    const std::vector<Part> none;
    if (s->received) CKR(group_turn(h, G, tn, 0, 0, H, none, P0, false, h->dev, false, 0u, n_pos_all, list_cap, want_cross, sb, &s1, s->newbits));
    CK(cudaEventRecord(h->ev1, st));
    CKR(read_ctrl(h));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->ingest_ms += ms;
    if (h->h_ctrl->overflow) {
        const unsigned bits = (unsigned)(h->h_ctrl->overflow & 3ull);
        CK(cudaMemsetAsync(&h->d_ctrl->overflow, 0, sizeof(unsigned long long), st));
        h->n_regroups++;
        CKR(group_turn(h, G, tn, 0, 0, H, none, P0, false, h->dev, false, bits, n_pos_all, list_cap, want_cross, sb, &s1, s->newbits));
        CKR(read_ctrl(h));
        if (h->h_ctrl->overflow) return fail(KMGPU_ECUDA, "internal: regrouping run overflowed");
        // bucket regions get more slack from the next round on
        const uint32_t cap_now = s->G.L.cap;
        s->G.L.cap = (uint32_t)std::min<uint64_t>(((uint64_t)cap_now * 3 / 2 + 1) & ~1ull, (uint64_t)n_pos_all + 2);
        s->G.wide = s->G.L.cap > 65535;
        s->G.sparse = s->G.sparse && s->G.L.cap <= SPARSE_MAX_RECORDS;
    }
    h->n_occupied += h->h_ctrl->n_new_t[0];   // the apply kernels of the grouped path count newly occupied bins per table
    if (want_cross) {
        // after any regrouping run (it reads the arena's records as they were pushed); no touch found a saturated byte: nothing to mark
        const Ctrl c = *h->h_ctrl;
        if (c.n_events > list_cap) return fail(KMGPU_ECUDA, "internal: crossing list overflow");
        if (c.n_sat) CKR(shard_satmark(s, c.n_events, c.n_cross, n_pos_all));
    }
    CK(cudaMemsetAsync(s->demand, 0, n_dem * 4, st));   // ranks without reads in a later round post nothing for tables they do not reach
    CK(cudaStreamSynchronize(st));
    h->satbits_valid = false;
    return KMGPU_OK;
}

// after every rank has applied the round: the positions of THIS rank's reads that any owner marked new (a k-mer is new iff
// one of its bins was empty when it arrived, whichever rank owns that bin)
extern "C" int kmgpu_shard_count_new(kmgpu_shard_t* s, uint64_t* n_new_out)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    const size_t words = (size_t)s->max_positions / 32, w0 = (size_t)s->rank * words;
    CKR(h->d_newbits.ensure(words));
    CK(cudaMemcpyAsync(h->d_newbits.p, s->newbits + w0, words * 4, cudaMemcpyDeviceToDevice, st));
    PeerPtrs pp;
    pp.n = 0;
    for (int q = 0; q < s->world; q++) {   // OR of the peers' bitmaps over NVLink, eight peers per pass
        if (q != s->rank) pp.p[pp.n++] = s->peers[q].newbits + w0;
        if (pp.n == 8 || (q == s->world - 1 && pp.n)) {
            unsigned gsz = (unsigned)std::min<uint64_t>((words + 255) / 256, 148 * 16);
            k_merge_peers<<<gsz, 256, 0, st>>>(BIT, h->d_newbits.p, pp, 0, words);
            h->all_launches += 1;
            pp.n = 0;
        }
    }
    CK(cudaMemsetAsync(&h->d_ctrl->n_unique, 0, sizeof(unsigned long long), st));
    k_popc<<<(unsigned)std::min<size_t>((words + 255) / 256, 148 * 8), 256, 0, st>>>(h->d_newbits.p, words, &h->d_ctrl->n_unique);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CKR(read_ctrl(h));
    s->n_unique += h->h_ctrl->n_unique;
    s->counted = true;
    if (n_new_out) *n_new_out = h->h_ctrl->n_unique;
    return KMGPU_OK;
}

// lookup (owner, query rounds): every record of my arena gets the counter it addresses in my slices, in place.  Tables, counters
// and the new-position bitmap are not touched.
extern "C" int kmgpu_shard_lookup(kmgpu_shard_t* s)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    const size_t n_dem = (size_t)s->n_sb_local * s->world;
    if (s->refused) {
        // the refusal flag stays up: the senders read it in kmgpu_shard_pull (kmgpu_shard_offsets writes it anew every round)
        s->refused = false;
        CK(cudaMemsetAsync(s->demand, 0, n_dem * 4, st));
        CK(cudaStreamSynchronize(st));
        return fail(KMGPU_ENOMEM, "rank %d was sent %llu records in one round, its arena holds %llu (this rank owns far more than its share of the "
                                  "k-mers): the round was not answered; create the shards with a smaller max_positions_per_route",
                    s->rank, (unsigned long long)s->received, (unsigned long long)s->arena);
    }
    if (s->received) {
        const int sbb = BKT_SHIFT + s->GF.L.sb_shift;
        const dim3 grid(s->n_sb_local, 8);
        if (h->kind == BYTE) k_shard_lookup<BYTE><<<grid, 256, 0, st>>>(s->geom, h->dev, s->rec1, s->sb_off.p, s->sb_cnt.p, sbb);
        else if (h->kind == NIBBLE) k_shard_lookup<NIBBLE><<<grid, 256, 0, st>>>(s->geom, h->dev, s->rec1, s->sb_off.p, s->sb_cnt.p, sbb);
        else k_shard_lookup<BIT><<<grid, 256, 0, st>>>(s->geom, h->dev, s->rec1, s->sb_off.p, s->sb_cnt.p, sbb);
        h->all_launches += 1;
        CK(cudaGetLastError());
    }
    CK(cudaMemsetAsync(s->demand, 0, n_dem * 4, st));   // as after an apply: ranks without reads in a later round post nothing
    CK(cudaStreamSynchronize(st));
    return KMGPU_OK;
}

// pull (sender, query rounds): read my answered records back from every owner; count per position = min over the tables
extern "C" int kmgpu_shard_pull(kmgpu_shard_t* s)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    cudaStream_t st = h->stream;
    s->pulled = false;
    const uint32_t n_pos = s->q.n_pos;
    CKR(h->d_counts.ensure(std::max<uint32_t>(n_pos, 1)));
    if (n_pos) {
        const uint64_t stride = s->max_positions;
        if (!try_ensure(s->planes, (size_t)s->nt * stride)) return fail(KMGPU_ENOMEM, "no room for the answers of a query round");
        ShardPeers PP;
        shard_peers(s, &PP);
        const Store src = s->exact_s ? Store{s->rec_s.p, s->off_s.p, s->cur_s.p, 0, 0} : Store{s->rec_s.p, nullptr, s->cur_s.p, s->GF.L.cap1, 0};
        CK(cudaMemsetAsync(&h->d_ctrl->overflow, 0, sizeof(unsigned long long), st));
        k_shard_pull<<<dim3(s->GF.n_sb, 8), 256, 0, st>>>(s->geom, src, PP, BKT_SHIFT + s->GF.L.sb_shift,
                                                         (uint32_t)((uint64_t)s->rank * s->max_positions), stride, s->planes.p,
                                                         &h->d_ctrl->overflow, 0ull);
        h->all_launches += 1;
        CK(cudaGetLastError());
        CKR(read_ctrl(h));
        if (h->h_ctrl->overflow)
            return fail(KMGPU_ENOMEM, "rank %d: an owner's arena could not hold this round (see its kmgpu_shard_lookup): no counts", s->rank);
        k_shard_fold<<<(unsigned)std::min<uint32_t>((n_pos + 255) / 256, 148 * 16), 256, 0, st>>>(s->planes.p, s->nt, stride, n_pos,
                                                                                                   h->d_counts.p);
        h->all_launches += 1;
        if (h->kind == BYTE && h->use_bigcount) {
            CKR(sync_big_to_device(h));
            if (h->n_big_dev) {
                Input in = make_input(s->q);
                const unsigned gb = (unsigned)std::min<uint32_t>((n_pos + 255) / 256, 148 * 16);
                if (h->hash == MURMUR) {
                    in.hashes = h->d_hash64.p;
                    k_shard_bigcount<TWOBIT, 1><<<gb, 256, 0, st>>>(h->d_counts.p, in, h->k, h->big_keys.p, h->big_vals.p, h->n_big_dev);
                } else {
                    k_shard_bigcount<TWOBIT, 0><<<gb, 256, 0, st>>>(h->d_counts.p, in, h->k, h->big_keys.p, h->big_vals.p, h->n_big_dev);
                }
                h->all_launches += 1;
            }
        }
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(st));
    }
    s->pulled = true;
    return KMGPU_OK;
}

// bigcount events (sender, ingest rounds): after every owner has applied the round, the k-mers of MY reads whose N bytes were all
// 255 before they arrived.  The answers of the owners that marked their arenas are pulled, ANDed over the tables and aggregated per
// k-mer; the list (one entry per distinct hash, in the order of its first event) is kept until the next route.
static int shard_bigcount_events(kmgpu_shard* s)
{
    kmgpu_sketch* h = s->local;
    cudaStream_t st = h->stream;
    constexpr uint64_t WS_MIN = 1ull << 20;
    s->big_ev.clear();
    const uint32_t n_pos = s->q.n_pos;
    if (n_pos == 0) return KMGPU_OK;
    unsigned long long fl[MAX_WORLD];
    for (int q = 0; q < s->world; q++) CK(cudaMemcpyAsync(&fl[q], s->peers[q].flags, 8, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));
    bool any = false;
    for (int q = 0; q < s->world; q++) any |= (fl[q] & 3ull) != 0;
    if (!any) return KMGPU_OK;   // no owner marked anything, and none refused the round
    const uint64_t stride = s->max_positions;
    if (!try_ensure(s->planes, (size_t)s->nt * stride)) return fail(KMGPU_ENOMEM, "no room for the bigcount answers of a round");
    CK(cudaMemset2DAsync(s->planes.p, stride, 0, n_pos, s->nt, st));   // positions whose owners marked nothing stay 0
    ShardPeers PP;
    shard_peers(s, &PP);
    const Store src = s->exact_s ? Store{s->rec_s.p, s->off_s.p, s->cur_s.p, 0, 0} : Store{s->rec_s.p, nullptr, s->cur_s.p, s->GF.L.cap1, 0};
    CK(cudaMemsetAsync(&h->d_ctrl->overflow, 0, sizeof(unsigned long long), st));
    k_shard_pull<<<dim3(s->GF.n_sb, 8), 256, 0, st>>>(s->geom, src, PP, BKT_SHIFT + s->GF.L.sb_shift, (uint32_t)((uint64_t)s->rank * s->max_positions),
                                                     stride, s->planes.p, &h->d_ctrl->overflow, 2ull);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CKR(read_ctrl(h));
    if (h->h_ctrl->overflow)
        return fail(KMGPU_ENOMEM, "rank %d: an owner's arena could not hold this round (see its kmgpu_shard_apply): no bigcount events", s->rank);
    CKR(h->d_counts.ensure(n_pos));
    const unsigned gp = (unsigned)std::min<uint32_t>((n_pos + 255) / 256, 148 * 16);
    k_shard_fold<<<gp, 256, 0, st>>>(s->planes.p, s->nt, stride, n_pos, h->d_counts.p);
    h->all_launches += 1;
    Input in = make_input(s->q);
    if (h->hash == MURMUR) in.hashes = h->d_hash64.p;   // the route's hashes: nothing restages or rehashes before the next route
    unsigned long long* n_ctr = &h->d_ctrl->n_events;
    uint64_t n_rec = 0;
    for (int pass = 0; pass < 2; pass++) {   // the event buffer grows (and the pass runs again) when the events do not fit
        CKR(h->d_events.ensure(std::max<uint64_t>(n_rec, WS_MIN)));
        CK(cudaMemsetAsync(n_ctr, 0, sizeof(unsigned long long), st));
        if (h->hash == MURMUR) k_shard_events<TWOBIT, 1><<<gp, 256, 0, st>>>(h->d_counts.p, in, h->k, h->d_events.p, h->d_events.cap, n_ctr);
        else k_shard_events<TWOBIT, 0><<<gp, 256, 0, st>>>(h->d_counts.p, in, h->k, h->d_events.p, h->d_events.cap, n_ctr);
        h->all_launches += 1;
        CK(cudaGetLastError());
        CKR(read_ctrl(h));
        n_rec = h->h_ctrl->n_events;
        if (n_rec <= h->d_events.cap) break;
    }
    if (n_rec > h->d_events.cap) return fail(KMGPU_ECUDA, "internal: bigcount events overflowed");
    if (n_rec == 0) return KMGPU_OK;
    // aggregate per k-mer: count and first position (as the single sketch's resolution does)
    const uint64_t evslots = pow2_at_least(2 * n_rec);
    CKR(h->d_evkeys.ensure(std::max<uint64_t>(evslots, WS_MIN)));
    CKR(h->d_evvals.ensure(std::max<uint64_t>(2 * evslots, 2 * WS_MIN)));
    CK(cudaMemsetAsync(h->d_evkeys.p, 0xFF, evslots * 8, st));
    CK(cudaMemsetAsync(h->d_evvals.p, 0, evslots * 4, st));
    CK(cudaMemsetAsync(h->d_evvals.p + evslots, 0xFF, evslots * 4, st));
    CK(cudaMemsetAsync(&h->d_ctrl->n_unique, 0, sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(n_ctr, 0, sizeof(unsigned long long), st));
    EvTable ev{h->d_evkeys.p, h->d_evvals.p, h->d_evvals.p + evslots, evslots - 1};
    k_ev_decide<<<(unsigned)((n_rec + 255) / 256), 256, 0, st>>>(h->d_events.p, n_rec, h->nt, nullptr, nullptr, 0, ev, h->d_ctrl);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CKR(read_ctrl(h));
    const uint64_t n_distinct = h->h_ctrl->n_unique;
    CKR(h->d_evout.ensure(std::max<uint64_t>(n_distinct, WS_MIN / 4)));
    CKR(h->h_evout.ensure(std::max<uint64_t>(n_distinct, WS_MIN / 4)));
    k_ev_compact<<<(unsigned)((evslots + 255) / 256), 256, 0, st>>>(ev, h->d_evout.p, h->d_ctrl);
    h->all_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_evout.p, h->d_evout.p, n_distinct * sizeof(EvOut), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    s->big_ev.assign(h->h_evout.p, h->h_evout.p + n_distinct);
    std::sort(s->big_ev.begin(), s->big_ev.end(), [](const EvOut& a, const EvOut& b) { return a.first < b.first; });
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_bigcount_events(kmgpu_shard_t* s, uint64_t* hashes, uint32_t* counts, uint64_t cap, uint64_t* n_out)
{
    if (!s || !n_out) return fail(KMGPU_EINVAL, "null argument");
    *n_out = 0;
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    if (!(h->kind == BYTE && h->use_bigcount)) return fail(KMGPU_EINVAL, "bigcount is off on this shard");
    if (hashes && !counts) return fail(KMGPU_EINVAL, "null counts");
    CKR(set_device(h->device));
    if (!s->big_ev_ready) {
        CKR(shard_bigcount_events(s));
        s->big_ev_ready = true;
    }
    const uint64_t n = s->big_ev.size();
    for (uint64_t i = 0; hashes && i < n && i < cap; i++) {
        hashes[i] = s->big_ev[i].hash;
        counts[i] = s->big_ev[i].count;
    }
    *n_out = n;
    return KMGPU_OK;
}

// the events of every rank, concatenated in rank order: new keys enter the map in the order of their first event in the stream
extern "C" int kmgpu_shard_bigcount_apply(kmgpu_shard_t* s, const uint64_t* hashes, const uint32_t* counts, uint64_t n)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    if (n && (!hashes || !counts)) return fail(KMGPU_EINVAL, "null input");
    kmgpu_sketch* h = s->local;
    if (h->kind != BYTE) return fail(KMGPU_EUNSUPPORTED, "bigcount is not supported for this storage.");
    std::lock_guard<std::mutex> g(h->mu);
    for (uint64_t i = 0; i < n; i++) big_events(h, hashes[i], std::min<uint32_t>(counts[i], 65535u));
    return KMGPU_OK;
}

static int shard_pulled(const kmgpu_shard* s)
{
    if (!s->pulled) return fail(KMGPU_EINVAL, "no query round was pulled since the last kmgpu_shard_route");
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_kmer_counts(kmgpu_shard_t* s, uint16_t* counts_out, uint64_t* n_kmers_out)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    if (n_kmers_out) *n_kmers_out = 0;
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(shard_pulled(s));
    const uint32_t nr = s->q.n_reads;
    if (nr == 0) return KMGPU_OK;
    if (!counts_out) return fail(KMGPU_EINVAL, "null output");
    CKR(set_device(h->device));
    std::vector<uint32_t> offs(nr + 1);
    std::vector<uint16_t> hc(s->q.n_pos);
    CK(cudaMemcpyAsync(offs.data(), s->q.offs, 4ull * (nr + 1), cudaMemcpyDeviceToHost, h->stream));
    if (s->q.n_pos) CK(cudaMemcpyAsync(hc.data(), h->d_counts.p, 2ull * s->q.n_pos, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const uint64_t w = compact_kmers(hc.data(), offs.data(), nr, h->k, counts_out);
    if (n_kmers_out) *n_kmers_out = w;
    return KMGPU_OK;
}

extern "C" int kmgpu_shard_read_medians(kmgpu_shard_t* s, uint16_t* median_out, float* average_out, float* stddev_out, uint32_t* n_kmers_out)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(shard_pulled(s));
    if (s->q.n_reads == 0) return KMGPU_OK;
    CKR(set_device(h->device));
    return read_stats_counts(h, h->d_counts.p, s->q, 0, median_out, average_out, stddev_out, n_kmers_out, false, 0, nullptr);
}

extern "C" int kmgpu_shard_median_at_least(kmgpu_shard_t* s, uint32_t cutoff, uint8_t* out)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(shard_pulled(s));
    if (s->q.n_reads == 0) return KMGPU_OK;
    if (!out) return fail(KMGPU_EINVAL, "null output");
    CKR(set_device(h->device));
    return read_stats_counts(h, h->d_counts.p, s->q, 0, nullptr, nullptr, nullptr, nullptr, true, cutoff, out);
}

extern "C" int kmgpu_shard_trim(kmgpu_shard_t* s, uint32_t abund, int below, uint32_t* trim_pos_out)
{
    if (!s) return fail(KMGPU_EINVAL, "null shard");
    kmgpu_sketch* h = s->local;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(shard_pulled(s));
    if (s->q.n_reads == 0) return KMGPU_OK;
    if (!trim_pos_out) return fail(KMGPU_EINVAL, "null output");
    CKR(set_device(h->device));
    return trim_counts(h, h->d_counts.p, s->q, 0, abund, below, trim_pos_out);
}

// abundance_distribution over one run of reads: `tracking` has ingested it (up to count_new: its local sketch holds this rank's
// new positions), `counts` has answered it (pull): hist[count] += 1 for every new position
extern "C" int kmgpu_shard_abundance_hist(kmgpu_shard_t* counts, kmgpu_shard_t* tracking, uint64_t* hist)
{
    if (!counts || !tracking || !hist) return fail(KMGPU_EINVAL, "null argument");
    if (counts == tracking) return fail(KMGPU_EINVAL, "tracking shard must differ from the counting shard");
    kmgpu_sketch* c = counts->local;
    kmgpu_sketch* t = tracking->local;
    if (c->device != t->device) return fail(KMGPU_EINVAL, "shards live on different devices");
    if (counts->max_positions != tracking->max_positions)
        return fail(KMGPU_EINVAL, "shards were created for different max_positions (%llu, %llu)", (unsigned long long)counts->max_positions,
                    (unsigned long long)tracking->max_positions);
    if (c->hash != t->hash || c->k != t->k) return fail(KMGPU_EINVAL, "the tracking shard must hash k-mers as the counting shard does");
    kmgpu_sketch* a = c < t ? c : t;
    kmgpu_sketch* b = c < t ? t : c;
    std::lock_guard<std::mutex> ga(a->mu);
    std::lock_guard<std::mutex> gb(b->mu);
    CKR(shard_pulled(counts));
    if (!tracking->counted) return fail(KMGPU_EINVAL, "the tracking shard has not counted the new k-mers of its last route (kmgpu_shard_count_new)");
    if (counts->q.n_pos != tracking->q.n_pos || counts->q.n_reads != tracking->q.n_reads)
        return fail(KMGPU_EINVAL, "the shards last routed different reads");
    const uint32_t n_pos = counts->q.n_pos;
    if (n_pos == 0) return KMGPU_OK;
    CKR(set_device(c->device));
    cudaStream_t st = c->stream;
    CK(cudaStreamSynchronize(t->stream));
    CKR(c->d_hist.ensure(65536));
    CK(cudaMemsetAsync(c->d_hist.p, 0, 65536 * 8, st));
    k_hist<<<148 * 4, 256, 0, st>>>(c->d_counts.p, t->d_newbits.p, n_pos, c->d_hist.p);
    c->all_launches += 1;
    CK(cudaGetLastError());
    std::vector<unsigned long long> hh(65536);
    CK(cudaMemcpyAsync(hh.data(), c->d_hist.p, 65536 * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < 65536; i++) hist[i] += hh[i];
    return KMGPU_OK;
}

// ------------------------------------------------------------------------------------------------------
// HyperLogLog registers (unique-kmers.py's counter; SURVEY.md §8f.4)
// ------------------------------------------------------------------------------------------------------
struct kmgpu_hll {
    kmgpu_sketch* stage = nullptr;   // a one-bin sketch: device, stream and the staging buffers of the read feed
    int p = 0, k = 0;
    DevBuf<uint32_t> regs;
    DevBuf<uint8_t> bytes;
};

extern "C" int kmgpu_hll_destroy(kmgpu_hll_t* c)
{
    if (!c) return KMGPU_OK;
    if (c->stage) {
        cudaSetDevice(c->stage->device);
        c->regs.release();
        c->bytes.release();
        kmgpu_destroy(c->stage);
    }
    delete c;
    return KMGPU_OK;
}

extern "C" int kmgpu_hll_create(int device, int ksize, int n_counters_log2, kmgpu_hll_t** out)
{
    if (!out) return fail(KMGPU_EINVAL, "out is NULL");
    *out = nullptr;
    if (n_counters_log2 < 4 || n_counters_log2 > 26) return fail(KMGPU_EINVAL, "log2(counters) %d out of range [4, 26]", n_counters_log2);
    kmgpu_hll* c = new kmgpu_hll();
    c->p = n_counters_log2;
    c->k = ksize;
    const uint64_t one = 2;
    int rc = kmgpu_create(KMGPU_BIT, KMGPU_MURMUR, ksize, 1, &one, device, &c->stage);
    if (rc != KMGPU_OK) {
        delete c;
        return rc;
    }
    const size_t n = (size_t)1 << c->p;
    if (c->regs.ensure(n) != KMGPU_OK || c->bytes.ensure(n) != KMGPU_OK || cudaMemset(c->regs.p, 0, n * 4) != cudaSuccess) {
        kmgpu_hll_destroy(c);
        return fail(KMGPU_ENOMEM, "HLL registers");
    }
    *out = c;
    return KMGPU_OK;
}

extern "C" int kmgpu_hll_consume(kmgpu_hll_t* c, const char* seqs, const uint64_t* offsets, uint64_t n_reads, uint32_t flags, uint64_t* n_kmers_out)
{
    if (!c) return fail(KMGPU_EINVAL, "null handle");
    if (n_kmers_out) *n_kmers_out = 0;
    if (n_reads == 0) return KMGPU_OK;
    if (!seqs || !offsets) return fail(KMGPU_EINVAL, "null input");
    kmgpu_sketch* h = c->stage;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    const HashCfg H{h->hash, h->k};
    std::vector<ChunkPlan> plan;
    plan_chunks(offsets, n_reads, h->k, chunk_bases(), plan);
    uint64_t n_kmers = 0;
    for (const ChunkPlan& cp : plan) {
        ChunkDev cd;
        CKR(stage_chunk(h, seqs, cp, flags, &cd, needs_acgt_check(h, flags)));
        if (cd.n_pos == 0) continue;
        k_hll<MURMUR, 0><<<n_tiles(cd.n_pos), THREADS, 0, h->stream>>>(H, make_input(cd), c->p, c->regs.p);
        h->all_launches += 1;
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(h->stream));   // the staging buffers are reused by the next chunk
        for (size_t j = 0; j + 1 < cp.offs.size(); j++) {
            const uint32_t len = cp.offs[j + 1] - cp.offs[j];
            if (len >= (uint32_t)h->k) n_kmers += len - h->k + 1;
        }
    }
    if (n_kmers_out) *n_kmers_out = n_kmers;
    return KMGPU_OK;
}

extern "C" int kmgpu_hll_get_registers(kmgpu_hll_t* c, uint8_t* out)
{
    if (!c || !out) return fail(KMGPU_EINVAL, "null argument");
    kmgpu_sketch* h = c->stage;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    const uint32_t n = 1u << c->p;
    k_hll_bytes<<<(n + 255) / 256, 256, 0, h->stream>>>(c->regs.p, n, c->bytes.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, c->bytes.p, n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return KMGPU_OK;
}

extern "C" int kmgpu_hll_merge_registers(kmgpu_hll_t* c, const uint8_t* in, int replace)
{
    if (!c || !in) return fail(KMGPU_EINVAL, "null argument");
    kmgpu_sketch* h = c->stage;
    std::lock_guard<std::mutex> g(h->mu);
    CKR(set_device(h->device));
    const uint32_t n = 1u << c->p;
    CK(cudaMemcpyAsync(c->bytes.p, in, n, cudaMemcpyHostToDevice, h->stream));
    k_hll_max_bytes<<<(n + 255) / 256, 256, 0, h->stream>>>(c->regs.p, n, c->bytes.p, replace);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return KMGPU_OK;
}

