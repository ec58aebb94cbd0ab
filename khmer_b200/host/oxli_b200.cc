// Host layer implementation: hashing helpers, GpuStorage over the C ABI, table file formats, Hashtable.
#include "oxli_b200.hh"

#include <zlib.h>

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstring>
#include <fstream>
#include <future>
#include <limits>
#include <sstream>

#include "../../include/kmgpu.h"

namespace oxli_b200 {

using namespace read_parsers;

// ---------------------------------------------------------------------------------------------------------
// C ABI errors -> exceptions (what oxli_exception_convert.cc then maps to Python exceptions)
// ---------------------------------------------------------------------------------------------------------
static void check(int rc)
{
    if (rc == KMGPU_OK) return;
    std::string msg = kmgpu_last_error();
    if (rc == KMGPU_EINVAL || rc == KMGPU_ENONACGT) throw oxli_value_exception(msg);
    throw oxli_exception(msg);
}

static int pick_device()
{
    const char* e = getenv("KMGPU_DEVICE");
    if (e && *e) return atoi(e);
    e = getenv("LOCAL_RANK");
    if (e && *e) return atoi(e);
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// hashing helpers — scalar host versions for the single-k-mer API (hash(), reverse_hash(), get(kmer) ...)
// ---------------------------------------------------------------------------------------------------------
static inline HashIntoType code_fwd(char c) { return c == 'A' ? 0 : c == 'T' ? 1 : c == 'C' ? 2 : 3; }  // kmer_hash.hh:70-72
static inline HashIntoType code_cmp(char c) { return c == 'A' ? 1 : c == 'T' ? 0 : c == 'C' ? 3 : 2; }  // kmer_hash.hh:86-88

HashIntoType _hash(const char* kmer, WordLength k, HashIntoType& _h, HashIntoType& _r)
{
    if (k > sizeof(HashIntoType) * 4) throw oxli_exception("Supplied kmer string doesn't match the underlying k-size.");
    if (strlen(kmer) < k) throw oxli_exception("k-mer is too short to hash.");
    HashIntoType h = 0, r = 0;
    for (unsigned i = 0; i < k; i++) {
        h = (h << 2) | code_fwd(kmer[i]);
        r = (r << 2) | code_cmp(kmer[k - 1 - i]);
    }
    _h = h;
    _r = r;
    return h < r ? h : r;
}
HashIntoType _hash(const char* kmer, WordLength k)
{
    HashIntoType h, r;
    return _hash(kmer, k, h, r);
}
HashIntoType _hash_forward(const char* kmer, WordLength k)
{
    HashIntoType h, r;
    _hash(kmer, k, h, r);
    return h;
}
std::string _revhash(HashIntoType hash, WordLength k)
{
    static const char L[4] = {'A', 'T', 'C', 'G'};
    std::string s(k, 'A');
    for (int i = k - 1; i >= 0; i--) {
        s[i] = L[hash & 3];
        hash >>= 2;
    }
    return s;
}
std::string _revcomp(const std::string& kmer)
{
    // src/oxli/kmer_hash.cc:52-55,152-166: complement through a 128-entry IUPAC table that maps both cases to
    // the UPPER-case complement and every other byte to a blank; rebuilt here from the letter pairs.
    static char table[256];
    static bool ready = false;
    if (!ready) {
        memset(table, ' ', sizeof table);
        const char* pairs = "ATBVCGDHFFGCHDKMMKNNRYSSTAUAVBWWYR";
        for (const char* p = pairs; *p; p += 2) {
            table[(unsigned char)p[0]] = p[1];
            table[(unsigned char)(p[0] + 32)] = p[1];
        }
        ready = true;
    }
    std::string out(kmer.size(), ' ');
    for (size_t i = 0; i < kmer.size(); i++) out[i] = table[(unsigned char)kmer[kmer.size() - 1 - i]];
    return out;
}

static inline uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
static inline uint64_t fmix64(uint64_t v)
{
    v ^= v >> 33;
    v *= 0xff51afd7ed558ccdULL;
    v ^= v >> 33;
    v *= 0xc4ceb9fe1a85ec53ULL;
    v ^= v >> 33;
    return v;
}
// MurmurHash3_x64_128, first 64 bits (third-party/smhasher/MurmurHash3.cc:56-144), seed 0
static uint64_t murmur64(const char* key, size_t len)
{
    const uint8_t* p = (const uint8_t*)key;
    const uint64_t C1 = 0x87c37b91114253d5ULL, C2 = 0x4cf5ad432745937fULL;
    uint64_t h1 = 0, h2 = 0;
    size_t nb = len / 16;
    for (size_t b = 0; b < nb; b++) {
        uint64_t k1, k2;
        memcpy(&k1, p + 16 * b, 8);
        memcpy(&k2, p + 16 * b + 8, 8);
        k1 *= C1; k1 = rotl64(k1, 31); k1 *= C2; h1 ^= k1;
        h1 = rotl64(h1, 27); h1 += h2; h1 = h1 * 5 + 0x52dce729;
        k2 *= C2; k2 = rotl64(k2, 33); k2 *= C1; h2 ^= k2;
        h2 = rotl64(h2, 31); h2 += h1; h2 = h2 * 5 + 0x38495ab5;
    }
    const uint8_t* t = p + 16 * nb;
    size_t rem = len & 15;
    uint64_t k1 = 0, k2 = 0;
    for (size_t i = rem; i > 8; i--) k2 ^= (uint64_t)t[i - 1] << (8 * (i - 9));
    if (rem > 8) { k2 *= C2; k2 = rotl64(k2, 33); k2 *= C1; h2 ^= k2; }
    for (size_t i = std::min<size_t>(rem, 8); i > 0; i--) k1 ^= (uint64_t)t[i - 1] << (8 * (i - 1));
    if (rem > 0) { k1 *= C1; k1 = rotl64(k1, 31); k1 *= C2; h1 ^= k1; }
    h1 ^= len; h2 ^= len;
    h1 += h2; h2 += h1;
    h1 = fmix64(h1); h2 = fmix64(h2);
    h1 += h2;
    return h1;
}
HashIntoType _hash_murmur(const std::string& kmer, WordLength k, HashIntoType& h, HashIntoType& r)
{
    h = murmur64(kmer.c_str(), k);
    std::string rev = _revcomp(kmer.substr(0, k));
    if (rev == kmer.substr(0, k)) {
        r = h;
        return h;
    }
    r = murmur64(rev.c_str(), k);
    return h ^ r;
}
HashIntoType _hash_murmur(const std::string& kmer, WordLength k)
{
    HashIntoType h, r;
    return _hash_murmur(kmer, k, h, r);
}
HashIntoType _hash_murmur_forward(const std::string& kmer, WordLength k)
{
    HashIntoType h, r;
    _hash_murmur(kmer, k, h, r);
    return h;
}

std::pair<uint64_t, uint64_t> compute_band_interval(unsigned int num_bands, unsigned int band)
{
    if (band > num_bands) {
        std::string message = "'band' must be in the interval [0, 'num_bands')";
        message += ", " + std::to_string(band) + " not in [0, " + std::to_string(num_bands) + ")";
        throw InvalidValue(message);
    }
    uint64_t band_size = std::numeric_limits<uint64_t>::max() / num_bands;
    return std::make_pair(band_size * band, band_size * (band + 1));
}

bool is_prime(uint64_t n)
{
    if (n < 2) return false;
    if (n == 2) return true;
    if (n % 2 == 0) return false;
    for (unsigned long long i = 3; i < sqrt((double)n) + 1; i += 2)
        if (n % i == 0) return false;
    return true;
}
std::vector<uint64_t> get_n_primes_near_x(uint32_t n, uint64_t x)
{
    std::vector<uint64_t> primes;
    if (x == 1) {
        primes.push_back(1);
        return primes;
    }
    uint64_t i = x - 1;
    if (i % 2 == 0) i--;
    while (primes.size() != n) {
        if (is_prime(i)) primes.push_back(i);
        if (i == 1) break;
        i -= 2;
    }
    return primes;
}

// ---------------------------------------------------------------------------------------------------------
// GpuStorage
// ---------------------------------------------------------------------------------------------------------
GpuStorage::GpuStorage(StorageKind kind, HashKind hash, WordLength ksize, const std::vector<uint64_t>& tablesizes, int device)
    : _kind(kind), _hash(hash), _device(device < 0 ? pick_device() : device)
{
    recreate(ksize, tablesizes);
}

GpuStorage::~GpuStorage()
{
    if (_h) kmgpu_destroy(_h);
}

void GpuStorage::recreate(WordLength ksize, const std::vector<uint64_t>& sizes)
{
    kmgpu_sketch* nh = nullptr;
    check(kmgpu_create((int)_kind, (int)_hash, ksize, (int)sizes.size(), sizes.data(), _device, &nh));
    if (_h) kmgpu_destroy(_h);
    _h = nh;
    _tablesizes = sizes;
    _mirror.clear();
    _mirror_ptrs.clear();
}

void GpuStorage::set_ksize(WordLength k) { check(kmgpu_set_ksize(_h, k)); }
void GpuStorage::reset() { check(kmgpu_reset(_h)); }

uint64_t GpuStorage::table_nbytes(size_t i) const
{
    uint64_t n = 0;
    check(kmgpu_table_nbytes(_h, (int)i, &n));
    return n;
}

const uint64_t GpuStorage::n_occupied() const
{
    uint64_t a = 0, b = 0;
    check(kmgpu_stats(_h, &a, &b));
    return a;
}
const uint64_t GpuStorage::n_unique_kmers() const
{
    uint64_t a = 0, b = 0;
    check(kmgpu_stats(_h, &a, &b));
    return b;
}

bool GpuStorage::add(HashIntoType khash)
{
    uint64_t h = khash;
    uint8_t is_new = 0;
    check(kmgpu_add_hashes(_h, &h, 1, &is_new));
    return is_new != 0;
}

BoundedCounterType GpuStorage::test_and_set_bits(HashIntoType khash)
{
    // BitStorage returns "was new" (storage.hh:172-199); the counting storages return !count-before
    // (storage.hh:564-569, :313-318) — both are exactly what add() reports... except that a counting
    // storage's add() says "new" when ANY table was empty while !get_count says ALL-min was zero; those agree.
    return add(khash) ? 1 : 0;
}

const BoundedCounterType GpuStorage::get_count(HashIntoType khash) const
{
    uint64_t h = khash;
    uint16_t c = 0;
    check(kmgpu_get_counts(_h, &h, 1, &c));
    return c;
}

Byte** GpuStorage::get_raw_tables()
{
    _mirror.resize(_tablesizes.size());
    _mirror_ptrs.resize(_tablesizes.size());
    for (size_t i = 0; i < _tablesizes.size(); i++) {
        uint64_t n = table_nbytes(i);
        _mirror[i].resize(n);
        check(kmgpu_download_table(_h, (int)i, _mirror[i].data(), 0, n));
        _mirror_ptrs[i] = _mirror[i].data();
    }
    return _mirror_ptrs.data();
}

void GpuStorage::set_use_bigcount(bool b)
{
    if (!_supports_bigcount) throw oxli_exception("bigcount is not supported for this storage.");  // storage.cc:52-54
    check(kmgpu_set_use_bigcount(_h, b ? 1 : 0));
}
bool GpuStorage::get_use_bigcount()
{
    int on = 0;
    check(kmgpu_get_use_bigcount(_h, &on));
    return on != 0;
}

void GpuStorage::update_from(const GpuStorage& other)
{
    if (_tablesizes != other._tablesizes) throw oxli_exception("both nodegraphs must have same table sizes");
    check(kmgpu_merge(_h, other._h));
}

// ---- table files -------------------------------------------------------------------------------------
// Layout: doc/dev/binary-file-formats.rst; writers src/oxli/storage.cc:99-136 (bits), :582-638 and :640-743
// (count, plain and gz), :772-803 (smallcount).  Little-endian, packed.
namespace {

struct Sink {  // plain or gz writer
    bool gz = false;
    std::ofstream f;
    gzFile g = nullptr;
    std::string name;
    void open(const std::string& fn, bool use_gz)
    {
        name = fn;
        gz = use_gz;
        if (gz) {
            g = gzopen(fn.c_str(), "wb");
            if (g == NULL) throw oxli_file_exception(strerror(errno));
        } else {
            f.open(fn.c_str(), std::ios::binary);
        }
    }
    void write(const void* p, size_t n)
    {
        if (gz) {
            const char* c = (const char*)p;
            while (n) {  // gzwrite takes unsigned; the reference chunks at INT_MAX too (storage.cc:700-724)
                unsigned m = (unsigned)std::min<size_t>(n, 1u << 30);
                if (gzwrite(g, c, m) <= 0) {
                    int errnum = 0;
                    const char* e = gzerror(g, &errnum);
                    std::string msg = errnum == Z_ERRNO ? strerror(errno) : e;
                    gzclose(g);
                    g = nullptr;
                    throw oxli_file_exception(msg);
                }
                c += m;
                n -= m;
            }
        } else {
            f.write((const char*)p, (std::streamsize)n);
        }
    }
    void close(bool check_fail)
    {
        if (gz) {
            if (g) gzclose(g);
            g = nullptr;
        } else {
            if (check_fail && f.fail()) throw oxli_file_exception(strerror(errno));
            f.close();
        }
    }
};

struct Source {  // plain or gz reader with the reference's error texts
    bool gz = false;
    std::ifstream f;
    gzFile g = nullptr;
    std::string name;
    const char* what;  // "k-mer count file" / "k-mer graph file"
    void read(void* p, size_t n)
    {
        if (gz) {
            char* c = (char*)p;
            while (n) {
                unsigned m = (unsigned)std::min<size_t>(n, 1u << 30);
                int got = gzread(g, c, m);
                if (got <= 0 || (unsigned)got != m) {
                    std::string err = std::string("K-mer count file read error: ") + name + " " + strerror(errno);
                    int errnum = 0;
                    const char* e = gzerror(g, &errnum);
                    if (got >= 0 && (unsigned)got != m) err = "Unexpected end of " + std::string(what) + ": " + name;
                    else if (errnum != Z_ERRNO && e) err = std::string("K-mer count file read error: ") + name + " " + e;
                    throw oxli_file_exception(err);
                }
                c += m;
                n -= m;
            }
        } else {
            f.read((char*)p, (std::streamsize)n);
            if ((size_t)f.gcount() != n || f.fail()) {
                if (f.eof()) throw oxli_file_exception("Unexpected end of " + std::string(what) + ": " + name);
                throw oxli_file_exception("Error reading from " + std::string(what) + ": " + name + " " + strerror(errno));
            }
        }
    }
};

bool ends_with_gz(const std::string& fn)
{
    size_t found = fn.find_last_of(".");
    return found != std::string::npos && fn.substr(found + 1) == "gz";
}

}  // namespace

void GpuStorage::save(std::string outfilename, WordLength ksize)
{
    // ByteStorage dispatches on the ".gz" suffix (storage.cc:254-268); the other two always write plain files
    bool gz = _kind == BYTE_STORAGE && ends_with_gz(outfilename);
    Sink out;
    out.open(outfilename, gz);
    unsigned char version = SAVED_FORMAT_VERSION;
    unsigned char ht_type = _kind == BYTE_STORAGE ? SAVED_COUNTING_HT : _kind == BIT_STORAGE ? SAVED_HASHBITS : SAVED_SMALLCOUNT;
    out.write(SAVED_SIGNATURE, 4);
    out.write(&version, 1);
    out.write(&ht_type, 1);
    if (_kind == BYTE_STORAGE) {
        unsigned char use_bigcount = get_use_bigcount() ? 1 : 0;
        out.write(&use_bigcount, 1);
    }
    unsigned int save_ksize = ksize;
    unsigned char save_n_tables = (unsigned char)_tablesizes.size();
    unsigned long long save_occupied_bins = n_occupied();
    out.write(&save_ksize, sizeof(save_ksize));
    out.write(&save_n_tables, sizeof(save_n_tables));
    out.write(&save_occupied_bins, sizeof(save_occupied_bins));
    std::vector<Byte> buf;
    for (size_t i = 0; i < _tablesizes.size(); i++) {
        unsigned long long save_tablesize = _tablesizes[i];
        out.write(&save_tablesize, sizeof(save_tablesize));
        uint64_t n = table_nbytes(i);
        const uint64_t step = 256ull << 20;  // stream the table out of HBM in 256 MB pieces
        for (uint64_t o = 0; o < n; o += step) {
            uint64_t m = std::min(step, n - o);
            buf.resize(m);
            check(kmgpu_download_table(_h, (int)i, buf.data(), o, m));
            out.write(buf.data(), m);
        }
    }
    if (_kind == BYTE_STORAGE) {
        uint64_t n_counts = 0;
        check(kmgpu_bigcount_size(_h, &n_counts));
        out.write(&n_counts, sizeof(n_counts));
        if (n_counts) {
            std::vector<uint64_t> keys(n_counts);
            std::vector<uint16_t> vals(n_counts);
            check(kmgpu_bigcount_export(_h, keys.data(), vals.data(), n_counts));
            for (uint64_t j = 0; j < n_counts; j++) {
                out.write(&keys[j], sizeof(uint64_t));
                out.write(&vals[j], sizeof(uint16_t));
            }
        }
    }
    // NibbleStorage::save never checks fail() (storage.cc:772-803); the others do
    out.close(_kind != NIBBLE_STORAGE);
}

void GpuStorage::load(std::string infilename, WordLength& ksize)
{
    const bool count_like = _kind != BIT_STORAGE;
    Source in;
    in.name = infilename;
    in.what = count_like ? "k-mer count file" : "k-mer graph file";
    in.gz = _kind == BYTE_STORAGE && ends_with_gz(infilename);
    if (in.gz) {
        in.g = gzopen(infilename.c_str(), "rb");
        if (in.g == Z_NULL) throw oxli_file_exception("Cannot open k-mer count file: " + infilename);
    } else {
        in.f.open(infilename.c_str(), std::ios::binary);
        if (!in.f.is_open()) {
            std::string err = std::string("Cannot open ") + in.what + ": " + infilename;
            if (count_like) err += std::string(" ") + strerror(errno);
            throw oxli_file_exception(err);
        }
    }
    struct Closer {
        Source& s;
        ~Closer()
        {
            if (s.g) gzclose(s.g);
        }
    } closer{in};

    char signature[4];
    unsigned char version = 0, ht_type = 0, use_bigcount = 0;
    in.read(signature, 4);
    in.read(&version, 1);
    in.read(&ht_type, 1);
    const unsigned char want_type = _kind == BYTE_STORAGE ? SAVED_COUNTING_HT : _kind == BIT_STORAGE ? SAVED_HASHBITS : SAVED_SMALLCOUNT;
    if (!(std::string(signature, 4) == SAVED_SIGNATURE)) {
        std::ostringstream err;
        err << "Does not start with signature for a oxli file: 0x";
        for (size_t i = 0; i < 4; ++i) err << std::hex << (int)signature[i];
        err << " Should be: " << SAVED_SIGNATURE;
        throw oxli_file_exception(err.str());
    } else if (!(version == SAVED_FORMAT_VERSION)) {
        std::ostringstream err;
        err << "Incorrect file format version " << (int)version << " while reading " << in.what << " from " << infilename
            << "; should be " << (int)SAVED_FORMAT_VERSION;
        throw oxli_file_exception(err.str());
    } else if (!(ht_type == want_type)) {
        std::ostringstream err;
        err << "Incorrect file format type " << (int)ht_type << " while reading " << in.what << " from " << infilename;
        throw oxli_file_exception(err.str());
    }
    if (_kind == BYTE_STORAGE) in.read(&use_bigcount, 1);
    unsigned int save_ksize = 0;
    unsigned char save_n_tables = 0;
    unsigned long long save_occupied_bins = 0;
    in.read(&save_ksize, sizeof(save_ksize));
    in.read(&save_n_tables, sizeof(save_n_tables));
    in.read(&save_occupied_bins, sizeof(save_occupied_bins));

    // tables are read to host memory first (sizes are only known table by table), then the sketch is rebuilt
    std::vector<uint64_t> sizes;
    std::vector<std::vector<Byte>> tables;
    for (unsigned i = 0; i < save_n_tables; i++) {
        unsigned long long save_tablesize = 0;
        in.read(&save_tablesize, sizeof(save_tablesize));
        uint64_t nbytes = _kind == BYTE_STORAGE ? save_tablesize : _kind == NIBBLE_STORAGE ? save_tablesize / 2 + 1 : save_tablesize / 8 + 1;
        sizes.push_back(save_tablesize);
        tables.emplace_back();
        try {
            tables.back().resize(nbytes);
        } catch (const std::exception&) {
            throw oxli_file_exception(std::string("Error reading from ") + in.what + ": " + infilename + " table too large");
        }
        in.read(tables.back().data(), nbytes);
    }
    std::vector<uint64_t> keys;
    std::vector<uint16_t> vals;
    if (_kind == BYTE_STORAGE) {
        uint64_t n_counts = 0;
        in.read(&n_counts, sizeof(n_counts));
        for (uint64_t n = 0; n < n_counts; n++) {
            uint64_t kmer;
            uint16_t count;
            in.read(&kmer, sizeof(kmer));
            in.read(&count, sizeof(count));
            keys.push_back(kmer);
            vals.push_back(count);
        }
    }
    ksize = (WordLength)save_ksize;
    recreate(ksize, sizes);
    for (size_t i = 0; i < sizes.size(); i++) check(kmgpu_upload_table(_h, (int)i, tables[i].data(), 0, tables[i].size()));
    check(kmgpu_set_stats(_h, save_occupied_bins, 0));
    if (_kind == BYTE_STORAGE) {
        check(kmgpu_set_use_bigcount(_h, use_bigcount ? 1 : 0));
        if (!keys.empty()) check(kmgpu_bigcount_import(_h, keys.data(), vals.data(), keys.size()));
    }
}

// ---------------------------------------------------------------------------------------------------------
// Hashtable
// ---------------------------------------------------------------------------------------------------------
HashIntoType Hashtable::hash_dna(const char* kmer) const
{
    if (_hashkind == TWOBIT_HASH) return _hash(kmer, _ksize);
    if (strlen(kmer) < _ksize) throw oxli_exception("k-mer is too short to hash.");
    return _hash_murmur(std::string(kmer, _ksize), _ksize);
}
HashIntoType Hashtable::hash_dna_top_strand(const char* kmer) const
{
    HashIntoType f = 0, r = 0;
    if (_hashkind == TWOBIT_HASH) _hash(kmer, _ksize, f, r);
    else _hash_murmur(std::string(kmer, _ksize), _ksize, f, r);
    return f;
}
HashIntoType Hashtable::hash_dna_bottom_strand(const char* kmer) const
{
    HashIntoType f = 0, r = 0;
    if (_hashkind == TWOBIT_HASH) _hash(kmer, _ksize, f, r);
    else _hash_murmur(std::string(kmer, _ksize), _ksize, f, r);
    return r;
}
std::string Hashtable::unhash_dna(HashIntoType hashval) const
{
    if (_hashkind == MURMUR_HASH) throw oxli_exception("This hash function is not reversible.");  // hashtable.hh:521-526
    return _revhash(hashval, _ksize);
}

void Hashtable::load(std::string filename)
{
    store->load(filename, _ksize);
}

// sequences without cleaning go to the device as they are; a Murmur table refuses non-ACGT bytes there, in
// which case the (rare) sequence is hashed here, letter for letter as the reference does, and added by hash
static bool device_can_hash_raw(HashKind hk, const std::string& s)
{
    if (hk == TWOBIT_HASH) return true;
    for (char c : s)
        if (!(c == 'A' || c == 'C' || c == 'G' || c == 'T')) return false;
    return true;
}

unsigned int Hashtable::consume_string(const std::string& s)
{
    if (s.size() < _ksize) return 0;
    if (device_can_hash_raw(_hashkind, s)) {
        uint64_t offs[2] = {0, s.size()};
        uint64_t n = 0;
        check(kmgpu_consume_reads(store->handle(), s.data(), offs, 1, 0, nullptr, nullptr, &n));
        return (unsigned int)n;
    }
    std::vector<HashIntoType> hs;
    get_kmer_hashes(s, hs);
    std::vector<uint64_t> h64(hs.begin(), hs.end());
    check(kmgpu_add_hashes(store->handle(), h64.data(), h64.size(), nullptr));
    return (unsigned int)hs.size();
}

void Hashtable::get_kmers(const std::string& s, std::vector<std::string>& kmers_vec) const
{
    if (s.length() < _ksize) return;
    for (unsigned int i = 0; i < s.length() - _ksize + 1; i++) kmers_vec.push_back(s.substr(i, _ksize));
}

void Hashtable::get_kmer_hashes(const std::string& s, std::vector<HashIntoType>& kmers_vec) const
{
    if (s.size() < _ksize) return;
    size_t n = s.size() - _ksize + 1;
    if (device_can_hash_raw(_hashkind, s) && n > 64) {
        std::vector<uint64_t> out(n);
        uint64_t offs[2] = {0, s.size()}, got = 0;
        check(kmgpu_kmer_hashes(store->handle(), s.data(), offs, 1, 0, out.data(), &got));
        kmers_vec.insert(kmers_vec.end(), out.begin(), out.begin() + got);
        return;
    }
    for (size_t i = 0; i < n; i++) {
        if (_hashkind == TWOBIT_HASH) kmers_vec.push_back(_hash(s.c_str() + i, _ksize));
        else kmers_vec.push_back(_hash_murmur(s.substr(i, _ksize), _ksize));
    }
}

void Hashtable::get_kmer_counts(const std::string& s, std::vector<BoundedCounterType>& counts) const
{
    if (s.size() < _ksize) return;
    size_t n = s.size() - _ksize + 1;
    std::vector<uint16_t> out(n);
    if (device_can_hash_raw(_hashkind, s)) {
        uint64_t offs[2] = {0, s.size()}, got = 0;
        check(kmgpu_kmer_counts(store->handle(), s.data(), offs, 1, 0, out.data(), &got));
    } else {
        std::vector<HashIntoType> hs;
        get_kmer_hashes(s, hs);
        std::vector<uint64_t> h64(hs.begin(), hs.end());
        check(kmgpu_get_counts(store->handle(), h64.data(), h64.size(), out.data()));
    }
    counts.insert(counts.end(), out.begin(), out.end());
}

void Hashtable::get_median_count(const std::string& s, BoundedCounterType& median, float& average, float& stddev)
{
    if (s.size() < _ksize) throw oxli_exception("no k-mer counts for this string; too short?");
    if (device_can_hash_raw(_hashkind, s)) {
        uint64_t offs[2] = {0, s.size()};
        uint16_t m = 0;
        uint32_t nk = 0;
        check(kmgpu_read_medians(store->handle(), s.data(), offs, 1, 0, &m, &average, &stddev, &nk));
        median = m;
        return;
    }
    // non-ACGT letters under a Murmur table: counts by hash, statistics exactly as hashtable.cc:299-328
    std::vector<BoundedCounterType> counts;
    get_kmer_counts(s, counts);
    average = 0;
    for (auto c : counts) average += c;
    average /= float(counts.size());
    stddev = 0;
    for (auto c : counts) stddev += (float(c) - average) * (float(c) - average);
    stddev /= float(counts.size());
    stddev = sqrt(stddev);
    std::sort(counts.begin(), counts.end());
    median = counts[counts.size() / 2];
}

bool Hashtable::median_at_least(const std::string& s, unsigned int cutoff)
{
    if (s.size() < _ksize) throw oxli_exception("past end of iterator");
    if (device_can_hash_raw(_hashkind, s)) {
        uint64_t offs[2] = {0, s.size()};
        uint8_t out = 0;
        check(kmgpu_median_at_least(store->handle(), s.data(), offs, 1, 0, cutoff, &out));
        return out == 1;
    }
    std::vector<BoundedCounterType> counts;
    get_kmer_counts(s, counts);
    unsigned int min_req = 0.5 + float(s.size() - _ksize + 1) / 2;
    unsigned int num = 0;
    for (auto c : counts) num += c >= cutoff;
    return num >= min_req;
}

static void pack_strings(const std::vector<std::string>& seqs, std::string& buf, std::vector<uint64_t>& offs)
{
    offs.assign(1, 0);
    size_t total = 0;
    for (auto& s : seqs) total += s.size();
    buf.clear();
    buf.reserve(total);
    for (auto& s : seqs) {
        buf += s;
        offs.push_back(buf.size());
    }
}

void Hashtable::get_median_counts(const std::vector<std::string>& seqs, std::vector<BoundedCounterType>& median,
                                  std::vector<float>& average, std::vector<float>& stddev, std::vector<uint32_t>& n_kmers)
{
    std::string buf;
    std::vector<uint64_t> offs;
    pack_strings(seqs, buf, offs);
    size_t n = seqs.size();
    std::vector<uint16_t> m(n);
    average.assign(n, 0.f);
    stddev.assign(n, 0.f);
    n_kmers.assign(n, 0);
    if (n) check(kmgpu_read_medians(store->handle(), buf.data(), offs.data(), n, 0, m.data(), average.data(), stddev.data(), n_kmers.data()));
    median.assign(m.begin(), m.end());
}

void Hashtable::median_at_least_batch(const std::vector<std::string>& seqs, unsigned int cutoff, std::vector<uint8_t>& out)
{
    std::string buf;
    std::vector<uint64_t> offs;
    pack_strings(seqs, buf, offs);
    out.assign(seqs.size(), 0);
    if (!seqs.empty()) check(kmgpu_median_at_least(store->handle(), buf.data(), offs.data(), seqs.size(), 0, cutoff, out.data()));
}

// The loop of scripts/normalize-by-median.py:155-179 (Normalizer.__call__ + ReadBundle.coverages_at_least, khmer/utils.py:178-180)
// over a batch of cleaned sequences in stream order, resolved on the device: keep[i] = 1 iff read i's bundle was kept (and consumed).
unsigned long long Hashtable::normalize_batch(const std::vector<std::string>& seqs, unsigned int cutoff, const std::vector<uint8_t>& pair_with_next,
                                              std::vector<uint8_t>& keep)
{
    std::string buf;
    std::vector<uint64_t> offs;
    pack_strings(seqs, buf, offs);
    keep.assign(seqs.size(), 0);
    if (seqs.empty()) return 0;
    if (!pair_with_next.empty() && pair_with_next.size() != seqs.size()) throw oxli_value_exception("pair flags: one per read");
    uint64_t kept = 0, kmers = 0;
    check(kmgpu_normalize_batch(store->handle(), buf.data(), offs.data(), seqs.size(), 0, pair_with_next.empty() ? nullptr : pair_with_next.data(), cutoff,
                                keep.data(), &kept, &kmers));
    return kmers;
}

unsigned long long Hashtable::trim_low_abund_pass1(const std::vector<std::string>& seqs, unsigned int trim_at_coverage, unsigned int cutoff,
                                                   unsigned int diginorm_coverage, const std::vector<uint8_t>& pair_with_next, bool clean,
                                                   std::vector<uint8_t>& action, std::vector<uint32_t>& trim_pos)
{
    std::string buf;
    std::vector<uint64_t> offs;
    pack_strings(seqs, buf, offs);
    action.assign(seqs.size(), 0);
    trim_pos.assign(seqs.size(), 0);
    if (seqs.empty()) return 0;
    if (!pair_with_next.empty() && pair_with_next.size() != seqs.size()) throw oxli_value_exception("pair flags: one per read");
    uint64_t kmers = 0;
    check(kmgpu_trim_low_abund_pass1(store->handle(), buf.data(), offs.data(), seqs.size(), clean ? KMGPU_CLEAN : 0,
                                     pair_with_next.empty() ? nullptr : pair_with_next.data(), trim_at_coverage, cutoff, diginorm_coverage,
                                     action.data(), trim_pos.data(), &kmers));
    return kmers;
}

void Hashtable::trim_low_abund_pass2(const std::vector<std::string>& seqs, unsigned int trim_at_coverage, unsigned int cutoff, bool variable_coverage,
                                     const std::vector<uint8_t>& pair_with_next, bool clean, std::vector<uint8_t>& action,
                                     std::vector<uint32_t>& trim_pos)
{
    std::string buf;
    std::vector<uint64_t> offs;
    pack_strings(seqs, buf, offs);
    action.assign(seqs.size(), 0);
    trim_pos.assign(seqs.size(), 0);
    if (seqs.empty()) return;
    if (!pair_with_next.empty() && pair_with_next.size() != seqs.size()) throw oxli_value_exception("pair flags: one per read");
    check(kmgpu_trim_low_abund_pass2(store->handle(), buf.data(), offs.data(), seqs.size(), clean ? KMGPU_CLEAN : 0,
                                     pair_with_next.empty() ? nullptr : pair_with_next.data(), trim_at_coverage, cutoff, variable_coverage ? 1 : 0,
                                     action.data(), trim_pos.data()));
}

BoundedCounterType Hashtable::get_min_count(const std::string& s)
{
    std::vector<BoundedCounterType> counts;
    get_kmer_counts(s, counts);
    BoundedCounterType mn = MAX_KCOUNT;  // hashtable.cc:419-434 starts from MAX_KCOUNT
    for (auto c : counts)
        if (c < mn) mn = c;
    return mn;
}
BoundedCounterType Hashtable::get_max_count(const std::string& s)
{
    std::vector<BoundedCounterType> counts;
    get_kmer_counts(s, counts);
    BoundedCounterType mx = 0;
    for (auto c : counts)
        if (c > mx) mx = c;
    return mx;
}

unsigned long Hashtable::trim_on_abundance(std::string seq, BoundedCounterType min_abund) const
{
    std::vector<BoundedCounterType> c;
    get_kmer_counts(seq, c);
    if (c.empty()) return 0;
    if (c.size() == 1 || c[0] < min_abund) return 0;
    unsigned long i = _ksize;
    for (size_t j = 1; j < c.size(); j++) {
        if (c[j] < min_abund) return i;
        i++;
    }
    return seq.length();
}
unsigned long Hashtable::trim_below_abundance(std::string seq, BoundedCounterType max_abund) const
{
    std::vector<BoundedCounterType> c;
    get_kmer_counts(seq, c);
    if (c.empty()) return 0;
    if (c.size() == 1 || c[0] > max_abund) return 0;
    unsigned long i = _ksize;
    for (size_t j = 1; j < c.size(); j++) {
        if (c[j] > max_abund) return i;
        i++;
    }
    return seq.length();
}
std::vector<unsigned int> Hashtable::find_spectral_error_positions(std::string seq, BoundedCounterType max_abund) const
{
    // restated from hashtable.cc:565-612 over the vector of counts: after the j-th next() the iterator's
    // start position is j-1 and its end position j-1+k; done() holds once the last k-mer has been returned
    std::vector<unsigned int> posns;
    std::vector<BoundedCounterType> c;
    get_kmer_counts(seq, c);
    if (c.empty()) throw oxli_exception("past end of iterator");
    size_t n = c.size(), cur = 0;
    if (n == 1) return posns;
    while (cur != n - 1) {
        if (c[cur] > max_abund) break;
        cur++;
    }
    if (cur == n - 1) return posns;
    if (cur > 0) posns.push_back((unsigned)cur - 1);
    while (cur != n - 1) {
        cur++;
        if (c[cur] <= max_abund) {
            posns.push_back((unsigned)(cur + _ksize - 1));
            while (cur != n - 1) {
                cur++;
                if (c[cur] > max_abund) break;
            }
        }
    }
    return posns;
}

// ---- bulk loaders -------------------------------------------------------------------------------------
static uint64_t feed_bases()
{
    const char* e = getenv("KMGPU_FEED_BASES");
    // half a device chunk per batch: the first batch's parse and the last batch's ingest are not overlapped with anything, so smaller
    // batches shorten a file's wall time until the per-chunk pass over the sketch takes over (measured on the headline table, 2 M
    // reads: 32 Mi 9.9, 48 Mi 10.7, 72 Mi 11.3, 144 Mi 9.7 G k-mers/s)
    return e && *e ? strtoull(e, nullptr, 10) : (72ull << 20);
}

template <typename SeqIO>
void Hashtable::bulk_consume(ReadParserPtr<SeqIO>& parser, const uint64_t* band, Hashtable* mask, unsigned int threshold,
                             bool consume_masked, unsigned int& total_reads, unsigned long long& n_consumed)
{
    // Hashtable::consume_seqfile (hashtable.cc:126-150): reads are cleaned (on the device) and all their
    // k-mers counted.  Reads are pulled from the shared parser a batch at a time, so several host threads
    // may run this on one table as the reference's scripts do.
    kmgpu_band_t b;
    kmgpu_mask_t m;
    if (band) {
        b.lo = band[0];
        b.hi = band[1];
    }
    if (mask) {
        m.mask = mask->store->handle();
        m.threshold = threshold;
        m.consume_masked = consume_masked ? 1 : 0;
    }
    // two pinned batches: the next one is parsed (by the reader's threads) while the device ingests the current one
    // the parser threads clean and 2-bit pack the reads as they copy them (KMGPU_FEED_PACKED=0: ASCII batches, cleaned and
    // packed on the device)
    static const bool packed = [] { const char* e = getenv("KMGPU_FEED_PACKED"); return !(e && *e == '0'); }();
    ReadBatch batch[2];
    batch[0].pack = batch[1].pack = packed;
    auto fetch = [&](int slot) -> size_t {
        batch[slot].clear();
        return parser->io().read_batch(feed_bases(), batch[slot]);
    };
    int cur = 0;
    size_t got = fetch(cur);
    while (got) {
        std::future<size_t> next = std::async(std::launch::async, fetch, cur ^ 1);
        uint64_t n = 0;
        int rc = packed ? kmgpu_consume_packed(store->handle(), batch[cur].words(), batch[cur].n_words(), batch[cur].offsets.data(), got,
                                               band ? &b : nullptr, mask ? &m : nullptr, &n)
                        : kmgpu_consume_reads(store->handle(), batch[cur].seqs, batch[cur].offsets.data(), got, KMGPU_CLEAN, band ? &b : nullptr,
                                              mask ? &m : nullptr, &n);
        __sync_add_and_fetch(&n_consumed, n);
        __sync_add_and_fetch(&total_reads, (unsigned int)got);
        size_t got_next = 0;
        try {
            got_next = next.get();
        } catch (...) {
            check(rc);
            throw;
        }
        check(rc);
        got = got_next;
        cur ^= 1;
    }
}

template <typename SeqIO>
void Hashtable::consume_seqfile(std::string const& filename, unsigned int& total_reads, unsigned long long& n_consumed)
{
    ReadParserPtr<SeqIO> parser = get_parser<SeqIO>(filename);
    consume_seqfile<SeqIO>(parser, total_reads, n_consumed);
}
template <typename SeqIO>
void Hashtable::consume_seqfile(ReadParserPtr<SeqIO>& parser, unsigned int& total_reads, unsigned long long& n_consumed)
{
    bulk_consume<SeqIO>(parser, nullptr, nullptr, 0, false, total_reads, n_consumed);
}
template <typename SeqIO>
void Hashtable::consume_seqfile_with_mask(std::string const& filename, Hashtable* mask, unsigned int threshold, unsigned int& total_reads,
                                          unsigned long long& n_consumed, bool consume_masked)
{
    ReadParserPtr<SeqIO> parser = get_parser<SeqIO>(filename);
    consume_seqfile_with_mask<SeqIO>(parser, mask, threshold, total_reads, n_consumed, consume_masked);
}
template <typename SeqIO>
void Hashtable::consume_seqfile_with_mask(ReadParserPtr<SeqIO>& parser, Hashtable* mask, unsigned int threshold, unsigned int& total_reads,
                                          unsigned long long& n_consumed, bool consume_masked)
{
    bulk_consume<SeqIO>(parser, nullptr, mask, threshold, consume_masked, total_reads, n_consumed);
}
template <typename SeqIO>
void Hashtable::consume_seqfile_banding(std::string const& filename, unsigned int num_bands, unsigned int band, unsigned int& total_reads,
                                        unsigned long long& n_consumed)
{
    ReadParserPtr<SeqIO> parser = get_parser<SeqIO>(filename);
    consume_seqfile_banding<SeqIO>(parser, num_bands, band, total_reads, n_consumed);
}
template <typename SeqIO>
void Hashtable::consume_seqfile_banding(ReadParserPtr<SeqIO>& parser, unsigned int num_bands, unsigned int band, unsigned int& total_reads,
                                        unsigned long long& n_consumed)
{
    std::pair<uint64_t, uint64_t> interval = compute_band_interval(num_bands, band);
    uint64_t b[2] = {interval.first, interval.second};
    bulk_consume<SeqIO>(parser, b, nullptr, 0, false, total_reads, n_consumed);
}
template <typename SeqIO>
void Hashtable::consume_seqfile_banding_with_mask(std::string const& filename, unsigned int num_bands, unsigned int band, Hashtable* mask,
                                                  unsigned int threshold, unsigned int& total_reads, unsigned long long& n_consumed,
                                                  bool consume_masked)
{
    ReadParserPtr<SeqIO> parser = get_parser<SeqIO>(filename);
    consume_seqfile_banding_with_mask<SeqIO>(parser, num_bands, band, mask, threshold, total_reads, n_consumed, consume_masked);
}
template <typename SeqIO>
void Hashtable::consume_seqfile_banding_with_mask(ReadParserPtr<SeqIO>& parser, unsigned int num_bands, unsigned int band, Hashtable* mask,
                                                  unsigned int threshold, unsigned int& total_reads, unsigned long long& n_consumed,
                                                  bool consume_masked)
{
    std::pair<uint64_t, uint64_t> interval = compute_band_interval(num_bands, band);
    uint64_t b[2] = {interval.first, interval.second};
    bulk_consume<SeqIO>(parser, b, mask, threshold, consume_masked, total_reads, n_consumed);
}

// ---------------------------------------------------------------------------------------------------------
// tagging
// ---------------------------------------------------------------------------------------------------------
void Hashtable::_set_tag_density(unsigned int d)
{
    // hashgraph.hh:128-135
    if (!(d % 2 == 0) || !all_tags.empty()) throw oxli_exception("Invalid tag density: must be even, and the tag set must be empty.");
    _tag_density = d;
}

// Hashgraph::consume_sequence_and_tag (hashgraph.cc:200-271) for every read of a batch, with store->test_and_set_bits(kmer)
// replaced by the bit the device returned for that k-mer.  Reads without a k-mer are skipped (the reference inserts an
// uninitialised hash value for them: undefined behaviour, consciously not reproduced).
void Hashtable::tag_batch(const char* seqs, const uint64_t* offsets, size_t n_reads, unsigned long long& n_consumed)
{
    if (_hashkind != TWOBIT_HASH) throw oxli_exception("tagging needs a two-bit hash sketch (Countgraph, SmallCountgraph, Nodegraph)");
    if (n_reads == 0) return;
    const uint64_t n_bases = offsets[n_reads] - offsets[0];
    std::vector<uint32_t> bits((n_bases + 31) / 32 + 1);
    uint64_t n_kmers = 0, n_new = 0;
    check(kmgpu_consume_reads_new(store->handle(), seqs, offsets, n_reads, KMGPU_CLEAN, bits.data(), &n_kmers, &n_new));
    n_consumed += n_new;
    const unsigned k = _ksize;
    const HashIntoType mask = k == 32 ? ~(HashIntoType)0 : (((HashIntoType)1 << (2 * k)) - 1);
    std::lock_guard<std::mutex> g(tags_mu);   // the reference takes a spin lock per k-mer; one batch at a time here
    auto clean = [](char c) -> char {
        switch (c) {
        case 'A': case 'C': case 'G': case 'T': return c;
        case 'a': return 'A';
        case 'c': return 'C';
        case 'g': return 'G';
        case 't': return 'T';
        default: return 'A';
        }
    };
    for (size_t r = 0; r < n_reads; r++) {
        const char* s = seqs + offsets[r];
        const uint64_t len = offsets[r + 1] - offsets[r], base = offsets[r] - offsets[0];
        if (len < k) continue;
        // KmerIterator (kmer_hash.cc:278-343) over the cleaned read (Read::set_clean_seq: ACGT kept, acgt upper-cased, else 'A')
        HashIntoType f = 0, rc = 0;
        for (unsigned i = 0; i + 1 < k; i++) {
            const char c = clean(s[i]);
            f = (f << 2) | code_fwd(c);
            rc = (rc >> 2) | (code_cmp(c) << (2 * k - 2));
        }
        unsigned int since = _tag_density / 2 + 1;
        HashIntoType kmer = 0;
        for (uint64_t i = 0; i + k <= len; i++) {
            const char c = clean(s[i + k - 1]);
            f = ((f << 2) | code_fwd(c)) & mask;
            rc = (rc >> 2) | (code_cmp(c) << (2 * k - 2));
            kmer = f < rc ? f : rc;
            const uint64_t p = base + i;
            const bool is_new = (bits[p >> 5] >> (p & 31)) & 1u;
            if (is_new) {
                ++since;
            } else if (all_tags.count(kmer)) {
                since = 1;
            } else {
                ++since;
            }
            if (since >= _tag_density) {
                all_tags.insert(kmer);
                since = 1;
            }
        }
        if (since >= _tag_density / 2 - 1) all_tags.insert(kmer);   // the last k-mer, too
    }
}

void Hashtable::consume_sequence_and_tag(const std::string& cleaned_seq, unsigned long long& n_consumed)
{
    const uint64_t offs[2] = {0, cleaned_seq.size()};
    tag_batch(cleaned_seq.data(), offs, 1, n_consumed);
}

template <typename SeqIO>
void Hashtable::consume_seqfile_and_tag(std::string const& filename, unsigned int& total_reads, unsigned long long& n_consumed)
{
    ReadParserPtr<SeqIO> parser = get_parser<SeqIO>(filename);
    consume_seqfile_and_tag<SeqIO>(parser, total_reads, n_consumed);
}
template <typename SeqIO>
void Hashtable::consume_seqfile_and_tag(ReadParserPtr<SeqIO>& parser, unsigned int& total_reads, unsigned long long& n_consumed)
{
    total_reads = 0;      // hashgraph.cc:300-301
    n_consumed = 0;
    ReadBatch batch;      // ASCII: the tag scan hashes the reads on the host
    while (true) {
        batch.clear();
        size_t got = parser->io().read_batch(feed_bases(), batch);
        if (got == 0) break;
        unsigned long long n = 0;
        tag_batch(batch.seqs, batch.offsets.data(), got, n);
        __sync_add_and_fetch(&n_consumed, n);
        __sync_add_and_fetch(&total_reads, (unsigned int)got);
    }
}

void Hashtable::save_tagset(std::string filename)
{
    // hashgraph.cc:55-88: "OXLI", version, SAVED_TAGS, ksize (u32), number of tags (u64), tag density (u32), the tags in set order
    std::ofstream out(filename.c_str(), std::ios::binary);
    const size_t n = all_tags.size();
    unsigned int save_ksize = _ksize;
    out.write(SAVED_SIGNATURE, 4);
    unsigned char version = SAVED_FORMAT_VERSION, ht_type = SAVED_TAGS;
    out.write((const char*)&version, 1);
    out.write((const char*)&ht_type, 1);
    out.write((const char*)&save_ksize, sizeof save_ksize);
    out.write((const char*)&n, sizeof n);
    out.write((const char*)&_tag_density, sizeof _tag_density);
    std::vector<HashIntoType> buf(all_tags.begin(), all_tags.end());
    out.write((const char*)buf.data(), sizeof(HashIntoType) * n);
    if (out.fail()) throw oxli_file_exception(strerror(errno));
    out.close();
}

void Hashtable::load_tagset(std::string filename, bool clear)
{
    // hashgraph.cc:90-175
    std::ifstream in(filename.c_str(), std::ios::binary);
    if (!in.is_open()) throw oxli_file_exception("Cannot open tagset file: " + filename);
    char sig[4];
    unsigned char version = 0, ht_type = 0;
    unsigned int save_ksize = 0, density = 0;
    size_t n = 0;
    in.read(sig, 4);
    in.read((char*)&version, 1);
    in.read((char*)&ht_type, 1);
    if (!in || std::string(sig, 4) != SAVED_SIGNATURE) throw oxli_file_exception("Does not start with signature for a oxli file: " + filename);
    if (version != SAVED_FORMAT_VERSION) throw oxli_file_exception("Incorrect file format version " + std::to_string((int)version) + " while reading tagset from " + filename);
    if (ht_type != SAVED_TAGS) throw oxli_file_exception("Incorrect file format type " + std::to_string((int)ht_type) + " while reading tagset from " + filename);
    in.read((char*)&save_ksize, sizeof save_ksize);
    if (!in || save_ksize != _ksize) throw oxli_file_exception("Incorrect k-mer size " + std::to_string(save_ksize) + " while reading tagset from " + filename);
    in.read((char*)&n, sizeof n);
    in.read((char*)&density, sizeof density);
    std::vector<HashIntoType> buf(n);
    in.read((char*)buf.data(), sizeof(HashIntoType) * n);
    if (!in) throw oxli_file_exception("Error reading tagset file: " + filename);
    if (clear) all_tags.clear();
    _tag_density = density;
    all_tags.insert(buf.begin(), buf.end());
}

template <typename SeqIO>
uint64_t* Hashtable::abundance_distribution(ReadParserPtr<SeqIO>& parser, Hashtable* tracking)
{
    uint64_t* dist = new uint64_t[MAX_BIGCOUNT + 1];
    for (uint64_t i = 0; i <= MAX_BIGCOUNT; i++) dist[i] = 0;
    ReadBatch batch;
    try {
        while (true) {
            batch.clear();
            size_t got = parser->io().read_batch(feed_bases(), batch);
            if (got == 0) break;
            check(kmgpu_abundance_distribution(store->handle(), tracking->store->handle(), batch.seqs, batch.offsets.data(), got, KMGPU_CLEAN, dist));
        }
    } catch (...) {
        delete[] dist;
        throw;
    }
    return dist;
}
template <typename SeqIO>
uint64_t* Hashtable::abundance_distribution(std::string filename, Hashtable* tracking)
{
    ReadParserPtr<SeqIO> parser = get_parser<SeqIO>(filename);
    return abundance_distribution(parser, tracking);
}

void Nodegraph::update_from(const Nodegraph& other)
{
    store->update_from(*other.store);
}

// template instantiations used by the bindings (cf. hashtable.cc:615-697)
template void Hashtable::consume_seqfile<FastxReader>(std::string const&, unsigned int&, unsigned long long&);
template void Hashtable::consume_seqfile<FastxReader>(ReadParserPtr<FastxReader>&, unsigned int&, unsigned long long&);
template void Hashtable::consume_seqfile_with_mask<FastxReader>(std::string const&, Hashtable*, unsigned int, unsigned int&,
                                                                unsigned long long&, bool);
template void Hashtable::consume_seqfile_with_mask<FastxReader>(ReadParserPtr<FastxReader>&, Hashtable*, unsigned int, unsigned int&,
                                                                unsigned long long&, bool);
template void Hashtable::consume_seqfile_banding<FastxReader>(std::string const&, unsigned int, unsigned int, unsigned int&,
                                                              unsigned long long&);
template void Hashtable::consume_seqfile_banding<FastxReader>(ReadParserPtr<FastxReader>&, unsigned int, unsigned int, unsigned int&,
                                                              unsigned long long&);
template void Hashtable::consume_seqfile_banding_with_mask<FastxReader>(std::string const&, unsigned int, unsigned int, Hashtable*,
                                                                        unsigned int, unsigned int&, unsigned long long&, bool);
template void Hashtable::consume_seqfile_banding_with_mask<FastxReader>(ReadParserPtr<FastxReader>&, unsigned int, unsigned int,
                                                                        Hashtable*, unsigned int, unsigned int&, unsigned long long&,
                                                                        bool);
template void Hashtable::consume_seqfile_and_tag<FastxReader>(std::string const&, unsigned int&, unsigned long long&);
template void Hashtable::consume_seqfile_and_tag<FastxReader>(ReadParserPtr<FastxReader>&, unsigned int&, unsigned long long&);
template uint64_t* Hashtable::abundance_distribution<FastxReader>(ReadParserPtr<FastxReader>&, Hashtable*);
template uint64_t* Hashtable::abundance_distribution<FastxReader>(std::string, Hashtable*);

}  // namespace oxli_b200
