// liboxli-compatible host layer over the kmgpu C ABI (include/kmgpu.h).
//
// Mirrors, for the ingestion path only, the reference's C++ interface:
//   oxli::Storage            include/oxli/storage.hh:56-78      -> oxli_b200::Storage / GpuStorage
//   oxli::Hashtable          include/oxli/hashtable.hh:127-433  -> oxli_b200::Hashtable
//   Countgraph & friends     include/oxli/hashgraph.hh:273-296, hashtable.hh:591-627
//   read_parsers             include/oxli/read_parsers.hh       -> oxli_b200::read_parsers (own FASTA/FASTQ reader)
//   exceptions               include/oxli/oxli_exception.hh:47-141
// Same names, argument meaning and error behaviour; the tables live in GPU memory behind the C ABI and there
// is no CPU implementation of the hot path here.  No CUDA headers are needed to build this layer.
#pragma once
#include <cstdint>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <utility>
#include <set>
#include <mutex>
#include <vector>

struct kmgpu_sketch;

namespace oxli_b200 {

typedef unsigned long long HashIntoType;   // include/oxli/oxli.hh
typedef unsigned short BoundedCounterType;
typedef unsigned char WordLength;
typedef unsigned char Byte;

constexpr unsigned MAX_KCOUNT = 255;
constexpr unsigned MAX_BIGCOUNT = 65535;
// file format constants, include/oxli/oxli.hh:89-98
constexpr const char* SAVED_SIGNATURE = "OXLI";
constexpr unsigned char SAVED_FORMAT_VERSION = 4;
constexpr unsigned char SAVED_COUNTING_HT = 1;
constexpr unsigned char SAVED_HASHBITS = 2;
constexpr unsigned char SAVED_TAGS = 3;
constexpr unsigned char SAVED_SMALLCOUNT = 7;

// ---- exceptions (include/oxli/oxli_exception.hh) -------------------------------------------------------
class oxli_exception : public std::exception {
public:
    explicit oxli_exception(const std::string& msg = "Generic oxli exception") : _msg(msg) {}
    const char* what() const noexcept override { return _msg.c_str(); }
protected:
    std::string _msg;
};
class oxli_file_exception : public oxli_exception {
public:
    explicit oxli_file_exception(const std::string& msg) : oxli_exception(msg) {}
};
class oxli_value_exception : public oxli_exception {
public:
    explicit oxli_value_exception(const std::string& msg) : oxli_exception(msg) {}
};
class InvalidValue : public oxli_value_exception {
public:
    explicit InvalidValue(const std::string& msg) : oxli_value_exception(msg) {}
};
class InvalidStream : public oxli_file_exception {
public:
    explicit InvalidStream(const std::string& msg = "Generic InvalidStream error") : oxli_file_exception(msg) {}
};
class StreamReadError : public oxli_file_exception {
public:
    explicit StreamReadError(const std::string& msg = "Generic StreamReadError error") : oxli_file_exception(msg) {}
};
class NoMoreReadsAvailable : public oxli_file_exception {
public:
    explicit NoMoreReadsAvailable(const std::string& msg = "No more reads available in this stream.") : oxli_file_exception(msg) {}
};
class InvalidRead : public oxli_value_exception {
public:
    explicit InvalidRead(const std::string& msg = "Invalid FASTA/Q read") : oxli_value_exception(msg) {}
};

// ---- hashing helpers (src/oxli/kmer_hash.cc, include/oxli/hashtable.hh:79-123) ---------------------------
HashIntoType _hash(const char* kmer, WordLength k);
HashIntoType _hash(const char* kmer, WordLength k, HashIntoType& h, HashIntoType& r);
HashIntoType _hash_forward(const char* kmer, WordLength k);
std::string _revhash(HashIntoType hash, WordLength k);
std::string _revcomp(const std::string& kmer);
HashIntoType _hash_murmur(const std::string& kmer, WordLength k);
HashIntoType _hash_murmur(const std::string& kmer, WordLength k, HashIntoType& h, HashIntoType& r);
HashIntoType _hash_murmur_forward(const std::string& kmer, WordLength k);
std::pair<uint64_t, uint64_t> compute_band_interval(unsigned int num_bands, unsigned int band);
bool is_prime(uint64_t n);
std::vector<uint64_t> get_n_primes_near_x(uint32_t n, uint64_t x);

// ---- reads (include/oxli/read_parsers.hh) ------------------------------------------------------------
namespace read_parsers {

struct Read {
    std::string name, description, sequence, quality, cleaned_seq;
    void reset();
    void set_clean_seq();  // read_parsers.hh:128-133
};
typedef std::pair<Read, Read> ReadPair;

// A batch of raw (uncleaned) reads, concatenated, for the device feed.  The sequence buffer is page-locked host
// memory obtained through the C ABI (kmgpu_alloc_pinned) so that uploads are asynchronous and run at PCIe speed;
// it is reused from batch to batch.
struct ReadBatch {
    char* seqs = nullptr;            // ASCII bases — or, when `pack` is set, the 2-bit stream (see words())
    size_t n_bases = 0, cap = 0;     // cap in bytes
    std::vector<uint64_t> offsets;   // n_reads + 1 entries once filled
    bool pinned = false;
    // pack: the parser threads write the CLEANED reads (Read::set_clean_seq, read_parsers.hh:128-133) straight into the
    // device's stream format — 64-bit words, 32 bases per word, first base in the top two bits, A0 T1 C2 G3
    // (kmer_hash.hh:70-72) — so a batch crosses PCIe at 2 bits per base (kmgpu_consume_packed)
    bool pack = false;
    uint64_t* words() const { return reinterpret_cast<uint64_t*>(seqs); }
    size_t n_words() const { return (n_bases + 31) / 32; }
    ReadBatch() {}
    ~ReadBatch();
    ReadBatch(const ReadBatch&) = delete;
    ReadBatch& operator=(const ReadBatch&) = delete;
    void clear()
    {
        n_bases = 0;
        offsets.clear();
    }
    void reserve(size_t n);          // keeps the first n_bases bytes
    size_t n_reads() const { return offsets.empty() ? 0 : offsets.size() - 1; }
};

// FASTA / FASTQ reader for plain, gzip and bzip2 files.  Thread-safe like the reference's (one lock around
// the stream); additionally hands out whole batches of reads so that the device feed does not pay a lock per read.
class FastxReader {
public:
    explicit FastxReader(const std::string& filename);
    ~FastxReader();
    Read get_next_read();
    bool is_complete();
    size_t get_num_reads();
    void close();
    // append reads until at least max_bases bases are buffered or the stream ends; raw (uncleaned) sequences,
    // concatenated, offsets has one more entry than reads.  Returns the number of reads appended.  Plain files are
    // memory-mapped and a batch is parsed by several threads (KMGPU_PARSE_THREADS).
    size_t read_batch(uint64_t max_bases, ReadBatch& out);

private:
    struct Impl;
    std::unique_ptr<Impl> _impl;
};

template <typename SeqIO>
class ReadParser {
public:
    explicit ReadParser(std::unique_ptr<SeqIO> pf) : _parser(std::move(pf)) {}
    Read get_next_read() { return _parser->get_next_read(); }
    ReadPair get_next_read_pair();
    size_t get_num_reads() { return _parser->get_num_reads(); }
    bool is_complete() { return _parser->is_complete(); }
    void close() { _parser->close(); }
    SeqIO& io() { return *_parser; }

private:
    std::unique_ptr<SeqIO> _parser;
};
template <typename SeqIO>
using ReadParserPtr = std::shared_ptr<ReadParser<SeqIO>>;
typedef ReadParserPtr<FastxReader> FastxParserPtr;

template <typename SeqIO>
ReadParserPtr<SeqIO> get_parser(const std::string& filename)
{
    return ReadParserPtr<SeqIO>(new ReadParser<SeqIO>(std::unique_ptr<SeqIO>(new SeqIO(filename))));
}

}  // namespace read_parsers

// ---- storage (include/oxli/storage.hh:56-78) ---------------------------------------------------------
class Storage {
protected:
    bool _supports_bigcount = false;

public:
    virtual ~Storage() {}
    virtual std::vector<uint64_t> get_tablesizes() const = 0;
    virtual const size_t n_tables() const = 0;
    virtual void save(std::string, WordLength) = 0;
    virtual void load(std::string, WordLength&) = 0;
    virtual const uint64_t n_occupied() const = 0;
    virtual const uint64_t n_unique_kmers() const = 0;
    virtual BoundedCounterType test_and_set_bits(HashIntoType khash) = 0;
    virtual bool add(HashIntoType khash) = 0;
    virtual const BoundedCounterType get_count(HashIntoType khash) const = 0;
    virtual Byte** get_raw_tables() = 0;
    virtual void set_use_bigcount(bool b) = 0;
    virtual bool get_use_bigcount() = 0;
};

enum StorageKind { BYTE_STORAGE = 0, NIBBLE_STORAGE = 1, BIT_STORAGE = 2 };
enum HashKind { TWOBIT_HASH = 0, MURMUR_HASH = 1 };

// Device-resident storage: every Storage virtual is served by the C ABI.  The raw table mirror handed out
// by get_raw_tables() is refreshed from the device on every call.
class GpuStorage : public Storage {
public:
    GpuStorage(StorageKind kind, HashKind hash, WordLength ksize, const std::vector<uint64_t>& tablesizes, int device = -1);
    ~GpuStorage() override;
    std::vector<uint64_t> get_tablesizes() const override { return _tablesizes; }
    const size_t n_tables() const override { return _tablesizes.size(); }
    void save(std::string, WordLength) override;
    void load(std::string, WordLength&) override;
    const uint64_t n_occupied() const override;
    const uint64_t n_unique_kmers() const override;
    BoundedCounterType test_and_set_bits(HashIntoType khash) override;
    bool add(HashIntoType khash) override;
    const BoundedCounterType get_count(HashIntoType khash) const override;
    Byte** get_raw_tables() override;
    void set_use_bigcount(bool b) override;
    bool get_use_bigcount() override;
    void update_from(const GpuStorage& other);  // BitStorage::update_from, src/oxli/storage.cc:63-96
    void reset();

    StorageKind kind() const { return _kind; }
    kmgpu_sketch* handle() const { return _h; }
    uint64_t table_nbytes(size_t i) const;
    void set_ksize(WordLength k);

private:
    void recreate(WordLength ksize, const std::vector<uint64_t>& sizes);
    StorageKind _kind;
    HashKind _hash;
    int _device;
    kmgpu_sketch* _h = nullptr;
    std::vector<uint64_t> _tablesizes;
    std::vector<std::vector<Byte>> _mirror;
    std::vector<Byte*> _mirror_ptrs;
};

class ByteStorage : public GpuStorage {  // storage.hh:480
public:
    ByteStorage(HashKind hash, WordLength k, const std::vector<uint64_t>& sizes) : GpuStorage(BYTE_STORAGE, hash, k, sizes)
    {
        _supports_bigcount = true;
    }
};
class NibbleStorage : public GpuStorage {  // storage.hh:241
public:
    NibbleStorage(HashKind hash, WordLength k, const std::vector<uint64_t>& sizes) : GpuStorage(NIBBLE_STORAGE, hash, k, sizes) {}
};
class BitStorage : public GpuStorage {  // storage.hh:92
public:
    BitStorage(HashKind hash, WordLength k, const std::vector<uint64_t>& sizes) : GpuStorage(BIT_STORAGE, hash, k, sizes) {}
};

// ---- Hashtable (include/oxli/hashtable.hh:127-433) -----------------------------------------------------
class Hashtable {
protected:
    WordLength _ksize;
    GpuStorage* store;
    HashKind _hashkind;

public:
    Hashtable(WordLength ksize, GpuStorage* s, HashKind hk) : _ksize(ksize), store(s), _hashkind(hk) {}
    virtual ~Hashtable() { delete store; }
    Hashtable(const Hashtable&) = delete;
    Hashtable& operator=(const Hashtable&) = delete;

    const WordLength ksize() const { return _ksize; }
    HashKind hashkind() const { return _hashkind; }
    GpuStorage* storage() { return store; }

    HashIntoType hash_dna(const char* kmer) const;
    HashIntoType hash_dna_top_strand(const char* kmer) const;
    HashIntoType hash_dna_bottom_strand(const char* kmer) const;
    std::string unhash_dna(HashIntoType hashval) const;

    void count(const char* kmer) { store->add(hash_dna(kmer)); }
    void count(HashIntoType khash) { store->add(khash); }
    bool add(const char* kmer) { return store->add(hash_dna(kmer)); }
    bool add(HashIntoType khash) { return store->add(khash); }
    const BoundedCounterType get_count(const char* kmer) const { return store->get_count(hash_dna(kmer)); }
    const BoundedCounterType get_count(HashIntoType khash) const { return store->get_count(khash); }

    void save(std::string filename) { store->save(filename, _ksize); }
    void load(std::string filename);

    unsigned int consume_string(const std::string& s);
    bool check_and_normalize_read(std::string& read) const;

    // bulk loaders (src/oxli/hashtable.cc:126-274)
    template <typename SeqIO>
    void consume_seqfile(std::string const& filename, unsigned int& total_reads, unsigned long long& n_consumed);
    template <typename SeqIO>
    void consume_seqfile(read_parsers::ReadParserPtr<SeqIO>& parser, unsigned int& total_reads, unsigned long long& n_consumed);
    template <typename SeqIO>
    void consume_seqfile_with_mask(std::string const& filename, Hashtable* mask, unsigned int threshold, unsigned int& total_reads,
                                   unsigned long long& n_consumed, bool consume_masked = false);
    template <typename SeqIO>
    void consume_seqfile_with_mask(read_parsers::ReadParserPtr<SeqIO>& parser, Hashtable* mask, unsigned int threshold,
                                   unsigned int& total_reads, unsigned long long& n_consumed, bool consume_masked = false);
    template <typename SeqIO>
    void consume_seqfile_banding(std::string const& filename, unsigned int num_bands, unsigned int band, unsigned int& total_reads,
                                 unsigned long long& n_consumed);
    template <typename SeqIO>
    void consume_seqfile_banding(read_parsers::ReadParserPtr<SeqIO>& parser, unsigned int num_bands, unsigned int band,
                                 unsigned int& total_reads, unsigned long long& n_consumed);
    template <typename SeqIO>
    void consume_seqfile_banding_with_mask(std::string const& filename, unsigned int num_bands, unsigned int band, Hashtable* mask,
                                           unsigned int threshold, unsigned int& total_reads, unsigned long long& n_consumed,
                                           bool consume_masked = false);
    template <typename SeqIO>
    void consume_seqfile_banding_with_mask(read_parsers::ReadParserPtr<SeqIO>& parser, unsigned int num_bands, unsigned int band,
                                           Hashtable* mask, unsigned int threshold, unsigned int& total_reads,
                                           unsigned long long& n_consumed, bool consume_masked = false);

    void set_use_bigcount(bool b) { store->set_use_bigcount(b); }
    bool get_use_bigcount() { return store->get_use_bigcount(); }

    const size_t n_tables() const { return store->n_tables(); }
    const uint64_t n_occupied() const { return store->n_occupied(); }
    const uint64_t n_unique_kmers() const { return store->n_unique_kmers(); }
    std::vector<uint64_t> get_tablesizes() const { return store->get_tablesizes(); }
    Byte** get_raw_tables() { return store->get_raw_tables(); }

    // queries (src/oxli/hashtable.cc:299-448)
    void get_median_count(const std::string& s, BoundedCounterType& median, float& average, float& stddev);
    bool median_at_least(const std::string& s, unsigned int cutoff);
    void get_kmers(const std::string& s, std::vector<std::string>& kmers) const;
    void get_kmer_hashes(const std::string& s, std::vector<HashIntoType>& kmers) const;
    void get_kmer_counts(const std::string& s, std::vector<BoundedCounterType>& counts) const;
    BoundedCounterType get_min_count(const std::string& s);
    BoundedCounterType get_max_count(const std::string& s);

    // batched forms of the above (one device call for many reads) — what normalize-by-median-like loops want
    void get_median_counts(const std::vector<std::string>& seqs, std::vector<BoundedCounterType>& median, std::vector<float>& average,
                           std::vector<float>& stddev, std::vector<uint32_t>& n_kmers);
    void median_at_least_batch(const std::vector<std::string>& seqs, unsigned int cutoff, std::vector<uint8_t>& out);

    // abundance histogram (src/oxli/hashtable.cc:451-503); returns new uint64_t[MAX_BIGCOUNT + 1]
    template <typename SeqIO>
    uint64_t* abundance_distribution(read_parsers::ReadParserPtr<SeqIO>& parser, Hashtable* tracking);
    template <typename SeqIO>
    uint64_t* abundance_distribution(std::string filename, Hashtable* tracking);

    // abundance trimming helpers (src/oxli/hashtable.cc:504-612)
    // digital normalization of a batch in stream order (scripts/normalize-by-median.py:155-179); returns the k-mers consumed
    unsigned long long normalize_batch(const std::vector<std::string>& seqs, unsigned int cutoff, const std::vector<uint8_t>& pair_with_next,
                                       std::vector<uint8_t>& keep);
    // trim-low-abund's two passes for a batch in stream order (scripts/trim-low-abund.py:196-271): per-read actions (KMGPU_TLA_*) and
    // trim lengths; pass 1 returns the k-mers consumed.  clean: Read::set_clean_seq on the device.
    unsigned long long trim_low_abund_pass1(const std::vector<std::string>& seqs, unsigned int trim_at_coverage, unsigned int cutoff,
                                            unsigned int diginorm_coverage, const std::vector<uint8_t>& pair_with_next, bool clean,
                                            std::vector<uint8_t>& action, std::vector<uint32_t>& trim_pos);
    void trim_low_abund_pass2(const std::vector<std::string>& seqs, unsigned int trim_at_coverage, unsigned int cutoff, bool variable_coverage,
                              const std::vector<uint8_t>& pair_with_next, bool clean, std::vector<uint8_t>& action,
                              std::vector<uint32_t>& trim_pos);
    unsigned long trim_on_abundance(std::string seq, BoundedCounterType min_abund) const;
    unsigned long trim_below_abundance(std::string seq, BoundedCounterType max_abund) const;
    std::vector<unsigned int> find_spectral_error_positions(std::string seq, BoundedCounterType min_abund) const;

    // ---- tagging (Hashgraph, include/oxli/hashgraph.hh:88-140, src/oxli/hashgraph.cc:200-320; two-bit hash sketches only) ----
    // The counting of every k-mer and its "was new" bit come from the device in one call per batch of reads
    // (kmgpu_consume_reads_new); the tag scan over those bits is the reference's, read by read in stream order, against the
    // std::set the tag file is written from.  n_consumed counts the NEW k-mers, like the reference's.
    void consume_sequence_and_tag(const std::string& cleaned_seq, unsigned long long& n_consumed);
    template <typename SeqIO>
    void consume_seqfile_and_tag(std::string const& filename, unsigned int& total_reads, unsigned long long& n_consumed);
    template <typename SeqIO>
    void consume_seqfile_and_tag(read_parsers::ReadParserPtr<SeqIO>& parser, unsigned int& total_reads, unsigned long long& n_consumed);
    size_t n_tags() const { return all_tags.size(); }
    const std::set<HashIntoType>& tags() const { return all_tags; }
    void add_tag(HashIntoType t) { all_tags.insert(t); }
    void clear_tags() { all_tags.clear(); }
    void _set_tag_density(unsigned int d);      // hashgraph.hh:128-135: even, and only while no tag exists
    unsigned int _get_tag_density() const { return _tag_density; }
    void save_tagset(std::string filename);     // hashgraph.cc:55-88
    void load_tagset(std::string filename, bool clear_tags = true);

private:
    template <typename SeqIO>
    void bulk_consume(read_parsers::ReadParserPtr<SeqIO>& parser, const uint64_t* band, Hashtable* mask, unsigned int threshold,
                      bool consume_masked, unsigned int& total_reads, unsigned long long& n_consumed);
    void tag_batch(const char* seqs, const uint64_t* offsets, size_t n_reads, unsigned long long& n_consumed);
    std::set<HashIntoType> all_tags;
    unsigned int _tag_density = 40;   // DEFAULT_TAG_DENSITY (include/oxli/oxli.hh:83)
    std::mutex tags_mu;
};

// class shells: (hash function, storage) pairs — hashgraph.hh:273-296, hashtable.hh:591-627
class Countgraph : public Hashtable {
public:
    Countgraph(WordLength k, std::vector<uint64_t> sizes) : Hashtable(k, new ByteStorage(TWOBIT_HASH, k, sizes), TWOBIT_HASH) {}
};
class SmallCountgraph : public Hashtable {
public:
    SmallCountgraph(WordLength k, std::vector<uint64_t> sizes) : Hashtable(k, new NibbleStorage(TWOBIT_HASH, k, sizes), TWOBIT_HASH) {}
};
class Nodegraph : public Hashtable {
public:
    Nodegraph(WordLength k, std::vector<uint64_t> sizes) : Hashtable(k, new BitStorage(TWOBIT_HASH, k, sizes), TWOBIT_HASH) {}
    void update_from(const Nodegraph& other);
};
class Counttable : public Hashtable {
public:
    Counttable(WordLength k, std::vector<uint64_t> sizes) : Hashtable(k, new ByteStorage(MURMUR_HASH, k, sizes), MURMUR_HASH) {}
};
class SmallCounttable : public Hashtable {
public:
    SmallCounttable(WordLength k, std::vector<uint64_t> sizes) : Hashtable(k, new NibbleStorage(MURMUR_HASH, k, sizes), MURMUR_HASH) {}
};
class Nodetable : public Hashtable {
public:
    Nodetable(WordLength k, std::vector<uint64_t> sizes) : Hashtable(k, new BitStorage(MURMUR_HASH, k, sizes), MURMUR_HASH) {}
};

}  // namespace oxli_b200
