// Python bindings of the host layer: the classes and free functions the reference exposes through
// khmer/_oxli/graphs.pyx (Hashtable and its six concrete table types), khmer/_oxli/parsing.pyx and
// src/khmer/_cpy_khmer.cc (ReadParser, hash helpers) — same names, arguments and exception types, so that
// code written against `khmer` runs against `khmer_b200` for the ingestion path.
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <execinfo.h>
#include <signal.h>
#include <unistd.h>

#include "oxli_b200.hh"

namespace py = pybind11;

// KMGPU_DEBUG_SEGV=1: print a native backtrace on SIGSEGV (debugging aid, off by default)
static void segv_backtrace(int sig)
{
    void* frames[64];
    int n = backtrace(frames, 64);
    backtrace_symbols_fd(frames, n, 2);
    signal(sig, SIG_DFL);
    raise(sig);
}

using namespace oxli_b200;
using namespace oxli_b200::read_parsers;

namespace {

bool is_str(const py::object& o) { return py::isinstance<py::str>(o) || py::isinstance<py::bytes>(o); }
bool is_num(const py::object& o) { return py::isinstance<py::int_>(o); }

std::string to_string(const py::object& o)
{
    if (py::isinstance<py::bytes>(o)) return o.cast<std::string>();
    return o.cast<std::string>();
}

struct PyParser {  // khmer.ReadParser (src/khmer/_cpy_readparsers.cc:392-416) / FastxParser (parsing.pyx)
    FastxParserPtr parser;
    explicit PyParser(const std::string& fn) : parser(get_parser<FastxReader>(fn)) {}
};

FastxParserPtr parser_of(const py::object& o)
{
    if (is_str(o)) return get_parser<FastxReader>(to_string(o));
    return o.cast<PyParser&>().parser;
}

// graphs.pyx:33-71 argument sanitising
std::string sanitize_seq_kmer(Hashtable& ht, const py::object& kmer)
{
    std::string s = to_string(kmer);
    if (s.size() != ht.ksize()) {
        throw py::value_error("Expected k-mer length " + std::to_string((int)ht.ksize()) + " but got " + std::to_string(s.size()) + ".");
    }
    return s;
}
HashIntoType sanitize_hash_kmer(Hashtable& ht, const py::object& kmer)
{
    if (is_num(kmer)) return kmer.cast<HashIntoType>();
    if (is_str(kmer)) return ht.hash_dna(sanitize_seq_kmer(ht, kmer).c_str());
    throw py::type_error("Object of type " + std::string(py::str(py::type::of(kmer))) + " can not be interpretted as  a k-mer");
}
std::string valid_sequence(Hashtable& ht, const std::string& seq)
{
    if (seq.size() < ht.ksize()) {
        throw py::value_error("sequence length (" + std::to_string(seq.size()) + ") must >= the hashtable k-mer size (" +
                              std::to_string((int)ht.ksize()) + ")");
    }
    return seq;
}

template <class T>
std::shared_ptr<T> make_table(int k, uint64_t starting_size, int n_tables, const py::object& primes)
{
    std::vector<uint64_t> sizes;
    if (!primes.is_none() && py::len(primes) > 0) sizes = primes.cast<std::vector<uint64_t>>();
    else sizes = get_n_primes_near_x((uint32_t)n_tables, starting_size);
    return std::make_shared<T>((WordLength)k, sizes);
}

template <class T>
void bind_table(py::module_& m, const char* name, py::class_<Hashtable, std::shared_ptr<Hashtable>>& base)
{
    py::class_<T, Hashtable, std::shared_ptr<T>> c(m, name);
    c.def(py::init([](int k, double starting_size, int n_tables, py::object primes) {
              return make_table<T>(k, (uint64_t)starting_size, n_tables, primes);
          }),
          py::arg("k"), py::arg("starting_size"), py::arg("n_tables"), py::arg("primes") = py::none());
    c.def_static(
        "load",
        [](const std::string& fn) {  // graphs.pyx:303-307: cls(1, 1, 1) then load
            auto t = std::make_shared<T>((WordLength)1, std::vector<uint64_t>{1});
            py::gil_scoped_release nogil;
            t->load(fn);
            return t;
        },
        py::arg("file_name"));
    (void)base;
}

}  // namespace

PYBIND11_MODULE(_oxli, m)
{
    if (getenv("KMGPU_DEBUG_SEGV")) signal(SIGSEGV, segv_backtrace);
    m.doc() = "khmer_b200 host layer: liboxli-compatible classes backed by the kmgpu C ABI (tables in GPU memory)";

    // exception mapping — khmer/_oxli/oxli_exception_convert.cc:9-31
    py::register_exception_translator([](std::exception_ptr p) {
        try {
            if (p) std::rethrow_exception(p);
        } catch (const oxli_file_exception& e) {
            PyErr_SetString(PyExc_OSError, e.what());
        } catch (const oxli_value_exception& e) {
            PyErr_SetString(PyExc_ValueError, e.what());
        } catch (const oxli_exception& e) {
            PyErr_SetString(PyExc_ValueError, e.what());
        }
    });

    m.attr("MAX_KCOUNT") = MAX_KCOUNT;
    m.attr("MAX_BIGCOUNT") = MAX_BIGCOUNT;

    // ---- free functions (src/khmer/_cpy_khmer.cc:60-311, khmer/_oxli/utils.pyx) ----------------------------
    m.def("forward_hash", [](const std::string& kmer, int k) {
        if (k > 32) throw py::value_error("k-mer size must be <= 32");
        if ((int)kmer.size() != k) throw py::value_error("k-mer length must equal the k-mer size");
        return _hash(kmer.c_str(), (WordLength)k);
    });
    m.def("forward_hash_no_rc", [](const std::string& kmer, int k) {
        if (k > 32) throw py::value_error("k-mer size must be <= 32");
        if ((int)kmer.size() != k) throw py::value_error("k-mer length must equal the k-mer size");
        return _hash_forward(kmer.c_str(), (WordLength)k);
    });
    m.def("reverse_hash", [](HashIntoType h, int k) {
        if (k > 32) throw py::value_error("k-mer size must be <= 32");
        return _revhash(h, (WordLength)k);
    });
    m.def("hash_murmur3", [](const std::string& kmer) { return _hash_murmur(kmer, (WordLength)kmer.size()); });
    m.def("hash_no_rc_murmur3", [](const std::string& kmer) { return _hash_murmur_forward(kmer, (WordLength)kmer.size()); });
    m.def("reverse_complement", [](const std::string& s) { return _revcomp(s); });
    m.def("get_n_primes_near_x", [](uint32_t n, uint64_t x) { return get_n_primes_near_x(n, x); });
    m.def("compute_band_interval", [](unsigned nb, unsigned b) { return compute_band_interval(nb, b); });

    // ---- reads -----------------------------------------------------------------------------------------
    py::class_<Read>(m, "Read")
        .def_readonly("name", &Read::name)
        .def_readonly("sequence", &Read::sequence)
        .def_readonly("quality", &Read::quality)
        .def_property_readonly("cleaned_seq", [](Read& r) {
            if (r.cleaned_seq.empty() && !r.sequence.empty()) r.set_clean_seq();
            return r.cleaned_seq;
        })
        .def("__len__", [](const Read& r) { return r.sequence.size(); });

    py::class_<PyParser>(m, "ReadParser")
        .def(py::init<const std::string&>(), py::arg("filename"))
        .def_property_readonly("num_reads", [](PyParser& p) { return p.parser->get_num_reads(); })
        .def("is_complete", [](PyParser& p) { return p.parser->is_complete(); })
        .def("close", [](PyParser& p) { p.parser->close(); })
        .def("read_batch", [](PyParser& p, uint64_t max_bases) {
            // the device feed's view of the file: raw sequences of the next batch (several parser threads on plain files)
            ReadBatch b;
            size_t n;
            {
                py::gil_scoped_release nogil;
                n = p.parser->io().read_batch(max_bases, b);
            }
            py::list out;
            for (size_t i = 0; i < n; i++) out.append(py::bytes(b.seqs + b.offsets[i], b.offsets[i + 1] - b.offsets[i]));
            return out;
        }, py::arg("max_bases") = (uint64_t)(64u << 20))
        .def("read_batch_packed", [](PyParser& p, uint64_t max_bases) {
            // the batch exactly as the device feed takes it: cleaned, 2-bit packed by the parser threads; returns (reads, bases)
            ReadBatch b;
            b.pack = true;
            size_t n;
            {
                py::gil_scoped_release nogil;
                n = p.parser->io().read_batch(max_bases, b);
            }
            if (!n) return py::make_tuple(n, (uint64_t)0, py::bytes(), py::bytes());
            return py::make_tuple(n, (uint64_t)b.n_bases, py::bytes((const char*)b.words(), b.n_words() * 8),
                                  py::bytes((const char*)b.offsets.data(), b.offsets.size() * 8));
        }, py::arg("max_bases") = (uint64_t)(64u << 20))
        .def("__iter__", [](py::object self) { return self; })
        .def("__next__", [](PyParser& p) {
            try {
                Read r = p.parser->get_next_read();
                r.set_clean_seq();
                return r;
            } catch (const NoMoreReadsAvailable&) {
                throw py::stop_iteration();
            }
        });
    m.attr("FastxParser") = m.attr("ReadParser");

    // ---- Hashtable (khmer/_oxli/graphs.pyx:31-390) -------------------------------------------------------
    py::class_<Hashtable, std::shared_ptr<Hashtable>> ht(m, "Hashtable");
    ht.def("ksize", [](Hashtable& h) { return (int)h.ksize(); })
        .def("hash", [](Hashtable& h, py::object kmer) -> HashIntoType {
            if (is_num(kmer)) return kmer.cast<HashIntoType>();
            return h.hash_dna(sanitize_seq_kmer(h, kmer).c_str());
        })
        .def("reverse_hash", [](Hashtable& h, HashIntoType v) { return h.unhash_dna(v); })
        .def("add", [](Hashtable& h, py::object kmer) { return h.add(sanitize_hash_kmer(h, kmer)); })
        .def("count", [](Hashtable& h, py::object kmer) { h.add(sanitize_hash_kmer(h, kmer)); })
        .def("get", [](Hashtable& h, py::object kmer) { return (int)h.get_count(sanitize_hash_kmer(h, kmer)); })
        .def("consume", [](Hashtable& h, const std::string& seq) {
            std::string s = valid_sequence(h, seq);
            py::gil_scoped_release nogil;
            return h.consume_string(s);
        })
        .def("get_kmers", [](Hashtable& h, const std::string& seq) {
            std::vector<std::string> out;
            h.get_kmers(seq, out);
            return out;
        })
        .def("get_kmer_hashes", [](Hashtable& h, const std::string& seq) {
            std::vector<HashIntoType> out;
            h.get_kmer_hashes(valid_sequence(h, seq), out);
            return out;
        })
        .def("get_kmer_counts", [](Hashtable& h, const std::string& seq) {
            std::vector<BoundedCounterType> out;
            h.get_kmer_counts(valid_sequence(h, seq), out);
            return out;
        })
        .def("get_min_count", [](Hashtable& h, const std::string& seq) { return (int)h.get_min_count(valid_sequence(h, seq)); })
        .def("get_max_count", [](Hashtable& h, const std::string& seq) { return (int)h.get_max_count(valid_sequence(h, seq)); })
        .def("get_median_count", [](Hashtable& h, const std::string& seq) {
            BoundedCounterType med = 0;
            float avg = 0, sd = 0;
            h.get_median_count(valid_sequence(h, seq), med, avg, sd);
            return py::make_tuple((int)med, avg, sd);
        })
        .def("median_at_least", [](Hashtable& h, const std::string& seq, unsigned cutoff) {
            return h.median_at_least(valid_sequence(h, seq), cutoff);
        })
        .def("get_median_counts", [](Hashtable& h, const std::vector<std::string>& seqs) {
            std::vector<BoundedCounterType> med;
            std::vector<float> avg, sd;
            std::vector<uint32_t> nk;
            {
                py::gil_scoped_release nogil;
                h.get_median_counts(seqs, med, avg, sd, nk);
            }
            return py::make_tuple(med, avg, sd, nk);
        })
        .def("median_at_least_batch", [](Hashtable& h, const std::vector<std::string>& seqs, unsigned cutoff) {
            std::vector<uint8_t> out;
            {
                py::gil_scoped_release nogil;
                h.median_at_least_batch(seqs, cutoff, out);
            }
            return out;
        })
        .def("consume_seqfile_and_tag", [](Hashtable& h, py::object file_or_parser) {
            // graphs.pyx:588-600: (total_reads, n_consumed) with n_consumed = the NEW k-mers
            unsigned int total_reads = 0;
            unsigned long long n_consumed = 0;
            if (py::isinstance<py::str>(file_or_parser)) {
                std::string fn = file_or_parser.cast<std::string>();
                py::gil_scoped_release nogil;
                h.consume_seqfile_and_tag<FastxReader>(fn, total_reads, n_consumed);
            } else {
                PyParser& p = file_or_parser.cast<PyParser&>();
                py::gil_scoped_release nogil;
                h.consume_seqfile_and_tag<FastxReader>(p.parser, total_reads, n_consumed);
            }
            return py::make_tuple(total_reads, n_consumed);
        })
        .def("consume_and_tag", [](Hashtable& h, const std::string& seq) {
            unsigned long long n = 0;
            h.consume_sequence_and_tag(seq, n);
            return n;
        })
        .def("n_tags", &Hashtable::n_tags)
        .def("get_tagset", [](Hashtable& h) { return std::vector<HashIntoType>(h.tags().begin(), h.tags().end()); })
        .def("add_tag", [](Hashtable& h, py::object kmer) { h.add_tag(sanitize_hash_kmer(h, kmer)); })
        .def("save_tagset", &Hashtable::save_tagset)
        .def("load_tagset", &Hashtable::load_tagset, py::arg("filename"), py::arg("clear_tags") = true)
        .def("_get_tag_density", &Hashtable::_get_tag_density)
        .def("_set_tag_density", &Hashtable::_set_tag_density)
        .def("normalize_batch", [](Hashtable& h, const std::vector<std::string>& seqs, unsigned cutoff, const std::vector<uint8_t>& paired) {
            std::vector<uint8_t> keep;
            unsigned long long kmers;
            {
                py::gil_scoped_release nogil;
                kmers = h.normalize_batch(seqs, cutoff, paired, keep);
            }
            return py::make_tuple(keep, kmers);
        }, py::arg("seqs"), py::arg("cutoff"), py::arg("paired") = std::vector<uint8_t>())
        .def("trim_low_abund_pass1", [](Hashtable& h, const std::vector<std::string>& seqs, unsigned trim_at_coverage, unsigned cutoff,
                                        unsigned diginorm_coverage, const std::vector<uint8_t>& paired, bool clean) {
            std::vector<uint8_t> action;
            std::vector<uint32_t> trim_pos;
            unsigned long long kmers;
            {
                py::gil_scoped_release nogil;
                kmers = h.trim_low_abund_pass1(seqs, trim_at_coverage, cutoff, diginorm_coverage, paired, clean, action, trim_pos);
            }
            return py::make_tuple(py::bytes(reinterpret_cast<const char*>(action.data()), action.size()), trim_pos, kmers);
        }, py::arg("seqs"), py::arg("trim_at_coverage"), py::arg("cutoff"), py::arg("diginorm_coverage") = 0,
           py::arg("paired") = std::vector<uint8_t>(), py::arg("clean") = false)
        .def("trim_low_abund_pass2", [](Hashtable& h, const std::vector<std::string>& seqs, unsigned trim_at_coverage, unsigned cutoff,
                                        bool variable_coverage, const std::vector<uint8_t>& paired, bool clean) {
            std::vector<uint8_t> action;
            std::vector<uint32_t> trim_pos;
            {
                py::gil_scoped_release nogil;
                h.trim_low_abund_pass2(seqs, trim_at_coverage, cutoff, variable_coverage, paired, clean, action, trim_pos);
            }
            return py::make_tuple(py::bytes(reinterpret_cast<const char*>(action.data()), action.size()), trim_pos);
        }, py::arg("seqs"), py::arg("trim_at_coverage"), py::arg("cutoff"), py::arg("variable_coverage") = false,
           py::arg("paired") = std::vector<uint8_t>(), py::arg("clean") = false)
        .def("n_unique_kmers", &Hashtable::n_unique_kmers)
        .def("n_occupied", &Hashtable::n_occupied)
        .def("n_tables", &Hashtable::n_tables)
        .def("hashsizes", &Hashtable::get_tablesizes)
        .def("set_use_bigcount", &Hashtable::set_use_bigcount)
        .def("get_use_bigcount", &Hashtable::get_use_bigcount)
        .def("save", [](Hashtable& h, const std::string& fn) {
            py::gil_scoped_release nogil;
            h.save(fn);
        })
        .def("consume_seqfile", [](Hashtable& h, py::object file_or_parser) {
            FastxParserPtr p = parser_of(file_or_parser);
            unsigned int total_reads = 0;
            unsigned long long n_consumed = 0;
            {
                py::gil_scoped_release nogil;  // graphs.pyx:235-238
                h.consume_seqfile<FastxReader>(p, total_reads, n_consumed);
            }
            return py::make_tuple(total_reads, n_consumed);
        })
        .def("consume_seqfile_with_mask", [](Hashtable& h, py::object file_or_parser, Hashtable& mask, unsigned threshold, bool consume_masked) {
            FastxParserPtr p = parser_of(file_or_parser);
            unsigned int total_reads = 0;
            unsigned long long n_consumed = 0;
            {
                py::gil_scoped_release nogil;
                h.consume_seqfile_with_mask<FastxReader>(p, &mask, threshold, total_reads, n_consumed, consume_masked);
            }
            return py::make_tuple(total_reads, n_consumed);
        }, py::arg("file_name"), py::arg("mask"), py::arg("threshold") = 0, py::arg("consume_masked") = false)
        .def("consume_seqfile_banding", [](Hashtable& h, py::object file_or_parser, unsigned num_bands, unsigned band) {
            FastxParserPtr p = parser_of(file_or_parser);
            unsigned int total_reads = 0;
            unsigned long long n_consumed = 0;
            {
                py::gil_scoped_release nogil;
                h.consume_seqfile_banding<FastxReader>(p, num_bands, band, total_reads, n_consumed);
            }
            return py::make_tuple(total_reads, n_consumed);
        })
        .def("consume_seqfile_banding_with_mask", [](Hashtable& h, py::object file_or_parser, unsigned num_bands, unsigned band,
                                                    Hashtable& mask, unsigned threshold, bool consume_masked) {
            FastxParserPtr p = parser_of(file_or_parser);
            unsigned int total_reads = 0;
            unsigned long long n_consumed = 0;
            {
                py::gil_scoped_release nogil;
                h.consume_seqfile_banding_with_mask<FastxReader>(p, num_bands, band, &mask, threshold, total_reads, n_consumed, consume_masked);
            }
            return py::make_tuple(total_reads, n_consumed);
        }, py::arg("file_name"), py::arg("num_bands"), py::arg("band"), py::arg("mask"), py::arg("threshold") = 0,
           py::arg("consume_masked") = false)
        .def("abundance_distribution", [](Hashtable& h, py::object file_or_parser, Hashtable& tracking) {
            FastxParserPtr p = parser_of(file_or_parser);
            uint64_t* dist;
            {
                py::gil_scoped_release nogil;  // graphs.pyx:282-296
                dist = h.abundance_distribution<FastxReader>(p, &tracking);
            }
            py::list out;
            for (unsigned i = 0; i < MAX_BIGCOUNT; i++) out.append(dist[i]);  // the reference returns 65535 entries
            delete[] dist;
            return out;
        })
        .def("trim_on_abundance", [](Hashtable& h, const std::string& seq, unsigned abund) {
            unsigned long pos = h.trim_on_abundance(valid_sequence(h, seq), (BoundedCounterType)abund);
            return py::make_tuple(seq.substr(0, pos), pos);
        })
        .def("trim_below_abundance", [](Hashtable& h, const std::string& seq, unsigned abund) {
            unsigned long pos = h.trim_below_abundance(valid_sequence(h, seq), (BoundedCounterType)abund);
            return py::make_tuple(seq.substr(0, pos), pos);
        })
        .def("find_spectral_error_positions", [](Hashtable& h, const std::string& seq, unsigned max_count) {
            return h.find_spectral_error_positions(valid_sequence(h, seq), (BoundedCounterType)max_count);
        })
        .def("get_raw_tables", [](Hashtable& h) {
            // graphs.pyx:333-347: a list of read-only views, one per table (here: snapshots downloaded from HBM)
            Byte** t = h.get_raw_tables();
            py::list out;
            for (size_t i = 0; i < h.n_tables(); i++) {
                uint64_t n = h.storage()->table_nbytes(i);
                out.append(py::memoryview(py::bytes((const char*)t[i], n)));
            }
            return out;
        });

    bind_table<Countgraph>(m, "Countgraph", ht);
    bind_table<SmallCountgraph>(m, "SmallCountgraph", ht);
    bind_table<Counttable>(m, "Counttable", ht);
    bind_table<SmallCounttable>(m, "SmallCounttable", ht);
    bind_table<Nodetable>(m, "Nodetable", ht);
    {
        py::class_<Nodegraph, Hashtable, std::shared_ptr<Nodegraph>> c(m, "Nodegraph");
        c.def(py::init([](int k, double starting_size, int n_tables, py::object primes) {
                  return make_table<Nodegraph>(k, (uint64_t)starting_size, n_tables, primes);
              }),
              py::arg("k"), py::arg("starting_size"), py::arg("n_tables"), py::arg("primes") = py::none());
        c.def_static("load", [](const std::string& fn) {
            auto t = std::make_shared<Nodegraph>((WordLength)1, std::vector<uint64_t>{1});
            py::gil_scoped_release nogil;
            t->load(fn);
            return t;
        });
        c.def("update", [](Nodegraph& a, Nodegraph& b) { a.update_from(b); });  // graphs.pyx:899-900
    }
}
