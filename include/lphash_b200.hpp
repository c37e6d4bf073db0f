// lphash_b200.hpp — C++ host-side mirror of the reference's interface for the hot path, on top of
// the C ABI (include/lphash_b200.h -> lphash_b200/liblphash_b200.so).  Header-only; C++17.
//
// The reference is compiled C++ whose seam for this path is a member function and two free
// function templates, so the drop-in keeps their names, argument meaning and error behaviour:
//
//   reference (jermp/lphash)                                   here (namespace lphash_b200)
//   ---------------------------------------------------------  -------------------------------------
//   lphash::mphf hf; essentials::load(hf, file)                mphf hf; hf.load(file)      (query.cpp:36-38)
//   hf(contig, length, streaming=true) -> vector<uint64_t>     same   (partitioned_mphf.hpp:21-26, 73-184)
//   hf(std::string const&, streaming=true)                     same   (partitioned_mphf.hpp:199-202)
//   hf.get_kmer_count(), hf.get_minimizer_L0()                 same   (partitioned_mphf.hpp:17-18)
//   minimizer::from_string<H>(contig, n, k, m, seed,           minimizer::from_string(...) same argument
//       canonical, mm_count, accumulator)                      list; accumulator = anything with
//                                                              push_back(mm_record_t)  (minimizer.hpp:11-170)
//   minimizer::get_colliding_kmers<H>(contig, n, k, m, seed,   minimizer::get_colliding_kmers(...) same
//       canonical, itr, stop, mm_count, accumulator)           argument list           (minimizer.hpp:172-319)
//
// Errors surface as std::runtime_error, like the reference (partitioned_mphf.cpp:67, :335).  There
// is no CPU path behind this header: without the CUDA library / a GPU every call throws.
//
// kmer_t follows the reference's compile-time switch (include/compile_constants.tpd): define
// LPHASH_B200_KMER_BITS to 64 for a `typedef uint64_t kmer_t;` build; the default is 128
// (`__uint128_t`, the reference's default).
#pragma once

#include <cstddef>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "lphash_b200.h"

#ifndef LPHASH_B200_KMER_BITS
#define LPHASH_B200_KMER_BITS 128
#endif

namespace lphash_b200 {

#if LPHASH_B200_KMER_BITS == 64
typedef uint64_t kmer_t;
#else
typedef __uint128_t kmer_t;
#endif
constexpr int kmer_bits = LPHASH_B200_KMER_BITS;

// include/constants.hpp:26-33
#pragma pack(push, 2)
struct mm_record_t {
    uint64_t itself;
    uint64_t id;
    uint8_t p1;
    uint8_t size;
};
#pragma pack(pop)
static_assert(sizeof(mm_record_t) == 18, "mm_record_t is the reference's packed 18-byte record");

// include/constants.hpp:35-41
#pragma pack(push, 2)
struct mm_triplet_t {
    uint64_t itself;
    uint8_t p1;
    uint8_t size;
};
#pragma pack(pop)
static_assert(sizeof(mm_triplet_t) == 10, "mm_triplet_t is the reference's packed 10-byte triplet");

namespace detail {
[[noreturn]] inline void raise(const char* what, int rc) {
    throw std::runtime_error(std::string(what) + ": " + lphb_last_error() + " (code " +
                             std::to_string(rc) + ")");
}
}  // namespace detail

class mphf {
public:
    mphf() = default;
    mphf(mphf const&) = delete;
    mphf& operator=(mphf const&) = delete;
    mphf(mphf&& o) noexcept : h_(o.h_), info_(o.info_) { o.h_ = nullptr; }
    mphf& operator=(mphf&& o) noexcept {
        if (this != &o) {
            reset();
            h_ = o.h_;
            info_ = o.info_;
            o.h_ = nullptr;
        }
        return *this;
    }
    ~mphf() { reset(); }

    // essentials::load(hf, filename) (src/query.cpp:37).  `device` = CUDA device holding the image.
    void load(const char* filename, int device = 0) {
        reset();
        int rc = lphb_mphf_load_file(filename, kmer_bits, device, &h_);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::load", rc);
        lphb_mphf_info(h_, &info_);
    }
    // the same from an in-memory essentials image (what essentials::save writes)
    void load(const void* image, uint64_t nbytes, int device = 0) {
        reset();
        int rc = lphb_mphf_load_memory(image, nbytes, kmer_bits, device, &h_);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::load", rc);
        lphb_mphf_info(h_, &info_);
    }

    // the unpartitioned variant (lphash::mphf_alt, build-u / query-u): same handle, same queries
    void load_alt(const char* filename, int device = 0) {
        reset();
        int rc = lphb_mphf_alt_load_file(filename, kmer_bits, device, &h_);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::load_alt", rc);
        lphb_mphf_info(h_, &info_);
    }
    void load_alt(const void* image, uint64_t nbytes, int device = 0) {
        reset();
        int rc = lphb_mphf_alt_load_memory(image, nbytes, kmer_bits, device, &h_);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::load_alt", rc);
        lphb_mphf_info(h_, &info_);
    }

    uint64_t get_minimizer_L0() const noexcept { return info_.distinct_minimizers; }
    uint64_t get_kmer_count() const noexcept { return info_.nkmers; }
    uint32_t get_k() const noexcept { return info_.k; }
    uint32_t get_m() const noexcept { return info_.m; }
    lphb_info const& info() const noexcept { return info_; }

    // hf(contig, length, streaming).  streaming = true: the reference's streaming branch, non-ACGT quirk
    // included (partitioned_mphf.hpp:73-184); false: its non-streaming branch, where a non-ACGT byte
    // counts as 'A' (partitioned_mphf.hpp:185-195, mphf_utils.hpp:108).  Same codes on ACGT-only input.
    std::vector<uint64_t> operator()(const char* contig, std::size_t length, bool streaming = true) const {
        const uint64_t offsets[2] = {0, uint64_t(length)};
        std::vector<uint64_t> codes, code_offsets;
        query_batch(contig, offsets, 1, codes, code_offsets, streaming);
        return codes;
    }
    std::vector<uint64_t> operator()(std::string const& contig, bool streaming = true) const {
        return (*this)(contig.c_str(), contig.length(), streaming);
    }

    // Many contigs per call (what a throughput-minded driver uses instead of one call per kseq
    // record): bases = contigs concatenated without separators, offsets = n_contigs + 1 entries.
    // codes = all contigs' codes in contig order; contig c owns
    // [code_offsets[c], code_offsets[c+1]).
    void query_batch(const char* bases, const uint64_t* offsets, uint64_t n_contigs,
                     std::vector<uint64_t>& codes, std::vector<uint64_t>& code_offsets,
                     bool streaming = true) const {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        // a contig with non-ACGT bytes can emit up to L-m+1 codes (reference quirk, SURVEY.md Q1)
        uint64_t cap = 0;
        for (uint64_t c = 0; c < n_contigs; ++c) {
            uint64_t len = offsets[c + 1] - offsets[c];
            cap += len >= info_.m ? len - info_.m + 1 : 0;
        }
        codes.resize(cap);
        code_offsets.resize(n_contigs + 1);
        uint64_t n = 0;
        int rc = streaming ? lphb_query_stream(h_, bases, offsets, n_contigs, codes.data(), cap, code_offsets.data(), &n)
                           : lphb_query_nonstreaming(h_, bases, offsets, n_contigs, codes.data(), cap,
                                                     code_offsets.data(), &n);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::operator()", rc);
        codes.resize(n);
    }

    // The codes of n packed k-mers (lphb_lookup_kmers): codes[i] is what hf(window, k, false) gives for the
    // window of k bases kmers[i] encodes (first base in the most significant of its 2k bits, A=0 C=1 G=2 T=3;
    // partitioned_mphf.hpp:106-108, 185-195).  kmer_t is the width the handle was loaded with.
    std::vector<uint64_t> lookup(const kmer_t* kmers, std::size_t n) const {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        std::vector<uint64_t> codes(n);
        int rc = lphb_lookup_kmers(h_, kmers, n, codes.data());
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::lookup", rc);
        return codes;
    }

    // Batches already in device memory: d_* are device pointers on the handle's GPU, h_offsets the host copy of the
    // offsets, stream a cudaStream_t (nullptr: the default stream).  query_batch_device is hf(contig, len, true) for
    // every contig, the non-ACGT quirk included (lphb_query_stream_exact_device): synchronous, it returns the number
    // of codes; codes_capacity = sum of max(0, L-m+1) always suffices.
    uint64_t query_batch_device(const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                                uint64_t n_contigs, uint64_t* d_codes, uint64_t codes_capacity,
                                uint64_t* d_code_offsets, void* stream = nullptr) const {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        uint64_t n = 0;
        int rc = lphb_query_stream_exact_device(h_, d_bases, d_offsets, h_offsets, n_contigs, d_codes, codes_capacity,
                                                d_code_offsets, &n, stream);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::query_batch_device", rc);
        return n;
    }
    // The same as query_batch_device, asynchronous on `stream` (lphb_query_stream_exact_device_async): d_status (4
    // words) receives the number of codes and of contigs with non-ACGT bytes; codes_capacity must be at least
    // sum of max(0, L-m+1).
    void query_batch_device_async(const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                                  uint64_t n_contigs, uint64_t* d_codes, uint64_t codes_capacity,
                                  uint64_t* d_code_offsets, uint64_t* d_status, void* stream = nullptr) const {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        int rc = lphb_query_stream_exact_device_async(h_, d_bases, d_offsets, h_offsets, n_contigs, d_codes,
                                                      codes_capacity, d_code_offsets, d_status, stream);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::query_batch_device_async", rc);
    }
    // hf(contig, len, false) for every contig (lphb_query_nonstreaming_device): max(0, L-k+1) codes per contig,
    // asynchronous on `stream`; d_status (4 words) as lphb_query_stream_device fills it.
    void query_batch_device_nonstreaming(const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                                         uint64_t n_contigs, uint64_t* d_codes, uint64_t codes_capacity,
                                         uint64_t* d_code_offsets, uint64_t* d_status, void* stream = nullptr) const {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        int rc = lphb_query_nonstreaming_device(h_, d_bases, d_offsets, h_offsets, n_contigs, d_codes, codes_capacity,
                                                d_code_offsets, d_status, stream);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::query_batch_device_nonstreaming", rc);
    }

    // build-p --check (include/mphf_utils.hpp:51-100) as a session over any number of batches of the index's contigs
    // (lphb_check_*): check_begin, check_batch / check_batch_device per batch, check_end for the report.
    // check_batch takes host buffers and returns once they may be reused; check_batch_device takes device buffers
    // (as query_batch_device) and is asynchronous on `stream`, d_stream_codes optional (the caller's streaming codes
    // of the batch in the layout of lphb_query_stream_device, compared instead of the library's own streaming pass).
    void check_begin() {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        int rc = lphb_check_begin(h_);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::check_begin", rc);
    }
    void check_batch(const char* bases, const uint64_t* offsets, uint64_t n_contigs) {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        int rc = lphb_check_batch(h_, bases, offsets, n_contigs);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::check_batch", rc);
    }
    void check_batch_device(const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                            uint64_t n_contigs, const uint64_t* d_stream_codes = nullptr, void* stream = nullptr) {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        int rc = lphb_check_batch_device(h_, d_bases, d_offsets, h_offsets, n_contigs, d_stream_codes, stream);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::check_batch_device", rc);
    }
    lphb_check_report check_end() {
        if (!h_) throw std::runtime_error("lphash_b200::mphf: no index loaded");
        lphb_check_report r{};
        int rc = lphb_check_end(h_, &r);
        if (rc != LPHB_OK) detail::raise("lphash_b200::mphf::check_end", rc);
        return r;
    }

    lphb_mphf* handle() const noexcept { return h_; }

private:
    void reset() noexcept {
        if (h_) lphb_mphf_free(h_);
        h_ = nullptr;
    }
    lphb_mphf* h_ = nullptr;
    lphb_info info_{};
};

// Serializes any object that speaks the essentials visitor protocol (`template <class V> void visit(V&)`)
// into memory, byte for byte what essentials::save writes to a file (essentials.hpp:326-366: PODs raw,
// std::vector<T> = size_t count + elements): the `.lph` image of a reference lphash::mphf without a
// round trip through the file system.  mphf::load(image, nbytes) takes the result.
struct memory_saver {
    std::vector<unsigned char> bytes;
    template <typename T>
    void visit(T& val) {
        if constexpr (std::is_pod<T>::value) {
            const unsigned char* p = reinterpret_cast<const unsigned char*>(&val);
            bytes.insert(bytes.end(), p, p + sizeof(T));
        } else {
            val.visit(*this);
        }
    }
    template <typename T, typename Allocator>
    void visit(std::vector<T, Allocator>& vec) {
        size_t n = vec.size();
        visit(n);
        if constexpr (std::is_pod<T>::value) {
            const unsigned char* p = reinterpret_cast<const unsigned char*>(vec.data());
            bytes.insert(bytes.end(), p, p + n * sizeof(T));
        } else {
            for (auto& v : vec) visit(v);
        }
    }
};

// The inverse: essentials' loader protocol (essentials.hpp:280-324) over a byte image in memory.
struct memory_loader {
    const unsigned char* p;
    const unsigned char* end;
    memory_loader(const void* image, size_t nbytes)
        : p(static_cast<const unsigned char*>(image)), end(static_cast<const unsigned char*>(image) + nbytes) {}
    template <typename T>
    void visit(T& val) {
        if constexpr (std::is_pod<T>::value) {
            take(&val, sizeof(T));
        } else {
            val.visit(*this);
        }
    }
    template <typename T, typename Allocator>
    void visit(std::vector<T, Allocator>& vec) {
        size_t n = 0;
        visit(n);
        if constexpr (std::is_pod<T>::value) {
            if (n > size_t(end - p) / sizeof(T)) throw std::runtime_error("lphash_b200: truncated image");
            vec.resize(n);
            take(vec.data(), n * sizeof(T));
        } else {
            vec.resize(n);
            for (auto& v : vec) visit(v);
        }
    }

private:
    void take(void* dst, size_t n) {
        if (size_t(end - p) < n) throw std::runtime_error("lphash_b200: truncated image");
        if (n) std::memcpy(dst, p, n);
        p += n;
    }
};

// Parts 1 + 2 of build-p over an input fed batch by batch (lphb_build_*): end() gives what minimizer::classify gives
// over the whole record stream (src/minimizer.cpp:5-50), however the input was cut.  Move-only; the destructor frees
// the session.
class build_session {
public:
    build_session(uint32_t k, uint32_t m, uint64_t seed, int device = 0) {
        const int rc = lphb_build_begin(device, k, m, seed, &b_);
        if (rc != LPHB_OK) detail::raise("lphash_b200::build_session", rc);
    }
    build_session(build_session&& o) noexcept : b_(std::exchange(o.b_, nullptr)) {}
    build_session& operator=(build_session&& o) noexcept {
        if (this != &o) {
            lphb_build_free(b_);
            b_ = std::exchange(o.b_, nullptr);
        }
        return *this;
    }
    build_session(build_session const&) = delete;
    build_session& operator=(build_session const&) = delete;
    ~build_session() { lphb_build_free(b_); }

    // one batch of whole contigs in host memory
    void batch(const char* bases, const uint64_t* offsets, uint64_t n_contigs) {
        const int rc = lphb_build_batch(b_, bases, offsets, n_contigs);
        if (rc != LPHB_OK) detail::raise("lphash_b200::build_session::batch", rc);
    }
    // one batch in device memory, written by the caller on `stream` (a cudaStream_t)
    void batch_device(const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets, uint64_t n_contigs,
                      void* stream = nullptr) {
        const int rc = lphb_build_batch_device(b_, d_bases, d_offsets, h_offsets, n_contigs, stream);
        if (rc != LPHB_OK) detail::raise("lphash_b200::build_session::batch_device", rc);
    }
    // merges the batches and closes the session: triplets in ascending minimizer order, ids ascending
    lphb_build_report end(std::vector<mm_triplet_t>& triplets, std::vector<uint64_t>& ids) {
        lphb_build_report r{};
        int rc = lphb_build_end(b_, nullptr, 0, nullptr, 0, &r);
        if (rc == LPHB_E_CAPACITY) {
            triplets.resize(r.n_triplets);
            ids.resize(r.n_ids);
            rc = lphb_build_end(b_, triplets.data(), triplets.size(), ids.data(), ids.size(), &r);
        } else if (rc == LPHB_OK) {
            triplets.clear();
            ids.clear();
        }
        if (rc != LPHB_OK) detail::raise("lphash_b200::build_session::end", rc);
        return r;
    }
    // the same into caller-owned buffers: LPHB_OK (session closed) or LPHB_E_CAPACITY (r holds the sizes; the session
    // stays open for another end)
    int end(mm_triplet_t* triplets, uint64_t triplets_capacity, uint64_t* ids, uint64_t ids_capacity,
            lphb_build_report& r) {
        const int rc = lphb_build_end(b_, triplets, triplets_capacity, ids, ids_capacity, &r);
        if (rc != LPHB_OK && rc != LPHB_E_CAPACITY) detail::raise("lphash_b200::build_session::end", rc);
        return rc;
    }

private:
    lphb_build* b_ = nullptr;
};

namespace minimizer {

// minimizer::from_string (include/minimizer.hpp:11-170): appends one mm_record_t per super-k-mer
// of `contig` to `accumulator` (anything with push_back(mm_record_t), e.g. the reference's
// external_memory_vector<mm_record_t>), advances the running m-mer ordinal `mm_count`, returns the
// number of k-mers.  `canonical_m_mers` must be false (the reference never passes true:
// src/partitioned_mphf.cpp:34).
template <class Accumulator>
[[nodiscard]] uint64_t from_string(char const* contig, std::size_t contig_size, uint32_t k,
                                   uint32_t m, uint64_t seed, bool canonical_m_mers,
                                   uint64_t& mm_count, Accumulator& accumulator, int device = 0) {
    if (canonical_m_mers) throw std::runtime_error("lphash_b200: canonical m-mers are not supported");
    const uint64_t offsets[2] = {0, uint64_t(contig_size)};
    const uint64_t cap = contig_size >= k ? contig_size - k + 1 : 0;
    std::vector<mm_record_t> rec(cap ? cap : 1);
    uint64_t n_rec = 0, n_kmers = 0;
    int rc = lphb_scan_superkmers(device, k, m, seed, contig, offsets, 1, &mm_count, rec.data(),
                                  cap, &n_rec, &n_kmers);
    if (rc != LPHB_OK) detail::raise("lphash_b200::minimizer::from_string", rc);
    for (uint64_t i = 0; i < n_rec; ++i) accumulator.push_back(rec[i]);
    return n_kmers;
}

// Sort by minimizer + minimizer::classify (src/minimizer.cpp:5-50): unique minimizers in ascending
// order as triplets ({itself, 0, 0} for minimizers seen several times) and the ascending ids of the
// occurrences of the latter.  `records` may be in any order (scan order is fine).
inline void classify(std::vector<mm_record_t> const& records, std::vector<mm_triplet_t>& unique_minimizers,
                     std::vector<uint64_t>& colliding_minimizer_ids, int device = 0) {
    const uint64_t n = records.size();
    unique_minimizers.resize(n ? n : 1);
    colliding_minimizer_ids.resize(n ? n : 1);
    uint64_t nt = 0, ni = 0;
    int rc = lphb_classify(device, records.data(), n, unique_minimizers.data(), n, &nt,
                           colliding_minimizer_ids.data(), n, &ni);
    if (rc != LPHB_OK) detail::raise("lphash_b200::minimizer::classify", rc);
    unique_minimizers.resize(nt);
    colliding_minimizer_ids.resize(ni);
}

// Frees the device workspace the two build-side calls keep between calls (call after the loop over
// from_string / get_colliding_kmers, i.e. after src/partitioned_mphf.cpp:77 and :129).
inline void release_workspace(int device = 0) {
    int rc = lphb_scan_release(device);
    if (rc != LPHB_OK) detail::raise("lphash_b200::minimizer::release_workspace", rc);
}

// Batch form: the whole input (or a large slab of it) in one call; records land in `records` in
// scan order.  Returns the number of k-mers.
inline uint64_t from_batch(const char* bases, const uint64_t* offsets, uint64_t n_contigs, uint32_t k,
                           uint32_t m, uint64_t seed, uint64_t& mm_count,
                           std::vector<mm_record_t>& records, int device = 0) {
    uint64_t cap = 0;
    for (uint64_t c = 0; c < n_contigs; ++c) {
        uint64_t len = offsets[c + 1] - offsets[c];
        cap += len >= k ? len - k + 1 : 0;
    }
    records.resize(cap ? cap : 1);
    uint64_t n_rec = 0, n_kmers = 0;
    int rc = lphb_scan_superkmers(device, k, m, seed, bases, offsets, n_contigs, &mm_count,
                                  records.data(), cap, &n_rec, &n_kmers);
    if (rc != LPHB_OK) detail::raise("lphash_b200::minimizer::from_batch", rc);
    records.resize(n_rec);
    return n_kmers;
}

// minimizer::get_colliding_kmers (include/minimizer.hpp:172-319): appends to `accumulator` every
// k-mer of the super-k-mers of `contig` whose minimizer-occurrence id appears in the ascending id
// stream [itr, stop); advances `itr` past the ids consumed and `mm_count` past the contig's m-mers.
template <class IdIterator, class Accumulator>
void get_colliding_kmers(char const* contig, std::size_t contig_size, uint32_t k, uint32_t m,
                         uint64_t seed, bool canonical_m_mers, IdIterator& itr, IdIterator& stop,
                         uint64_t& mm_count, Accumulator& accumulator, int device = 0) {
    if (canonical_m_mers) throw std::runtime_error("lphash_b200: canonical m-mers are not supported");
    const uint64_t n_mmers = contig_size >= m ? contig_size - m + 1 : 0;
    const uint64_t id_end = mm_count + n_mmers;
    // ids that can belong to this contig: [mm_count, id_end)
    std::vector<uint64_t> ids;
    IdIterator probe = itr;
    while (probe != stop && *probe < id_end) {
        ids.push_back(*probe);
        ++probe;
    }
    const uint64_t offsets[2] = {0, uint64_t(contig_size)};
    const uint64_t cap = contig_size >= k ? contig_size - k + 1 : 0;
    std::vector<kmer_t> out(cap ? cap : 1);
    uint64_t n = 0;
    int rc = lphb_colliding_kmers(device, k, m, seed, contig, offsets, 1, &mm_count, ids.data(),
                                  ids.size(), kmer_bits, out.data(), cap, &n);
    if (rc != LPHB_OK) detail::raise("lphash_b200::minimizer::get_colliding_kmers", rc);
    for (uint64_t i = 0; i < n; ++i) accumulator.push_back(out[i]);
    itr = probe;
}

}  // namespace minimizer

}  // namespace lphash_b200
