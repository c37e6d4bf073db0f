// Shared by the two shadow headers of the literal drop-in (partitioned_mphf.hpp, unpartitioned_mphf.hpp): the parts
// of mphf::build / mphf_alt::build that are the same for both - Part 1 (minimizer::from_string over every record),
// Part 2 (sort + minimizer::classify, then PTHash on the distinct minimizers) and Part 4 (k-mers of the colliding
// minimizers, then PTHash on them) - with the scans on the GPU through the C ABI and the two PTHash constructions on
// the CPU through the reference's own pthash headers, called as the reference calls them
// (src/partitioned_mphf.cpp:45-52, 62-90, 108-135, 147-160; src/unpartitioned_mphf.cpp:31-75, 99-128, 140-150).
// Included after the reference's headers (configuration, kmer_t, pthash_*_mphf_t come from there).
#pragma once
#include <cstdlib>
#include <algorithm>
#include <iostream>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "lphash_b200.hpp"
#include "lphash_b200_fastx.hpp"

namespace lphash {
namespace gpu_build {

inline void check(int rc) {
    if (rc != LPHB_OK) throw std::runtime_error(std::string("lphash_b200: ") + lphb_last_error());
}

inline bool cpu_requested() {  // LPHASH_B200_CPU_BUILD=1 forwards the whole build to the reference's class
    const char* e = std::getenv("LPHASH_B200_CPU_BUILD");
    return e && e[0] == '1';
}

// text per batch of the streamed input; LPHASH_B200_BATCH_BYTES sets it (a test forces many batches with it)
inline size_t batch_bytes() {
    constexpr size_t kDefault = size_t(1) << 30;  // well under a batch's 2^32 bases
    const char* e = std::getenv("LPHASH_B200_BATCH_BYTES");
    const size_t v = e ? size_t(std::strtoull(e, nullptr, 10)) : 0;
    return v ? v : kDefault;
}

struct Parts {
    int device = 0;
    uint32_t k = 0, m = 0;
    pthash::build_configuration cfg;
    uint64_t n_records = 0, nkmers = 0;  // contigs of the input, k-mers of Part 1
    // one triplet per distinct minimizer, ascending; ids of every occurrence of a colliding minimizer, ascending
    // (uninitialised storage: at 2.5e9 k-mers a zero-filled worst-case vector would be tens of GB)
    struct Triplets {
        std::unique_ptr<lphash_b200::mm_triplet_t[]> p;
        uint64_t n = 0;
        const lphash_b200::mm_triplet_t* data() const { return p.get(); }
        uint64_t size() const { return n; }
        const lphash_b200::mm_triplet_t* begin() const { return p.get(); }
        const lphash_b200::mm_triplet_t* end() const { return p.get() + n; }
    } triplets;
    struct Ids {
        std::unique_ptr<uint64_t[]> p;
        uint64_t n = 0;
        const uint64_t* data() const { return p.get(); }
        uint64_t size() const { return n; }
    } coll_ids;
    std::vector<unsigned char> minimizer_order, fallback;  // the two serialized single_phf objects

    // Parts 1 and 2: the file streamed through a build session, one batch of at most batch_bytes() of text at a time,
    // so that host memory holds one batch and the result, never the whole input
    void scan_and_order(configuration const& config) {
        k = uint32_t(config.k);
        m = uint32_t(config.m);
        cfg.minimal_output = true;
        cfg.seed = constants::default_pthash_seed;
        cfg.c = config.c;
        cfg.alpha = 0.94;
        cfg.verbose_output = config.verbose;
        cfg.num_threads = config.num_threads;
        cfg.ram = static_cast<uint64_t>(config.max_memory) * essentials::GB;
        cfg.tmp_dir = config.tmp_dirname;
        if (config.verbose) std::cerr << "Part 1: file reading and info gathering\n";
        lphash_b200::build_session session(k, m, config.mm_seed, device);
        uint64_t max_kmers = 0;
        n_records = lphash_b200::fastx::stream_file(config.input_filename, batch_bytes(), [&](lphash_b200::fastx::Batch const& b) {
            for (uint64_t c = 0; c < b.n_records(); ++c) {
                const uint64_t len = b.offsets[c + 1] - b.offsets[c];
                if (len >= k) max_kmers += len - k + 1;
            }
            session.batch(b.bases.data(), b.offsets.data(), b.n_records());
        });
        // super-k-mers are about 2 / (k - m + 2) of the k-mers; a third is room enough for every window of 5 or
        // more (an input that needs more - LPHB_E_CAPACITY reports the counts - gets exactly that on the second end)
        uint64_t cap = max_kmers / 3 + 4096;
        if (const char* e = std::getenv("LPHASH_B200_FIRST_CAP")) cap = std::strtoull(e, nullptr, 10) + 1;  // test hook
        lphb_build_report report{};
        for (int attempt = 0;; ++attempt) {
            triplets.p.reset(new lphash_b200::mm_triplet_t[cap]);
            coll_ids.p.reset(new uint64_t[cap]);
            const int rc = session.end(triplets.p.get(), cap, coll_ids.p.get(), cap, report);
            if (rc == LPHB_E_CAPACITY && attempt == 0) {
                cap = std::max(report.n_triplets, report.n_ids) + 1;
                continue;
            }
            check(rc);
            break;
        }
        triplets.n = report.n_triplets;
        coll_ids.n = report.n_ids;
        nkmers = report.kmers;
        if (config.verbose) std::cerr << "Part 2: build MPHF\n";
        std::vector<uint64_t> keys(triplets.n);
        for (uint64_t i = 0; i < triplets.n; ++i) keys[i] = triplets.p[i].itself;
        pthash_minimizers_mphf_t f;
        f.build_in_external_memory(keys.begin(), triplets.n, cfg);
        lphash_b200::memory_saver saver;
        saver.visit(f);
        minimizer_order.swap(saver.bytes);
    }

    // Part 4: a second pass over the file in the same batches; each batch gets the colliding ids of its m-mer range
    void fallback_function(configuration const& config) {
        if (config.verbose) std::cerr << "Part 4: build fallback MPHF\n";
        uint64_t n_coll_kmers = 0, mm_count = 0;
        const uint64_t kcap = coll_ids.size() * (uint64_t(k) - m + 1) + 1;  // a super-k-mer holds at most k - m + 1 k-mers
        std::unique_ptr<kmer_t[]> kmers(new kmer_t[kcap]);
        const uint64_t* ids_end = coll_ids.data() + coll_ids.size();
        lphash_b200::fastx::stream_file(config.input_filename, batch_bytes(), [&](lphash_b200::fastx::Batch const& b) {
            uint64_t mm_bound = mm_count;  // the batch's ordinals end at or before this (non-ACGT bytes only remove m-mers)
            for (uint64_t c = 0; c < b.n_records(); ++c) {
                const uint64_t len = b.offsets[c + 1] - b.offsets[c];
                if (len >= m) mm_bound += len - m + 1;
            }
            const uint64_t* first = std::lower_bound(coll_ids.data(), ids_end, mm_count);
            const uint64_t* last = std::lower_bound(first, ids_end, mm_bound);
            uint64_t n = 0;
            check(lphb_colliding_kmers(device, k, m, config.mm_seed, b.bases.data(), b.offsets.data(), b.n_records(), &mm_count,
                                       first, uint64_t(last - first), int(sizeof(kmer_t) * 8), kmers.get() + n_coll_kmers,
                                       kcap - n_coll_kmers, &n));
            n_coll_kmers += n;
        });
        pthash_fallback_mphf_t f;
        f.build_in_external_memory(kmers.get(), n_coll_kmers, cfg);
        lphash_b200::memory_saver saver;
        saver.visit(f);
        fallback.swap(saver.bytes);
    }

    // the CSV line both builds print (src/partitioned_mphf.cpp:137-144, src/unpartitioned_mphf.cpp:130-138)
    void csv_line(configuration const& config, std::ostream& res_strm, uint64_t colliding_minimizers, double bits_per_kmer) const {
        const uint64_t n_triplets = triplets.size();
        const uint64_t total_minimizers = (n_triplets - colliding_minimizers) + coll_ids.size();  // records of Part 1
        const uint64_t total_contigs = n_records ? n_records - 1 : 0;
        res_strm << config.input_filename << "," << static_cast<uint32_t>(k) << "," << static_cast<uint32_t>(m) << ","
                 << static_cast<double>(coll_ids.size()) / n_triplets << "," << 2.0 / ((k - m + 1) + 1) << ","
                 << static_cast<double>(total_minimizers) / nkmers << "," << static_cast<double>(total_contigs) / nkmers << ","
                 << bits_per_kmer;
        res_strm << "\n";
    }
};

}  // namespace gpu_build
}  // namespace lphash
