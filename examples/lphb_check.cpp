// build-p --check on the GPU path, stand-alone: is <index.lph> a minimal perfect hash of the k-mers of <unitigs>, and do
// its streaming and non-streaming codes agree on them?  The reference runs the three tests of `check`
// (include/mphf_utils.hpp:51-100; src/build.cpp:36-43) with two operator() calls per record and a bit vector on one
// host thread; here the records stream through the ingest of include/lphash_b200_fastx.hpp into one lphb_check_*
// session (lphb_check_batch per chunk), so inflate + parse of one chunk overlap the check of the previous one.
//
//   lphb_check <index.lph> <kmer_bits: 64|128> <unitigs.fa|.fq[.gz]> [device] [chunk_MB] [alt]
//
// `alt`: the index is an unpartitioned one (build-u).  Prints one CSV line: unitig file, index file, k-mers checked,
// out-of-range codes, duplicate hits, missing codes, streaming mismatches, ms end to end (file open to the verdict).
// Then "[Info] Everything is ok" when the check passes, else the first failure: a record number (0-based, file
// order) and a position in the record for a code out of range or a streaming mismatch, a code for a duplicate or a
// missing code.  Exit status: 0 passed, 1 failed, 2 could not run.
//
//   g++ -std=c++17 -O2 -DLPHASH_B200_WITH_ZLIB -Iinclude examples/lphb_check.cpp -o lphb_check
//       (continued) -Llphash_b200 -llphash_b200 -Wl,-rpath,$PWD/lphash_b200 -lz -pthread
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "lphash_b200.hpp"
#include "lphash_b200_fastx.hpp"

int main(int argc, char** argv) {
    if (argc < 4) {
        std::fprintf(stderr, "usage: %s <index.lph> <kmer_bits> <unitigs.fa|.fq[.gz]> [device] [chunk_MB] [alt]\n",
                     argv[0]);
        return 2;
    }
    const int bits = std::atoi(argv[2]);
    const int device = argc > 4 ? std::atoi(argv[4]) : 0;
    const size_t chunk = (argc > 5 ? size_t(std::atoll(argv[5])) : 16) << 20;
    const bool alt = argc > 6 && std::strcmp(argv[6], "alt") == 0;
    lphb_mphf* f = nullptr;
    try {
        using clock = std::chrono::steady_clock;
        const auto t0 = clock::now();
        const int rc = alt ? lphb_mphf_alt_load_file(argv[1], bits, device, &f)
                           : lphb_mphf_load_file(argv[1], bits, device, &f);
        if (rc != LPHB_OK) {
            std::fprintf(stderr, "%s\n", lphb_last_error());
            return 2;
        }
        lphb_info info{};
        lphb_mphf_info(f, &info);
        auto check = [](int rc) {
            if (rc != LPHB_OK) throw std::runtime_error(lphb_last_error());
        };
        check(lphb_check_begin(f));
        // first k-mer ordinal of every record, to name the record a failing ordinal belongs to
        std::vector<uint64_t> record_start{0};
        lphash_b200::fastx::stream_file(argv[3], chunk, [&](lphash_b200::fastx::Batch& b) {
            for (uint64_t c = 0; c < b.n_records(); ++c) {
                const uint64_t len = b.offsets[c + 1] - b.offsets[c];
                record_start.push_back(record_start.back() + (len >= info.k ? len - info.k + 1 : 0));
            }
            check(lphb_check_batch(f, b.bases.data(), b.offsets.data(), b.n_records()));
        });
        lphb_check_report r{};
        check(lphb_check_end(f, &r));
        const double ms = std::chrono::duration<double, std::milli>(clock::now() - t0).count();
        std::printf("%s,%s,%llu,%llu,%llu,%llu,%llu,%.3f\n", argv[3], argv[1], (unsigned long long)r.kmers,
                    (unsigned long long)r.out_of_range, (unsigned long long)r.duplicates, (unsigned long long)r.missing,
                    (unsigned long long)r.stream_mismatches, ms);
        auto where = [&](uint64_t ordinal) {
            const uint64_t rec = uint64_t(std::upper_bound(record_start.begin(), record_start.end(), ordinal) -
                                          record_start.begin()) - 1;
            std::printf("record %llu, position %llu", (unsigned long long)rec,
                        (unsigned long long)(ordinal - record_start[rec]));
        };
        if (r.ok) {
            std::printf("[Info] Everything is ok\n");
        } else if (r.out_of_range) {
            std::printf("[Error] code out of range (>= %llu) at ", (unsigned long long)info.nkmers);
            where(r.first_out_of_range);
            std::printf("\n");
        } else if (r.stream_mismatches) {
            std::printf("[Error] streaming code differs from the non-streaming one at ");
            where(r.first_mismatch);
            std::printf("\n");
        } else if (r.duplicates) {
            std::printf("[Error] code %llu hit more than once (%llu duplicate hits)\n",
                        (unsigned long long)r.min_duplicate_code, (unsigned long long)r.duplicates);
        } else {
            std::printf("[Error] code %llu never hit (%llu codes missing)\n", (unsigned long long)r.min_missing_code,
                        (unsigned long long)r.missing);
        }
        if (r.dirty_contigs)
            std::printf("[Warning] %llu records hold bytes outside ACGT: their streaming codes were not compared\n",
                        (unsigned long long)r.dirty_contigs);
        lphb_mphf_free(f);
        return r.ok ? 0 : 1;
    } catch (std::exception const& e) {
        std::fprintf(stderr, "%s\n", e.what());
        if (f) lphb_mphf_free(f);
        return 2;
    }
}
