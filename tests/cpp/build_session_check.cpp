// lphash_b200::build_session (include/lphash_b200.hpp) fed one contig per batch.
// usage: build_session_check <batch.bin> <out.bin>
//   batch.bin: u64 k, m, n_contigs, offsets[n_contigs + 1], bases
//   out.bin:   u64 n_triplets, triplets (10 bytes each), u64 n_ids, ids, u64 kmers, mm_count, batches
#include <cstdio>
#include <fstream>
#include <iterator>
#include <vector>

#include "lphash_b200.hpp"

int main(int argc, char** argv) {
    if (argc != 3) return 2;
    std::ifstream in(argv[1], std::ios::binary);
    std::vector<char> raw((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
    const uint64_t* h = reinterpret_cast<const uint64_t*>(raw.data());
    const uint64_t k = h[0], m = h[1], n = h[2];
    const uint64_t* offsets = h + 3;
    const char* bases = reinterpret_cast<const char*>(offsets + n + 1);
    try {
        lphash_b200::build_session s(uint32_t(k), uint32_t(m), 42);
        for (uint64_t c = 0; c < n; ++c) s.batch(bases, offsets + c, 1);
        lphash_b200::build_session moved(std::move(s));
        std::vector<lphash_b200::mm_triplet_t> triplets;
        std::vector<uint64_t> ids;
        const lphb_build_report r = moved.end(triplets, ids);
        std::ofstream out(argv[2], std::ios::binary);
        auto u64 = [&](uint64_t v) { out.write(reinterpret_cast<const char*>(&v), 8); };
        u64(triplets.size());
        out.write(reinterpret_cast<const char*>(triplets.data()), std::streamsize(triplets.size() * 10));
        u64(ids.size());
        out.write(reinterpret_cast<const char*>(ids.data()), std::streamsize(ids.size() * 8));
        u64(r.kmers);
        u64(r.mm_count);
        u64(r.batches);
    } catch (std::exception const& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 3;
    }
    return 0;
}
