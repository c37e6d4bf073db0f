// Exercises the check session of lphash_b200::mphf (include/lphash_b200.hpp): check_begin, check_batch, check_end.
//   check_mirror <file.lph> <batch.bin> <n_batches>
// batch.bin: u64 n_contigs, n_contigs + 1 u64 offsets (offsets[0] = 0), then the bases.  The contigs are cut into
// n_batches batches of about equal contig counts.  Prints the report as `name value` lines.
// Exit code 3 = std::runtime_error from the library: printed to stderr.
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <vector>

#include "lphash_b200.hpp"

namespace lb = lphash_b200;

int main(int argc, char** argv) {
    if (argc != 4) return 1;
    try {
        std::ifstream in(argv[2], std::ios::binary);
        uint64_t n = 0;
        if (!in.read(reinterpret_cast<char*>(&n), 8)) throw std::logic_error("cannot read the contig count");
        std::vector<uint64_t> offsets(n + 1);
        if (!in.read(reinterpret_cast<char*>(offsets.data()), std::streamsize((n + 1) * 8)))
            throw std::logic_error("short offsets");
        std::vector<char> bases(offsets[n]);
        if (!in.read(bases.data(), std::streamsize(bases.size()))) throw std::logic_error("short bases");
        const uint64_t parts = uint64_t(std::atoll(argv[3]));
        lb::mphf hf;
        hf.load(argv[1]);
        hf.check_begin();
        for (uint64_t p = 0; p < parts; ++p) {
            const uint64_t c0 = n * p / parts, c1 = n * (p + 1) / parts;
            hf.check_batch(bases.data(), offsets.data() + c0, c1 - c0);
        }
        const lphb_check_report r = hf.check_end();
        std::cout << "kmers " << r.kmers << "\ncontigs " << r.contigs << "\ndirty_contigs " << r.dirty_contigs
                  << "\nout_of_range " << r.out_of_range << "\nduplicates " << r.duplicates << "\nmissing " << r.missing
                  << "\nstream_mismatches " << r.stream_mismatches << "\nfirst_out_of_range " << r.first_out_of_range
                  << "\nfirst_mismatch " << r.first_mismatch << "\nmin_duplicate_code " << r.min_duplicate_code
                  << "\nmin_missing_code " << r.min_missing_code << "\nok " << r.ok << "\n";
        // a batch outside a session is an argument error, reported as such
        try {
            hf.check_batch(bases.data(), offsets.data(), n);
            throw std::logic_error("check_batch outside a session did not throw");
        } catch (std::runtime_error const&) {
        }
    } catch (std::runtime_error const& e) {
        std::cerr << e.what() << "\n";
        return 3;
    } catch (std::exception const& e) {
        std::cerr << e.what() << "\n";
        return 2;
    }
    return 0;
}
