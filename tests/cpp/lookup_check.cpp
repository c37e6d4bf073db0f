// Exercises lphash_b200::mphf::lookup (include/lphash_b200.hpp) with the class's compile-time kmer_t:
//   lookup_check <file.lph> <kmers.bin> <codes.bin>
// kmers.bin: u64 n, then n packed k-mers of LPHASH_B200_KMER_BITS / 8 little-endian bytes each.
// codes.bin: the n codes.  Exit code 3 = std::runtime_error from the library: printed to stderr.
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
        if (!in.read(reinterpret_cast<char*>(&n), 8)) throw std::runtime_error("cannot read the k-mer count");
        std::vector<lb::kmer_t> kmers(n);
        if (!in.read(reinterpret_cast<char*>(kmers.data()), std::streamsize(n * sizeof(lb::kmer_t))))
            throw std::runtime_error("short k-mer file");
        lb::mphf hf;
        hf.load(argv[1]);
        const std::vector<uint64_t> codes = hf.lookup(kmers.data(), kmers.size());
        if (codes.size() != n) throw std::logic_error("lookup returned the wrong number of codes");
        std::ofstream out(argv[3], std::ios::binary);
        out.write(reinterpret_cast<const char*>(codes.data()), std::streamsize(n * 8));
    } catch (std::runtime_error const& e) {
        std::cerr << e.what() << "\n";
        return 3;
    } catch (std::exception const& e) {
        std::cerr << e.what() << "\n";
        return 2;
    }
    return 0;
}
