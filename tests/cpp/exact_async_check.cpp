// Exercises lphash_b200::mphf::query_batch_device_async (include/lphash_b200.hpp) on a batch the program moves to the
// device itself, on a stream of its own:
//   exact_async_check <file.lph> <batch.bin> <out.bin>
// batch.bin: u64 n_contigs, n_contigs + 1 u64 offsets, then the bases.  out.bin: the 4 status words, then the
// status[0] codes and the n_contigs + 1 code offsets.
// Exit code 3 = std::runtime_error from the library or the CUDA runtime: printed to stderr.
#include <cuda_runtime.h>

#include <fstream>
#include <iostream>
#include <stdexcept>
#include <vector>

#include "lphash_b200.hpp"

namespace lb = lphash_b200;

namespace {
void ck(cudaError_t e) {
    if (e != cudaSuccess) throw std::runtime_error(std::string("CUDA: ") + cudaGetErrorString(e));
}
struct Stream {  // declared before the handle, so destroyed after it: the handle refers to the streams it ran on
    cudaStream_t s = nullptr;
    Stream() { ck(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)); }
    ~Stream() { cudaStreamDestroy(s); }
};
template <class T>
struct Dev {
    T* p = nullptr;
    explicit Dev(size_t n) { ck(cudaMalloc(reinterpret_cast<void**>(&p), (n ? n : 1) * sizeof(T))); }
    ~Dev() { cudaFree(p); }
};
}  // namespace

int main(int argc, char** argv) {
    if (argc != 4) return 1;
    try {
        std::ifstream in(argv[2], std::ios::binary);
        uint64_t n_contigs = 0;
        if (!in.read(reinterpret_cast<char*>(&n_contigs), 8)) throw std::logic_error("cannot read the contig count");
        std::vector<uint64_t> offsets(n_contigs + 1);
        if (!in.read(reinterpret_cast<char*>(offsets.data()), std::streamsize(offsets.size() * 8)))
            throw std::logic_error("short offsets");
        std::vector<char> bases(offsets.back());
        if (!in.read(bases.data(), std::streamsize(bases.size()))) throw std::logic_error("short bases");
        Stream stream;
        const cudaStream_t s = stream.s;
        lb::mphf hf;
        hf.load(argv[1]);
        uint64_t cap = 0;
        for (uint64_t c = 0; c < n_contigs; ++c) {
            const uint64_t len = offsets[c + 1] - offsets[c];
            cap += len >= hf.get_m() ? len - hf.get_m() + 1 : 0;
        }
        Dev<char> d_bases(bases.size());
        Dev<uint64_t> d_off(n_contigs + 1), d_codes(cap), d_code_off(n_contigs + 1), d_status(4);
        ck(cudaMemcpyAsync(d_bases.p, bases.data(), bases.size(), cudaMemcpyHostToDevice, s));
        ck(cudaMemcpyAsync(d_off.p, offsets.data(), offsets.size() * 8, cudaMemcpyHostToDevice, s));
        hf.query_batch_device_async(d_bases.p, d_off.p, offsets.data(), n_contigs, d_codes.p, cap, d_code_off.p,
                                    d_status.p, s);
        std::vector<uint64_t> status(4);
        ck(cudaMemcpyAsync(status.data(), d_status.p, 32, cudaMemcpyDeviceToHost, s));
        ck(cudaStreamSynchronize(s));
        std::vector<uint64_t> codes(status[0]), code_off(n_contigs + 1);
        ck(cudaMemcpy(codes.data(), d_codes.p, codes.size() * 8, cudaMemcpyDeviceToHost));
        ck(cudaMemcpy(code_off.data(), d_code_off.p, code_off.size() * 8, cudaMemcpyDeviceToHost));
        std::ofstream out(argv[3], std::ios::binary);
        out.write(reinterpret_cast<const char*>(status.data()), 32);
        out.write(reinterpret_cast<const char*>(codes.data()), std::streamsize(codes.size() * 8));
        out.write(reinterpret_cast<const char*>(code_off.data()), std::streamsize(code_off.size() * 8));
        // a capacity one short of the bound is refused before anything runs
        if (cap) {
            try {
                hf.query_batch_device_async(d_bases.p, d_off.p, offsets.data(), n_contigs, d_codes.p, cap - 1,
                                            d_code_off.p, d_status.p, s);
                throw std::logic_error("a capacity below the bound was accepted");
            } catch (std::runtime_error const& e) {
                if (std::string(e.what()).find("code -5") == std::string::npos) throw;
            }
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
