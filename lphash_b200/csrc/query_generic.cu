// Generic query kernels: valid for every (k, m) the format allows.
//   k_query_generic  one thread per k-mer, stateless definition (SURVEY.md S1): the code of a
//                    k-mer is query(kmer, leftmost-minimum m-mer, its offset).  It is the
//                    always-available path for (k, m) pairs the tiled kernel (query_tiled.cu) is
//                    not instantiated for.
// (contigs with non-ACGT bytes, where the reference's output depends on stale state - SURVEY.md Q1 -
//  are finished by quirk_kernels.cu.)
#include <cub/device/device_scan.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "device_mphf.cuh"
#include "query_kernels.cuh"

namespace lphb {

namespace {

struct KmerCount {
    const uint64_t* offsets;
    uint32_t k;
    __host__ __device__ uint64_t operator()(uint64_t c) const {
        uint64_t len = offsets[c + 1] - offsets[c];
        return len >= k ? len - k + 1 : 0;
    }
};

__global__ void k_finish_code_offsets(const uint64_t* offsets, uint64_t n_contigs, uint32_t k,
                                      uint64_t* code_off, unsigned long long* status) {
    // ExclusiveSum wrote code_off[0..n); close the array and publish the total.
    uint64_t total = 0;
    if (n_contigs) {
        uint64_t len = offsets[n_contigs] - offsets[n_contigs - 1];
        total = code_off[n_contigs - 1] + (len >= k ? len - k + 1 : 0);
    }
    code_off[n_contigs] = total;
    status[0] = total;
    status[1] = 0;
}

// index of the contig containing stream position i (offsets[c] <= i < offsets[c+1])
__device__ __forceinline__ uint64_t find_contig(const uint64_t* offsets, uint64_t n, uint64_t i) {
    uint64_t lo = 0, hi = n;  // invariant: offsets[lo] <= i < offsets[hi]
    while (hi - lo > 1) {
        uint64_t mid = (lo + hi) >> 1;
        if (__ldg(offsets + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256) k_query_generic(const __grid_constant__ DevImage f,
                                                       const __grid_constant__ DevBatch b) {
    const uint32_t k = f.k;
    uint64_t span = b.end_base - b.first_base;
    for (uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; t < span;
         t += uint64_t(gridDim.x) * blockDim.x) {
        uint64_t i = b.first_base + t;
        uint64_t c = find_contig(b.offsets, b.n_contigs, i);
        uint64_t start = __ldg(b.offsets + c), end = __ldg(b.offsets + c + 1);
        if (i + k > end) continue;
        // forward k-mer, first base in the most significant bits (partitioned_mphf.hpp:106-108)
        uint64_t lo = 0, hi = 0;
        bool ok = true;
        for (uint32_t j = 0; j < k; ++j) {
            uint32_t code = nt4(uint8_t(b.bases[i + j]));
            if (code > 3) { ok = false; break; }
            hi = (hi << 2) | (lo >> 62);
            lo = (lo << 2) | code;
        }
        if (!ok) {
            b.dirty[c] = 1;  // plain store: every writer stores the same value
            continue;
        }
        const Minimizer mz = kmer_minimizer(k, f.m, f.mm_seed, lo, hi);
        Probe pr = probe_minimizer(f, mz.mmer);
        uint64_t hval = pr.slope == 0 ? pr.base + fallback_order(f, lo, hi) : probe_hval(pr, mz.pos);
        b.codes[__ldg(b.code_off + c) + (i - start)] = hval;
    }
}

// bytes outside ACGT/acgt/U/u -> 'A' (what the reference's non-streaming branch makes of them:
// include/mphf_utils.hpp:108, seq_nt4_table[c] & 3)
__global__ void k_sanitize(char* bases, uint64_t n) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x)
        if (nt4(uint8_t(bases[i])) > 3) bases[i] = 'A';
}

__device__ __forceinline__ uint32_t sanitize4(uint32_t w) {
    uint32_t out = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t ch = (w >> (8 * i)) & 0xFFu;
        out |= (nt4(ch) > 3 ? uint32_t('A') : ch) << (8 * i);
    }
    return out;
}

// dst[0..n) = src[0..n) with k_sanitize's mapping, then `pad` bytes of 'A' (the read-ahead of the last tile).  dst and
// src have the same address mod 16: the bytes before the first 16-byte boundary and after the last are copied one by
// one, everything between in 16-byte vectors, streamed (each byte is read and written once).
__global__ void __launch_bounds__(256) k_copy_sanitize(char* dst, const char* src, uint64_t n, uint32_t pad) {
    const uint64_t tid = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x, stride = uint64_t(gridDim.x) * blockDim.x;
    const uint64_t head = min(n, uint64_t((16u - uint32_t(reinterpret_cast<uintptr_t>(src) & 15u)) & 15u));
    const uint64_t n_vec = (n - head) / 16, tail = head + n_vec * 16;
    const uint4* s4 = reinterpret_cast<const uint4*>(src + head);
    uint4* d4 = reinterpret_cast<uint4*>(dst + head);
    for (uint64_t i = tid; i < n_vec; i += stride) {
        uint4 v = __ldcs(s4 + i);
        v.x = sanitize4(v.x);
        v.y = sanitize4(v.y);
        v.z = sanitize4(v.z);
        v.w = sanitize4(v.w);
        __stcs(d4 + i, v);
    }
    if (tid < head) dst[tid] = nt4(uint8_t(src[tid])) > 3 ? 'A' : src[tid];
    if (tid < n - tail) dst[tail + tid] = nt4(uint8_t(src[tail + tid])) > 3 ? 'A' : src[tail + tid];
    if (tid < pad) dst[n + tid] = 'A';
}

__global__ void k_count_dirty(const uint8_t* dirty, uint64_t n, unsigned long long* status) {
    unsigned long long local = 0;
    for (uint64_t c = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; c < n;
         c += uint64_t(gridDim.x) * blockDim.x)
        local += dirty[c] ? 1 : 0;
    for (int o = 16; o; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(status + 1, local);
}

}  // namespace

uint64_t code_offsets_tmp_bytes(uint64_t n_contigs) {
    size_t bytes = 0;
    KmerCount op{nullptr, 1};
    cub::CountingInputIterator<uint64_t> cnt(0);
    cub::TransformInputIterator<uint64_t, KmerCount, cub::CountingInputIterator<uint64_t>> it(cnt, op);
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, it, (uint64_t*)nullptr, n_contigs);
    return bytes + 256;
}

void launch_code_offsets(const uint64_t* d_offsets, uint64_t n_contigs, uint32_t k,
                         uint64_t* d_code_off, unsigned long long* d_status, void* d_tmp,
                         uint64_t tmp_bytes, cudaStream_t stream) {
    if (n_contigs) {
        KmerCount op{d_offsets, k};
        cub::CountingInputIterator<uint64_t> cnt(0);
        cub::TransformInputIterator<uint64_t, KmerCount, cub::CountingInputIterator<uint64_t>> it(cnt, op);
        size_t bytes = tmp_bytes;
        cub::DeviceScan::ExclusiveSum(d_tmp, bytes, it, d_code_off, n_contigs, stream);
    }
    k_finish_code_offsets<<<1, 1, 0, stream>>>(d_offsets, n_contigs, k, d_code_off, d_status);
}

void launch_query_generic(DevImage const& img, DevBatch const& b, cudaStream_t stream) {
    uint64_t span = b.end_base - b.first_base;
    if (span == 0) return;
    uint64_t blocks = (span + 255) / 256;
    if (blocks > 148ull * 64) blocks = 148ull * 64;
    k_query_generic<<<unsigned(blocks), 256, 0, stream>>>(img, b);
}

void launch_sanitize(char* d_bases, uint64_t n, cudaStream_t stream) {
    if (!n) return;
    uint64_t blocks = (n + 255) / 256;
    if (blocks > 148ull * 16) blocks = 148ull * 16;
    k_sanitize<<<unsigned(blocks), 256, 0, stream>>>(d_bases, n);
}

uint64_t copy_sanitize_at(const char* src) { return reinterpret_cast<uintptr_t>(src) & 15u; }

void launch_copy_sanitize(char* d_dst, const char* d_src, uint64_t n, cudaStream_t stream) {
    char* dst = d_dst + copy_sanitize_at(d_src);
    uint64_t blocks = (n / 16 + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 148ull * 16) blocks = 148ull * 16;
    k_copy_sanitize<<<unsigned(blocks), 256, 0, stream>>>(dst, d_src, n, kCopySanitizePad);
}

void launch_count_dirty(const uint8_t* dirty, uint64_t n, unsigned long long* status,
                        cudaStream_t stream) {
    if (!n) return;
    uint64_t blocks = (n + 255) / 256;
    if (blocks > 148ull * 8) blocks = 148ull * 8;
    k_count_dirty<<<unsigned(blocks), 256, 0, stream>>>(dirty, n, status);
}

}  // namespace lphb
