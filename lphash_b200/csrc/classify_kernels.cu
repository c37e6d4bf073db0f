// minimizer::classify on the device (ref src/minimizer.cpp:5-50, caller src/partitioned_mphf.cpp:86;
// SURVEY.md §8 row a16) together with the sort by minimizer it consumes (the reference sorts the
// mm_record_t stream in an external_memory_vector, src/partitioned_mphf.cpp:62-66):
//   records sorted by `itself`; a minimizer seen once -> triplet {itself, p1, size}; a minimizer seen
//   several times -> ONE triplet {itself, 0, 0} + the ids of all its occurrences; triplets come out in
//   ascending minimizer order (the key stream PTHash consumes), ids in ascending order.
// Radix sort of (itself, record index), neighbour compare for group heads / singletons, two prefix
// sums for the output slots, scatter, radix sort of the colliding ids.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "scan_kernels.cuh"

namespace lphb {

namespace {

__device__ __forceinline__ uint64_t rec_u64(const uint8_t* p) {  // records are 2-byte aligned
    const uint16_t* q = reinterpret_cast<const uint16_t*>(p);
    return uint64_t(q[0]) | (uint64_t(q[1]) << 16) | (uint64_t(q[2]) << 32) | (uint64_t(q[3]) << 48);
}

unsigned cgrid(uint64_t n) {
    uint64_t blocks = (n + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 148ull * 64) blocks = 148ull * 64;
    return unsigned(blocks);
}

__global__ void k_rec_keys(const uint8_t* records, uint64_t n, uint64_t* key, uint32_t* idx) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        key[i] = rec_u64(records + 18 * i);
        idx[i] = uint32_t(i);
    }
}

// flags[i] bit 0: first of its group (one triplet); bit 1: member of a group of several (one id)
__global__ void k_group_flags(const uint64_t* key, uint64_t n, uint8_t* flags) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint64_t v = key[i];
        const bool first = i == 0 || key[i - 1] != v;
        const bool last = i + 1 == n || key[i + 1] != v;
        flags[i] = uint8_t((first ? 1 : 0) | ((first && last) ? 0 : 2));
    }
}

struct Bit0 {
    __host__ __device__ uint32_t operator()(uint8_t f) const { return f & 1u; }
};
struct Bit1 {
    __host__ __device__ uint32_t operator()(uint8_t f) const { return (f >> 1) & 1u; }
};

__global__ void k_close_counts(const uint8_t* flags, uint64_t n, const uint32_t* gslot, const uint32_t* cslot,
                               unsigned long long* counts) {
    counts[0] = n ? gslot[n - 1] + (flags[n - 1] & 1u) : 0;         // triplets
    counts[1] = n ? cslot[n - 1] + ((flags[n - 1] >> 1) & 1u) : 0;  // colliding ids
}

__global__ void k_classify_emit(const uint8_t* records, const uint64_t* key, const uint32_t* idx,
                                const uint8_t* flags, const uint32_t* gslot, const uint32_t* cslot,
                                uint64_t n, uint8_t* triplets, uint64_t* ids) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint8_t f = flags[i];
        const uint8_t* r = records + 18ull * idx[i];
        if (f & 1u) {  // 10-byte packed mm_triplet_t (constants.hpp:35-41), 2-byte aligned
            uint16_t* q = reinterpret_cast<uint16_t*>(triplets + 10ull * gslot[i]);
            const uint64_t v = key[i];
            q[0] = uint16_t(v); q[1] = uint16_t(v >> 16); q[2] = uint16_t(v >> 32); q[3] = uint16_t(v >> 48);
            q[4] = (f & 2u) ? uint16_t(0) : *reinterpret_cast<const uint16_t*>(r + 16);  // p1 | size << 8
        }
        if (f & 2u) ids[cslot[i]] = rec_u64(r + 8);
    }
}

__global__ void k_group_singleton_ids(const uint8_t* records, const uint32_t* idx, const uint8_t* flags,
                                      const uint32_t* gslot, uint64_t n, uint64_t* sid) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint8_t f = flags[i];
        if (f & 1u) sid[gslot[i]] = (f & 2u) ? ~0ull : rec_u64(records + 18ull * idx[i] + 8);
    }
}

}  // namespace

uint64_t classify_tmp_bytes(uint64_t n) {
    size_t a = 0, b = 0, c = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                    (const uint32_t*)nullptr, (uint32_t*)nullptr, n);
    cub::TransformInputIterator<uint32_t, Bit0, const uint8_t*> it(nullptr, Bit0{});
    cub::DeviceScan::ExclusiveSum(nullptr, b, it, (uint32_t*)nullptr, n);
    cub::DeviceRadixSort::SortKeys(nullptr, c, (const uint64_t*)nullptr, (uint64_t*)nullptr, n);
    size_t m = a > b ? a : b;
    return (m > c ? m : c) + 256;
}

void launch_classify_groups(const uint8_t* records, uint64_t n, uint64_t* key, uint64_t* key_sorted,
                            uint32_t* idx, uint32_t* idx_sorted, uint8_t* flags, uint32_t* gslot,
                            uint32_t* cslot, unsigned long long* counts, void* d_tmp, uint64_t tmp_bytes,
                            int key_bits, cudaStream_t stream) {
    if (n) {
        k_rec_keys<<<cgrid(n), 256, 0, stream>>>(records, n, key, idx);
        size_t bytes = tmp_bytes;
        cub::DeviceRadixSort::SortPairs(d_tmp, bytes, key, key_sorted, idx, idx_sorted, n, 0, key_bits, stream);
        k_group_flags<<<cgrid(n), 256, 0, stream>>>(key_sorted, n, flags);
        cub::TransformInputIterator<uint32_t, Bit0, const uint8_t*> it0(flags, Bit0{});
        bytes = tmp_bytes;
        cub::DeviceScan::ExclusiveSum(d_tmp, bytes, it0, gslot, n, stream);
        cub::TransformInputIterator<uint32_t, Bit1, const uint8_t*> it1(flags, Bit1{});
        bytes = tmp_bytes;
        cub::DeviceScan::ExclusiveSum(d_tmp, bytes, it1, cslot, n, stream);
    }
    k_close_counts<<<1, 1, 0, stream>>>(flags, n, gslot, cslot, counts);
}

void launch_classify_emit(const uint8_t* records, const uint64_t* key_sorted, const uint32_t* idx_sorted,
                          const uint8_t* flags, const uint32_t* gslot, const uint32_t* cslot, uint64_t n,
                          uint8_t* triplets, uint64_t* ids_unsorted, uint64_t* ids_sorted, uint64_t n_ids,
                          void* d_tmp, uint64_t tmp_bytes, cudaStream_t stream) {
    if (!n) return;
    k_classify_emit<<<cgrid(n), 256, 0, stream>>>(records, key_sorted, idx_sorted, flags, gslot, cslot, n,
                                                   triplets, ids_unsorted);
    if (n_ids) {
        size_t bytes = tmp_bytes;
        cub::DeviceRadixSort::SortKeys(d_tmp, bytes, ids_unsorted, ids_sorted, n_ids, 0, 64, stream);
    }
}

void launch_classify_singleton_ids(const uint8_t* records, const uint32_t* idx_sorted, const uint8_t* flags,
                                   const uint32_t* gslot, uint64_t n, uint64_t* sid, cudaStream_t stream) {
    if (n) k_group_singleton_ids<<<cgrid(n), 256, 0, stream>>>(records, idx_sorted, flags, gslot, n, sid);
}

}  // namespace lphb
