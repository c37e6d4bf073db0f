// Build-side scan, generic form (any k, m): the stateless definition of the record stream that
// minimizer::from_string emits (SURVEY.md S2'; ref include/minimizer.hpp:11-170):
//   for k-mer i of a contig, b(i) = leftmost argmin of the m-mer hash over offsets i..i+w-1;
//   a record starts at every i with b(i) != b(i-1) (and at the contig's first k-mer);
//   record = {itself = m-mer at b, id = id_base(contig) + b, p1 = b - i, size = run length}.
// and of minimizer::get_colliding_kmers (ref include/minimizer.hpp:172-319): the forward k-mers
// of every record whose id is in the sorted id list, in scan order.
#include <cub/device/device_scan.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "device_mphf.cuh"
#include "scan_kernels.cuh"

namespace lphb {

namespace {

struct MmerCount {
    const uint64_t* offsets;
    uint32_t m;
    __host__ __device__ uint64_t operator()(uint64_t c) const {
        uint64_t len = offsets[c + 1] - offsets[c];
        return len >= m ? len - m + 1 : 0;
    }
};

struct AddBase {
    uint64_t base;
    __host__ __device__ uint64_t operator()(uint64_t a, uint64_t b) const { return a + b; }
};

__global__ void k_finish_id_base(const uint64_t* offsets, uint64_t n, uint32_t m, uint64_t mm_in,
                                 uint64_t* id_base) {
    // ExclusiveSum filled id_base[0..n) with sums starting at 0: shift by mm_in is folded into the
    // scan's initial value; only the closing entry is written here.
    uint64_t total = mm_in;
    if (n) {
        uint64_t len = offsets[n] - offsets[n - 1];
        total = id_base[n - 1] + (len >= m ? len - m + 1 : 0);
    }
    id_base[n] = total;
}

__device__ __forceinline__ uint64_t find_contig(const uint64_t* offsets, uint64_t n, uint64_t i) {
    uint64_t lo = 0, hi = n;
    while (hi - lo > 1) {
        uint64_t mid = (lo + hi) >> 1;
        if (__ldg(offsets + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// m-mer starting at base j (first base most significant), or false if a byte is invalid
__device__ __forceinline__ bool read_mmer(const char* s, uint32_t m, uint64_t& out) {
    uint64_t v = 0;
    for (uint32_t j = 0; j < m; ++j) {
        uint32_t code = nt4(uint8_t(s[j]));
        if (code > 3) return false;
        v = (v << 2) | code;
    }
    out = v;
    return true;
}

__global__ void __launch_bounds__(256) k_scan_heads(const __grid_constant__ ScanBatch b,
                                                    uint8_t* head, uint8_t* pos) {
    const uint32_t k = b.k, m = b.m, w = k - m + 1;
    const uint64_t mm_mask = (uint64_t(1) << (2 * m)) - 1;
    uint64_t span = b.end_base - b.first_base;
    for (uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; t < span;
         t += uint64_t(gridDim.x) * blockDim.x) {
        uint64_t i = b.first_base + t;
        uint64_t c = find_contig(b.offsets, b.n_contigs, i);
        uint64_t start = __ldg(b.offsets + c), end = __ldg(b.offsets + c + 1);
        if (i + k > end) continue;
        bool first = (i == start);
        // rolling m-mers over bases [i - 1, i + k): w + 1 hashes (the extra one is the m-mer that
        // left the window, needed for b(i-1))
        uint64_t from = first ? i : i - 1;
        uint64_t mm = 0;
        bool ok = true;
        uint64_t prev_best = 0, best = 0;
        uint32_t prev_p = 0, best_p = 0;  // offsets relative to i - 1 (prev) and i (cur)
        uint32_t run = 0;
        for (uint64_t j = from; j < i + k; ++j) {
            uint32_t code = nt4(uint8_t(b.bases[j]));
            if (code > 3) { ok = false; break; }
            mm = ((mm << 2) | code) & mm_mask;
            if (++run < m) continue;
            uint64_t q = j + 1 - m;  // start of this m-mer
            uint64_t h = murmur64(mm, b.seed);
            if (q >= i) {            // in the current window [i, i+w)
                if (q == i || h < best) { best = h; best_p = uint32_t(q - i); }
            }
            if (!first && q < i + w - 1) {  // in the previous window [i-1, i+w-1)
                if (q == i - 1 || h < prev_best) { prev_best = h; prev_p = uint32_t(q - (i - 1)); }
            }
        }
        if (!ok) {
            b.dirty[c] = 1;
            continue;
        }
        uint64_t d = __ldg(b.code_off + c) + (i - start);
        bool is_head = first || (uint64_t(best_p) + i != uint64_t(prev_p) + i - 1);
        head[d] = is_head ? 1 : 0;
        pos[d] = uint8_t(best_p);
    }
}

struct U8ToU32 {
    __host__ __device__ uint32_t operator()(uint8_t v) const { return v; }
};

__global__ void k_finish_ranks(const uint8_t* head, uint64_t n, uint32_t* rank) {
    rank[n] = n ? rank[n - 1] + head[n - 1] : 0;
}

__device__ __forceinline__ void store_record(uint8_t* rec, uint64_t itself, uint64_t id, uint8_t p1) {
    // 18-byte packed mm_record_t (constants.hpp:26-33); records are only 2-byte aligned
    uint16_t* q = reinterpret_cast<uint16_t*>(rec);
    q[0] = uint16_t(itself); q[1] = uint16_t(itself >> 16); q[2] = uint16_t(itself >> 32); q[3] = uint16_t(itself >> 48);
    q[4] = uint16_t(id); q[5] = uint16_t(id >> 16); q[6] = uint16_t(id >> 32); q[7] = uint16_t(id >> 48);
    rec[16] = p1;
}

// Pass 2.  A block takes 1024 consecutive k-mers (dense index) at a time; their records are
// consecutive too (rank is a prefix count).  Step 1 compacts the heads of the chunk into a list
// (rank - rank of the chunk's first k-mer is the list index), step 2 builds one record per thread
// with all lanes busy, in shared memory, step 3 writes the chunk's records as one contiguous,
// coalesced run.  size = distance to the next head (every contig's first k-mer is a head).
constexpr int kEmitChunk = 1024;
__global__ void __launch_bounds__(256) k_scan_emit(const __grid_constant__ ScanBatch b,
                                                   const uint8_t* head, const uint8_t* pos,
                                                   const uint32_t* rank, uint8_t* records,
                                                   uint32_t* start_pos) {
    __shared__ __align__(16) uint16_t s_rec[kEmitChunk * 9];
    __shared__ uint16_t s_list[kEmitChunk];
    __shared__ uint64_t s_c0;
    const uint32_t m = b.m;
    const uint64_t n = b.n_kmers;
    for (uint64_t d0 = uint64_t(blockIdx.x) * kEmitChunk; d0 < n; d0 += uint64_t(gridDim.x) * kEmitChunk) {
        const uint64_t d1 = d0 + kEmitChunk < n ? d0 + kEmitChunk : n;
        const uint32_t r0 = rank[d0], r1 = rank[d1];
        // contig of the chunk's first k-mer, once per chunk; a record then walks forward from it (a chunk
        // rarely spans more than a few contigs)
        if (threadIdx.x == 0) s_c0 = find_contig(b.code_off, b.n_contigs, d0);
        for (uint64_t d = d0 + threadIdx.x; d < d1; d += blockDim.x)
            if (head[d]) s_list[rank[d] - r0] = uint16_t(d - d0);
        __syncthreads();
        const uint64_t c0 = s_c0;
        for (uint32_t t = threadIdx.x; t < r1 - r0; t += blockDim.x) {
            const uint64_t d = d0 + s_list[t];
            // last contig whose first k-mer is at or before d (contigs without k-mers share their successor's offset)
            uint64_t c = c0;
            while (c + 1 < b.n_contigs && __ldg(b.code_off + c + 1) <= d) ++c;
            const uint64_t start = __ldg(b.offsets + c);
            const uint64_t i = start + (d - __ldg(b.code_off + c));
            const uint32_t p1 = pos[d];
            const char* s = b.bases + i + p1;
            uint64_t mm = 0;
#pragma unroll
            for (int j = 0; j < 31; ++j) {  // clean input only (a dirty batch was rejected before pass 2)
                const uint32_t ch = uint8_t(s[j < int(m) ? j : 0]);
                if (j < int(m)) mm = (mm << 2) | (((ch >> 1) ^ (ch >> 2)) & 3u);
            }
            uint64_t e;  // next head
            if (t + 1 < r1 - r0) {
                e = d0 + s_list[t + 1];
            } else {
                e = d1;
                while (e < n && !head[e]) ++e;
            }
            const uint64_t id = __ldg(b.id_base + c) + (i + p1 - start);
            uint16_t* q = s_rec + t * 9;  // 18-byte packed mm_record_t (constants.hpp:26-33)
            q[0] = uint16_t(mm); q[1] = uint16_t(mm >> 16); q[2] = uint16_t(mm >> 32); q[3] = uint16_t(mm >> 48);
            q[4] = uint16_t(id); q[5] = uint16_t(id >> 16); q[6] = uint16_t(id >> 32); q[7] = uint16_t(id >> 48);
            q[8] = uint16_t(p1 | (uint32_t(e - d) << 8));
            start_pos[r0 + t] = uint32_t(i - b.first_base);
        }
        __syncthreads();
        uint16_t* dst = reinterpret_cast<uint16_t*>(records) + uint64_t(r0) * 9;  // records are 2-byte aligned
        const uint32_t n16 = (r1 - r0) * 9;
        for (uint32_t t = threadIdx.x; t < n16; t += blockDim.x) dst[t] = s_rec[t];
        __syncthreads();
    }
}

__device__ __forceinline__ uint64_t load_u64_2(const uint8_t* p) {
    const uint16_t* q = reinterpret_cast<const uint16_t*>(p);
    return uint64_t(q[0]) | (uint64_t(q[1]) << 16) | (uint64_t(q[2]) << 32) | (uint64_t(q[3]) << 48);
}

__global__ void k_colliding_mark(const uint8_t* records, uint64_t n_records, const uint64_t* ids,
                                 uint64_t n_ids, uint32_t* take) {
    for (uint64_t r = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; r < n_records;
         r += uint64_t(gridDim.x) * blockDim.x) {
        uint64_t id = load_u64_2(records + 18 * r + 8);
        uint64_t lo = 0, hi = n_ids;  // first index with ids[idx] >= id
        while (lo < hi) {
            uint64_t mid = (lo + hi) >> 1;
            if (__ldg(ids + mid) < id) lo = mid + 1; else hi = mid;
        }
        bool in = lo < n_ids && __ldg(ids + lo) == id;
        take[r] = in ? uint32_t(records[18 * r + 17]) : 0u;
    }
}

// get_colliding_kmers: the forward k-mers of every taken record, in scan order.  One thread per record
// (about 1 % of them are taken; a record has at most k - m + 1 k-mers).
__global__ void __launch_bounds__(256) k_colliding_emit(const __grid_constant__ ScanBatch b, uint64_t n_records,
                                                        const uint32_t* start_pos, const uint32_t* take,
                                                        const uint64_t* out_off, int kmer_bits, uint8_t* kmers) {
    const uint32_t k = b.k;
    const uint64_t lo_mask = k >= 32 ? ~uint64_t(0) : ((uint64_t(1) << (2 * k)) - 1);
    const uint64_t hi_mask = k > 32 ? ((uint64_t(1) << (2 * k - 64)) - 1) : 0;
    for (uint64_t r = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; r < n_records;
         r += uint64_t(gridDim.x) * blockDim.x) {
        const uint32_t n = take[r];
        if (!n) continue;
        const char* s = b.bases + b.first_base + start_pos[r];
        uint64_t lo = 0, hi = 0;
        for (uint32_t j = 0; j + 1 < k; ++j) {  // first k - 1 bases
            const uint32_t code = nt4(uint8_t(s[j])) & 3u;
            hi = (hi << 2) | (lo >> 62);
            lo = (lo << 2) | code;
        }
        uint64_t o = out_off[r];
        for (uint32_t j = 0; j < n; ++j, ++o) {
            const uint32_t code = nt4(uint8_t(s[k - 1 + j])) & 3u;
            hi = ((hi << 2) | (lo >> 62)) & hi_mask;
            lo = ((lo << 2) | code) & lo_mask;
            if (kmer_bits == 64) {
                reinterpret_cast<uint64_t*>(kmers)[o] = lo;
            } else {
                reinterpret_cast<uint64_t*>(kmers)[2 * o] = lo;
                reinterpret_cast<uint64_t*>(kmers)[2 * o + 1] = hi;
            }
        }
    }
}

unsigned grid_for(uint64_t n, unsigned cap_blocks = 148 * 64) {
    uint64_t blocks = (n + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > cap_blocks) blocks = cap_blocks;
    return unsigned(blocks);
}

}  // namespace

void launch_id_base(const uint64_t* d_offsets, uint64_t n_contigs, uint32_t m, uint64_t mm_count_in,
                    uint64_t* d_id_base, void* d_tmp, uint64_t tmp_bytes, cudaStream_t stream) {
    if (n_contigs) {
        MmerCount op{d_offsets, m};
        cub::CountingInputIterator<uint64_t> cnt(0);
        cub::TransformInputIterator<uint64_t, MmerCount, cub::CountingInputIterator<uint64_t>> it(cnt, op);
        size_t bytes = tmp_bytes;
        cub::DeviceScan::ExclusiveScan(d_tmp, bytes, it, d_id_base, AddBase{0}, mm_count_in, n_contigs,
                                       stream);
    }
    k_finish_id_base<<<1, 1, 0, stream>>>(d_offsets, n_contigs, m, mm_count_in, d_id_base);
}

void launch_scan_heads(ScanBatch const& b, uint8_t* head, uint8_t* pos, cudaStream_t stream) {
    uint64_t span = b.end_base - b.first_base;
    if (!span) return;
    k_scan_heads<<<grid_for(span), 256, 0, stream>>>(b, head, pos);
}

uint64_t head_ranks_tmp_bytes(uint64_t n_kmers) {
    size_t bytes = 0;
    cub::TransformInputIterator<uint32_t, U8ToU32, const uint8_t*> it(nullptr, U8ToU32{});
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, it, (uint32_t*)nullptr, n_kmers);
    size_t bytes2 = 0;
    MmerCount op{nullptr, 1};
    cub::CountingInputIterator<uint64_t> cnt(0);
    cub::TransformInputIterator<uint64_t, MmerCount, cub::CountingInputIterator<uint64_t>> it2(cnt, op);
    cub::DeviceScan::ExclusiveScan(nullptr, bytes2, it2, (uint64_t*)nullptr, AddBase{0}, uint64_t(0), n_kmers);
    return (bytes > bytes2 ? bytes : bytes2) + 256;
}

void launch_head_ranks(const uint8_t* head, uint64_t n_kmers, uint32_t* rank, void* d_tmp,
                       uint64_t tmp_bytes, cudaStream_t stream) {
    if (n_kmers) {
        cub::TransformInputIterator<uint32_t, U8ToU32, const uint8_t*> it(head, U8ToU32{});
        size_t bytes = tmp_bytes;
        cub::DeviceScan::ExclusiveSum(d_tmp, bytes, it, rank, n_kmers, stream);
    }
    k_finish_ranks<<<1, 1, 0, stream>>>(head, n_kmers, rank);
}

void launch_scan_emit(ScanBatch const& b, const uint8_t* head, const uint8_t* pos,
                      const uint32_t* rank, uint8_t* records, uint32_t* start_pos, cudaStream_t stream) {
    if (!b.n_kmers) return;
    k_scan_emit<<<grid_for((b.n_kmers + 3) / 4), 256, 0, stream>>>(b, head, pos, rank, records, start_pos);
}

// every byte of the batch looked at once: contigs too short for a k-mer never reach the scan kernels, but an invalid
// byte in them still matters to the m-mer ordinals (include/minimizer.hpp:45-49 counts valid runs only)
__global__ void k_flag_invalid_bytes(const char* bases, uint64_t first, uint64_t span, const uint64_t* offsets,
                                     uint64_t n_contigs, uint8_t* dirty) {
    for (uint64_t p = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < span; p += uint64_t(gridDim.x) * blockDim.x) {
        if (nt4(uint8_t(bases[first + p])) < 4) continue;
        const uint64_t at = first + p;
        uint64_t lo = 0, hi = n_contigs;  // offsets[lo] <= at < offsets[hi]
        while (hi - lo > 1) {
            const uint64_t mid = (lo + hi) >> 1;
            if (__ldg(offsets + mid) <= at) lo = mid; else hi = mid;
        }
        dirty[lo] = 1;
    }
}
void launch_flag_invalid_bytes(const char* bases, uint64_t first, uint64_t span, const uint64_t* offsets, uint64_t n_contigs,
                               uint8_t* dirty, cudaStream_t stream) {
    if (!span || !n_contigs) return;
    k_flag_invalid_bytes<<<grid_for(span), 256, 0, stream>>>(bases, first, span, offsets, n_contigs, dirty);
}

void launch_colliding_mark(const uint8_t* records, uint64_t n_records, const uint64_t* ids,
                           uint64_t n_ids, uint32_t* take, cudaStream_t stream) {
    if (!n_records) return;
    k_colliding_mark<<<grid_for(n_records), 256, 0, stream>>>(records, n_records, ids, n_ids, take);
}

namespace {
struct U32ToU64 {
    __host__ __device__ uint64_t operator()(uint32_t v) const { return v; }
};
}  // namespace

uint64_t exclusive_u32_tmp_bytes(uint64_t n) {
    size_t bytes = 0;
    cub::TransformInputIterator<uint64_t, U32ToU64, const uint32_t*> it(nullptr, U32ToU64{});
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, it, (uint64_t*)nullptr, n);
    return bytes + 256;
}

namespace {
__global__ void k_finish_u32(const uint32_t* in, uint64_t n, uint64_t* out) {
    out[n] = n ? out[n - 1] + in[n - 1] : 0;
}
}  // namespace

void launch_exclusive_u32(const uint32_t* in, uint64_t n, uint64_t* out, void* d_tmp,
                          uint64_t tmp_bytes, cudaStream_t stream) {
    if (n) {
        cub::TransformInputIterator<uint64_t, U32ToU64, const uint32_t*> it(in, U32ToU64{});
        size_t bytes = tmp_bytes;
        cub::DeviceScan::ExclusiveSum(d_tmp, bytes, it, out, n, stream);
    }
    k_finish_u32<<<1, 1, 0, stream>>>(in, n, out);
}

void launch_colliding_emit(ScanBatch const& b, uint64_t n_records, const uint32_t* start_pos,
                           const uint32_t* take, const uint64_t* out_off, int kmer_bits,
                           uint8_t* kmers, cudaStream_t stream) {
    if (!n_records) return;
    k_colliding_emit<<<grid_for(n_records), 256, 0, stream>>>(b, n_records, start_pos, take, out_off, kmer_bits, kmers);
}

}  // namespace lphb
