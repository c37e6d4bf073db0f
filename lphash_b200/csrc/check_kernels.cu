// The self-check of build-p --check (check, include/mphf_utils.hpp:51-100) over a batch of the index's contigs, in
// one pass over every window of k bytes: the non-streaming code of the window (a non-ACGT byte counts as 'A',
// mphf_utils.hpp:108), compared with the streaming code of the same window when its contig is clean
// (check_streaming_correctness), and marked in a bitmap of nkmers bits (check_collisions); k_check_missing then
// counts the codes of [0, nkmers) never marked (check_perfection).  The per-window evaluation is the one of
// k_query_generic and k_lookup_kmers: kmer_minimizer, probe_minimizer, probe_hval / fallback_order.
#include "check_kernels.cuh"
#include "device_mphf.cuh"

namespace lphb {

namespace {

constexpr int kCheckThreads = 256;
constexpr unsigned kFull = 0xffffffffu;

// contig holding k-mer ordinal j: code_off[c] <= j < code_off[c + 1] (empty contigs have equal entries)
__device__ __forceinline__ uint64_t contig_of_kmer(const uint64_t* code_off, uint64_t n, uint64_t j) {
    uint64_t lo = 0, hi = n;  // invariant: code_off[lo] <= j < code_off[hi]
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (__ldg(code_off + mid) <= j) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ uint64_t warp_sum(uint64_t v) {
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ uint64_t warp_min(uint64_t v) {
    for (int o = 16; o; o >>= 1) v = min(v, __shfl_down_sync(kFull, v, o));
    return v;
}

// Grid-stride over warp spans of 32 k-mer ordinals of [j0, j1) (warp-uniform, so that every lane reaches the warp
// intrinsics).  Consecutive k-mers of a super-k-mer get consecutive codes: a warp's in-range codes fall into few
// 32-bit words of the bitmap, one atomicOr per distinct word (__match_any_sync).  A hit is a duplicate when its bit
// was set in the word before that atomicOr, or when a lower lane holds the same code: every code hit h >= 1 times is
// flagged exactly h - 1 times, whatever the order of the atomics.  Counters stay in registers until the end.
template <int KmerWords>
__global__ void __launch_bounds__(kCheckThreads) k_check_windows(const __grid_constant__ DevImage f,
                                                                 const __grid_constant__ CheckBatch b) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
    const uint64_t n_warps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
    const uint32_t k = f.k;
    const uint64_t nkmers = f.nkmers;
    const unsigned lower = (1u << lane) - 1u;
    uint64_t kmers = 0, out_of_range = 0, dups = 0, mismatches = 0;
    uint64_t first_oor = ~uint64_t(0), first_mm = ~uint64_t(0), min_dup = ~uint64_t(0);
#pragma unroll 1
    for (uint64_t span = b.j0 + warp * 32; span < b.j1; span += n_warps * 32) {
        const uint64_t j = span + lane;
        bool in_range = false;
        uint64_t code = 0;
        if (j < b.j1) {
            const uint64_t c = contig_of_kmer(b.code_off, b.n_contigs, j);
            const uint64_t at = __ldg(b.offsets + c) + (j - __ldg(b.code_off + c));
            // forward k-mer, first base in the most significant bits; non-ACGT -> 'A' (nt4 gives 4, & 3 = 0)
            uint64_t lo = 0, hi = 0;
            for (uint32_t i = 0; i < k; ++i) {
                const uint32_t x = nt4(uint8_t(__ldg(b.bases + at + i))) & 3u;
                if (KmerWords == 2) hi = (hi << 2) | (lo >> 62);
                lo = (lo << 2) | x;
            }
            const Minimizer mz = kmer_minimizer(k, f.m, f.mm_seed, lo, hi);
            const Probe pr = probe_minimizer(f, mz.mmer);
            code = pr.slope == 0 ? pr.base + fallback_order(f, lo, hi) : probe_hval(pr, mz.pos);
            const uint64_t ordinal = b.ordinal_base + j;
            ++kmers;
            in_range = code < nkmers;
            if (!in_range) {
                ++out_of_range;
                first_oor = min(first_oor, ordinal);
            }
            if (b.stream_codes && !b.dirty[c] && __ldcs(reinterpret_cast<const unsigned long long*>(b.stream_codes) + j) != code) {
                ++mismatches;
                first_mm = min(first_mm, ordinal);
            }
        }
        // lanes without an in-range code take keys no in-range code can equal (codes < nkmers < 2^64 - 32, which
        // lphb_check_begin enforces on the header's nkmers)
        const unsigned word_peers = __match_any_sync(kFull, in_range ? code >> 5 : ~uint64_t(lane));
        const unsigned code_peers = __match_any_sync(kFull, in_range ? code : ~uint64_t(lane));
        if (in_range) {
            const uint32_t bit = 1u << (code & 31);
            const uint32_t bits = __reduce_or_sync(word_peers, bit);
            const int leader = __ffs(word_peers) - 1;
            uint32_t old = 0;
            if (int(lane) == leader) old = atomicOr(b.bitmap + (code >> 5), bits);
            old = __shfl_sync(word_peers, old, leader);
            if ((old & bit) || (code_peers & lower)) {
                ++dups;
                min_dup = min(min_dup, code);
            }
        }
    }
    kmers = warp_sum(kmers);
    out_of_range = warp_sum(out_of_range);
    dups = warp_sum(dups);
    mismatches = warp_sum(mismatches);
    first_oor = warp_min(first_oor);
    first_mm = warp_min(first_mm);
    min_dup = warp_min(min_dup);
    if (lane == 0) {
        unsigned long long* cnt = b.counters;
        if (kmers) atomicAdd(cnt + kCheckKmers, kmers);
        if (out_of_range) {
            atomicAdd(cnt + kCheckOutOfRange, out_of_range);
            atomicMin(cnt + kCheckFirstOutOfRange, first_oor);
        }
        if (dups) {
            atomicAdd(cnt + kCheckDuplicates, dups);
            atomicMin(cnt + kCheckMinDuplicate, min_dup);
        }
        if (mismatches) {
            atomicAdd(cnt + kCheckMismatches, mismatches);
            atomicMin(cnt + kCheckFirstMismatch, first_mm);
        }
    }
}

// popcount of the bitmap's nkmers bits and the smallest code never hit
__global__ void __launch_bounds__(kCheckThreads) k_check_missing(const uint32_t* __restrict__ bitmap, uint64_t nkmers,
                                                                 unsigned long long* counters) {
    const uint64_t n_words = (nkmers + 31) / 32;
    const uint32_t last_mask = nkmers % 32 ? (1u << (nkmers % 32)) - 1u : ~0u;
    uint64_t hits = 0, first_missing = ~uint64_t(0);
    const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
    for (uint64_t w = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; w < n_words; w += stride) {
        const uint32_t valid = w + 1 == n_words ? last_mask : ~0u;
        const uint32_t word = __ldcs(bitmap + w) & valid;
        hits += __popc(word);
        const uint32_t miss = ~word & valid;
        if (miss) first_missing = min(first_missing, w * 32 + uint64_t(__ffs(miss) - 1));
    }
    hits = warp_sum(hits);
    first_missing = warp_min(first_missing);
    if ((threadIdx.x & 31) == 0) {
        if (hits) atomicAdd(counters + kCheckHits, hits);
        if (first_missing != ~uint64_t(0)) atomicMin(counters + kCheckMinMissing, first_missing);
    }
}

template <int KmerWords>
void launch_windows(DevImage const& img, CheckBatch const& b, cudaStream_t stream) {
    static unsigned resident = 0;  // blocks that fill the device
    if (!resident) {
        int dev = 0, sms = 0, per_sm = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_check_windows<KmerWords>, kCheckThreads, 0) !=
                cudaSuccess ||
            sms <= 0 || per_sm <= 0) {
            cudaGetLastError();
            sms = 148;
            per_sm = 4;
        }
        resident = unsigned(sms) * unsigned(per_sm);
    }
    uint64_t blocks = (b.j1 - b.j0 + kCheckThreads - 1) / kCheckThreads;
    if (blocks > resident) blocks = resident;
    k_check_windows<KmerWords><<<unsigned(blocks), kCheckThreads, 0, stream>>>(img, b);
}

}  // namespace

void launch_check_windows(DevImage const& img, CheckBatch const& b, cudaStream_t stream) {
    if (b.j1 <= b.j0) return;
    if (img.kmer_bits == 128) launch_windows<2>(img, b, stream);
    else launch_windows<1>(img, b, stream);
}

void launch_check_missing(const uint32_t* d_bitmap, uint64_t nkmers, unsigned long long* d_counters,
                          cudaStream_t stream) {
    if (!nkmers) return;
    uint64_t blocks = ((nkmers + 31) / 32 + kCheckThreads - 1) / kCheckThreads;
    if (blocks > 148ull * 8) blocks = 148ull * 8;
    k_check_missing<<<unsigned(blocks), kCheckThreads, 0, stream>>>(d_bitmap, nkmers, d_counters);
}

}  // namespace lphb
