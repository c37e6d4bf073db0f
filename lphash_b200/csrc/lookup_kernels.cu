// Lookup of packed k-mers (lphb_lookup_kmers): the code of every k-mer is what the reference's non-streaming
// branch (include/partitioned_mphf.hpp:185-195) returns for the window that encodes it.  Of its three steps the
// first, the integer k-mer (string_to_integer_no_reverse, include/mphf_utils.hpp:110-116), is the caller's input;
// the leftmost-minimum m-mer (compute_minimizer_triplet, mphf_utils.hpp:118-137) and mphf::query
// (src/partitioned_mphf.cpp:292-339) run here, over the same image reads as the query kernels.
#include "device_mphf.cuh"
#include "query_kernels.cuh"

namespace lphb {

namespace {

constexpr int kLookupThreads = 256;
// k-mers per thread in flight: the two dependent gathers of each (hashed pilot, then bucket word) overlap with
// those of the others instead of queueing up
constexpr int kLookupGroup = 4;

template <int KmerWords>
__device__ __forceinline__ void load_kmer(const uint64_t* kmers, uint64_t i, uint64_t& lo, uint64_t& hi) {
    if (KmerWords == 1) {
        lo = __ldcs(reinterpret_cast<const unsigned long long*>(kmers) + i);
        hi = 0;
    } else {
        const ulonglong2 v = __ldcs(reinterpret_cast<const ulonglong2*>(kmers) + i);
        lo = v.x;
        hi = v.y;
    }
}

// Persistent grid, grid-stride over warp spans of 32 * kLookupGroup k-mers: lane l takes k-mers span + 32 g + l,
// so that every load and store instruction of a warp covers one contiguous stretch.  The stages run across the
// group: 1. k-mer, minimizer, bucket of the minimizer PHF; 2. hashed-pilot gathers; 3. table slot and bucket-word
// gathers (the bucket table is indexed by the raw slot: no free-slot remap, device_image.h); 4. the code, through
// fallback_kmer_order for the k-mers of colliding minimizers.
// The w murmur hashes of the minimizer search dominate, not the gathers: one probe per distinct minimizer of a warp
// (__match_any_sync, the others' words by __shfl_sync) gained at most 0.6 % on contig-ordered input and lost up to
// 7 % on both orders at k=31 (DESIGN.md 4.9), so every lane probes for itself.
template <int KmerWords>
__global__ void __launch_bounds__(kLookupThreads) k_lookup_kmers(const __grid_constant__ DevImage f,
                                                                 const uint64_t* __restrict__ kmers, uint64_t n,
                                                                 uint64_t* __restrict__ codes) {
    constexpr int G = kLookupGroup;
    constexpr uint64_t kSpan = 32 * G;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
    const uint64_t n_warps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
    const uint32_t k = f.k, m = f.m;
    // the k-mer is the low 2k bits of its word(s): fallback_kmer_order hashes whole words
    const uint64_t lo_mask = 2 * k >= 64 ? ~uint64_t(0) : (uint64_t(1) << (2 * k)) - 1;
    const uint64_t hi_mask = 2 * k > 64 ? (uint64_t(1) << (2 * k - 64)) - 1 : 0;
    const DevPhf& P = f.minimizer_order;
    const uint64_t keep = l2_keep_policy();
    const bool wide = f.buckets.wide != 0;
#pragma unroll 1
    for (uint64_t span = warp * kSpan; span < n; span += n_warps * kSpan) {  // warp-uniform
        uint64_t lo[G], hi[G], h[G], e[G];
        uint32_t pos[G], slot[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const uint64_t i = span + 32 * g + lane;
            lo[g] = hi[g] = 0;
            if (i < n) load_kmer<KmerWords>(kmers, i, lo[g], hi[g]);
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
            lo[g] &= lo_mask;
            hi[g] &= hi_mask;
            const Minimizer mz = kmer_minimizer(k, m, f.mm_seed, lo[g], hi[g]);
            pos[g] = mz.pos;
            h[g] = murmur64(mz.mmer, P.seed);
            slot[g] = phf_bucket(P, h[g]);
        }
        uint64_t hp[G];
#pragma unroll
        for (int g = 0; g < G; ++g) hp[g] = ldg_keep(P.pilot_hash + slot[g], keep);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const uint32_t ts = phf_table_slot(P, h[g] ^ hp[g]);
            e[g] = wide ? ldg_keep(reinterpret_cast<const uint64_t*>(f.buckets.entries) + ts, keep)
                        : ldg_keep(reinterpret_cast<const uint32_t*>(f.buckets.entries) + ts, keep);
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const uint64_t i = span + 32 * g + lane;
            if (i < n) {
                const Probe pr = probe_decode(f, e[g]);
                const uint64_t code = pr.slope == 0 ? pr.base + fallback_order(f, lo[g], hi[g]) : probe_hval(pr, pos[g]);
                __stcs(reinterpret_cast<unsigned long long*>(codes) + i, code);
            }
        }
    }
}

template <int KmerWords>
void launch_lookup(DevImage const& img, const void* d_kmers, uint64_t n, uint64_t* d_codes, cudaStream_t stream) {
    static unsigned resident = 0;  // blocks that fill the device
    if (!resident) {
        int dev = 0, sms = 0, per_sm = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_lookup_kmers<KmerWords>, kLookupThreads,
                                                          0) != cudaSuccess ||
            sms <= 0 || per_sm <= 0) {
            cudaGetLastError();
            sms = 148;
            per_sm = 4;
        }
        resident = unsigned(sms) * unsigned(per_sm);
    }
    const uint64_t per_block = uint64_t(kLookupThreads) * kLookupGroup;
    uint64_t blocks = (n + per_block - 1) / per_block;
    if (blocks > resident) blocks = resident;
    k_lookup_kmers<KmerWords><<<unsigned(blocks), kLookupThreads, 0, stream>>>(
        img, static_cast<const uint64_t*>(d_kmers), n, d_codes);
}

}  // namespace

void launch_lookup_kmers(DevImage const& img, const void* d_kmers, uint64_t n, uint64_t* d_codes, cudaStream_t stream) {
    if (n == 0) return;
    if (img.kmer_bits == 128) launch_lookup<2>(img, d_kmers, n, d_codes, stream);
    else launch_lookup<1>(img, d_kmers, n, d_codes, stream);
}

}  // namespace lphb
