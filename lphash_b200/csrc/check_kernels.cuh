// Launchers of the index self-check (check_kernels.cu; C ABI lphb_check_*).  All pointers are device pointers; all
// launches are asynchronous on `stream`.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_image.h"

namespace lphb {

// Slots of the session's counter array (unsigned long long): sums first, then minima (reset to UINT64_MAX).
enum CheckCounter {
    kCheckKmers = 0,
    kCheckDirty = 1,  // launch_count_dirty adds to status[1]: pass the array itself as its status
    kCheckOutOfRange,
    kCheckDuplicates,
    kCheckMismatches,
    kCheckHits,  // distinct codes of [0, nkmers) hit (k_check_missing)
    kCheckFirstOutOfRange,
    kCheckFirstMismatch,
    kCheckMinDuplicate,
    kCheckMinMissing,
    kCheckCounters
};
constexpr int kCheckFirstMin = kCheckFirstOutOfRange;

// One batch (or one chunk of it) of the session.  bases / offsets as in DevBatch (bases indexed by the offsets);
// code_off: exclusive sum of max(0, L-k+1) over the n_contigs contigs, k-mer ordinals of the batch; the launch
// checks ordinals [j0, j1), the session ordinal of ordinal j being ordinal_base + j.  stream_codes: the streaming
// codes of the batch in the clean layout (indexed by the ordinal), or null (no comparison); dirty: per contig,
// nonzero if it holds a non-ACGT byte (its windows are not compared).
struct CheckBatch {
    const char* bases;
    const uint64_t* offsets;
    const uint64_t* code_off;
    uint64_t n_contigs;
    uint64_t j0, j1, ordinal_base;
    const uint64_t* stream_codes;
    const uint8_t* dirty;
    uint32_t* bitmap;  // nkmers bits, the session's
    unsigned long long* counters;
};

// k_check_windows<1 or 2 words per k-mer, by img.kmer_bits>: every window of the batch, see check_kernels.cu
void launch_check_windows(DevImage const& img, CheckBatch const& b, cudaStream_t stream);
// k_check_missing: counters[kCheckHits] += popcount of the bitmap's nkmers bits, counters[kCheckMinMissing] = smallest
// code of [0, nkmers) whose bit is clear
void launch_check_missing(const uint32_t* d_bitmap, uint64_t nkmers, unsigned long long* d_counters,
                          cudaStream_t stream);

}  // namespace lphb
