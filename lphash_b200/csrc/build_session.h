// The state behind lphb_build (include/lphash_b200.h, build session): the classify of each batch reduced to one
// entry per distinct minimizer, and the merge of those summaries into the session's triplets and ids
// (build_session.cu).  The batch entry points live in scan_api.cu, next to the scan they run first.  Also the
// classify workspace, which lphb_classify and lphb_scan_classify use too.
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "api_internal.h"

namespace lphb {

// Workspace of minimizer::classify (classify_kernels.cu) over n records on the device.
struct Classify {
    DevBuf key, key2, idx, idx2, flags, gslot, cslot, counts, tmp, idu;
    uint64_t tmp_bytes = 0;           // what step 2 may use of tmp
    uint64_t groups = 0, members = 0;  // of step 1: groups (triplets), members of groups of several (ids)
    // Step 1 (sort by minimizer, group) on stream s, its counts read back; returns after the device finished.
    void group(const uint8_t* rec, uint64_t n, int key_bits, cudaStream_t s);
    // Step 2 on s: the groups' triplets; the members' ids unsorted in idu and, unless ids is null, sorted into ids.
    void emit(const uint8_t* rec, uint64_t n, uint8_t* triplets, uint64_t* ids, cudaStream_t s);
    uint64_t bytes() const;
};

// One batch after its classify: G entries sorted by minimizer, L local collision ids.
struct BatchSummary {
    DevBuf trip;  // G 10-byte triplets: {itself, p1, size}, {itself, 0, 0} for a minimizer seen several times in the batch
    DevBuf sid;   // G ids: the occurrence id of a minimizer seen once in the batch, UINT64_MAX otherwise
    DevBuf lids;  // L ascending ids of the occurrences of the batch's locally colliding minimizers
    uint64_t n_groups = 0, n_lids = 0;
};

// Everything the session holds on the device; dropped as a whole when the session closes.
struct BuildDevice {
    std::vector<BatchSummary> batches;
    Classify cls;                                                   // classify of one batch or one slice
    DevBuf rec, bounds, desc, marks, idw, nsel, res_trip, res_ids;  // the merge
    Stream s;                                                       // the merge's stream
    bool merged = false;
    uint64_t n_triplets = 0, n_ids = 0, colliding = 0;
    uint64_t bytes() const;
};

}  // namespace lphb

struct lphb_build {
    int device = 0;
    uint32_t k = 0, m = 0;
    uint64_t seed = 0;
    lphb_build_report totals{};  // batches, contigs, kmers, mm_count, records
    std::unique_ptr<lphb::BuildDevice> dev;  // null once the session is closed
};

namespace lphb {

// Classifies the n records of one scanned batch (device memory, ordered on stream s) and appends the batch's
// summary to the session.  Returns after the device finished; on an exception the session is unchanged.
void build_add_batch(lphb_build* b, const uint8_t* d_records, uint64_t n, cudaStream_t s);

// guarded() that reports a failed device allocation as LPHB_E_NOMEM with its size
template <class F>
int guarded_nomem(F&& body) {
    return guarded([&]() -> int {
        try {
            return body();
        } catch (DeviceOom const& e) {
            cudaGetLastError();
            return fail(LPHB_E_NOMEM, "cannot allocate " + std::to_string(e.bytes) + " bytes of device memory");
        }
    });
}

}  // namespace lphb
