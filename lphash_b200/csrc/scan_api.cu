// C ABI of the handle-less build side (include/lphash_b200.h): the super-k-mer scan, classify and colliding k-mers,
// and the batch entry points of build sessions, which run that scan first.  Their device workspace is kept per device.
#include <cuda_runtime.h>

#include <algorithm>
#include <mutex>
#include <stdexcept>

#include "../../include/lphash_b200.h"
#include "api_internal.h"
#include "build_session.h"
#include "query_kernels.cuh"
#include "scan_kernels.cuh"

using namespace lphb;

namespace {

// Device workspace of the build-side scan, kept per device between calls.
struct ScanSession {
    DevBuf bases, offsets, code_off, id_base, dirty, head, pos, rank, records, start_pos, tmp, status, tile_ws;
    DevBuf r_starts, r_flag, r_voff, r_vstart, r_tmp, r_cnt, r_poff, r_pid;  // contigs with non-ACGT bytes: runs, pieces
    Stream s;
    ScanBatch b{};
    uint64_t n_records = 0, n_kmers = 0, tmp_bytes = 0;
    Event ev0, ev1;  // bracket the record-producing kernels of the last scan
    double kernel_ms = 0;
};

// The scan entry points have no handle: their device workspace (a few bytes per base) is kept per
// device between calls, so that a caller streaming batches does not pay cudaMalloc / cudaFree
// (both synchronizing) on every batch.  One mutex PER DEVICE: scans on different GPUs driven from
// different host threads run concurrently, scans on one GPU take turns; lphb_scan_release frees.
struct ClassifySession;
struct DeviceSessions {
    std::mutex mu;
    ScanSession* scan = nullptr;
    ClassifySession* classify = nullptr;
};
DeviceSessions g_dev[64];
DeviceSessions& device_sessions(int device) {
    if (device < 0 || device >= 64) throw std::invalid_argument("device index out of range");
    return g_dev[device];
}
ScanSession& scan_session(int device) {
    DeviceSessions& d = device_sessions(device);
    if (!d.scan) d.scan = new ScanSession();
    return *d.scan;
}

// Checks a scan batch (host offsets) and counts its k-mers and m-mers; the session starts on it.
ContigCounts begin_scan(ScanSession& S, uint32_t k, uint32_t m, const uint64_t* offsets, uint64_t n_contigs) {
    if (const char* e = scan_km_error(k, m)) throw std::invalid_argument(e);
    const ContigCounts n = contig_layout(offsets, n_contigs, k, m);
    if (n.kmers >= (1ull << 32) || (n_contigs && offsets[n_contigs] - offsets[0] >= (1ull << 32)))
        throw std::invalid_argument("batch holds >= 2^32 k-mers or bases: split it");
    S.n_kmers = n.kmers;
    S.n_records = 0;
    S.s.create();
    return n;
}

// The scan of one batch whose bases and offsets are ALREADY on the device (d_bases indexed by the
// offsets, i.e. d_bases + offsets[0] is the first base): leaves the records (scan order) and the
// stream position of every record's first k-mer in the session, returns after the device finished.
// Instantiated (k, m): one fused kernel (query_tiled.cu, kScan form); others: the generic passes.
// One pass of the scan kernels over a partition of the stream into contigs.  d_bases is indexed by the offsets;
// n_kmers = k-mers of the partition; d_id_base = m-mer ordinal of every contig's first m-mer, or null (then
// mm_count_in + the m-mers of the contigs before it).  *n_dirty = contigs with non-ACGT bytes (their records are
// meaningless; with `pieces` the partition was cut so that such contigs hold no k-mer at all).
int scan_pass(ScanSession& S, uint32_t k, uint32_t m, uint64_t seed, const char* d_bases, const uint64_t* d_offsets,
              uint64_t n_contigs, uint64_t first, uint64_t span, uint64_t n_kmers, uint64_t n_kmers_cap,
              const uint64_t* d_id_base, uint64_t mm_count_in, bool pieces, uint64_t* n_dirty) {
    cudaStream_t s = S.s;
    S.code_off.reserve((n_contigs + 1) * 8);
    S.id_base.reserve((n_contigs + 1) * 8);
    S.dirty.reserve(n_contigs + 8);
    S.status.reserve(64);
    S.records.reserve(n_kmers_cap * 18 + 64);       // capacity: one record per k-mer (low-complexity worst case)
    S.start_pos.reserve((n_kmers_cap + 2) * 4);
    const bool tiled = scan_tiled_available(k, m);
    uint64_t t1 = tiled ? 0 : head_ranks_tmp_bytes(n_kmers_cap > n_contigs ? n_kmers_cap : n_contigs);
    uint64_t t2 = code_offsets_tmp_bytes(n_contigs);
    uint64_t t3 = head_ranks_tmp_bytes(n_contigs);  // the m-mer ordinal scan over contigs
    S.tmp_bytes = std::max(std::max(t1, t2), t3);
    S.tmp.reserve(S.tmp_bytes);
    if (!tiled) {
        S.head.reserve(n_kmers_cap + 8);
        S.pos.reserve(n_kmers_cap + 8);
        S.rank.reserve((n_kmers_cap + 2) * 4);
    }
    S.tile_ws.reserve(query_tiled_ws_bytes(span));
    S.ev0.create(cudaEventDefault);
    S.ev1.create(cudaEventDefault);
    CK(cudaMemsetAsync(S.dirty.p, 0, n_contigs + 8, s));
    auto* st = S.status.as<unsigned long long>();
    CK(cudaMemsetAsync(st, 0, 64, s));
    launch_code_offsets(d_offsets, n_contigs, k, S.code_off.as<uint64_t>(), st, S.tmp.p, S.tmp_bytes, s);
    if (!d_id_base) {
        launch_id_base(d_offsets, n_contigs, m, mm_count_in, S.id_base.as<uint64_t>(), S.tmp.p, S.tmp_bytes, s);
        d_id_base = S.id_base.as<uint64_t>();
    }
    if (pieces) {  // the partition's k-mer count is only known on the device
        CK(cudaMemcpyAsync(&n_kmers, S.code_off.as<uint64_t>() + n_contigs, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    ScanBatch& b = S.b;
    b.bases = d_bases;
    b.offsets = d_offsets;
    b.code_off = S.code_off.as<uint64_t>();
    b.id_base = d_id_base;
    b.n_contigs = n_contigs;
    b.first_base = first;
    b.end_base = first + span;
    b.n_kmers = n_kmers;
    b.k = k;
    b.m = m;
    b.seed = seed;
    b.dirty = S.dirty.as<uint8_t>();
    S.n_records = 0;
    *n_dirty = 0;
    // the generic kernels (and a batch without any k-mer) never see the bytes of contigs shorter than k: look at them here
    if (!pieces && (!tiled || n_kmers == 0)) launch_flag_invalid_bytes(d_bases, first, span, d_offsets, n_contigs, b.dirty, s);
    if (n_kmers == 0) {
        if (!pieces) {
            launch_count_dirty(b.dirty, n_contigs, st, s);
            unsigned long long h_st[2] = {0, 0};
            CK(cudaMemcpyAsync(h_st, st, sizeof(h_st), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            *n_dirty = h_st[1];
        }
        return LPHB_OK;
    }
    CK(cudaEventRecord(S.ev0, s));
    unsigned long long h_nrec = 0;
    if (tiled) {
        DevBatch qb{};
        qb.bases = b.bases;
        qb.offsets = b.offsets;
        qb.code_off = b.code_off;
        qb.n_contigs = n_contigs;
        qb.first_base = b.first_base;
        qb.end_base = b.end_base;
        qb.dirty = b.dirty;
        qb.status = st;
        qb.tile_ws = S.tile_ws.p;
        qb.tile_ws_bytes = S.tile_ws.cap;
        if (!launch_scan_records_tiled(k, m, seed, qb, b.id_base, S.records.as<uint8_t>(), S.start_pos.as<uint32_t>(),
                                       st + 2, s))
            return fail(LPHB_E_ARG, "scan: batch too large for one launch");
        CK(cudaEventRecord(S.ev1, s));
        launch_count_dirty(b.dirty, n_contigs, st, s);
    } else {
        CK(cudaMemsetAsync(S.head.p, 0, n_kmers + 8, s));
        launch_scan_heads(b, S.head.as<uint8_t>(), S.pos.as<uint8_t>(), s);
        launch_count_dirty(b.dirty, n_contigs, st, s);
        launch_head_ranks(S.head.as<uint8_t>(), n_kmers, S.rank.as<uint32_t>(), S.tmp.p, S.tmp_bytes, s);
    }
    unsigned long long h_st[3] = {0, 0, 0};
    uint32_t n_rec32 = 0;
    CK(cudaMemcpyAsync(h_st, st, sizeof(h_st), cudaMemcpyDeviceToHost, s));
    if (!tiled) CK(cudaMemcpyAsync(&n_rec32, S.rank.as<uint32_t>() + n_kmers, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    *n_dirty = h_st[1];
    if (h_st[1] != 0 && !pieces) return LPHB_OK;  // the caller cuts the batch at the invalid bytes and comes back
    h_nrec = tiled ? h_st[2] : n_rec32;
    S.n_records = h_nrec;
    if (!tiled) {
        launch_scan_emit(b, S.head.as<uint8_t>(), S.pos.as<uint8_t>(), S.rank.as<uint32_t>(),
                         S.records.as<uint8_t>(), S.start_pos.as<uint32_t>(), s);
        CK(cudaEventRecord(S.ev1, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
    }
    float ms = 0;
    if (cudaEventElapsedTime(&ms, S.ev0, S.ev1) == cudaSuccess) S.kernel_ms = ms; else cudaGetLastError();
    return LPHB_OK;
}

int run_scan_device(ScanSession& S, uint32_t k, uint32_t m, uint64_t seed, const char* d_bases,
                    const uint64_t* d_offsets, const uint64_t* offsets, uint64_t n_contigs, uint64_t mm_count_in,
                    uint64_t* mm_count_out) {
    cudaStream_t s = S.s;
    const uint64_t first = offsets[0], span = offsets[n_contigs] - first;
    const uint64_t n_kmers = S.n_kmers;
    uint64_t n_dirty = 0;
    int rc = scan_pass(S, k, m, seed, d_bases, d_offsets, n_contigs, first, span, n_kmers, n_kmers, nullptr, mm_count_in,
                       false, &n_dirty);
    if (rc != LPHB_OK || n_dirty == 0) return rc;
    // Contigs with non-ACGT bytes (include/minimizer.hpp:138-151): every maximal valid run is scanned as a contig
    // of its own (quirk_kernels.cu, build side); k-mer and m-mer totals come from the runs.
    if (k < 2) return fail(LPHB_E_ARG, "build input with non-ACGT bytes needs k >= 2");
    const char* rel = d_bases + first;  // positions below are relative to the batch
    S.r_starts.reserve((n_contigs + 2) * 8);
    S.r_flag.reserve(span + 8);
    S.r_voff.reserve((span + 2) * 8);
    S.r_vstart.reserve((n_contigs + 2) * 4);
    const uint64_t qt = quirk_tmp_bytes(span + 2);
    S.r_tmp.reserve(qt);
    auto* st = S.status.as<unsigned long long>();
    launch_shift_starts(d_offsets, n_contigs, first, S.r_starts.as<uint64_t>(), s);
    launch_find_runs(rel, span, S.r_starts.as<uint64_t>(), n_contigs, S.r_flag.as<uint8_t>(), S.r_voff.as<uint64_t>(), st + 4,
                     S.r_vstart.as<uint32_t>(), S.r_tmp.p, qt, s);
    unsigned long long n_v = 0;
    CK(cudaMemcpyAsync(&n_v, st + 4, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    S.r_cnt.reserve(3 * (n_v + 1) * 8);
    uint64_t *d_pieces = S.r_cnt.as<uint64_t>(), *d_ids = d_pieces + (n_v + 1), *d_kmers = d_ids + (n_v + 1);
    launch_build_run_counts(rel, S.r_voff.as<uint64_t>(), st + 4, S.r_vstart.as<uint32_t>(), n_contigs, n_v, k, m, d_pieces,
                            d_ids, d_kmers, S.r_tmp.p, qt, s);
    uint64_t totals[3] = {0, 0, 0};
    CK(cudaMemcpyAsync(&totals[0], d_pieces + n_v, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&totals[1], d_ids + n_v, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&totals[2], d_kmers + n_v, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const uint64_t n_pieces = totals[0];
    S.r_poff.reserve((n_pieces + 2) * 8);
    S.r_pid.reserve((n_pieces + 2) * 8);
    launch_build_pieces(S.r_voff.as<uint64_t>(), st + 4, n_v, k, d_pieces, d_ids, mm_count_in, span, S.r_poff.as<uint64_t>(),
                        S.r_pid.as<uint64_t>(), s);
    *mm_count_out = mm_count_in + totals[1];
    rc = scan_pass(S, k, m, seed, rel, S.r_poff.as<uint64_t>(), n_pieces, 0, span, 0, n_kmers, S.r_pid.as<uint64_t>(),
                   mm_count_in, true, &n_dirty);
    S.n_kmers = totals[2];  // what from_string returns: the swallowed k-mers of exactly-k runs included
    return rc;
}

// Validates a host batch, moves it to the device and scans it.
int run_scan(ScanSession& S, uint32_t k, uint32_t m, uint64_t seed, const char* bases,
             const uint64_t* offsets, uint64_t n_contigs, uint64_t mm_count_in,
             uint64_t* mm_count_out) {
    const ContigCounts n = begin_scan(S, k, m, offsets, n_contigs);
    *mm_count_out = mm_count_in + n.mmers;
    if (n_contigs == 0 || n.mmers == 0) return LPHB_OK;  // (without a k-mer there is no record, but an invalid byte
    if (!bases) return fail(LPHB_E_ARG, "bases is null");  //  still changes the m-mer ordinals: the device decides)
    cudaStream_t s = S.s;
    const uint64_t first = offsets[0], span = offsets[n_contigs] - first;
    S.bases.reserve(span + 64);
    S.offsets.reserve((n_contigs + 1) * 8);
    CK(cudaMemcpyAsync(S.bases.p, bases + first, span, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(S.offsets.p, offsets, (n_contigs + 1) * 8, cudaMemcpyHostToDevice, s));
    return run_scan_device(S, k, m, seed, S.bases.as<char>() - first, S.offsets.as<uint64_t>(), offsets, n_contigs,
                           mm_count_in, mm_count_out);
}

struct ClassifySession {
    DevBuf rec;        // lphb_classify's records
    Classify cls;
    DevBuf trip, ids;  // the results on their way to the host
};
ClassifySession& classify_session(int device) {
    DeviceSessions& d = device_sessions(device);
    if (!d.classify) d.classify = new ClassifySession();
    return *d.classify;
}

// Sort by minimizer + classify of n records that are already on the device (stream s); results to host.
int classify_device(const uint8_t* d_rec, uint64_t n, void* triplets, uint64_t triplets_capacity,
                    uint64_t* n_triplets, uint64_t* ids, uint64_t ids_capacity, uint64_t* n_ids,
                    int key_bits, cudaStream_t s) {
    // workspace kept per device between calls (freed by lphb_scan_release); callers hold the device's mutex
    int dev = 0;
    CK(cudaGetDevice(&dev));
    ClassifySession& cs = classify_session(dev);
    Classify& C = cs.cls;
    C.group(d_rec, n, key_bits, s);
    *n_triplets = C.groups;
    *n_ids = C.members;
    if (C.groups > triplets_capacity) return fail(LPHB_E_CAPACITY, "triplets buffer too small");
    if (C.members > ids_capacity) return fail(LPHB_E_CAPACITY, "ids buffer too small");
    if (!triplets || (C.members && !ids)) return fail(LPHB_E_ARG, "null output buffer");
    cs.trip.reserve(C.groups * 10 + 64);
    cs.ids.reserve(C.members * 8 + 64);
    C.emit(d_rec, n, cs.trip.as<uint8_t>(), cs.ids.as<uint64_t>(), s);
    CK(cudaMemcpyAsync(triplets, cs.trip.p, C.groups * 10, cudaMemcpyDeviceToHost, s));
    if (C.members) CK(cudaMemcpyAsync(ids, cs.ids.p, C.members * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    return LPHB_OK;
}

// Adds the batch the scan session holds (records still on the device) to a build session.
int build_take_scan(lphb_build* b, ScanSession& S, uint64_t n_contigs, uint64_t mm_out) {
    build_add_batch(b, S.records.as<uint8_t>(), S.n_records, S.s);
    lphb_build_report& t = b->totals;
    t.batches += 1;
    t.contigs += n_contigs;
    t.kmers += S.n_kmers;
    t.records += S.n_records;
    t.mm_count = mm_out;
    return LPHB_OK;
}

}  // namespace

extern "C" {

int lphb_scan_superkmers(int device, uint32_t k, uint32_t m, uint64_t seed, const char* bases,
                         const uint64_t* offsets, uint64_t n_contigs, uint64_t* mm_count,
                         void* records, uint64_t records_capacity, uint64_t* n_records,
                         uint64_t* n_kmers) {
    if (!offsets || !mm_count || !n_records || !n_kmers) return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(device);
        std::lock_guard<std::mutex> lock(device_sessions(device).mu);
        ScanSession& S = scan_session(device);
        uint64_t mm_out = *mm_count;
        int rc = run_scan(S, k, m, seed, bases, offsets, n_contigs, *mm_count, &mm_out);
        if (rc != LPHB_OK) return rc;
        *n_kmers = S.n_kmers;
        *n_records = S.n_records;
        if (S.n_records > records_capacity) return fail(LPHB_E_CAPACITY, "records buffer too small");
        if (S.n_records) {
            if (!records) return fail(LPHB_E_ARG, "records is null");
            CK(cudaMemcpyAsync(records, S.records.p, S.n_records * 18, cudaMemcpyDeviceToHost, S.s));
        }
        CK(cudaStreamSynchronize(S.s));
        *mm_count = mm_out;
        return LPHB_OK;
    });
}

int lphb_scan_superkmers_device(int device, uint32_t k, uint32_t m, uint64_t seed, const char* d_bases,
                                const uint64_t* d_offsets, const uint64_t* h_offsets, uint64_t n_contigs,
                                uint64_t* mm_count, const void** d_records, uint64_t* n_records, uint64_t* n_kmers,
                                double* kernel_ms) {
    if (!h_offsets || !d_offsets || !mm_count || !d_records || !n_records || !n_kmers)
        return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(device);
        std::lock_guard<std::mutex> lock(device_sessions(device).mu);
        ScanSession& S = scan_session(device);
        const ContigCounts n = begin_scan(S, k, m, h_offsets, n_contigs);
        *n_kmers = n.kmers;
        *n_records = 0;
        *d_records = nullptr;
        if (kernel_ms) *kernel_ms = 0;
        uint64_t mm_out = *mm_count + n.mmers;
        if (n_contigs && n.mmers) {
            if (!d_bases) return fail(LPHB_E_ARG, "d_bases is null");
            CK(cudaDeviceSynchronize());  // the caller's buffers may still be written on other streams
            int rc = run_scan_device(S, k, m, seed, d_bases, d_offsets, h_offsets, n_contigs, *mm_count, &mm_out);
            if (rc != LPHB_OK) return rc;
            *d_records = S.records.p;
            *n_records = S.n_records;
            *n_kmers = S.n_kmers;  // (differs from the count above when contigs hold non-ACGT bytes)
            if (kernel_ms) *kernel_ms = S.kernel_ms;
        }
        *mm_count = mm_out;
        return LPHB_OK;
    });
}

int lphb_scan_release(int device) {
    return guarded([&]() -> int {
        if (device < 0 || device >= 64) return LPHB_OK;
        DeviceSessions& d = device_sessions(device);
        std::lock_guard<std::mutex> lock(d.mu);
        if (!d.scan && !d.classify) return LPHB_OK;
        DeviceGuard g(device);
        delete d.scan;
        d.scan = nullptr;
        delete d.classify;
        d.classify = nullptr;
        return LPHB_OK;
    });
}

int lphb_classify(int device, const void* records, uint64_t n_records, void* triplets,
                  uint64_t triplets_capacity, uint64_t* n_triplets, uint64_t* ids, uint64_t ids_capacity,
                  uint64_t* n_ids) {
    if (!n_triplets || !n_ids || (n_records && !records)) return fail(LPHB_E_ARG, "null argument");
    if (n_records >= (1ull << 32)) return fail(LPHB_E_ARG, "batch holds >= 2^32 records: split it");
    return guarded([&]() -> int {
        DeviceGuard g(device);
        *n_triplets = 0;
        *n_ids = 0;
        if (n_records == 0) return LPHB_OK;
        std::lock_guard<std::mutex> lock(device_sessions(device).mu);
        DevBuf& rec = classify_session(device).rec;
        Stream s;
        s.create();
        rec.reserve(n_records * 18 + 64);
        CK(cudaMemcpyAsync(rec.p, records, n_records * 18, cudaMemcpyHostToDevice, s));
        return classify_device(rec.as<uint8_t>(), n_records, triplets, triplets_capacity, n_triplets, ids,
                               ids_capacity, n_ids, 64, s);  // m unknown here: all key bits
    });
}

int lphb_scan_classify(int device, uint32_t k, uint32_t m, uint64_t seed, const char* bases,
                       const uint64_t* offsets, uint64_t n_contigs, uint64_t* mm_count, void* triplets,
                       uint64_t triplets_capacity, uint64_t* n_triplets, uint64_t* ids,
                       uint64_t ids_capacity, uint64_t* n_ids, uint64_t* n_kmers) {
    if (!offsets || !mm_count || !n_triplets || !n_ids || !n_kmers) return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(device);
        std::lock_guard<std::mutex> lock(device_sessions(device).mu);
        ScanSession& S = scan_session(device);
        uint64_t mm_out = *mm_count;
        int rc = run_scan(S, k, m, seed, bases, offsets, n_contigs, *mm_count, &mm_out);
        if (rc != LPHB_OK) return rc;
        *n_kmers = S.n_kmers;
        *n_triplets = 0;
        *n_ids = 0;
        if (S.n_records) {  // the records never leave the device
            rc = classify_device(S.records.as<uint8_t>(), S.n_records, triplets, triplets_capacity, n_triplets,
                                 ids, ids_capacity, n_ids, int(2 * m), S.s);  // a minimizer is 2m bits
            if (rc != LPHB_OK) return rc;
        }
        *mm_count = mm_out;
        return LPHB_OK;
    });
}

int lphb_build_batch(lphb_build* b, const char* bases, const uint64_t* offsets, uint64_t n_contigs) {
    if (!b || !offsets) return fail(LPHB_E_ARG, "null argument");
    if (!b->dev) return fail(LPHB_E_ARG, "the build session has ended");
    return guarded_nomem([&]() -> int {
        DeviceGuard g(b->device);
        std::lock_guard<std::mutex> lock(device_sessions(b->device).mu);
        ScanSession& S = scan_session(b->device);
        uint64_t mm_out = b->totals.mm_count;
        int rc = run_scan(S, b->k, b->m, b->seed, bases, offsets, n_contigs, b->totals.mm_count, &mm_out);
        if (rc != LPHB_OK) return rc;
        return build_take_scan(b, S, n_contigs, mm_out);
    });
}

int lphb_build_batch_device(lphb_build* b, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                            uint64_t n_contigs, void* stream) {
    if (!b || !d_offsets || !h_offsets) return fail(LPHB_E_ARG, "null argument");
    if (!b->dev) return fail(LPHB_E_ARG, "the build session has ended");
    return guarded_nomem([&]() -> int {
        DeviceGuard g(b->device);
        std::lock_guard<std::mutex> lock(device_sessions(b->device).mu);
        ScanSession& S = scan_session(b->device);
        const ContigCounts n = begin_scan(S, b->k, b->m, h_offsets, n_contigs);
        uint64_t mm_out = b->totals.mm_count + n.mmers;
        if (n_contigs && n.mmers) {
            if (!d_bases) return fail(LPHB_E_ARG, "d_bases is null");
            CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));  // the caller wrote its buffers on `stream`
            int rc = run_scan_device(S, b->k, b->m, b->seed, d_bases, d_offsets, h_offsets, n_contigs, b->totals.mm_count,
                                     &mm_out);
            if (rc != LPHB_OK) return rc;
        }
        return build_take_scan(b, S, n_contigs, mm_out);
    });
}

int lphb_colliding_kmers(int device, uint32_t k, uint32_t m, uint64_t seed, const char* bases,
                         const uint64_t* offsets, uint64_t n_contigs, uint64_t* mm_count,
                         const uint64_t* ids, uint64_t n_ids, int kmer_bits, void* kmers,
                         uint64_t kmers_capacity, uint64_t* n_kmers) {
    if (!offsets || !mm_count || !n_kmers || (n_ids && !ids)) return fail(LPHB_E_ARG, "null argument");
    if (kmer_bits != 64 && kmer_bits != 128) return fail(LPHB_E_ARG, "kmer_bits must be 64 or 128");
    if (k > uint32_t(kmer_bits / 2 - 1)) return fail(LPHB_E_ARG, "k too large for this kmer_t");
    return guarded([&]() -> int {
        DeviceGuard g(device);
        std::lock_guard<std::mutex> lock(device_sessions(device).mu);
        ScanSession& S = scan_session(device);
        uint64_t mm_out = *mm_count;
        int rc = run_scan(S, k, m, seed, bases, offsets, n_contigs, *mm_count, &mm_out);
        if (rc != LPHB_OK) return rc;
        *n_kmers = 0;
        if (S.n_records == 0 || n_ids == 0) {
            *mm_count = mm_out;
            return LPHB_OK;
        }
        DevBuf d_ids, take, out_off, out;
        cudaStream_t s = S.s;
        d_ids.reserve(n_ids * 8);
        take.reserve((S.n_records + 1) * 4);
        out_off.reserve((S.n_records + 1) * 8);
        CK(cudaMemcpyAsync(d_ids.p, ids, n_ids * 8, cudaMemcpyHostToDevice, s));
        launch_colliding_mark(S.records.as<uint8_t>(), S.n_records, d_ids.as<uint64_t>(), n_ids,
                              take.as<uint32_t>(), s);
        uint64_t tb = exclusive_u32_tmp_bytes(S.n_records);
        S.tmp.reserve(tb);
        launch_exclusive_u32(take.as<uint32_t>(), S.n_records, out_off.as<uint64_t>(), S.tmp.p, tb, s);
        uint64_t total = 0;
        CK(cudaMemcpyAsync(&total, out_off.as<uint64_t>() + S.n_records, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        *n_kmers = total;
        if (total > kmers_capacity) return fail(LPHB_E_CAPACITY, "kmers buffer too small");
        if (total) {
            if (!kmers) return fail(LPHB_E_ARG, "kmers is null");
            const uint64_t bytes = total * uint64_t(kmer_bits / 8);
            out.reserve(bytes + 64);
            launch_colliding_emit(S.b, S.n_records, S.start_pos.as<uint32_t>(), take.as<uint32_t>(),
                                  out_off.as<uint64_t>(), kmer_bits, out.as<uint8_t>(), s);
            CK(cudaMemcpyAsync(kmers, out.p, bytes, cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            CK(cudaGetLastError());
        }
        *mm_count = mm_out;
        return LPHB_OK;
    });
}

}  // extern "C"
