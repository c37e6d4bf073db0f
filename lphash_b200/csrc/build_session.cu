// Build session (include/lphash_b200.h, "build-p Parts 1 + 2 over a stream of batches"): minimizer::classify
// (src/minimizer.cpp:5-50) over a record stream that arrives batch by batch and never exists as a whole.
//
// Per batch (build_add_batch): the classify of classify_kernels.cu on the batch's records, kept as a summary - one
// entry per distinct minimizer of the batch, sorted by minimizer: its triplet ({itself, 0, 0} when it collides inside
// the batch) and, when it does not, the id of its one occurrence; plus the batch's local collision ids, ascending.
// The records themselves are not needed again.
//
// At the end (build_merge): the summaries are merged in minimizer-range slices.  A slice is a contiguous range of
// every batch's summary (binary search), halved until it holds at most LPHB_BUILD_SLICE entries, so that it fits the
// 32-bit indices of the classify kernels and a bounded workspace.  The slice's entries, packed as records
// {itself, origin, p1 | size}, go through the same classify: a minimizer seen once in the session keeps the triplet
// of its one entry (which already says whether it collided inside its batch), one seen in several batches becomes
// {itself, 0, 0}, and every entry of such a group that was a singleton in its batch is marked - its id collides
// globally.  Triplets come out slice by slice in ascending order.  Ids: batches hold disjoint, ascending ranges of
// m-mer ordinals (mm_count runs through the session), so the session's ids are, batch by batch, the sorted union of
// the batch's local collision ids and its marked singleton ids.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <cstdlib>
#include <utility>

#include "build_session.h"
#include "scan_kernels.cuh"

namespace lphb {

namespace {

constexpr uint64_t kSliceEntries = 1ull << 26;   // default slice: about 5 GB of classify workspace
constexpr uint64_t kLocalCollision = 1ull << 63;  // origin flag: the entry collided inside its batch (no id of its own)

struct BatchDesc {
    const uint8_t* trip;
    uint64_t n;
};

unsigned grid(uint64_t n) {
    uint64_t blocks = (n + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 148ull * 64) blocks = 148ull * 64;
    return unsigned(blocks);
}

// triplets and records are 2-byte aligned
__device__ __forceinline__ uint64_t u64_at(const uint8_t* p) {
    const uint16_t* q = reinterpret_cast<const uint16_t*>(p);
    return uint64_t(q[0]) | (uint64_t(q[1]) << 16) | (uint64_t(q[2]) << 32) | (uint64_t(q[3]) << 48);
}
__device__ __forceinline__ void put_u64(uint8_t* p, uint64_t v) {
    uint16_t* q = reinterpret_cast<uint16_t*>(p);
    q[0] = uint16_t(v); q[1] = uint16_t(v >> 16); q[2] = uint16_t(v >> 32); q[3] = uint16_t(v >> 48);
}

// bounds[2j] = first entry of batch j with minimizer >= lo, bounds[2j + 1] = first with minimizer >= hi
__global__ void k_slice_bounds(const BatchDesc* d, uint32_t nb, uint64_t lo, uint64_t hi, uint64_t* bounds) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * nb) return;
    const BatchDesc b = d[t >> 1];
    const uint64_t key = (t & 1) ? hi : lo;
    uint64_t a = 0, e = b.n;
    while (a < e) {
        const uint64_t mid = a + (e - a) / 2;
        if (u64_at(b.trip + 10 * mid) < key) a = mid + 1;
        else e = mid;
    }
    bounds[t] = a;
}

// n summary entries -> 18-byte records {itself, origin, p1 | size}; origin = the entry's index in the session
__global__ void k_pack_slice(const uint8_t* trip, const uint64_t* sid, uint64_t n, uint64_t origin0, uint8_t* rec) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint8_t* t = trip + 10 * i;
        uint8_t* r = rec + 18 * i;
        put_u64(r, u64_at(t));
        put_u64(r + 8, (origin0 + i) | (sid[i] == ~0ull ? kLocalCollision : 0));
        *reinterpret_cast<uint16_t*>(r + 16) = *reinterpret_cast<const uint16_t*>(t + 8);
    }
}

// origins of the entries in groups of several: a batch singleton among them collides globally
__global__ void k_mark(const uint64_t* origin, uint64_t n, uint8_t* marks) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint64_t o = origin[i];
        if (!(o & kLocalCollision)) marks[o] = 1;
    }
}

__global__ void k_count_colliding(const uint8_t* trip, uint64_t n, unsigned long long* count) {
    unsigned long long c = 0;
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x)
        c += *reinterpret_cast<const uint16_t*>(trip + 10 * i + 8) == 0;
    if (c) atomicAdd(count, c);
}

uint64_t slice_entries() {
    const char* e = std::getenv("LPHB_BUILD_SLICE");
    const uint64_t v = e ? std::strtoull(e, nullptr, 10) : 0;
    return v ? v : kSliceEntries;
}

}  // namespace

void Classify::group(const uint8_t* rec, uint64_t n, int key_bits, cudaStream_t s) {
    key.reserve(n * 8);
    key2.reserve(n * 8);
    idx.reserve(n * 4);
    idx2.reserve(n * 4);
    flags.reserve(n + 8);
    gslot.reserve(n * 4);
    cslot.reserve(n * 4);
    counts.reserve(64);
    tmp_bytes = classify_tmp_bytes(n);
    tmp.reserve(tmp_bytes);
    launch_classify_groups(rec, n, key.as<uint64_t>(), key2.as<uint64_t>(), idx.as<uint32_t>(), idx2.as<uint32_t>(),
                           flags.as<uint8_t>(), gslot.as<uint32_t>(), cslot.as<uint32_t>(), counts.as<unsigned long long>(),
                           tmp.p, tmp_bytes, key_bits, s);
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(h, counts.p, sizeof(h), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    groups = h[0];
    members = h[1];
}

void Classify::emit(const uint8_t* rec, uint64_t n, uint8_t* triplets, uint64_t* ids, cudaStream_t s) {
    idu.reserve(members * 8);
    launch_classify_emit(rec, key2.as<uint64_t>(), idx2.as<uint32_t>(), flags.as<uint8_t>(), gslot.as<uint32_t>(),
                         cslot.as<uint32_t>(), n, triplets, idu.as<uint64_t>(), ids, ids ? members : 0, tmp.p, tmp_bytes, s);
}

uint64_t Classify::bytes() const {
    uint64_t n = 0;
    for (const DevBuf* d : {&key, &key2, &idx, &idx2, &flags, &gslot, &cslot, &counts, &tmp, &idu}) n += d->cap;
    return n;
}

uint64_t BuildDevice::bytes() const {
    uint64_t n = cls.bytes();
    for (auto const& b : batches) n += b.trip.cap + b.sid.cap + b.lids.cap;
    for (const DevBuf* d : {&rec, &bounds, &desc, &marks, &idw, &nsel, &res_trip, &res_ids}) n += d->cap;
    return n;
}

void build_add_batch(lphb_build* b, const uint8_t* rec, uint64_t n, cudaStream_t s) {
    BuildDevice& D = *b->dev;
    BatchSummary sum;
    if (n) {
        D.cls.group(rec, n, int(2 * b->m), s);  // a minimizer is 2m bits
        sum.n_groups = D.cls.groups;
        sum.n_lids = D.cls.members;
        sum.trip.reserve(sum.n_groups * 10);
        sum.sid.reserve(sum.n_groups * 8);
        sum.lids.reserve(sum.n_lids * 8);
        D.cls.emit(rec, n, sum.trip.as<uint8_t>(), sum.lids.as<uint64_t>(), s);
        launch_classify_singleton_ids(rec, D.cls.idx2.as<uint32_t>(), D.cls.flags.as<uint8_t>(), D.cls.gslot.as<uint32_t>(),
                                      n, sum.sid.as<uint64_t>(), s);
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
    }
    D.batches.push_back(std::move(sum));
    D.merged = false;
}

namespace {

void build_merge(lphb_build* b) {
    BuildDevice& D = *b->dev;
    cudaStream_t s = D.s;
    const uint64_t nb = D.batches.size();
    const int key_bits = int(2 * b->m);
    std::vector<uint64_t> base(nb + 1, 0);
    std::vector<BatchDesc> desc(nb);
    uint64_t ids_bound = 0, ids_batch_max = 0;
    for (uint64_t j = 0; j < nb; ++j) {
        BatchSummary const& B = D.batches[j];
        base[j + 1] = base[j] + B.n_groups;
        desc[j] = {B.trip.as<uint8_t>(), B.n_groups};
        ids_bound += B.n_lids + B.n_groups;
        ids_batch_max = std::max(ids_batch_max, B.n_lids + B.n_groups);
    }
    const uint64_t E = base[nb];
    D.n_triplets = D.n_ids = D.colliding = 0;
    if (E == 0) {
        D.merged = true;
        return;
    }

    // triplets, slice by slice in ascending minimizer order
    D.marks.reserve(E);
    D.res_trip.reserve(E * 10);
    D.desc.reserve(nb * sizeof(BatchDesc));
    D.bounds.reserve(nb * 16);
    CK(cudaMemsetAsync(D.marks.p, 0, E, s));
    CK(cudaMemcpyAsync(D.desc.p, desc.data(), nb * sizeof(BatchDesc), cudaMemcpyHostToDevice, s));
    const uint64_t cap = slice_entries();
    std::vector<std::pair<uint64_t, uint64_t>> todo{{0, (1ull << key_bits) - 1}};  // inclusive ranges, last = next
    std::vector<uint64_t> bnd(2 * nb);
    uint64_t T = 0;
    while (!todo.empty()) {
        const auto [lo, hi] = todo.back();
        todo.pop_back();
        k_slice_bounds<<<unsigned((2 * nb + 255) / 256), 256, 0, s>>>(D.desc.as<BatchDesc>(), uint32_t(nb), lo, hi + 1,
                                                                      D.bounds.as<uint64_t>());
        CK(cudaMemcpyAsync(bnd.data(), D.bounds.p, nb * 16, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        uint64_t n = 0;
        for (uint64_t j = 0; j < nb; ++j) n += bnd[2 * j + 1] - bnd[2 * j];
        if (n == 0) continue;
        if (n > cap && lo < hi) {  // one minimizer has at most one entry per batch, so halving always ends
            const uint64_t mid = lo + (hi - lo) / 2;
            todo.push_back({mid + 1, hi});
            todo.push_back({lo, mid});
            continue;
        }
        D.rec.reserve(n * 18);
        uint64_t at = 0;
        for (uint64_t j = 0; j < nb; ++j) {
            const uint64_t a = bnd[2 * j], cnt = bnd[2 * j + 1] - a;
            if (!cnt) continue;
            BatchSummary const& B = D.batches[j];
            k_pack_slice<<<grid(cnt), 256, 0, s>>>(B.trip.as<uint8_t>() + 10 * a, B.sid.as<uint64_t>() + a, cnt, base[j] + a,
                                                   D.rec.as<uint8_t>() + 18 * at);
            at += cnt;
        }
        Classify& C = D.cls;
        C.group(D.rec.as<uint8_t>(), n, key_bits, s);
        C.emit(D.rec.as<uint8_t>(), n, D.res_trip.as<uint8_t>() + 10 * T, nullptr, s);  // the origins are only marked
        if (C.members) k_mark<<<grid(C.members), 256, 0, s>>>(C.idu.as<uint64_t>(), C.members, D.marks.as<uint8_t>());
        T += C.groups;
    }
    D.nsel.reserve(64);
    auto* d_cnt = D.nsel.as<unsigned long long>();
    CK(cudaMemsetAsync(d_cnt, 0, 16, s));
    k_count_colliding<<<grid(T), 256, 0, s>>>(D.res_trip.as<uint8_t>(), T, d_cnt);

    // ids, batch by batch: local collision ids + the batch singletons marked above, sorted
    size_t t_sel = 0, t_sort = 0;
    CK(cub::DeviceSelect::Flagged(nullptr, t_sel, (const uint64_t*)nullptr, (const uint8_t*)nullptr, (uint64_t*)nullptr,
                                  (long long*)nullptr, (int64_t)ids_batch_max));
    CK(cub::DeviceRadixSort::SortKeys(nullptr, t_sort, (const uint64_t*)nullptr, (uint64_t*)nullptr, ids_batch_max));
    D.cls.tmp.reserve(std::max<uint64_t>(t_sel, t_sort));
    D.idw.reserve(ids_batch_max * 8);
    D.res_ids.reserve(ids_bound * 8);
    auto* d_sel = reinterpret_cast<long long*>(d_cnt + 1);
    uint64_t I = 0;
    for (uint64_t j = 0; j < nb; ++j) {
        BatchSummary const& B = D.batches[j];
        if (!B.n_groups) continue;
        if (B.n_lids)
            CK(cudaMemcpyAsync(D.idw.p, B.lids.p, B.n_lids * 8, cudaMemcpyDeviceToDevice, s));
        size_t bytes = D.cls.tmp.cap;
        CK(cub::DeviceSelect::Flagged(D.cls.tmp.p, bytes, B.sid.as<uint64_t>(), D.marks.as<uint8_t>() + base[j],
                                      D.idw.as<uint64_t>() + B.n_lids, d_sel, (int64_t)B.n_groups, s));
        long long sel = 0;
        CK(cudaMemcpyAsync(&sel, d_sel, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        const uint64_t n = B.n_lids + uint64_t(sel);
        if (n) {
            bytes = D.cls.tmp.cap;
            CK(cub::DeviceRadixSort::SortKeys(D.cls.tmp.p, bytes, D.idw.as<uint64_t>(), D.res_ids.as<uint64_t>() + I, n, 0, 64, s));
        }
        I += n;
    }
    unsigned long long colliding = 0;
    CK(cudaMemcpyAsync(&colliding, d_cnt, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    D.n_triplets = T;
    D.n_ids = I;
    D.colliding = colliding;
    D.merged = true;
}

}  // namespace

}  // namespace lphb

using namespace lphb;

extern "C" {

int lphb_build_begin(int device, uint32_t k, uint32_t m, uint64_t seed, lphb_build** out) {
    if (!out) return fail(LPHB_E_ARG, "null argument");
    *out = nullptr;
    if (const char* e = scan_km_error(k, m)) return fail(LPHB_E_ARG, e);
    if (device < 0 || device >= 64) return fail(LPHB_E_ARG, "device index out of range");
    return guarded([&]() -> int {
        DeviceGuard g(device);
        std::unique_ptr<lphb_build> b(new lphb_build());
        b->device = device;
        b->k = k;
        b->m = m;
        b->seed = seed;
        b->dev.reset(new BuildDevice());
        b->dev->s.create();
        *out = b.release();
        return LPHB_OK;
    });
}

int lphb_build_end(lphb_build* b, void* triplets, uint64_t triplets_capacity, uint64_t* ids, uint64_t ids_capacity,
                   lphb_build_report* report) {
    if (!b || !report) return fail(LPHB_E_ARG, "null argument");
    if (!b->dev) return fail(LPHB_E_ARG, "the build session has ended");
    return guarded_nomem([&]() -> int {
        DeviceGuard g(b->device);
        BuildDevice& D = *b->dev;
        if (!D.merged) build_merge(b);
        *report = b->totals;
        report->n_triplets = D.n_triplets;
        report->n_ids = D.n_ids;
        report->colliding_minimizers = D.colliding;
        report->device_bytes = D.bytes();
        if (D.n_triplets > triplets_capacity) return fail(LPHB_E_CAPACITY, "triplets buffer too small");
        if (D.n_ids > ids_capacity) return fail(LPHB_E_CAPACITY, "ids buffer too small");
        if ((D.n_triplets && !triplets) || (D.n_ids && !ids)) return fail(LPHB_E_ARG, "null output buffer");
        if (D.n_triplets) CK(cudaMemcpyAsync(triplets, D.res_trip.p, D.n_triplets * 10, cudaMemcpyDeviceToHost, D.s));
        if (D.n_ids) CK(cudaMemcpyAsync(ids, D.res_ids.p, D.n_ids * 8, cudaMemcpyDeviceToHost, D.s));
        CK(cudaStreamSynchronize(D.s));
        b->dev.reset();
        return LPHB_OK;
    });
}

int lphb_build_free(lphb_build* b) {
    if (!b) return LPHB_OK;
    const int rc = guarded([&]() -> int {
        if (b->dev) {
            DeviceGuard g(b->device);
            b->dev.reset();
        }
        return LPHB_OK;
    });
    b->dev.reset();
    delete b;
    return rc;
}

}  // extern "C"
