// C ABI, build-p Part 3 and the `.lph` writer (include/lphash_b200.h): kernel sequencing for
// lphb_build_inverted_index, host-only assembly of the serialized image.
#include <cuda_runtime.h>

#include <cstring>
#include <vector>

#include "api_internal.h"
#include "image_decode.cuh"
#include "invindex_kernels.cuh"

using namespace lphb;

namespace {

uint64_t words_for(uint64_t bits) { return (bits + 63) / 64; }

// the image of one rs_bit_vector / of the Elias-Fano sequence while it is being laid out in the caller's buffer
struct Writer {
    uint8_t* out;
    uint64_t cap, at = 0;
    bool overflow = false;
    void u64(uint64_t v) { raw(&v, 8); }
    void raw(const void* p, uint64_t n) {
        if (at + n <= cap && !overflow) std::memcpy(out + at, p, n);
        else overflow = true;
        at += n;
    }
    // n bytes that live on the device
    void dev(const void* d, uint64_t n) {
        if (at + n <= cap && !overflow) {
            if (n) CK(cudaMemcpy(out + at, d, n, cudaMemcpyDeviceToHost));
        } else {
            overflow = true;
        }
        at += n;
    }
};

// one device allocation for the whole call, handed out 256-byte aligned (sizes are known up front from n; the
// only data-dependent one, the darray1 overflow list, is allocated on its own in the rare case it is needed)
struct Bump {
    uint8_t* base = nullptr;
    uint64_t at = 0, cap = 0;
    template <class T>
    T* take(uint64_t bytes) {
        at = (at + 255) & ~uint64_t(255);
        if (at + bytes > cap) throw std::runtime_error("internal: Part-3 workspace bound too small");
        T* p = reinterpret_cast<T*>(base + at);
        at += bytes;
        return p;
    }
};

struct BitsOnDevice {  // one wavelet-tree level
    uint64_t nbits = 0, words = 0, blocks = 0;
    uint64_t *bits = nullptr, *pairs = nullptr, *pop = nullptr;
    void alloc(Bump& w, uint64_t n) {
        nbits = n;
        words = words_for(n);
        blocks = (words + 7) / 8;
        bits = w.take<uint64_t>(blocks * 64 + 64);
        pairs = w.take<uint64_t>((2 * blocks + 2) * 8);
        pop = w.take<uint64_t>((blocks + 1) * 8);
    }
};


// Elias-Fano image of the prefix sums of n_ef byte values (ef_sequence::encode with its leading zero,
// include/ef_sequence.hpp:36-75) + darray1 over the high bits, built in the caller's workspace
struct EfOnDevice {
    uint64_t n_ef = 0, universe = 0, n_enc = 0, high_bits = 0, high_words = 0, low_words = 0, d_blocks = 0, n_sub = 0, n_ovf = 0;
    uint32_t l = 0;
    uint64_t *high = nullptr, *low = nullptr;
    int64_t* binv = nullptr;
    uint16_t* sinv = nullptr;
    DevBuf overflow;  // sparse blocks only: never seen on sequence data
};

void ef_encode(Bump& w, const uint8_t* vals, uint64_t n_ef, void* tmp, uint64_t tmp_bytes, cudaStream_t s, EfOnDevice& e) {
    e.n_ef = n_ef;
    if (!n_ef) return;
    auto* cum = w.take<uint64_t>(8 * n_ef + 16);
    launch_cumulative(vals, n_ef, cum, tmp, tmp_bytes, s);
    CK(cudaMemcpyAsync(&e.universe, cum + (n_ef - 1), 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    e.n_enc = n_ef + 1;
    const uint64_t q = e.universe / e.n_enc;
    e.l = q ? uint32_t(63 - __builtin_clzll(q)) : 0;  // pthash::util::msb, ef_sequence.hpp:44
    e.high_bits = e.n_enc + (e.universe >> e.l) + 1;
    e.high_words = words_for(e.high_bits);
    e.low_words = words_for(e.n_enc * e.l) + 1;  // compact_vector::builder keeps one spare word
    e.high = w.take<uint64_t>(8 * e.high_words + 16);
    e.low = w.take<uint64_t>(8 * e.low_words + 16);
    CK(cudaMemsetAsync(e.high, 0, 8 * e.high_words, s));
    launch_ef_encode(cum, e.n_enc, e.l, e.high, e.low, e.low_words, s);
    e.d_blocks = (e.n_enc + 1023) / 1024;
    e.n_sub = (e.d_blocks - 1) * 32 + ((e.n_enc - (e.d_blocks - 1) * 1024) + 31) / 32;
    auto* sparse = w.take<uint64_t>(8 * (e.d_blocks + 1));
    auto* ovf_off = w.take<uint64_t>(8 * (e.d_blocks + 1));
    e.binv = w.take<int64_t>(8 * e.d_blocks);
    e.sinv = w.take<uint16_t>(2 * e.d_blocks * 32 + 16);
    launch_darray(cum, e.n_enc, e.l, e.d_blocks, sparse, ovf_off, tmp, tmp_bytes, s);
    CK(cudaMemcpyAsync(&e.n_ovf, ovf_off + e.d_blocks, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (e.n_ovf) e.overflow.reserve(8 * e.n_ovf + 16);
    launch_darray_fill(cum, e.n_enc, e.l, e.d_blocks, sparse, ovf_off, e.binv, e.sinv, e.overflow.as<uint64_t>(), s);
}

// visitor order: include/ef_sequence.hpp:107-112, darray.hpp:90-96, compact_vector.hpp:278-283
void ef_write(Writer& wr, EfOnDevice const& e) {
    wr.u64(e.high_bits);
    wr.u64(e.high_words);
    wr.dev(e.high, 8 * e.high_words);
    wr.u64(e.n_enc);  // darray1::m_positions
    wr.u64(e.d_blocks);
    wr.dev(e.binv, 8 * e.d_blocks);
    wr.u64(e.n_sub);
    wr.dev(e.sinv, 2 * e.n_sub);
    wr.u64(e.n_ovf);
    wr.dev(e.overflow.p, 8 * e.n_ovf);
    wr.u64(e.n_enc);  // compact_vector: size, width, mask, words
    wr.u64(e.l);
    wr.u64(e.n_ef ? (uint64_t(1) << e.l) - 1 : 0);
    wr.u64(e.low_words);
    wr.dev(e.low, 8 * e.low_words);
}

// bytes of device workspace that suffice for the Part-3 pipeline over n minimizers (n_seq Elias-Fano sequences of at
// most v_max values each, every value < 256)
uint64_t part3_tmp_bytes(uint64_t n, uint64_t v_max) {
    uint64_t t = inv_scan_tmp_bytes((n + kInvBlock - 1) / kInvBlock);
    t = std::max(t, cum_tmp_bytes(v_max));
    t = std::max(t, darray_tmp_bytes(v_max / 1024 + 2));
    return std::max(t, rank_tmp_bytes(n / 512 + 2));
}
uint64_t ef_work_bytes(uint64_t v_max) {
    return v_max + 8 * v_max + 8 * (words_for(3 * v_max + 2) + 1) + 8 * (words_for(8 * v_max) + 2) +
           (v_max / 1024 + 2) * (8 + 8 + 8 + 64) + 16 * 256;
}

// One call of an inverted-index build (build-p Part 3) on the legacy stream: minimizer_order decoded on the device,
// the n triplets (10 bytes each) uploaded, the serialized index written to the caller's buffer through wr.
struct Part3 {
    DevPhf phf;
    const uint8_t* trip;
    Writer wr;
    DevBuf work;
    Event ev0, ev1;
    // `bytes` of device workspace; the device clock starts
    Bump start(uint64_t bytes) {
        work.reserve(bytes);
        ev0.create(cudaEventDefault);
        ev1.create(cudaEventDefault);
        CK(cudaEventRecord(ev0, nullptr));
        return Bump{work.as<uint8_t>(), 0, work.cap};
    }
    // milliseconds of device time since start(), once the device has finished
    float stop() {
        CK(cudaEventRecord(ev1, nullptr));
        CK(cudaStreamSynchronize(nullptr));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ev0, ev1));
        return ms;
    }
};

// Runs body(Part3&) on `device` after the checks both builds share; *out_bytes = what the index needs.
template <class Body>
int build_part3(int device, const void* minimizer_order, uint64_t minimizer_order_bytes, const void* triplets, uint64_t n,
                void* out, uint64_t out_capacity, uint64_t* out_bytes, Body&& body) {
    return guarded([&]() -> int {
        const ImagePlan plan = ImageBuilder::plan_phf(static_cast<const uint8_t*>(minimizer_order), minimizer_order_bytes);
        int count = 0;
        CK(cudaGetDeviceCount(&count));
        if (device < 0 || device >= count) return fail(LPHB_E_CUDA, "no such CUDA device");
        DeviceGuard g(device);
        DevBuf arena, trip;
        arena.reserve(plan.arena_bytes + 256);
        decode_phf_on_device(plan, arena.p);  // pilots and free slots decoded on the GPU (image_decode.cu)
        const DevPhf phf = rebase_image(plan.img, arena.p).minimizer_order;
        if (phf.num_keys != n) return fail(LPHB_E_ARG, "minimizer_order was built on a different number of keys");
        trip.reserve(10 * n + 16);
        if (n) CK(cudaMemcpy(trip.p, triplets, 10 * n, cudaMemcpyHostToDevice));
        Part3 p{phf, trip.as<uint8_t>(), Writer{static_cast<uint8_t*>(out), out_capacity}};
        const int rc = body(p);
        if (rc != LPHB_OK) return rc;
        *out_bytes = p.wr.at;
        if (p.wr.overflow) return fail(LPHB_E_CAPACITY, "output buffer too small for the inverted index");
        return LPHB_OK;
    });
}

}  // namespace

extern "C" {

uint64_t lphb_inverted_index_bound(uint64_t n) {
    // three rs_bit_vectors over <= 2n bits in total (bits + 2 directory words per 8), Elias-Fano of <= 2n + 1
    // values: high bits <= 3 values' worth, low bits <= 8 per value, darray1 <= (8/1024 + 2/32 + 3*1024*8/65536) bytes
    const uint64_t v = 2 * n + 2;
    return 3 * 64 + (2 * n / 8 + 3 * 8) * 5 / 4 + 3 * 32 + 256 + (3 * v / 8 + 16) + (v + 16) + (v / 128 + v / 16 + 3 * v / 8 + 64);
}

int lphb_build_inverted_index(int device, uint32_t k, uint32_t m, const void* minimizer_order,
                              uint64_t minimizer_order_bytes, const void* triplets, uint64_t n, void* out,
                              uint64_t out_capacity, uint64_t* out_bytes, lphb_inverted_index* info) {
    if (!minimizer_order || (!triplets && n) || !out_bytes || !info || (!out && out_capacity))
        return fail(LPHB_E_ARG, "null argument");
    if (m == 0 || k < m || k - m + 1 > 255) return fail(LPHB_E_ARG, "k/m out of range");
    return build_part3(device, minimizer_order, minimizer_order_bytes, triplets, n, out, out_capacity, out_bytes,
                       [&](Part3& p) -> int {
        cudaStream_t s = nullptr;  // the call is synchronous; the legacy stream orders it against the copies
        // workspace: everything below is bounded by n (at most 2n + 1 Elias-Fano values, each < 256)
        const uint64_t n_blocks = (n + kInvBlock - 1) / kInvBlock, v_max = 2 * n + 2;
        const uint64_t tmp_bytes = part3_tmp_bytes(n, v_max);
        Bump w = p.start(4 * n + 64 + (n_blocks + 1) * sizeof(InvCounts) + tmp_bytes + ef_work_bytes(v_max) +
                         3 * (n / 4 + 4096) + 16 * 256);
        auto* counters = w.take<unsigned long long>(64);  // [0] outside the range, [1] colliding, [2] unset cells
        auto* cells = w.take<uint32_t>(4 * n + 16);
        auto* blk = w.take<InvCounts>((n_blocks + 1) * sizeof(InvCounts));
        void* tmp = w.take<uint8_t>(tmp_bytes);

        // 1. re-key: the triplet of the minimizer with order i lands in cell i
        CK(cudaMemsetAsync(cells, 0, 4 * n + 16, s));
        CK(cudaMemsetAsync(counters, 0, 64, s));
        launch_rekey(p.phf, p.trip, n, k, m, cells, counters, counters + 1, s);
        // 2. how many of each type, per block of cells and in total
        launch_cell_counts(cells, n, blk, counters + 2, s);
        launch_counts_scan(blk, n_blocks, tmp, tmp_bytes, s);
        unsigned long long h_counters[3] = {0, 0, 0};
        InvCounts total{0, 0, 0, 0};
        CK(cudaMemcpyAsync(h_counters, counters, sizeof h_counters, cudaMemcpyDeviceToHost, s));
        if (n_blocks) CK(cudaMemcpyAsync(&total, blk + (n_blocks - 1), sizeof total, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (h_counters[0] || h_counters[2])
            return fail(LPHB_E_ARG, "minimizer_order does not map the triplets one to one onto [0, n)");
        const uint64_t n_left = total.left, n_rc = total.rc, n_none = total.none, n_msb = total.msb;
        const uint64_t rs = n_left, ns = rs + n_rc, np = ns + n_none, n_ef = np + n_none;
        info->n_maximal = n_msb - n_none;
        info->right_coll_sizes_start = rs;
        info->none_sizes_start = ns;
        info->none_pos_start = np;
        info->colliding_minimizers = h_counters[1];

        // 3. wavelet-tree bits and the four lists
        BitsOnDevice root, left_right, max_none;
        root.alloc(w, n);
        left_right.alloc(w, n - n_msb);
        max_none.alloc(w, n_msb);
        for (BitsOnDevice* b : {&root, &left_right, &max_none}) CK(cudaMemsetAsync(b->bits, 0, b->blocks * 64 + 64, s));
        auto* vals = w.take<uint8_t>(n_ef + 16);
        launch_place(cells, n, blk, rs, ns, np, reinterpret_cast<uint32_t*>(root.bits),
                     reinterpret_cast<uint32_t*>(left_right.bits), reinterpret_cast<uint32_t*>(max_none.bits), vals, s);
        for (BitsOnDevice* b : {&root, &left_right, &max_none})
            launch_rank_pairs(b->bits, b->blocks, b->pop, b->pairs, tmp, tmp_bytes, s);

        // 4. prefix sums -> Elias-Fano (ef_sequence::encode with a leading zero) -> darray1
        EfOnDevice ef;
        ef_encode(w, vals, n_ef, tmp, tmp_bytes, s, ef);
        info->device_ms = p.stop();
        info->universe = ef.universe;

        // 5. the serialized forms, in visitor order (include/quartet_wtree.hpp:43-48, include/rs_bit_vector.hpp:
        //    91-96, include/ef_sequence.hpp:107-112, darray.hpp:90-96, compact_vector.hpp:278-283)
        Writer& wr = p.wr;
        for (BitsOnDevice* b : {&root, &left_right, &max_none}) {
            wr.u64(b->nbits);
            wr.u64(b->words);
            wr.dev(b->bits, 8 * b->words);
            wr.u64(2 * b->blocks + 2);
            wr.dev(b->pairs, 8 * (2 * b->blocks + 2));
            wr.u64(0);  // select hints: never built (src/quartet_wtree.cpp:51-53)
        }
        info->wtree_bytes = wr.at;
        ef_write(wr, ef);
        info->ef_bytes = wr.at - info->wtree_bytes;
        return LPHB_OK;
    });
}

int lphb_build_inverted_index_alt(int device, const void* minimizer_order, uint64_t minimizer_order_bytes,
                                  const void* triplets, uint64_t n, void* out, uint64_t out_capacity, uint64_t* out_bytes,
                                  lphb_inverted_index_alt* info) {
    if (!minimizer_order || (!triplets && n) || !out_bytes || !info || (!out && out_capacity))
        return fail(LPHB_E_ARG, "null argument");
    return build_part3(device, minimizer_order, minimizer_order_bytes, triplets, n, out, out_capacity, out_bytes,
                       [&](Part3& p) -> int {
        cudaStream_t s = nullptr;
        const uint64_t v_max = n + 2, tmp_bytes = part3_tmp_bytes(n, v_max);
        Bump w = p.start(4 * n + 64 + tmp_bytes + 2 * ef_work_bytes(v_max) + 16 * 256);
        auto* counters = w.take<unsigned long long>(64);
        auto* cells = w.take<uint32_t>(4 * n + 16);
        void* tmp = w.take<uint8_t>(tmp_bytes);
        auto* p1 = w.take<uint8_t>(n + 16);
        auto* size = w.take<uint8_t>(n + 16);
        CK(cudaMemsetAsync(cells, 0, 4 * n + 16, s));
        CK(cudaMemsetAsync(counters, 0, 64, s));
        launch_rekey_alt(p.phf, p.trip, n, cells, counters, s);
        launch_split_alt(cells, n, p1, size, counters + 1, s);
        unsigned long long h_counters[2] = {0, 0};
        CK(cudaMemcpyAsync(h_counters, counters, sizeof h_counters, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (h_counters[0] || h_counters[1])
            return fail(LPHB_E_ARG, "minimizer_order does not map the triplets one to one onto [0, n)");
        EfOnDevice positions, sizes;
        ef_encode(w, p1, n, tmp, tmp_bytes, s, positions);  // build_pos_index, src/unpartitioned_mphf.cpp:152-159
        ef_encode(w, size, n, tmp, tmp_bytes, s, sizes);    // build_size_index, :161-169
        info->device_ms = p.stop();
        info->num_kmers_in_main_index = sizes.universe;  // sizes.access(sizes.size() - 1)
        ef_write(p.wr, positions);
        info->positions_bytes = p.wr.at;
        ef_write(p.wr, sizes);
        info->sizes_bytes = p.wr.at - info->positions_bytes;
        return LPHB_OK;
    });
}

int lphb_lph_assemble_alt(uint32_t k, uint32_t m, uint64_t mm_seed, uint64_t nkmers, uint64_t distinct_minimizers,
                          const lphb_inverted_index_alt* index, const void* minimizer_order, uint64_t minimizer_order_bytes,
                          const void* index_body, uint64_t index_body_bytes, const void* fallback_kmer_order,
                          uint64_t fallback_bytes, void* out, uint64_t out_capacity, uint64_t* out_bytes) {
    if (!index || !minimizer_order || !index_body || !fallback_kmer_order || !out_bytes || (!out && out_capacity))
        return fail(LPHB_E_ARG, "null argument");
    if (k > 255 || m > 255) return fail(LPHB_E_ARG, "k/m out of range");
    if (index_body_bytes != index->positions_bytes + index->sizes_bytes) return fail(LPHB_E_ARG, "index body size mismatch");
    return guarded([&]() -> int {
        // visitor order of lphash::mphf_alt (include/unpartitioned_mphf.hpp:198-210)
        Writer w{static_cast<uint8_t*>(out), out_capacity};
        const uint8_t k8 = uint8_t(k), m8 = uint8_t(m);
        w.raw(&k8, 1);
        w.raw(&m8, 1);
        w.u64(mm_seed);
        w.u64(nkmers);
        w.u64(distinct_minimizers);
        w.u64(index->num_kmers_in_main_index);
        w.raw(minimizer_order, minimizer_order_bytes);
        w.raw(index_body, index_body_bytes);
        w.raw(fallback_kmer_order, fallback_bytes);
        *out_bytes = w.at;
        if (w.overflow) return fail(LPHB_E_CAPACITY, "output buffer too small for the image");
        return LPHB_OK;
    });
}

int lphb_lph_sections(const void* image, uint64_t nbytes, int kmer_bits, int alt, uint64_t sections[5]) {
    if (!image || !sections) return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        const ImagePlan plan = ImageBuilder::plan(static_cast<const uint8_t*>(image), nbytes, kmer_bits, alt != 0);
        for (int i = 0; i < 5; ++i) sections[i] = plan.sections[i];
        return LPHB_OK;
    });
}

int lphb_lph_assemble(uint32_t k, uint32_t m, uint64_t mm_seed, uint64_t nkmers, uint64_t distinct_minimizers,
                      const lphb_inverted_index* index, const void* minimizer_order, uint64_t minimizer_order_bytes,
                      const void* index_body, uint64_t index_body_bytes, const void* fallback_kmer_order,
                      uint64_t fallback_bytes, void* out, uint64_t out_capacity, uint64_t* out_bytes) {
    if (!index || !minimizer_order || !index_body || !fallback_kmer_order || !out_bytes || (!out && out_capacity))
        return fail(LPHB_E_ARG, "null argument");
    if (k > 255 || m > 255) return fail(LPHB_E_ARG, "k/m out of range");
    if (index_body_bytes != index->wtree_bytes + index->ef_bytes) return fail(LPHB_E_ARG, "index body size mismatch");
    return guarded([&]() -> int {
        // visitor order of lphash::mphf (include/partitioned_mphf.hpp:204-219)
        Writer w{static_cast<uint8_t*>(out), out_capacity};
        const uint8_t k8 = uint8_t(k), m8 = uint8_t(m);
        w.raw(&k8, 1);
        w.raw(&m8, 1);
        w.u64(mm_seed);
        w.u64(nkmers);
        w.u64(distinct_minimizers);
        w.u64(index->n_maximal);
        w.u64(index->right_coll_sizes_start);
        w.u64(index->none_sizes_start);
        w.u64(index->none_pos_start);
        w.raw(minimizer_order, minimizer_order_bytes);
        w.raw(index_body, index_body_bytes);
        w.raw(fallback_kmer_order, fallback_bytes);
        *out_bytes = w.at;
        if (w.overflow) return fail(LPHB_E_CAPACITY, "output buffer too small for the .lph image");
        return LPHB_OK;
    });
}

}  // extern "C"
