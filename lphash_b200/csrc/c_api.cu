// C ABI of lphash_b200 (include/lphash_b200.h), the lphb_mphf handle: loading, host<->device staging and kernel
// sequencing of its queries, lookups and self-checks.  No CPU implementation of the path exists here: without a
// CUDA device every computing entry point fails with LPHB_E_CUDA.  The handle-less build side is in scan_api.cu.
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>
#include <fstream>
#include <new>
#include <algorithm>
#include <chrono>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/lphash_b200.h"
#include "api_internal.h"
#include "check_kernels.cuh"
#include "image_decode.cuh"
#include "lph_image.h"
#include "query_kernels.cuh"
#include "scan_kernels.cuh"

using namespace lphb;

namespace lphb {
std::string& last_error_slot() {
    thread_local std::string err;
    return err;
}
}  // namespace lphb

namespace {

struct Workspace {
    Stream stream;
    // a host call's batch in the clean layout (L-k+1 codes per contig)
    DevBuf bases, offsets, code_off, codes, dirty, status, tile;
    HostBuf h_status;     // 4 words
    DevBuf offsets_tmp;   // scan scratch of the code offsets (lphb_query_stream_device)
    // small batches (one record per call, as the reference's own loop makes them): one device block and its pinned
    // mirror, so that a call is one copy up, the kernels, one copy down
    struct Small {
        static constexpr uint64_t kBytes = uint64_t(1) << 20;
        DevBuf d;
        HostBuf h;
    } small;
    // run-length form of the codes (lphb_query_stream_runs); chunks alternate between two scratch sets
    struct Runs {
        DevBuf start, head, rank, head_at, tmp, records, count;
        HostBuf h_count;              // runs per chunk
        std::vector<Event> ev_count;  // per chunk: its run count has reached h_count
    } runs;
    // repair of contigs with non-ACGT bytes (quirk_kernels.cu): its scratch, and the host forms' final codes
    struct Repair {
        DevBuf scratch, out;
    } repair;
    // chunk pipeline of lphb_query_stream: two extra streams so that the H2D copy of chunk j+1,
    // the kernels of chunk j and the D2H copy of chunk j-1 overlap (PCIe is full duplex)
    Stream cs[2];
    Event ev_ready, ev_done[2];
    // session of the index self-check (lphb_check_begin .. lphb_check_end)
    struct Check {
        bool open = false;
        DevBuf bitmap;    // one bit per code of [0, nkmers): hit
        DevBuf counters;  // kCheckCounters words (check_kernels.cuh)
        HostBuf h_counters;
        uint64_t kmers = 0, contigs = 0;  // of the batches so far: the next batch's first k-mer ordinal
        uint64_t host_dirty = 0;          // dirty contigs the host form counted (the device form counts in `counters`)
    } check;
    // The handle has ONE device workspace (dirty flags, tile records, scan scratch).  Calls may arrive
    // on different streams (lphb_query_stream_device takes the caller's): every call first makes its
    // stream wait for the previous call's last kernel, so that two calls never share the workspace
    // in time; their device work is ordered, whatever the streams.
    Event ev_last;
    bool have_last = false;
    void order_after_previous(cudaStream_t st) {
        if (have_last) CK(cudaStreamWaitEvent(st, ev_last, 0));
    }
    void mark_last(cudaStream_t st) {
        CK(cudaEventRecord(ev_last, st));
        have_last = true;
    }
    // Stream of chunk j of a batch of n_chunks, called for j = 0, 1, ... in order: one chunk runs on s itself; several
    // alternate between cs[0] and cs[1], which first wait for what s holds at chunk 0.  join_chunks then makes s wait
    // for both.
    cudaStream_t chunk_stream(cudaStream_t s, uint64_t j, uint64_t n_chunks) {
        if (n_chunks < 2) return s;
        if (j == 0) {
            for (int i = 0; i < 2; ++i) {
                cs[i].create();
                ev_done[i].create(cudaEventDisableTiming);
            }
            ev_ready.create(cudaEventDisableTiming);
            CK(cudaEventRecord(ev_ready, s));
        }
        if (j < 2) CK(cudaStreamWaitEvent(cs[j & 1], ev_ready, 0));
        return cs[j & 1];
    }
    void join_chunks(cudaStream_t s, uint64_t n_chunks) {
        if (n_chunks < 2) return;
        for (int i = 0; i < 2; ++i) {
            CK(cudaEventRecord(ev_done[i], cs[i]));
            CK(cudaStreamWaitEvent(s, ev_done[i], 0));
        }
    }
    // A call through the small block on s, ordered after the previous call: up(h) writes its input to [at, end) of
    // the pinned mirror h, which goes up in one copy; kernels(d) enqueues its work on the device block d; [0, down)
    // comes back in one copy to h, and the call returns after the device finished.  Returns false, doing nothing,
    // when the block cannot hold `end` bytes or LPHB_NO_SMALL_PATH is set.
    template <class Up, class Kernels>
    bool small_round_trip(cudaStream_t s, uint64_t at, uint64_t end, uint64_t down, Up&& up, Kernels&& kernels) {
        if (end > Small::kBytes || getenv("LPHB_NO_SMALL_PATH")) return false;
        small.d.reserve(Small::kBytes);
        small.h.reserve(Small::kBytes);
        auto* h = small.h.as<unsigned char>();
        auto* d = small.d.as<unsigned char>();
        up(h);
        order_after_previous(s);
        CK(cudaMemcpyAsync(d + at, h + at, end - at, cudaMemcpyHostToDevice, s));
        kernels(d);
        mark_last(s);
        CK(cudaMemcpyAsync(h, d, down, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        return true;
    }
    // ring of event pairs bracketing the main kernel of the last kEvRing calls
    static constexpr int kEvRing = 128;
    Event ev0[kEvRing], ev1[kEvRing];
    uint64_t ev_next = 0, ev_pending = 0;  // next slot; pairs recorded since the last stats read
    void init() {
        stream.create();
        h_status.reserve(4 * sizeof(unsigned long long));
        ev_last.create(cudaEventDisableTiming);
        for (int i = 0; i < kEvRing; ++i) {
            ev0[i].create(cudaEventDefault);
            ev1[i].create(cudaEventDefault);
        }
        status.reserve(4 * sizeof(unsigned long long));
    }
};

// bases per chunk of the lphb_query_stream pipeline (LPHB_CHUNK_BASES overrides; 0: one chunk)
uint64_t pipeline_chunk_bases() {
    const char* e = getenv("LPHB_CHUNK_BASES");  // read per call: tests vary it
    uint64_t x = e ? strtoull(e, nullptr, 10) : (uint64_t(8) << 20);
    return x ? x : ~uint64_t(0);
}

}  // namespace

struct lphb_mphf {
    int device = 0;
    DevImage img{};
    void* d_arena = nullptr;
    uint64_t arena_bytes = 0;
    uint64_t l2_window_bytes = 0;      // 0: persistence not available
    float l2_hit_ratio = 1.0f;         // share of the window that may persist (carve-out / window)
    std::vector<cudaStream_t> l2_streams;  // streams the window is attached to
    lphb_info info{};
    lphb_stats stats{};
    uint64_t last_dirty_n = 0;  // contigs of the last query call (length of the dirty-flag array)
    const uint8_t* last_dirty = nullptr;  // where its flags are (device)
    Workspace ws;
    ~lphb_mphf() {
        if (d_arena) cudaFree(d_arena);
    }
};

namespace {

int load_image(const uint8_t* data, uint64_t n, int kmer_bits, int device, lphb_mphf** out, bool alt = false) {
    if (!out) return fail(LPHB_E_ARG, "out is null");
    *out = nullptr;
    return guarded([&]() -> int {
        // The structure of the file is walked on the host (sizes, ranges: format errors surface before any CUDA
        // call); the decoding - compact vectors, Elias-Fano, wavelet-tree ranks, one word per bucket - runs on the
        // GPU (image_decode.cu).  LPHB_HOST_DECODE=1 decodes on the host instead (lph_image.cpp; tests compare the
        // two images byte for byte), and so does a machine without a usable device, so that a malformed file is
        // reported as such before the missing device is.
        ImageBuilder builder;
        ImagePlan plan;
        const auto t_parse0 = std::chrono::steady_clock::now();
        int count = 0;
        const bool have_device = cudaGetDeviceCount(&count) == cudaSuccess && device >= 0 && device < count;
        if (!have_device) cudaGetLastError();
        const char* hd = getenv("LPHB_HOST_DECODE");
        const bool host_decode = !have_device || (hd && hd[0] && hd[0] != '0');
        if (host_decode) {
            if (alt) builder.parse_alt(data, n, kmer_bits);
            else builder.parse(data, n, kmer_bits);
        } else {
            plan = ImageBuilder::plan(data, n, kmer_bits, alt);
        }
        const auto t_parse1 = std::chrono::steady_clock::now();
        if (!have_device) return fail(LPHB_E_CUDA, "no such CUDA device");
        DeviceGuard g(device);
        std::unique_ptr<lphb_mphf> f(new lphb_mphf());
        f->device = device;
        const uint64_t arena_bytes = host_decode ? builder.arena().size() : plan.arena_bytes;
        CK(cudaMalloc(&f->d_arena, arena_bytes + 256));
        if (host_decode) {
            CK(cudaMemcpy(f->d_arena, builder.arena().data(), arena_bytes, cudaMemcpyHostToDevice));
            f->img = builder.rebased(f->d_arena);
        } else {
            uint64_t collision_base = 0;
            decode_image_on_device(plan, f->d_arena, &collision_base);
            f->img = rebase_image(plan.img, f->d_arena);
            f->img.collision_base = collision_base;
        }
        f->arena_bytes = arena_bytes;
        f->info.load_host_ms = std::chrono::duration<double, std::milli>(t_parse1 - t_parse0).count();
        f->info.load_h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_parse1).count();
        {
            int max_persist = 0, max_window = 0;
            cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, device);
            cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, device);
            // window = the whole image (clamped to the device's maximum window); carve-out =
            // as much of it as may persist; hitRatio = carve-out / window so that an image
            // larger than the carve-out does not thrash it
            uint64_t window = arena_bytes;
            if (uint64_t(max_window) < window) window = uint64_t(max_window);
            uint64_t carve = window;
            if (uint64_t(max_persist) < carve) carve = uint64_t(max_persist);
            if (carve && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve) == cudaSuccess) {
                f->l2_window_bytes = window;
                f->l2_hit_ratio = float(double(carve) / double(window));
            } else {
                cudaGetLastError();
            }
        }
        f->ws.init();
        lphb_info& i = f->info;
        i.k = f->img.k;
        i.m = f->img.m;
        i.kmer_bits = uint32_t(kmer_bits);
        i.device = device;
        i.mm_seed = f->img.mm_seed;
        i.nkmers = f->img.nkmers;
        i.distinct_minimizers = f->img.distinct_minimizers;
        i.n_maximal = f->img.n_maximal;
        i.right_coll_sizes_start = f->img.right_start;
        i.none_sizes_start = f->img.none_sizes_start;
        i.none_pos_start = f->img.none_pos_start;
        i.fallback_keys = host_decode ? builder.fallback_keys() : plan.fallback_keys;
        i.file_bytes = host_decode ? builder.file_bytes() : plan.file_bytes;
        i.device_bytes = arena_bytes;
        *out = f.release();
        return LPHB_OK;
    });
}

int load_file(const char* path, int kmer_bits, int device, lphb_mphf** out, bool alt) {
    if (!path) return fail(LPHB_E_ARG, "path is null");
    if (!out) return fail(LPHB_E_ARG, "out is null");
    *out = nullptr;
    std::vector<uint8_t> buf;
    int rc = guarded([&]() -> int {  // allocation failures must not cross the C boundary either
        std::ifstream in(path, std::ios::binary | std::ios::ate);
        if (!in.good()) return fail(LPHB_E_IO, std::string("cannot open ") + path);
        const std::streamoff n = in.tellg();
        if (n < 0) return fail(LPHB_E_IO, std::string("cannot size ") + path);
        in.seekg(0);
        buf.resize(static_cast<size_t>(n));
        if (n && !in.read(reinterpret_cast<char*>(buf.data()), n)) return fail(LPHB_E_IO, "short read");
        return LPHB_OK;
    });
    if (rc != LPHB_OK) return rc;
    return load_image(buf.data(), uint64_t(buf.size()), kmer_bits, device, out, alt);
}

// main kernel bracketed by the handle's events (elapsed time is read lazily by lphb_mphf_stats)
// Keep the image (a few bits per k-mer, gathered at random) resident in L2 while the base stream
// and the codes (streamed once, marked evict-first in the kernels) flow through it.
void attach_l2_window(lphb_mphf* f, cudaStream_t s) {
    if (!f->l2_window_bytes) return;
    for (cudaStream_t t : f->l2_streams)
        if (t == s) return;
    cudaStreamAttrValue attr{};
    attr.accessPolicyWindow.base_ptr = f->d_arena;
    attr.accessPolicyWindow.num_bytes = f->l2_window_bytes;
    attr.accessPolicyWindow.hitRatio = f->l2_hit_ratio;
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    if (cudaStreamSetAttribute(s, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess)
        cudaGetLastError();  // a hint only
    if (f->l2_streams.size() >= 16) f->l2_streams.clear();  // caller cycles through many streams
    f->l2_streams.push_back(s);
}

// `launch` enqueues the main kernel of a call on s, between the next pair of the handle's events
template <class Launch>
void timed_launch(lphb_mphf* f, cudaStream_t s, Launch&& launch) {
    attach_l2_window(f, s);
    const int slot = int(f->ws.ev_next % Workspace::kEvRing);
    CK(cudaEventRecord(f->ws.ev0[slot], s));
    launch();
    CK(cudaEventRecord(f->ws.ev1[slot], s));
    ++f->ws.ev_next;
    ++f->ws.ev_pending;
}

// the streaming query kernel over a batch: tiled where (k, m) is instantiated, else generic
void launch_stream_pass(lphb_mphf* f, DevBatch const& b, cudaStream_t s) {
    // A batch of a few tiles would leave one or two warps of the tiled kernel to walk its whole (cold) code
    // alone, about 40 us whatever the size; below 256 K bases the one-thread-per-k-mer kernel answers sooner
    // (10 us for a record of 8,000 bases; tools/ubench/call_latency.cpp).  LPHB_GENERIC_BELOW overrides (tests: 0).
    const char* gb = getenv("LPHB_GENERIC_BELOW");
    const uint64_t generic_below = gb ? strtoull(gb, nullptr, 10) : (uint64_t(1) << 18);
    if (b.end_base - b.first_base < generic_below || !launch_query_tiled(f->img, b, s))
        launch_query_generic(f->img, b, s);
}

void run_kernels(lphb_mphf* f, DevBatch const& b, cudaStream_t s) {
    timed_launch(f, s, [&] { launch_stream_pass(f, b, s); });
    launch_count_dirty(b.dirty, b.n_contigs, b.status, s);
    f->stats.kernel_launches += 2;
}

// ---- the index self-check (lphb_check_*) -----------------------------------------------------------------------
// One batch or chunk b (bases, offsets, code_off from ordinal j0 of the batch on, n_contigs, dirty zeroed) through
// the check: the contigs' dirty flags (any non-ACGT byte, whatever the contig's length) counted into
// dirty_status[1]; unless the caller gave its own streaming codes, the streaming pass into b.codes; then the check
// kernel, timed, over the ordinals [j0, j1) of the batch.
void check_chunk(lphb_mphf* f, DevBatch const& b, uint64_t j0, uint64_t j1, const uint64_t* caller_codes,
                 unsigned long long* dirty_status, cudaStream_t s) {
    Workspace::Check& C = f->ws.check;
    launch_flag_invalid_bytes(b.bases, b.first_base, b.end_base - b.first_base, b.offsets, b.n_contigs, b.dirty, s);
    launch_count_dirty(b.dirty, b.n_contigs, dirty_status, s);
    f->stats.kernel_launches += 2;
    if (!caller_codes && j1 > j0) {
        launch_stream_pass(f, b, s);
        f->stats.kernel_launches += 1;
    }
    CheckBatch cb{};
    cb.bases = b.bases;
    cb.offsets = b.offsets;
    cb.code_off = b.code_off;
    cb.n_contigs = b.n_contigs;
    cb.j0 = j0;
    cb.j1 = j1;
    cb.ordinal_base = C.kmers;
    cb.stream_codes = caller_codes ? caller_codes : b.codes;
    cb.dirty = b.dirty;
    cb.bitmap = C.bitmap.as<uint32_t>();
    cb.counters = C.counters.as<unsigned long long>();
    timed_launch(f, s, [&] { launch_check_windows(f->img, cb, s); });
    f->stats.kernel_launches += 1;
}

// ---- contigs with non-ACGT bytes (SURVEY.md Q1; quirk_kernels.cu) ----------------------------------------------
// Every form runs the same two device stages after its clean pass: launch_repair_layout (the dirty contigs listed,
// their spurious codes replayed, the final layout into the code offsets and its total into a status word), then
// launch_repair_assemble (the codes in that layout).  Nothing between them needs the host; the synchronous forms
// read the total back there for their capacity check.

// The repair scratch of a batch (n_contigs contigs over `span` bases with clean_total clean codes), sized from the
// host offsets alone, over the batch's bytes (indexed by the offsets) and the clean pass's dirty flags.
RepairWs reserve_repair(lphb_mphf* f, const char* bases, const uint64_t* d_offsets, const uint8_t* dirty,
                        uint64_t n_contigs, uint64_t span, uint64_t clean_total, bool in_place) {
    RepairWs w{};
    w.bases = bases;
    w.offsets = d_offsets;
    w.n_contigs = n_contigs;
    w.dirty = dirty;
    DevBuf& buf = f->ws.repair.scratch;
    buf.reserve(repair_scratch(n_contigs, span, clean_total, in_place, nullptr, nullptr));
    repair_scratch(n_contigs, span, clean_total, in_place, buf.as<char>(), &w);
    return w;
}

// the layout stage on s, its counters cleared first
void repair_layout(lphb_mphf* f, RepairWs const& w, uint64_t* d_code_off, const uint64_t* codes, uint64_t clean_total,
                   bool in_place, unsigned long long* d_total, cudaStream_t s) {
    CK(cudaMemsetAsync(w.ctr, 0, sizeof(RepairCounters), s));
    f->stats.kernel_launches += launch_repair_layout(f->img, w, d_code_off, codes, clean_total, in_place, d_total, s);
}

// What the caller wants back: the codes themselves (8 B per k-mer) or their run-length form (12-byte
// records, about 2 B per k-mer: runs_kernels.cu).
struct RunSink {
    void* runs = nullptr;        // null: codes mode
    uint64_t capacity = 0;
    uint64_t* n_runs = nullptr;
    // the reference's NON-streaming branch (include/partitioned_mphf.hpp:185-195): every window of k bytes is a
    // k-mer, a non-ACGT byte counts as 'A' (include/mphf_utils.hpp:108); no streaming state, hence no quirk
    bool non_streaming = false;
    // the index self-check (lphb_check_batch): every chunk goes through check_chunk; no code leaves the device
    bool check = false;
};

// One call of lphb_query_stream, lphb_query_nonstreaming or lphb_query_stream_runs with its batch on the host.
// Stages: the layout (run), then either the small-batch block (small_call) or the clean pass (clean_pass); when
// a contig holds a non-ACGT byte, the repair of such contigs (launch_repair_layout, launch_repair_assemble); the
// output (output).
struct HostQuery {
    lphb_mphf* f;
    const char* bases;
    const uint64_t* offsets;
    uint64_t n_contigs;
    uint64_t* codes;
    uint64_t codes_capacity;
    uint64_t* code_offsets;  // the layout on the host: clean first, final after the repair
    uint64_t* n_codes;
    RunSink sink;
    Workspace& ws = f->ws;
    cudaStream_t s = ws.stream;
    const bool want_runs = sink.runs != nullptr || sink.n_runs != nullptr;
    uint64_t first = 0, span = 0, total = 0;  // bases of the batch, codes of the clean layout
    bool copied_out = false;  // the clean pass copied every chunk's results out (a check: ran its chunks piped)
    uint64_t n_chunks = 1;
    uint64_t runs_per = 0;    // codes per scratch set of the run-length pass
    uint64_t runs_done = 0;   // run records already placed in the caller's buffer
    bool runs_overflow = false;

    int run() {
        f->stats = lphb_stats{};
        if (want_runs) *sink.n_runs = 0;
        // layout for clean input: L-k+1 codes per contig (partitioned_mphf.hpp:79-80)
        total = contig_layout(offsets, n_contigs, f->img.k, 0, code_offsets).kmers;
        *n_codes = total;
        if (n_contigs == 0) return LPHB_OK;
        first = offsets[0];
        span = offsets[n_contigs] - first;
        if (span && !bases) return fail(LPHB_E_ARG, "bases is null");
        if (want_runs && total >= (1ull << 31)) return fail(LPHB_E_ARG, "batch holds >= 2^31 k-mers: split it");
        f->last_dirty = nullptr;
        if (small_call()) return LPHB_OK;
        const uint64_t n_dirty = clean_pass();
        if (sink.check) {
            ws.check.host_dirty += n_dirty;
            return LPHB_OK;
        }
        if (n_dirty == 0) return copied_out ? finish(total, n_chunks, 0) : output(ws.codes.as<uint64_t>(), total, 0);
        const RepairWs w = reserve_repair(f, ws.bases.as<char>() - first, ws.offsets.as<uint64_t>(), ws.dirty.as<uint8_t>(),
                                          n_contigs, span, total, false);
        repair_layout(f, w, ws.code_off.as<uint64_t>(), ws.codes.as<uint64_t>(), total, false,
                      ws.status.as<unsigned long long>(), s);
        CK(cudaMemcpyAsync(code_offsets, ws.code_off.p, (n_contigs + 1) * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        const uint64_t new_total = code_offsets[n_contigs];
        *n_codes = new_total;
        if (!want_runs && new_total > codes_capacity) return fail(LPHB_E_CAPACITY, "codes buffer too small");
        if (want_runs && new_total >= (1ull << 31)) return fail(LPHB_E_ARG, "batch holds >= 2^31 codes: split it");
        ws.repair.out.reserve(new_total * 8 + 64);
        f->stats.kernel_launches += launch_repair_assemble(f->img, w, ws.code_off.as<uint64_t>(), ws.codes.as<uint64_t>(),
                                                           false, ws.repair.out.as<uint64_t>(), new_total, s);
        if (want_runs) reserve_runs(new_total + 16, 1, new_total, 1);
        return output(ws.repair.out.as<uint64_t>(), new_total, (n_contigs + 1) * 8);
    }

    // ---- small batch (the reference's own loop hands over one record per call, src/query.cpp:48-56): one device
    // block [codes | status | dirty flags | offsets | code offsets | bases] with a pinned mirror - one copy up (status
    // and flags arrive zeroed with it), the kernels, one copy down [codes | status].  Returns false when the batch
    // does not qualify, or when a contig holds a non-ACGT byte: the call then starts over on the general path.
    bool small_call() {
        if (want_runs || sink.check || !codes || !total || total > codes_capacity) return false;
        const uint64_t codes_b = (total * 8 + 63) & ~uint64_t(63), dirty_b = (n_contigs + 8 + 63) & ~uint64_t(63);
        const uint64_t off_b = (n_contigs + 1) * 8;
        const uint64_t in_b = 64 + dirty_b + 2 * off_b + span + 64;
        const uint64_t at_status = codes_b, at_dirty = at_status + 64, at_off = at_dirty + dirty_b,
                       at_coff = at_off + off_b, at_bases = at_coff + off_b;
        auto up = [&](unsigned char* h) {
            std::memset(h + at_status, 0, 64 + dirty_b);
            std::memcpy(h + at_off, offsets, off_b);
            std::memcpy(h + at_coff, code_offsets, off_b);
            if (span) std::memcpy(h + at_bases, bases + first, span);
            std::memset(h + at_bases + span, 'A', 64);
        };
        auto kernels = [&](unsigned char* d) {
            if (sink.non_streaming) launch_sanitize(reinterpret_cast<char*>(d + at_bases), span, s);
            DevBatch b{};
            b.bases = reinterpret_cast<const char*>(d + at_bases) - first;
            b.offsets = reinterpret_cast<const uint64_t*>(d + at_off);
            b.code_off = reinterpret_cast<const uint64_t*>(d + at_coff);
            b.n_contigs = n_contigs;
            b.first_base = first;
            b.end_base = first + span;
            b.codes = reinterpret_cast<uint64_t*>(d);
            b.dirty = d + at_dirty;
            b.status = reinterpret_cast<unsigned long long*>(d + at_status);
            ws.tile.reserve(query_tiled_ws_bytes(span));
            b.tile_ws = ws.tile.p;
            b.tile_ws_bytes = ws.tile.cap;
            run_kernels(f, b, s);
        };
        if (!ws.small_round_trip(s, at_status, codes_b + in_b, codes_b + 64, up, kernels)) return false;
        const auto* h = ws.small.h.as<unsigned char>();
        const auto* st = reinterpret_cast<const unsigned long long*>(h + at_status);
        f->last_dirty_n = n_contigs;
        f->last_dirty = ws.small.d.as<uint8_t>() + at_dirty;
        f->stats.h2d_bytes = in_b;
        f->stats.d2h_bytes = codes_b + 64;
        if (st[1] == 0) {
            std::memcpy(codes, h, total * 8);
            return true;
        }
        f->last_dirty = nullptr;
        f->stats = lphb_stats{};
        return false;
    }

    // ---- clean pass: every contig in the clean layout, the batch cut (on contig boundaries) into chunks.  Several
    // chunks flow through two streams: the H2D copy of chunk j+1, the kernels of chunk j and the D2H copy of chunk
    // j-1's results overlap.  Their results are copied out optimistically; if some contig turns out to contain a
    // non-ACGT byte the repair rewrites them.  A batch whose results cannot be copied out per chunk is one chunk on
    // the handle's stream, and nothing leaves the device before its status is known.  Returns the contigs with
    // non-ACGT bytes.
    uint64_t clean_pass() {
        ws.bases.reserve(span + 64);
        ws.offsets.reserve((n_contigs + 1) * 8);
        ws.code_off.reserve((n_contigs + 1) * 8);
        ws.codes.reserve(total * 8 + 64);
        ws.dirty.reserve(n_contigs + 8);
        ws.order_after_previous(s);  // a device-resident call may still be running on the caller's stream
        CK(cudaMemcpyAsync(ws.offsets.p, offsets, (n_contigs + 1) * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(ws.code_off.p, code_offsets, (n_contigs + 1) * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemsetAsync(ws.dirty.p, 0, n_contigs + 8, s));
        CK(cudaMemsetAsync(ws.status.p, 0, 4 * sizeof(unsigned long long), s));
        f->last_dirty_n = n_contigs;
        f->stats.h2d_bytes = span + 2 * (n_contigs + 1) * 8;
        std::vector<uint64_t> cuts{0};
        const uint64_t chunk = pipeline_chunk_bases();
        for (uint64_t c = 0; c < n_contigs; ++c)
            if (offsets[c + 1] - offsets[cuts.back()] >= chunk && c + 1 < n_contigs) cuts.push_back(c + 1);
        cuts.push_back(n_contigs);
        copied_out = cuts.size() > 2 && (sink.check || (want_runs ? sink.runs != nullptr : (total <= codes_capacity && codes)));
        if (!copied_out) cuts = {0, n_contigs};
        n_chunks = cuts.size() - 1;
        std::vector<uint64_t> tile_at(n_chunks + 1, 0);
        uint64_t max_codes = 0;
        for (uint64_t j = 0; j < n_chunks; ++j) {
            const uint64_t bytes = query_tiled_ws_bytes(offsets[cuts[j + 1]] - offsets[cuts[j]]);
            tile_at[j + 1] = tile_at[j] + (bytes + 255) / 256 * 256;
            max_codes = std::max<uint64_t>(max_codes, code_offsets[cuts[j + 1]] - code_offsets[cuts[j]]);
        }
        ws.tile.reserve(tile_at[n_chunks]);
        if (want_runs) reserve_runs(max_codes + 16, copied_out ? 2 : 1, total, n_chunks);
        for (uint64_t j = 0; j < n_chunks; ++j) {
            const cudaStream_t st = ws.chunk_stream(s, j, n_chunks);
            const uint64_t c0 = cuts[j], c1 = cuts[j + 1];
            const uint64_t b0 = offsets[c0], b1 = offsets[c1];
            if (b1 > b0) {
                CK(cudaMemcpyAsync(ws.bases.as<char>() + (b0 - first), bases + b0, b1 - b0, cudaMemcpyHostToDevice, st));
                if (sink.non_streaming) launch_sanitize(ws.bases.as<char>() + (b0 - first), b1 - b0, st);
            }
            DevBatch b{};
            b.bases = ws.bases.as<char>() - first;  // kernels index bases[offsets[c] + ...]
            b.offsets = ws.offsets.as<uint64_t>() + c0;
            b.code_off = ws.code_off.as<uint64_t>() + c0;
            b.n_contigs = c1 - c0;
            b.first_base = b0;
            b.end_base = b1;
            b.codes = ws.codes.as<uint64_t>();
            b.dirty = ws.dirty.as<uint8_t>() + c0;
            b.status = ws.status.as<unsigned long long>();
            b.tile_ws = static_cast<char*>(ws.tile.p) + tile_at[j];
            b.tile_ws_bytes = tile_at[j + 1] - tile_at[j];
            if (sink.check) {
                check_chunk(f, b, code_offsets[c0], code_offsets[c1], nullptr, b.status, st);
                continue;
            }
            run_kernels(f, b, st);
            if (copied_out) {
                emit(j, j & 1, ws.codes.as<uint64_t>(), code_offsets[c0], code_offsets[c1], b.code_off, b.n_contigs, st);
                // the previous chunk's records leave while this chunk computes
                if (want_runs && j >= 1) fetch_runs(j - 1, code_offsets[cuts[j - 1]], ws.cs[(j - 1) & 1]);
            }
        }
        if (copied_out && want_runs) fetch_runs(n_chunks - 1, code_offsets[cuts[n_chunks - 1]], ws.cs[(n_chunks - 1) & 1]);
        ws.join_chunks(s, n_chunks);
        auto* h_status = ws.h_status.as<unsigned long long>();
        CK(cudaMemcpyAsync(h_status, ws.status.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        f->stats.dirty_contigs = h_status[1];
        return h_status[1];
    }

    // ---- output: the n codes d_codes of the batch, laid out as ws.code_off says, to the caller as codes or runs
    int output(const uint64_t* d_codes, uint64_t n, uint64_t d2h_before) {
        if (!want_runs && n > codes_capacity) return fail(LPHB_E_CAPACITY, "codes buffer too small");
        runs_done = 0;
        runs_overflow = false;
        emit(0, 0, d_codes, 0, n, ws.code_off.as<uint64_t>(), n_contigs, s);
        if (want_runs) fetch_runs(0, 0, s);
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        return finish(n, 1, d2h_before);
    }

    int finish(uint64_t n, uint64_t n_counts, uint64_t d2h_before) {
        const uint64_t d2h_status = 4 * sizeof(unsigned long long);
        if (!want_runs) {
            f->stats.d2h_bytes = d2h_status + d2h_before + n * 8;
            return LPHB_OK;
        }
        *sink.n_runs = runs_done;
        if (runs_overflow) return fail(LPHB_E_CAPACITY, "runs buffer too small");
        f->stats.d2h_bytes = d2h_status + d2h_before + runs_done * 12 + n_counts * 8;
        return LPHB_OK;
    }

    // scratch of the run-length pass: `sets` sets of `per` codes each, records for n_codes codes, n_counts counts
    void reserve_runs(uint64_t per, uint64_t sets, uint64_t n_codes, uint64_t n_counts) {
        Workspace::Runs& R = ws.runs;
        const uint64_t n = sets * per;
        runs_per = per;
        R.start.reserve(n + 8);
        R.head.reserve(n + 8);
        R.rank.reserve((n + 2) * 4);
        R.head_at.reserve((n + 2) * 4);
        R.tmp.reserve(2 * ((runs_tmp_bytes(n) + 255) / 256 * 256));  // one half per scratch set
        R.records.reserve(n_codes * 12 + 64);
        R.count.reserve((n_counts + 1) * 8);
        R.h_count.reserve((n_counts + 1) * 8);
        while (R.ev_count.size() < n_counts + 1) {
            R.ev_count.emplace_back();
            R.ev_count.back().create(cudaEventDisableTiming);
        }
    }

    // The codes [o0, o1) of chunk j (nc contigs from d_code_off) leave the device: copied to the caller's buffer, or
    // through the run-length pass on scratch set `set`, its count to the host
    void emit(uint64_t j, uint64_t set, const uint64_t* d_codes, uint64_t o0, uint64_t o1, const uint64_t* d_code_off,
              uint64_t nc, cudaStream_t st) {
        if (!want_runs) {
            if (o1 > o0) CK(cudaMemcpyAsync(codes + o0, d_codes + o0, (o1 - o0) * 8, cudaMemcpyDeviceToHost, st));
            return;
        }
        Workspace::Runs& R = ws.runs;
        const uint64_t at = set * runs_per, tmp_half = R.tmp.cap / 2 / 256 * 256;
        launch_runs(d_codes + o0, o1 - o0, d_code_off, nc, o0, R.start.as<uint8_t>() + at, R.head.as<uint8_t>() + at,
                    R.rank.as<uint32_t>() + at, R.head_at.as<uint32_t>() + at, static_cast<char*>(R.tmp.p) + set * tmp_half,
                    tmp_half, R.records.as<uint8_t>() + o0 * 12, R.count.as<unsigned long long>() + j, st);
        f->stats.kernel_launches += 5;
        CK(cudaMemcpyAsync(R.h_count.as<unsigned long long>() + j, R.count.as<unsigned long long>() + j, 8,
                           cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(R.ev_count[j], st));
    }

    // once chunk j's run count is known: its records to the caller's buffer, behind the earlier chunks'
    void fetch_runs(uint64_t j, uint64_t o0, cudaStream_t st) {
        Workspace::Runs& R = ws.runs;
        CK(cudaEventSynchronize(R.ev_count[j]));
        const uint64_t n = R.h_count.as<unsigned long long>()[j];
        if (runs_done + n > sink.capacity || !sink.runs) {
            runs_overflow = true;
        } else if (n) {
            CK(cudaMemcpyAsync(static_cast<char*>(sink.runs) + runs_done * 12, R.records.as<uint8_t>() + o0 * 12, n * 12,
                               cudaMemcpyDeviceToHost, st));
        }
        runs_done += n;
    }
};

int query_stream_host(lphb_mphf* f, const char* bases, const uint64_t* offsets, uint64_t n_contigs,
                      uint64_t* codes, uint64_t codes_capacity, uint64_t* code_offsets, uint64_t* n_codes,
                      RunSink sink) {
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        HostQuery q{f, bases, offsets, n_contigs, codes, codes_capacity, code_offsets, n_codes, sink};
        return q.run();
    });
}

// ---- batches in the caller's device buffers ------------------------------------------------------

// What every call on a batch in the caller's device buffers runs first on s, ordered after the previous call: the
// dirty flags cleared, the code offsets into code_off with status[0] = the k-mer total.  Reserves the workspace the
// kernels use (with tile, the streaming pass's too) and returns the batch, its codes going to `codes`.
// (growing a workspace buffer frees the old one: cudaFree waits for the device, so a previous call still running
// never loses its buffer)
DevBatch start_device_batch(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                            uint64_t n_contigs, uint64_t* code_off, uint64_t* codes, unsigned long long* status,
                            bool tile, cudaStream_t s) {
    Workspace& ws = f->ws;
    ws.offsets_tmp.reserve(code_offsets_tmp_bytes(n_contigs));
    ws.dirty.reserve(n_contigs + 8);
    if (tile) ws.tile.reserve(query_tiled_ws_bytes(h_offsets[n_contigs] - h_offsets[0]));
    ws.order_after_previous(s);
    CK(cudaMemsetAsync(ws.dirty.p, 0, n_contigs + 8, s));
    launch_code_offsets(d_offsets, n_contigs, f->img.k, code_off, status, ws.offsets_tmp.p, ws.offsets_tmp.cap, s);
    f->stats.kernel_launches += 2;
    f->last_dirty_n = n_contigs;
    f->last_dirty = nullptr;
    DevBatch b{};
    b.bases = d_bases;
    b.offsets = d_offsets;
    b.code_off = code_off;
    b.n_contigs = n_contigs;
    b.first_base = h_offsets[0];
    b.end_base = h_offsets[n_contigs];
    b.codes = codes;
    b.dirty = ws.dirty.as<uint8_t>();
    b.status = status;
    b.tile_ws = ws.tile.p;
    b.tile_ws_bytes = ws.tile.cap;
    return b;
}

// lphb_query_stream_device, lphb_query_nonstreaming_device and (n_codes not null) lphb_query_stream_exact_device.
// The stateless forms enqueue the codes of the batch on s and count its dirty contigs into the caller's st.
// non_streaming: the kernels read a copy of the batch's bytes in the workspace with every non-ACGT byte made 'A',
// so that every window has its code and the caller's bytes stay as they are.
// The exact form: the same clean pass, one read-back of its status and, when a contig holds a non-ACGT byte, the
// repair's layout stage, one read-back of the final total (the capacity check), the assemble stage.  The clean pass
// writes straight into d_codes when the clean layout fits there, so a clean batch costs one device call more than
// the stateless form: the status read.  The layout stage then saves the clean codes the assemble overwrites.
int device_query(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                 uint64_t n_contigs, uint64_t* d_codes, uint64_t codes_capacity, uint64_t* d_code_offsets,
                 unsigned long long* st, uint64_t* n_codes, bool non_streaming, cudaStream_t s) {
    f->stats = lphb_stats{};
    Workspace& ws = f->ws;
    const bool exact = n_codes != nullptr;
    const uint64_t total = contig_layout(h_offsets, n_contigs, f->img.k).kmers;
    const uint64_t first = h_offsets[0], span = h_offsets[n_contigs] - first;
    if (exact) *n_codes = total;
    else if (total > codes_capacity) return fail(LPHB_E_CAPACITY, "codes buffer too small");
    // (a contig shorter than k yields no code, spurious ones included: without a clean code there is none at all;
    // the stateless streaming form reads no byte of a batch without a k-mer)
    if ((total && !d_codes) || (span && !d_bases && (total || exact || non_streaming)))
        return fail(LPHB_E_ARG, "null data pointer");
    const bool in_place = total <= codes_capacity;  // (only the exact form gets here with a clean layout too large)
    if (non_streaming) ws.bases.reserve(span + 16 + kCopySanitizePad);
    if (!in_place) ws.codes.reserve(total * 8 + 64);
    if (exact) st = ws.status.as<unsigned long long>();
    DevBatch b = start_device_batch(f, d_bases, d_offsets, h_offsets, n_contigs, d_code_offsets,
                                    in_place ? d_codes : ws.codes.as<uint64_t>(), st, true, s);
    if (non_streaming && span) {
        launch_copy_sanitize(ws.bases.as<char>(), d_bases + first, span, s);
        b.bases = ws.bases.as<char>() + copy_sanitize_at(d_bases + first) - first;  // indexed by the offsets
        f->stats.kernel_launches += 1;
    }
    if (n_contigs) run_kernels(f, b, s);
    ws.mark_last(s);
    if (!exact) {
        CK(cudaGetLastError());
        return LPHB_OK;
    }
    auto* h_status = ws.h_status.as<unsigned long long>();
    CK(cudaMemcpyAsync(h_status, st, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    f->stats.d2h_bytes = 4 * sizeof(unsigned long long);
    f->stats.dirty_contigs = h_status[1];
    if (h_status[1] == 0) return in_place ? LPHB_OK : fail(LPHB_E_CAPACITY, "codes buffer too small");
    uint64_t* clean = in_place ? d_codes : ws.codes.as<uint64_t>();
    const RepairWs w = reserve_repair(f, d_bases, d_offsets, b.dirty, n_contigs, span, total, in_place);
    repair_layout(f, w, d_code_offsets, clean, total, in_place, st, s);
    CK(cudaMemcpyAsync(h_status, st, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    const uint64_t new_total = h_status[0];
    *n_codes = new_total;
    f->stats.d2h_bytes += sizeof(unsigned long long);
    if (new_total > codes_capacity) return fail(LPHB_E_CAPACITY, "codes buffer too small");
    f->stats.kernel_launches += launch_repair_assemble(f->img, w, d_code_offsets, clean, in_place, d_codes, new_total, s);
    ws.mark_last(s);
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    return LPHB_OK;
}

// lphb_query_stream_exact_device_async: the exact form with nothing on the host between the stages.  The capacity
// is checked against the bound, Σ max(0, L-m+1), before anything is enqueued, so the clean pass always writes in
// place and the assemble never needs the total on the host; the scratch is sized from h_offsets alone.
int device_query_exact_async(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                             uint64_t n_contigs, uint64_t* d_codes, uint64_t codes_capacity, uint64_t* d_code_offsets,
                             unsigned long long* st, cudaStream_t s) {
    f->stats = lphb_stats{};
    const ContigCounts n = contig_layout(h_offsets, n_contigs, f->img.k, f->img.m);
    const uint64_t span = h_offsets[n_contigs] - h_offsets[0];
    if (n.mmers > codes_capacity)
        return fail(LPHB_E_CAPACITY, "codes_capacity = " + std::to_string(codes_capacity) +
                                         " is below the bound sum of max(0, L-m+1) = " + std::to_string(n.mmers));
    if ((n.kmers && !d_codes) || (span && !d_bases)) return fail(LPHB_E_ARG, "null data pointer");
    const DevBatch b = start_device_batch(f, d_bases, d_offsets, h_offsets, n_contigs, d_code_offsets, d_codes, st, true, s);
    if (n_contigs) {
        const RepairWs w = reserve_repair(f, d_bases, d_offsets, b.dirty, n_contigs, span, n.kmers, true);
        run_kernels(f, b, s);
        repair_layout(f, w, d_code_offsets, d_codes, n.kmers, true, st, s);
        f->stats.kernel_launches += launch_repair_assemble(f->img, w, d_code_offsets, d_codes, true, d_codes, n.mmers, s);
    }
    f->ws.mark_last(s);
    CK(cudaGetLastError());
    return LPHB_OK;
}

// ---- lookup of packed k-mers ---------------------------------------------------------------------

// the lookup kernel, bracketed by the handle's events like a query's main kernel
void lookup_launch(lphb_mphf* f, const void* d_kmers, uint64_t n, uint64_t* d_codes, cudaStream_t s) {
    timed_launch(f, s, [&] { launch_lookup_kmers(f->img, d_kmers, n, d_codes, s); });
    f->stats.kernel_launches += 1;
}

// lphb_lookup_kmers, n > 0.  When the k-mers and their codes fit the small block, one copy up, the kernel and one
// copy down.  Otherwise the k-mers flow in chunks of pipeline_chunk_bases() input bytes through two streams (as in
// HostQuery::clean_pass), so that the upload of chunk j+1, the kernel of chunk j and the download of chunk j-1
// overlap; one chunk runs on the handle's stream alone.
int lookup_host(lphb_mphf* f, const void* kmers, uint64_t n, uint64_t* codes) {
    Workspace& ws = f->ws;
    const cudaStream_t s = ws.stream;
    const uint64_t kb = f->img.kmer_bits / 8, in_b = n * kb, out_b = n * 8;
    f->stats = lphb_stats{};
    f->last_dirty_n = 0;
    f->last_dirty = nullptr;
    f->stats.h2d_bytes = in_b;
    f->stats.d2h_bytes = out_b;
    const uint64_t codes_b = (out_b + 63) & ~uint64_t(63);  // [codes | k-mers]: the k-mers 16-byte aligned
    if (ws.small_round_trip(
            s, codes_b, codes_b + in_b, out_b, [&](unsigned char* h) { std::memcpy(h + codes_b, kmers, in_b); },
            [&](unsigned char* d) { lookup_launch(f, d + codes_b, n, reinterpret_cast<uint64_t*>(d), s); })) {
        std::memcpy(codes, ws.small.h.p, out_b);
        return LPHB_OK;
    }
    const uint64_t per = std::max<uint64_t>(1, pipeline_chunk_bases() / kb);  // k-mers per chunk
    const uint64_t n_chunks = n / per + (n % per != 0);
    ws.bases.reserve(in_b + 64);
    ws.codes.reserve(out_b + 64);
    ws.order_after_previous(s);
    const auto* src = static_cast<const unsigned char*>(kmers);
    for (uint64_t j = 0; j < n_chunks; ++j) {
        const cudaStream_t st = ws.chunk_stream(s, j, n_chunks);
        const uint64_t i0 = j * per, c = std::min(per, n - i0);
        unsigned char* d_in = ws.bases.as<unsigned char>() + i0 * kb;
        uint64_t* d_out = ws.codes.as<uint64_t>() + i0;
        CK(cudaMemcpyAsync(d_in, src + i0 * kb, c * kb, cudaMemcpyHostToDevice, st));
        lookup_launch(f, d_in, c, d_out, st);
        CK(cudaMemcpyAsync(codes + i0, d_out, c * 8, cudaMemcpyDeviceToHost, st));
    }
    ws.join_chunks(s, n_chunks);
    ws.mark_last(s);
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    return LPHB_OK;
}

// ---- the index self-check: sessions ----------------------------------------------------------------------------

// lphb_check_begin: the bitmap and the counters cleared on the handle's stream, ordered after the previous call.
// nkmers comes from the file header: k_check_windows needs nkmers < 2^64 - 32 (its match keys), and the bitmap's
// size is computed without wrap-around and refused with LPHB_E_NOMEM when the device cannot hold it.
int check_begin(lphb_mphf* f) {
    Workspace& ws = f->ws;
    Workspace::Check& C = ws.check;
    const cudaStream_t s = ws.stream;
    const uint64_t nkmers = f->img.nkmers;
    C.open = false;  // a failed begin leaves no session, not the previous one over a freed bitmap
    if (nkmers >= ~uint64_t(0) - 31)
        return fail(LPHB_E_ARG, "check: nkmers = " + std::to_string(nkmers) + " in the header: at most 2^64 - 33 can be checked");
    const uint64_t bitmap_bytes = (nkmers / 32 + (nkmers % 32 != 0)) * 4;
    try {
        C.bitmap.reserve(bitmap_bytes + 8);
    } catch (CudaError const& e) {
        if (e.e != cudaErrorMemoryAllocation) throw;
        cudaGetLastError();
        return fail(LPHB_E_NOMEM, "check: cannot allocate the " + std::to_string(bitmap_bytes + 8) +
                                      "-byte bitmap of nkmers = " + std::to_string(nkmers) + " on the device");
    }
    C.counters.reserve(kCheckCounters * 8);
    C.h_counters.reserve(kCheckCounters * 8);
    f->stats = lphb_stats{};
    ws.order_after_previous(s);
    CK(cudaMemsetAsync(C.bitmap.p, 0, bitmap_bytes + 8, s));
    CK(cudaMemsetAsync(C.counters.p, 0, kCheckFirstMin * 8, s));
    CK(cudaMemsetAsync(C.counters.as<unsigned long long>() + kCheckFirstMin, 0xFF, (kCheckCounters - kCheckFirstMin) * 8, s));
    ws.mark_last(s);
    CK(cudaGetLastError());
    C.kmers = C.contigs = C.host_dirty = 0;
    C.open = true;
    return LPHB_OK;
}

// lphb_check_batch_device: asynchronous on s.  The code offsets of the batch go to ws.code_off, the streaming pass
// (without caller codes) to ws.codes.
int check_batch_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                       uint64_t n_contigs, const uint64_t* d_stream_codes, cudaStream_t s) {
    Workspace& ws = f->ws;
    Workspace::Check& C = ws.check;
    f->stats = lphb_stats{};
    const uint64_t total = contig_layout(h_offsets, n_contigs, f->img.k).kmers;
    const uint64_t span = h_offsets[n_contigs] - h_offsets[0];
    if (span && !d_bases) return fail(LPHB_E_ARG, "d_bases is null");
    if (n_contigs == 0) {
        f->last_dirty_n = 0;
        f->last_dirty = nullptr;
        return LPHB_OK;
    }
    ws.code_off.reserve((n_contigs + 1) * 8);
    if (!d_stream_codes) ws.codes.reserve(total * 8 + 64);
    const DevBatch b = start_device_batch(f, d_bases, d_offsets, h_offsets, n_contigs, ws.code_off.as<uint64_t>(),
                                          ws.codes.as<uint64_t>(), ws.status.as<unsigned long long>(), !d_stream_codes, s);
    check_chunk(f, b, 0, total, d_stream_codes, C.counters.as<unsigned long long>(), s);
    ws.mark_last(s);
    CK(cudaGetLastError());
    C.kmers += total;
    C.contigs += n_contigs;
    return LPHB_OK;
}

// lphb_check_end: the missing codes, the counters to the host, the session closed
int check_end(lphb_mphf* f, lphb_check_report* r) {
    Workspace& ws = f->ws;
    Workspace::Check& C = ws.check;
    const cudaStream_t s = ws.stream;
    const uint64_t nkmers = f->img.nkmers;
    C.open = false;
    ws.order_after_previous(s);
    launch_check_missing(C.bitmap.as<uint32_t>(), nkmers, C.counters.as<unsigned long long>(), s);
    auto* h = C.h_counters.as<unsigned long long>();
    CK(cudaMemcpyAsync(h, C.counters.p, kCheckCounters * 8, cudaMemcpyDeviceToHost, s));
    ws.mark_last(s);
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    f->stats = lphb_stats{};
    f->stats.kernel_launches = 1;
    f->stats.d2h_bytes = kCheckCounters * 8;
    *r = lphb_check_report{};
    r->kmers = h[kCheckKmers];
    r->contigs = C.contigs;
    r->dirty_contigs = h[kCheckDirty] + C.host_dirty;
    r->out_of_range = h[kCheckOutOfRange];
    r->duplicates = h[kCheckDuplicates];
    r->missing = nkmers - h[kCheckHits];
    r->stream_mismatches = h[kCheckMismatches];
    r->first_out_of_range = h[kCheckFirstOutOfRange];
    r->first_mismatch = h[kCheckFirstMismatch];
    r->min_duplicate_code = h[kCheckMinDuplicate];
    r->min_missing_code = h[kCheckMinMissing];
    r->ok = r->out_of_range == 0 && r->duplicates == 0 && r->missing == 0 && r->stream_mismatches == 0;
    return LPHB_OK;
}

}  // namespace

extern "C" {

const char* lphb_last_error(void) { return last_error_slot().c_str(); }
const char* lphb_version(void) { return "lphash_b200 0.1 (sm_100a)"; }

int lphb_device_count(int* count) {
    if (!count) return fail(LPHB_E_ARG, "count is null");
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *count = 0;
        return fail(LPHB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e));
    }
    return LPHB_OK;
}

int lphb_mphf_load_memory(const void* image, uint64_t nbytes, int kmer_bits, int device,
                          lphb_mphf** out) {
    if (!image) return fail(LPHB_E_ARG, "image is null");
    return load_image(static_cast<const uint8_t*>(image), nbytes, kmer_bits, device, out);
}

int lphb_mphf_load_file(const char* path, int kmer_bits, int device, lphb_mphf** out) {
    return load_file(path, kmer_bits, device, out, false);
}
int lphb_mphf_alt_load_file(const char* path, int kmer_bits, int device, lphb_mphf** out) {
    return load_file(path, kmer_bits, device, out, true);
}
int lphb_mphf_alt_load_memory(const void* image, uint64_t nbytes, int kmer_bits, int device, lphb_mphf** out) {
    if (!image) return fail(LPHB_E_ARG, "image is null");
    return load_image(static_cast<const uint8_t*>(image), nbytes, kmer_bits, device, out, true);
}

int lphb_mphf_free(lphb_mphf* f) {
    if (!f) return LPHB_OK;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(f->device);
    cudaDeviceSynchronize();  // no call of this handle may still be in flight
    if (f->l2_window_bytes) {
        // the access-policy window points into the arena that is about to be freed
        cudaStreamAttrValue attr{};
        attr.accessPolicyWindow.num_bytes = 0;
        for (cudaStream_t t : f->l2_streams)
            if (t != f->ws.stream && t != f->ws.cs[0] && t != f->ws.cs[1])
                if (cudaStreamSetAttribute(t, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
        cudaCtxResetPersistingL2Cache();
    }
    delete f;
    if (prev >= 0) cudaSetDevice(prev);
    return LPHB_OK;
}

int lphb_mphf_info(const lphb_mphf* f, lphb_info* info) {
    if (!f || !info) return fail(LPHB_E_ARG, "null argument");
    *info = f->info;
    return LPHB_OK;
}

int lphb_mphf_stats(const lphb_mphf* cf, lphb_stats* stats) {
    if (!cf || !stats) return fail(LPHB_E_ARG, "null argument");
    auto* f = const_cast<lphb_mphf*>(cf);
    if (f->ws.ev_pending) {
        // mean device time of the main kernel over the calls made since the last stats read (at
        // most the kEvRing most recent); waits for the last of them to finish
        Workspace& ws = f->ws;
        uint64_t n = ws.ev_pending < uint64_t(Workspace::kEvRing) ? ws.ev_pending : uint64_t(Workspace::kEvRing);
        double sum = 0;
        uint64_t got = 0;
        for (uint64_t i = 0; i < n; ++i) {
            const int slot = int((ws.ev_next - 1 - i) % Workspace::kEvRing);
            float ms = 0;
            if (cudaEventSynchronize(ws.ev1[slot]) == cudaSuccess &&
                cudaEventElapsedTime(&ms, ws.ev0[slot], ws.ev1[slot]) == cudaSuccess) {
                sum += ms;
                ++got;
            } else {
                cudaGetLastError();
            }
        }
        if (got) f->stats.kernel_ms = sum / double(got);
        ws.ev_pending = 0;
    }
    *stats = f->stats;
    return LPHB_OK;
}

int lphb_mphf_device_image(const lphb_mphf* f, const void** d_image, uint64_t* nbytes) {
    if (!f || !d_image || !nbytes) return fail(LPHB_E_ARG, "null argument");
    *d_image = f->d_arena;
    *nbytes = f->arena_bytes;
    return LPHB_OK;
}

int lphb_mphf_dirty_flags(const lphb_mphf* f, const uint8_t** d_flags, uint64_t* n_contigs) {
    if (!f || !d_flags || !n_contigs) return fail(LPHB_E_ARG, "null argument");
    *d_flags = f->last_dirty ? f->last_dirty : f->ws.dirty.as<uint8_t>();
    *n_contigs = f->last_dirty_n;
    return LPHB_OK;
}

int lphb_host_alloc(void** ptr, uint64_t nbytes) {
    if (!ptr) return fail(LPHB_E_ARG, "ptr is null");
    cudaError_t e = cudaMallocHost(ptr, nbytes ? nbytes : 1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(LPHB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e));
    }
    return LPHB_OK;
}

int lphb_copy_to_host(int device, void* dst, const void* d_src, uint64_t nbytes) {
    if (nbytes && (!dst || !d_src)) return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(device);
        if (nbytes) CK(cudaMemcpy(dst, d_src, nbytes, cudaMemcpyDeviceToHost));
        return LPHB_OK;
    });
}

int lphb_host_free(void* ptr) {
    if (ptr) cudaFreeHost(ptr);
    return LPHB_OK;
}

int lphb_query_stream_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                             const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                             uint64_t codes_capacity, uint64_t* d_code_offsets, uint64_t* d_status,
                             void* stream) {
    if (!f || !d_offsets || !h_offsets || !d_code_offsets || !d_status)
        return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return device_query(f, d_bases, d_offsets, h_offsets, n_contigs, d_codes, codes_capacity, d_code_offsets,
                            reinterpret_cast<unsigned long long*>(d_status), nullptr, false, static_cast<cudaStream_t>(stream));
    });
}

int lphb_query_nonstreaming_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                                   const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                                   uint64_t codes_capacity, uint64_t* d_code_offsets, uint64_t* d_status,
                                   void* stream) {
    if (!f || !d_offsets || !h_offsets || !d_code_offsets || !d_status)
        return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return device_query(f, d_bases, d_offsets, h_offsets, n_contigs, d_codes, codes_capacity, d_code_offsets,
                            reinterpret_cast<unsigned long long*>(d_status), nullptr, true, static_cast<cudaStream_t>(stream));
    });
}

int lphb_query_stream_exact_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                                   const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                                   uint64_t codes_capacity, uint64_t* d_code_offsets, uint64_t* n_codes,
                                   void* stream) {
    if (!f || !d_offsets || !h_offsets || !d_code_offsets || !n_codes)
        return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return device_query(f, d_bases, d_offsets, h_offsets, n_contigs, d_codes, codes_capacity, d_code_offsets,
                            nullptr, n_codes, false, static_cast<cudaStream_t>(stream));
    });
}

int lphb_query_stream_exact_device_async(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                                         const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                                         uint64_t codes_capacity, uint64_t* d_code_offsets, uint64_t* d_status,
                                         void* stream) {
    if (!f || !d_offsets || !h_offsets || !d_code_offsets || !d_status)
        return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return device_query_exact_async(f, d_bases, d_offsets, h_offsets, n_contigs, d_codes, codes_capacity,
                                        d_code_offsets, reinterpret_cast<unsigned long long*>(d_status),
                                        static_cast<cudaStream_t>(stream));
    });
}

int lphb_query_stream(lphb_mphf* f, const char* bases, const uint64_t* offsets, uint64_t n_contigs,
                      uint64_t* codes, uint64_t codes_capacity, uint64_t* code_offsets,
                      uint64_t* n_codes) {
    if (!f || !offsets || !code_offsets || !n_codes) return fail(LPHB_E_ARG, "null argument");
    return query_stream_host(f, bases, offsets, n_contigs, codes, codes_capacity, code_offsets, n_codes, RunSink{});
}

int lphb_query_nonstreaming(lphb_mphf* f, const char* bases, const uint64_t* offsets, uint64_t n_contigs,
                            uint64_t* codes, uint64_t codes_capacity, uint64_t* code_offsets, uint64_t* n_codes) {
    if (!f || !offsets || !code_offsets || !n_codes) return fail(LPHB_E_ARG, "null argument");
    RunSink sink;
    sink.non_streaming = true;
    return query_stream_host(f, bases, offsets, n_contigs, codes, codes_capacity, code_offsets, n_codes, sink);
}

int lphb_query_stream_runs(lphb_mphf* f, const char* bases, const uint64_t* offsets, uint64_t n_contigs,
                           void* runs, uint64_t runs_capacity, uint64_t* n_runs, uint64_t* code_offsets,
                           uint64_t* n_codes) {
    if (!f || !offsets || !code_offsets || !n_codes || !n_runs) return fail(LPHB_E_ARG, "null argument");
    RunSink sink;
    sink.runs = runs;
    sink.capacity = runs ? runs_capacity : 0;
    sink.n_runs = n_runs;
    return query_stream_host(f, bases, offsets, n_contigs, nullptr, 0, code_offsets, n_codes, sink);
}

int lphb_check_begin(lphb_mphf* f) {
    if (!f) return fail(LPHB_E_ARG, "null handle");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return check_begin(f);
    });
}

int lphb_check_batch(lphb_mphf* f, const char* bases, const uint64_t* offsets, uint64_t n_contigs) {
    if (!f || !offsets) return fail(LPHB_E_ARG, "null argument");
    if (!f->ws.check.open) return fail(LPHB_E_ARG, "no check session open: call lphb_check_begin first");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        std::vector<uint64_t> code_offsets(n_contigs + 1);
        uint64_t n_codes = 0;
        RunSink sink;
        sink.check = true;
        HostQuery q{f, bases, offsets, n_contigs, nullptr, 0, code_offsets.data(), &n_codes, sink};
        const int rc = q.run();
        if (rc != LPHB_OK) return rc;
        f->ws.check.kmers += n_codes;
        f->ws.check.contigs += n_contigs;
        return LPHB_OK;
    });
}

int lphb_check_batch_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                            uint64_t n_contigs, const uint64_t* d_stream_codes, void* stream) {
    if (!f || !d_offsets || !h_offsets) return fail(LPHB_E_ARG, "null argument");
    if (!f->ws.check.open) return fail(LPHB_E_ARG, "no check session open: call lphb_check_begin first");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return check_batch_device(f, d_bases, d_offsets, h_offsets, n_contigs, d_stream_codes,
                                  static_cast<cudaStream_t>(stream));
    });
}

int lphb_check_end(lphb_mphf* f, lphb_check_report* report) {
    if (!f || !report) return fail(LPHB_E_ARG, "null argument");
    if (!f->ws.check.open) return fail(LPHB_E_ARG, "no check session open: call lphb_check_begin first");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return check_end(f, report);
    });
}

int lphb_lookup_kmers(lphb_mphf* f, const void* kmers, uint64_t n, uint64_t* codes) {
    if (!f) return fail(LPHB_E_ARG, "null handle");
    if (n == 0) return LPHB_OK;
    if (!kmers || !codes) return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        return lookup_host(f, kmers, n, codes);
    });
}

int lphb_lookup_kmers_device(lphb_mphf* f, const void* d_kmers, uint64_t n, uint64_t* d_codes, void* stream) {
    if (!f) return fail(LPHB_E_ARG, "null handle");
    if (n == 0) return LPHB_OK;
    if (!d_kmers || !d_codes) return fail(LPHB_E_ARG, "null argument");
    if (reinterpret_cast<uintptr_t>(d_kmers) % (f->img.kmer_bits / 8) || reinterpret_cast<uintptr_t>(d_codes) % 8)
        return fail(LPHB_E_ARG, "d_kmers must be aligned to kmer_bits / 8 bytes, d_codes to 8");
    return guarded([&]() -> int {
        DeviceGuard g(f->device);
        cudaStream_t s = static_cast<cudaStream_t>(stream);
        f->stats = lphb_stats{};
        f->last_dirty_n = 0;
        f->last_dirty = nullptr;
        f->ws.order_after_previous(s);
        lookup_launch(f, d_kmers, n, d_codes, s);
        f->ws.mark_last(s);
        CK(cudaGetLastError());
        return LPHB_OK;
    });
}

// Host side of the run-length form: the uint64_t vector the reference returns, bit for bit.  Pure
// decoding of the device's output (no hashing happens here); `threads` host threads share the runs.
int lphb_expand_runs(const void* runs, uint64_t n_runs, uint64_t* codes, uint64_t codes_capacity,
                     uint64_t* n_codes, int threads) {
    if ((n_runs && !runs) || !n_codes) return fail(LPHB_E_ARG, "null argument");
    return guarded([&]() -> int {
        const unsigned char* p = static_cast<const unsigned char*>(runs);
        if (threads < 1) threads = 1;
        if (uint64_t(threads) > n_runs / 4096 + 1) threads = int(n_runs / 4096 + 1);
        // where each thread's slice of runs starts in the output
        std::vector<uint64_t> slice_at(size_t(threads) + 1, 0);
        auto run_len = [&](uint64_t r) -> uint64_t {
            int32_t n;
            memcpy(&n, p + r * 12 + 8, 4);
            return uint64_t(n < 0 ? -int64_t(n) : int64_t(n));
        };
        for (int t = 0; t < threads; ++t) {
            uint64_t r0 = n_runs * uint64_t(t) / threads, r1 = n_runs * uint64_t(t + 1) / threads, sum = 0;
            for (uint64_t r = r0; r < r1; ++r) sum += run_len(r);
            slice_at[size_t(t) + 1] = slice_at[size_t(t)] + sum;
        }
        const uint64_t total = slice_at[size_t(threads)];
        *n_codes = total;
        if (total > codes_capacity) return fail(LPHB_E_CAPACITY, "codes buffer too small");
        if (total && !codes) return fail(LPHB_E_ARG, "codes is null");
        auto work = [&](int t) {
            uint64_t at = slice_at[size_t(t)];
            const uint64_t r0 = n_runs * uint64_t(t) / threads, r1 = n_runs * uint64_t(t + 1) / threads;
            for (uint64_t r = r0; r < r1; ++r) {
                uint64_t first;
                int32_t n;
                memcpy(&first, p + r * 12, 8);
                memcpy(&n, p + r * 12 + 8, 4);
                if (n >= 0) {
                    for (int32_t j = 0; j < n; ++j) codes[at + uint64_t(j)] = first + uint64_t(j);
                    at += uint64_t(n);
                } else {
                    for (int32_t j = 0; j < -n; ++j) codes[at + uint64_t(j)] = first - uint64_t(j);
                    at += uint64_t(-int64_t(n));
                }
            }
        };
        if (threads == 1) {
            work(0);
        } else {
            std::vector<std::thread> pool;
            for (int t = 0; t < threads; ++t) pool.emplace_back(work, t);
            for (auto& th : pool) th.join();
        }
        return LPHB_OK;
    });
}

}  // extern "C"
