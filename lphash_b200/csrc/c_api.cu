// C ABI of lphash_b200 (include/lphash_b200.h): handle management, host<->device staging and
// kernel sequencing.  No CPU implementation of the path exists here: without a CUDA device every
// computing entry point fails with LPHB_E_CUDA.
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>
#include <fstream>
#include <new>
#include <algorithm>
#include <chrono>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/lphash_b200.h"
#include "api_internal.h"
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
    // repair of contigs with non-ACGT bytes
    struct Repair {
        DevBuf contigs, starts;                          // the contigs, where each starts in `bases`
        DevBuf bases, flag, run_off, run_first, status;  // their bytes gathered, cut into maximal runs
        DevBuf tmp;                                      // scan scratch
        DevBuf run_code_off, run_dirty, run_codes, tile;  // the runs through the query kernel
        DevBuf spur, spur_count, out_off, out;           // the runs' final codes
        DevBuf out_at, counts;                           // per contig: where its codes are in `out`, how many
        DevBuf src_off, assembled;                       // the batch's codes in their final layout
    } repair;
    // chunk pipeline of lphb_query_stream: two extra streams so that the H2D copy of chunk j+1,
    // the kernels of chunk j and the D2H copy of chunk j-1 overlap (PCIe is full duplex)
    Stream cs[2];
    Event ev_ready, ev_done[2];
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
    void ensure_pipeline() {
        for (int i = 0; i < 2; ++i) {
            cs[i].create();
            ev_done[i].create(cudaEventDisableTiming);
        }
        ev_ready.create(cudaEventDisableTiming);
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

void run_kernels(lphb_mphf* f, DevBatch const& b, cudaStream_t s) {
    attach_l2_window(f, s);
    const int slot = int(f->ws.ev_next % Workspace::kEvRing);
    CK(cudaEventRecord(f->ws.ev0[slot], s));
    // A batch of a few tiles would leave one or two warps of the tiled kernel to walk its whole (cold) code alone,
    // about 40 us whatever the size; below 256 K bases the one-thread-per-k-mer kernel answers sooner (10 us for a
    // record of 8,000 bases; tools/ubench/call_latency.cpp).  LPHB_GENERIC_BELOW overrides (tests: 0).
    const char* gb = getenv("LPHB_GENERIC_BELOW");
    const uint64_t generic_below = gb ? strtoull(gb, nullptr, 10) : (uint64_t(1) << 18);
    if (b.end_base - b.first_base < generic_below || !launch_query_tiled(f->img, b, s)) launch_query_generic(f->img, b, s);
    CK(cudaEventRecord(f->ws.ev1[slot], s));
    ++f->ws.ev_next;
    ++f->ws.ev_pending;
    launch_count_dirty(b.dirty, b.n_contigs, b.status, s);
    f->stats.kernel_launches += 2;
}

// Layout of a batch of contigs (host offsets): max(0, L-k+1) k-mers per contig and, with m, max(0, L-m+1) m-mers.
// With code_offsets, writes where each contig's codes start (n_contigs + 1 entries).  Offsets that decrease are
// an argument error (thrown; guarded() reports it as LPHB_E_ARG).
struct ContigCounts {
    uint64_t kmers = 0, mmers = 0;
};
ContigCounts contig_layout(const uint64_t* offsets, uint64_t n_contigs, uint32_t k, uint32_t m = 0,
                           uint64_t* code_offsets = nullptr) {
    ContigCounts n;
    for (uint64_t c = 0; c < n_contigs; ++c) {
        if (offsets[c + 1] < offsets[c]) throw std::invalid_argument("offsets must be non-decreasing");
        const uint64_t len = offsets[c + 1] - offsets[c];
        if (code_offsets) code_offsets[c] = n.kmers;
        n.kmers += len >= k ? len - k + 1 : 0;
        if (m) n.mmers += len >= m ? len - m + 1 : 0;
    }
    if (code_offsets) code_offsets[n_contigs] = n.kmers;
    return n;
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
};

// One call of lphb_query_stream, lphb_query_nonstreaming or lphb_query_stream_runs with its batch on the host.
// Stages: the layout (run), then either the small-batch block (small_call) or the clean pass (clean_pass); when
// a contig holds a non-ACGT byte, the repair of such contigs (repair); the output (output).
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
    bool copied_out = false;  // the clean pass copied every chunk's results out
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
        if (n_dirty == 0) return copied_out ? finish(total, n_chunks, 0) : output(ws.codes.as<uint64_t>(), total, 0);
        uint64_t new_total = 0, d2h_repair = 0;
        const int rc = repair(&new_total, &d2h_repair);
        if (rc != LPHB_OK) return rc;
        return output(ws.repair.assembled.as<uint64_t>(), new_total, d2h_repair);
    }

    // ---- small batch (the reference's own loop hands over one record per call, src/query.cpp:48-56): one device
    // block [codes | status | dirty flags | offsets | code offsets | bases] with a pinned mirror - one copy up (status
    // and flags arrive zeroed with it), the kernels, one copy down [codes | status].  Returns false when the batch
    // does not qualify, or when a contig holds a non-ACGT byte: the call then starts over on the general path.
    bool small_call() {
        const uint64_t codes_b = (total * 8 + 63) & ~uint64_t(63), dirty_b = (n_contigs + 8 + 63) & ~uint64_t(63);
        const uint64_t off_b = (n_contigs + 1) * 8;
        const uint64_t in_b = 64 + dirty_b + 2 * off_b + span + 64, all_b = codes_b + in_b;
        if (want_runs || !codes || !total || total > codes_capacity || all_b > Workspace::Small::kBytes ||
            getenv("LPHB_NO_SMALL_PATH"))
            return false;
        ws.small.d.reserve(Workspace::Small::kBytes);
        ws.small.h.reserve(Workspace::Small::kBytes);
        auto* h = ws.small.h.as<unsigned char>();
        auto* d = ws.small.d.as<unsigned char>();
        const uint64_t at_status = codes_b, at_dirty = at_status + 64, at_off = at_dirty + dirty_b,
                       at_coff = at_off + off_b, at_bases = at_coff + off_b;
        std::memset(h + at_status, 0, 64 + dirty_b);
        std::memcpy(h + at_off, offsets, off_b);
        std::memcpy(h + at_coff, code_offsets, off_b);
        if (span) std::memcpy(h + at_bases, bases + first, span);
        std::memset(h + at_bases + span, 'A', 64);
        ws.order_after_previous(s);
        CK(cudaMemcpyAsync(d + at_status, h + at_status, in_b, cudaMemcpyHostToDevice, s));
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
        ws.mark_last(s);
        CK(cudaMemcpyAsync(h, d, codes_b + 64, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        const auto* st = reinterpret_cast<const unsigned long long*>(h + at_status);
        f->last_dirty_n = n_contigs;
        f->last_dirty = d + at_dirty;
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
        copied_out = cuts.size() > 2 && (want_runs ? sink.runs != nullptr : (total <= codes_capacity && codes));
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
        if (copied_out) {
            ws.ensure_pipeline();
            CK(cudaEventRecord(ws.ev_ready, s));
        }
        for (uint64_t j = 0; j < n_chunks; ++j) {
            const cudaStream_t st = copied_out ? cudaStream_t(ws.cs[j & 1]) : s;
            if (copied_out && j < 2) CK(cudaStreamWaitEvent(st, ws.ev_ready, 0));
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
            run_kernels(f, b, st);
            if (copied_out) {
                emit(j, j & 1, ws.codes.as<uint64_t>(), code_offsets[c0], code_offsets[c1], b.code_off, b.n_contigs, st);
                // the previous chunk's records leave while this chunk computes
                if (want_runs && j >= 1) fetch_runs(j - 1, code_offsets[cuts[j - 1]], ws.cs[(j - 1) & 1]);
            }
        }
        if (copied_out) {
            if (want_runs) fetch_runs(n_chunks - 1, code_offsets[cuts[n_chunks - 1]], ws.cs[(n_chunks - 1) & 1]);
            for (int i = 0; i < 2; ++i) {
                CK(cudaEventRecord(ws.ev_done[i], ws.cs[i]));
                CK(cudaStreamWaitEvent(s, ws.ev_done[i], 0));
            }
        }
        auto* h_status = ws.h_status.as<unsigned long long>();
        CK(cudaMemcpyAsync(h_status, ws.status.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        f->stats.dirty_contigs = h_status[1];
        return h_status[1];
    }

    // ---- contigs with non-ACGT bytes (SURVEY.md Q1; quirk_kernels.cu) ----------------------------------------
    // Their valid k-mers are ordinary work: the contigs are gathered into a compact batch, cut into maximal runs of
    // valid / invalid bytes, and the runs go through the same query kernel as contigs of their own.  Only the
    // reference's spurious codes (pushed while a run is shorter than k) need the sequential state machine, one
    // thread per episode of a few dozen bases.  Leaves the batch's codes in ws.repair.assembled, their layout in
    // code_offsets and ws.code_off; *d2h_bytes = what it copied to the host.
    int repair(uint64_t* new_total_out, uint64_t* d2h_bytes) {
        Workspace::Repair& R = ws.repair;
        const uint32_t k = f->img.k, w_cap = f->img.w;
        std::vector<uint8_t> dirty(n_contigs);
        CK(cudaMemcpy(dirty.data(), ws.dirty.p, n_contigs, cudaMemcpyDeviceToHost));
        std::vector<uint64_t> list, starts;
        uint64_t q_bytes = 0;
        for (uint64_t c = 0; c < n_contigs; ++c)
            if (dirty[c]) {
                list.push_back(c);
                starts.push_back(q_bytes);
                q_bytes += offsets[c + 1] - offsets[c];
            }
        starts.push_back(q_bytes);
        const uint64_t n_list = list.size();
        R.contigs.reserve(n_list * 8);
        R.starts.reserve((n_list + 1) * 8);
        R.out_at.reserve(n_list * 8);
        R.counts.reserve(n_list * 8);
        R.bases.reserve(q_bytes + 64);
        R.flag.reserve(q_bytes + 8);
        R.run_off.reserve((q_bytes + 2) * 8);
        R.run_first.reserve((n_list + 2) * 4);
        R.status.reserve(64);
        R.tmp.reserve(std::max<uint64_t>(quirk_tmp_bytes(q_bytes + 1), code_offsets_tmp_bytes(q_bytes + 1)));
        CK(cudaMemcpyAsync(R.contigs.p, list.data(), n_list * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(R.starts.p, starts.data(), (n_list + 1) * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemsetAsync(R.bases.as<char>() + q_bytes, 'A', 64, s));  // read-ahead of the last tile
        launch_gather_contigs(ws.bases.as<char>() - first, ws.offsets.as<uint64_t>(), R.contigs.as<uint64_t>(),
                              R.starts.as<uint64_t>(), n_list, q_bytes, R.bases.as<char>(), s);
        auto* qst = R.status.as<unsigned long long>();
        launch_find_runs(R.bases.as<char>(), q_bytes, R.starts.as<uint64_t>(), n_list, R.flag.as<uint8_t>(),
                         R.run_off.as<uint64_t>(), qst + 4, R.run_first.as<uint32_t>(), R.tmp.p, R.tmp.cap, s);
        unsigned long long n_v = 0;
        CK(cudaMemcpyAsync(&n_v, qst + 4, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        f->stats.kernel_launches += 7;
        // the runs as a batch of their own: valid k-mers of every run, clean layout per run
        R.run_code_off.reserve((n_v + 2) * 8);
        R.run_dirty.reserve(n_v + 8);
        R.run_codes.reserve(q_bytes * 8 + 64);
        R.tile.reserve(query_tiled_ws_bytes(q_bytes));
        CK(cudaMemsetAsync(R.run_dirty.p, 0, n_v + 8, s));
        launch_code_offsets(R.run_off.as<uint64_t>(), n_v, k, R.run_code_off.as<uint64_t>(), qst, R.tmp.p, R.tmp.cap, s);
        DevBatch bq{};
        bq.bases = R.bases.as<char>();
        bq.offsets = R.run_off.as<uint64_t>();
        bq.code_off = R.run_code_off.as<uint64_t>();
        bq.n_contigs = n_v;
        bq.first_base = 0;
        bq.end_base = q_bytes;
        bq.codes = R.run_codes.as<uint64_t>();
        bq.dirty = R.run_dirty.as<uint8_t>();
        bq.status = qst;
        bq.tile_ws = R.tile.p;
        bq.tile_ws_bytes = R.tile.cap;
        if (!launch_query_tiled(f->img, bq, s)) launch_query_generic(f->img, bq, s);
        f->stats.kernel_launches += 3;
        R.spur.reserve((n_v + 1) * uint64_t(w_cap) * 8);
        R.spur_count.reserve((n_v + 2) * 4);
        R.out_off.reserve((n_v + 2) * 8);
        R.out.reserve((q_bytes + n_v * uint64_t(w_cap)) * 8 + 64);
        launch_quirk_finish(f->img, R.bases.as<char>(), R.run_off.as<uint64_t>(), n_v, qst + 4, R.run_first.as<uint32_t>(),
                            n_list, R.run_code_off.as<uint64_t>(), R.run_codes.as<uint64_t>(), R.spur.as<uint64_t>(),
                            R.spur_count.as<uint32_t>(), w_cap, R.out_off.as<uint64_t>(), R.out.as<uint64_t>(),
                            R.out_at.as<uint64_t>(), R.counts.as<uint64_t>(), R.tmp.p, R.tmp.cap, s);
        launch_quirk_emit(R.run_code_off.as<uint64_t>(), R.run_codes.as<uint64_t>(), R.spur.as<uint64_t>(),
                          R.spur_count.as<uint32_t>(), w_cap, n_v, qst + 4, R.out_off.as<uint64_t>(), q_bytes,
                          R.out.as<uint64_t>(), s);
        f->stats.kernel_launches += 6;
        std::vector<uint64_t> counts(n_list), out_at(n_list);
        CK(cudaMemcpyAsync(out_at.data(), R.out_at.p, n_list * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(counts.data(), R.counts.p, n_list * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        // final layout + where each contig's codes come from (clean layout or the repaired runs)
        std::vector<uint64_t> src_off(n_contigs);
        uint64_t new_total = 0, clean_run = 0;
        for (uint64_t c = 0, j = 0; c < n_contigs; ++c) {
            uint64_t len = offsets[c + 1] - offsets[c];
            uint64_t clean_cnt = len >= k ? len - k + 1 : 0;
            uint64_t cnt = clean_cnt;
            if (dirty[c]) {
                src_off[c] = out_at[j];
                cnt = counts[j++];
            } else {
                src_off[c] = clean_run;
            }
            clean_run += clean_cnt;
            code_offsets[c] = new_total;
            new_total += cnt;
        }
        code_offsets[n_contigs] = new_total;
        *n_codes = new_total;
        if (!want_runs && new_total > codes_capacity) return fail(LPHB_E_CAPACITY, "codes buffer too small");
        if (want_runs && new_total >= (1ull << 31)) return fail(LPHB_E_ARG, "batch holds >= 2^31 codes: split it");
        R.src_off.reserve((n_contigs + 1) * 8);
        R.assembled.reserve(new_total * 8 + 64);
        CK(cudaMemcpyAsync(R.src_off.p, src_off.data(), n_contigs * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(ws.code_off.p, code_offsets, (n_contigs + 1) * 8, cudaMemcpyHostToDevice, s));
        launch_assemble(R.assembled.as<uint64_t>(), ws.code_off.as<uint64_t>(), ws.codes.as<uint64_t>(), R.out.as<uint64_t>(),
                        R.src_off.as<uint64_t>(), ws.dirty.as<uint8_t>(), n_contigs, new_total, s);
        f->stats.kernel_launches += 1;
        if (want_runs) reserve_runs(new_total + 16, 1, new_total, 1);
        *new_total_out = new_total;
        *d2h_bytes = n_contigs + n_list * 8;
        return LPHB_OK;
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

// ---- build-side scan ---------------------------------------------------------------------------

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
    if (m == 0 || m > 31 || k < m || k > 63) throw std::invalid_argument("need 1 <= m <= 31, m <= k <= 63");
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
    DevBuf rec, key, key2, idx, idx2, flags, gslot, cslot, counts, tmp, trip, idu, ids_s;
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
    DevBuf &key = cs.key, &key2 = cs.key2, &idx = cs.idx, &idx2 = cs.idx2, &flags = cs.flags, &gslot = cs.gslot,
           &cslot = cs.cslot, &counts = cs.counts, &tmp = cs.tmp, &trip = cs.trip, &idu = cs.idu, &ids_s = cs.ids_s;
    key.reserve(n * 8);
    key2.reserve(n * 8);
    idx.reserve(n * 4);
    idx2.reserve(n * 4);
    flags.reserve(n + 8);
    gslot.reserve(n * 4);
    cslot.reserve(n * 4);
    counts.reserve(64);
    const uint64_t tb = classify_tmp_bytes(n);
    tmp.reserve(tb);
    launch_classify_groups(d_rec, n, key.as<uint64_t>(), key2.as<uint64_t>(), idx.as<uint32_t>(),
                           idx2.as<uint32_t>(), flags.as<uint8_t>(), gslot.as<uint32_t>(), cslot.as<uint32_t>(),
                           counts.as<unsigned long long>(), tmp.p, tb, key_bits, s);
    unsigned long long h_counts[2] = {0, 0};
    CK(cudaMemcpyAsync(h_counts, counts.p, sizeof(h_counts), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    *n_triplets = h_counts[0];
    *n_ids = h_counts[1];
    if (h_counts[0] > triplets_capacity) return fail(LPHB_E_CAPACITY, "triplets buffer too small");
    if (h_counts[1] > ids_capacity) return fail(LPHB_E_CAPACITY, "ids buffer too small");
    if (!triplets || (h_counts[1] && !ids)) return fail(LPHB_E_ARG, "null output buffer");
    trip.reserve(h_counts[0] * 10 + 64);
    idu.reserve(h_counts[1] * 8 + 64);
    ids_s.reserve(h_counts[1] * 8 + 64);
    launch_classify_emit(d_rec, key2.as<uint64_t>(), idx2.as<uint32_t>(), flags.as<uint8_t>(),
                         gslot.as<uint32_t>(), cslot.as<uint32_t>(), n, trip.as<uint8_t>(), idu.as<uint64_t>(),
                         ids_s.as<uint64_t>(), h_counts[1], tmp.p, tb, s);
    CK(cudaMemcpyAsync(triplets, trip.p, h_counts[0] * 10, cudaMemcpyDeviceToHost, s));
    if (h_counts[1]) CK(cudaMemcpyAsync(ids, ids_s.p, h_counts[1] * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
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
        cudaStream_t s = static_cast<cudaStream_t>(stream);
        f->stats = lphb_stats{};
        const uint32_t k = f->img.k;
        const uint64_t total = contig_layout(h_offsets, n_contigs, k).kmers;
        if (total > codes_capacity) return fail(LPHB_E_CAPACITY, "codes buffer too small");
        if (total && (!d_bases || !d_codes)) return fail(LPHB_E_ARG, "null data pointer");
        Workspace& ws = f->ws;
        // (growing a workspace buffer frees the old one: cudaFree waits for the device, so a previous
        // call still running never loses its buffer)
        ws.offsets_tmp.reserve(code_offsets_tmp_bytes(n_contigs));
        ws.dirty.reserve(n_contigs + 8);
        ws.tile.reserve(query_tiled_ws_bytes(h_offsets[n_contigs] - h_offsets[0]));
        ws.order_after_previous(s);
        CK(cudaMemsetAsync(ws.dirty.p, 0, n_contigs + 8, s));
        auto* st = reinterpret_cast<unsigned long long*>(d_status);
        launch_code_offsets(d_offsets, n_contigs, k, d_code_offsets, st, ws.offsets_tmp.p, ws.offsets_tmp.cap, s);
        f->stats.kernel_launches += 2;
        DevBatch b{};
        b.bases = d_bases;
        b.offsets = d_offsets;
        b.code_off = d_code_offsets;
        b.n_contigs = n_contigs;
        b.first_base = h_offsets[0];
        b.end_base = h_offsets[n_contigs];
        b.codes = d_codes;
        b.dirty = ws.dirty.as<uint8_t>();
        b.status = st;
        b.tile_ws = ws.tile.p;
        b.tile_ws_bytes = ws.tile.cap;
        if (n_contigs) run_kernels(f, b, s);
        ws.mark_last(s);
        f->last_dirty_n = n_contigs;
        CK(cudaGetLastError());
        return LPHB_OK;
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
