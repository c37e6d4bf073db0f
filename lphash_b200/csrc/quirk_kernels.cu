// Contigs with non-ACGT bytes, run-parallel (SURVEY.md Q1).
//
// The reference's streaming loop (include/partitioned_mphf.hpp:103-184) resets only its base counter
// and ring cursor at an invalid byte; the ring, the minimum's slot, and the rolling registers stay.
// What follows from the code:
//   (i)  inside a maximal ACGT run, every k-mer window gets exactly its stateless code (the first full
//        window rescans w fresh slots) - so the VALID codes of a dirty contig are the clean pass's codes
//        of those windows;
//   (ii) the only state-dependent outputs are the SPURIOUS codes pushed while m <= run < k, when the
//        cursor meets the stale minimum slot (:117-118, :146-171).  They depend on the state the
//        previous runs left, and that state is fully rewritten by any run of >= k bases (w fresh slots,
//        slot = m-mer index mod w, minimum = leftmost minimum of the last window).
// Hence one thread per EPISODE - the end of a run of >= k bases, the shorter runs after it, and the first k-1
// bases of the next long run - replays just those bases through the line-exact state machine (QuirkState
// below, the same code the one-thread-per-contig kernel of round 1 ran over whole contigs) to get the
// spurious codes, and the final sequence of a dirty contig is, byte by byte, the code pushed at that byte.
// An episode walks its bytes one by one only inside a chunk of 1024 bytes: a stretch of non-ACGT bytes counts as one
// (the state machine's reset is idempotent) and is crossed with per-chunk summaries, so a record with one N in
// 5 Mbases costs a few dozen sequential bases and a gap of 20 Mbases a few hundred steps, not millions.
#include <algorithm>

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "device_mphf.cuh"
#include "query_kernels.cuh"

namespace lphb {

namespace {

// ---- line-exact restatement of the streaming loop's state ------------------------------------------
// ref: include/partitioned_mphf.hpp:73-184.  feed() is one iteration of its `for` loop for a valid
// base, invalid() its else-branch.  `push` is called with every code the reference pushes.
struct QuirkState {
    uint32_t k, m, w;
    uint64_t mm_mask, lo_mask, hi_mask;
    uint64_t ring_mm[64], ring_h[64];
    uint32_t cursor, min_slot, p1;
    uint64_t mmer, lo, hi, run;
    uint64_t g_rank, l_rank;  // last probe context (mm_context_t, partitioned_mphf.hpp:55-60)
    int32_t ctx_slope;        // slope of the last probe (0: colliding minimizer)

    __device__ void init(DevImage const& f) {
        k = f.k;
        m = f.m;
        w = f.w;
        mm_mask = (uint64_t(1) << (2 * m)) - 1;
        lo_mask = k >= 32 ? ~uint64_t(0) : ((uint64_t(1) << (2 * k)) - 1);
        hi_mask = k > 32 ? ((uint64_t(1) << (2 * k - 64)) - 1) : 0;
        for (uint32_t q = 0; q < w; ++q) ring_mm[q] = 0, ring_h[q] = 0;
        cursor = 0;
        min_slot = w;
        p1 = 0;
        mmer = lo = hi = run = 0;
        g_rank = l_rank = 0;
        ctx_slope = 1;
    }
    __device__ void invalid() {  // :179-183
        run = 0;
        cursor = 0;
    }
    // kProbe = false: only the state is advanced (codes are not wanted: no image access at all)
    template <bool kProbe, class Push>
    __device__ void feed(DevImage const& f, uint32_t code, Push&& push) {
        mmer = ((mmer << 2) | code) & mm_mask;
        hi = ((hi << 2) | (lo >> 62)) & hi_mask;
        lo = ((lo << 2) | code) & lo_mask;
        ++run;
        if (run < m) return;
        int action = 0;  // 0 keep, 1 rescan, 2 newcomer
        if (cursor == min_slot) action = 1;
        ring_mm[cursor] = mmer;
        ring_h[cursor] = murmur64(mmer, f.mm_seed);
        if (run == k) {
            action = 1;
        } else if (run > k && ring_h[min_slot] > ring_h[cursor]) {
            p1 = k - m;
            min_slot = cursor;
            action = 2;
        }
        if (action == 0) {
            if (run >= k) {
                if (kProbe) {
                    if (ctx_slope == 0) l_rank = fallback_order(f, lo, hi);
                    else if (ctx_slope < 0) ++l_rank;  // RIGHT, NONE
                    else --l_rank;                     // LEFT, MAXIMAL
                    push(g_rank + l_rank);
                }
            }
        } else {
            if (action == 1) {
                min_slot = (cursor + 1) % w;
                p1 = 0;
                uint32_t step = 1;
                for (uint32_t q = (cursor + 2) % w; q < w; ++q, ++step)
                    if (ring_h[min_slot] > ring_h[q]) { min_slot = q; p1 = step; }
                for (uint32_t q = 0; q <= (cursor + 2) % w; ++q, ++step)
                    if (ring_h[min_slot] > ring_h[q]) { min_slot = q; p1 = step; }
            }
            if (kProbe) {
                Probe pr = probe_minimizer(f, ring_mm[min_slot]);
                ctx_slope = pr.slope;
                // split hval back into the reference's (global_rank, local_rank) so that the
                // +-1 continuation above reproduces :131-145 (mod 2^64)
                if (pr.slope == 0) { g_rank = pr.base; l_rank = fallback_order(f, lo, hi); }
                else if (pr.slope > 0) { g_rank = pr.base; l_rank = p1; }
                else { g_rank = pr.base; l_rank = uint64_t(0) - uint64_t(p1); }
                push(g_rank + l_rank);
            }
        }
        cursor = (cursor + 1) % w;
    }
};

// flag[p] = 1 where a run (of valid or of invalid bytes) or a contig begins
__global__ void k_run_boundaries(const char* bases, uint64_t n, uint8_t* flag) {
    for (uint64_t p = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < n; p += uint64_t(gridDim.x) * blockDim.x) {
        if (p == 0) { flag[p] = 1; continue; }
        const bool a = nt4(uint8_t(bases[p - 1])) < 4, b = nt4(uint8_t(bases[p])) < 4;
        if (a != b) flag[p] = 1;  // (contig starts were set before: the array is zeroed, then marked)
    }
}
__global__ void k_mark_starts(const uint64_t* starts, uint64_t n_list, uint64_t n, uint8_t* flag) {
    uint64_t j = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (j < n_list && starts[j] < n) flag[starts[j]] = 1;
}
__global__ void k_close_offsets(uint64_t* voff, const unsigned long long* n_v, uint64_t n) { voff[*n_v] = n; }

// first run (virtual contig) of every dirty contig: its start is a boundary, so the search is exact
__global__ void k_first_run(const uint64_t* voff, const unsigned long long* n_v_p, const uint64_t* starts, uint64_t n_list,
                            uint64_t n, uint32_t* vstart) {
    const uint64_t n_v = *n_v_p;
    uint64_t j = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (j > n_list) return;
    const uint64_t target = j < n_list ? starts[j] : n;
    uint64_t lo = 0, hi = n_v;  // first v with voff[v] >= target
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (voff[mid] < target) lo = mid + 1; else hi = mid;
    }
    vstart[j] = uint32_t(lo);
}

// ---- build side: minimizer::from_string over contigs with non-ACGT bytes (include/minimizer.hpp:138-151) ----
// An invalid byte flushes the open super-k-mer and restarts the window, so every maximal valid run is scanned like
// a contig of its own, with two exceptions the reference's loop has: m-mer ordinals (`id`) advance over valid runs
// only, and a run of exactly k bases that is FOLLOWED by an invalid byte counts its k-mer but never emits it (the
// first window is only searched when base k+1 arrives or the contig ends, minimizer.hpp:59-74, 153-162).  The scan
// kernels take a partition of the stream into contigs; the partition handed to them cuts invalid runs and those
// swallowed runs into pieces shorter than k, which hold no k-mer.
__global__ void k_shift_starts(const uint64_t* offsets, uint64_t n_contigs, uint64_t first, uint64_t* starts) {
    const uint64_t c = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (c <= n_contigs) starts[c] = offsets[c] - first;
}
__global__ void k_build_run_counts(const char* bases, const uint64_t* voff, const unsigned long long* n_v_p,
                                   const uint32_t* vstart, uint64_t n_list, uint32_t k, uint32_t m, uint64_t* pieces,
                                   uint64_t* ids, uint64_t* kmers) {
    const uint64_t n_v = *n_v_p;
    const uint64_t r = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (r > n_v) return;
    if (r == n_v) {
        pieces[r] = ids[r] = kmers[r] = 0;
        return;
    }
    const uint64_t L = voff[r + 1] - voff[r];
    const bool valid = nt4(uint8_t(bases[voff[r]])) < 4;
    bool swallowed = false;
    if (valid && L == k) {  // followed by an invalid byte of the same contig?
        uint64_t lo = 0, hi = n_list;  // first j with vstart[j] >= r + 1 (vstart[n_list] = n_v)
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (vstart[mid] < r + 1) lo = mid + 1; else hi = mid;
        }
        swallowed = vstart[lo] != r + 1;
    }
    const uint64_t step = k - 1;
    pieces[r] = (valid && !swallowed) ? 1 : (L + step - 1) / step;
    ids[r] = valid && L >= m ? L - m + 1 : 0;
    kmers[r] = valid && L >= k ? L - k + 1 : 0;
}
__global__ void k_build_pieces(const uint64_t* voff, const unsigned long long* n_v_p, uint32_t k, const uint64_t* pieces,
                               const uint64_t* ids, uint64_t mm_count_in, uint64_t n, uint64_t* poff, uint64_t* pid) {
    const uint64_t n_v = *n_v_p;
    const uint64_t r = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (r > n_v) return;
    if (r == n_v) {
        poff[pieces[r]] = n;
        pid[pieces[r]] = mm_count_in + ids[r];
        return;
    }
    const uint64_t first = pieces[r], cnt = pieces[r + 1] - first, step = k - 1;
    for (uint64_t i = 0; i < cnt; ++i) {
        poff[first + i] = voff[r] + i * step;
        pid[first + i] = mm_count_in + ids[r] + i * step;  // only read for single-piece (scanned) runs
    }
}


// ---- the query side's repair, on the device -------------------------------------------------------------------
// Every byte of a dirty contig pushes at most one code, and the reference pushes them in byte order: at byte p a
// VALID code when the k bytes ending at p are ACGT (the window's code is the clean pass's), or a SPURIOUS one (the
// state machine, when the run at p is shorter than k).  So a chunk of a dirty contig yields the pushes of its bytes,
// its codes go after those of the contig's earlier chunks, and the final layout is two exclusive scans: over the
// chunks, then over the contigs.  Spurious codes come from episodes (see above), replayed one thread per episode by
// k_rep_episodes into a flag and a code slot per byte.  Counts live in RepairCounters; grids are sized from the host
// bounds and every block loops over what the counters say, so a clean batch costs a dozen empty launches.

constexpr uint32_t kRepLook = 64;                        // bytes before a chunk its windows reach (k <= 63)
constexpr uint32_t kRepMask = kRepairChunk + kRepLook;   // bytes of a chunk's mask
constexpr int kRepThreads = 256;                         // kRepairChunk / 4: 4 consecutive bytes per thread
constexpr uint16_t kRepNone = 0xFFFF;                    // a chunk summary's "no such byte"

struct ChunkAt {
    uint64_t c, j;      // contig, list entry
    uint64_t a, b;      // bytes [a, b) of the contig
    uint64_t len, d;    // the contig's length, its first scratch slot
    uint64_t start;     // where the contig starts in `bases`
};
__device__ __forceinline__ ChunkAt chunk_at(RepairWs const& w, uint64_t ch) {
    ChunkAt r;
    r.j = w.chunk_tab[ch];
    r.c = w.list[3 * r.j];
    r.d = w.list[3 * r.j + 1];
    r.start = w.offsets[r.c];
    r.len = w.offsets[r.c + 1] - r.start;
    r.a = (ch - w.list[3 * r.j + 2]) * kRepairChunk;
    r.b = min(r.a + kRepairChunk, r.len);
    return r;
}
__device__ __forceinline__ bool acgt(const char* bases, uint64_t i) { return nt4(uint8_t(bases[i])) < 4; }

// the dirty contigs listed, each given its scratch slots and chunks (warp-aggregated atomics: the list is in no
// particular order; everything downstream is keyed by contig)
__global__ void __launch_bounds__(256) k_rep_list(const __grid_constant__ RepairWs w) {
    const uint64_t n = w.n_contigs;
    const int lane = threadIdx.x & 31;
    const uint64_t warps = uint64_t(gridDim.x) * (blockDim.x / 32);
    for (uint64_t base = (uint64_t(blockIdx.x) * (blockDim.x / 32) + threadIdx.x / 32) * 32; base < n; base += warps * 32) {
        const uint64_t c = base + lane;
        const bool is = c < n && w.dirty[c];
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, is);
        if (!bal) continue;
        uint64_t len = 0, nch = 0;
        if (is) {
            len = w.offsets[c + 1] - w.offsets[c];
            nch = (len + kRepairChunk - 1) / kRepairChunk;
        }
        uint64_t sl = len, sn = nch;  // inclusive sums over the warp
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t x = __shfl_up_sync(0xFFFFFFFFu, sl, o), y = __shfl_up_sync(0xFFFFFFFFu, sn, o);
            if (lane >= o) sl += x, sn += y;
        }
        unsigned long long j0 = 0, d0 = 0, ch0 = 0;
        if (lane == 31) {
            j0 = atomicAdd(&w.ctr->n_list, (unsigned long long)__popc(bal));
            d0 = atomicAdd(&w.ctr->bytes, (unsigned long long)sl);
            ch0 = atomicAdd(&w.ctr->n_chunks, (unsigned long long)sn);
            atomicMax(&w.ctr->fd_rev, (unsigned long long)(n - (base + __ffs(bal) - 1)));
        }
        j0 = __shfl_sync(0xFFFFFFFFu, j0, 31);
        d0 = __shfl_sync(0xFFFFFFFFu, d0, 31);
        ch0 = __shfl_sync(0xFFFFFFFFu, ch0, 31);
        if (is) {
            const uint64_t j = j0 + __popc(bal & ((1u << lane) - 1u)), cb = ch0 + sn - nch;
            w.list[3 * j] = c;
            w.list[3 * j + 1] = d0 + sl - len;
            w.list[3 * j + 2] = cb;
            w.slot[c] = j;
            for (uint64_t i = 0; i < nch; ++i) w.chunk_tab[cb + i] = j;
        }
    }
}

// Before the final layout overwrites them: the clean code offsets of the contigs from the first dirty one on and, in
// place, their clean codes.  The copy goes in 16-byte vectors, 4 in flight per thread; the saved codes start at
// tail_codes + tail_shift(codes + c0), which has the address of codes + c0 mod 16.
__device__ __forceinline__ uint64_t tail_shift(const uint64_t* p) { return (reinterpret_cast<uintptr_t>(p) >> 3) & 1; }
__device__ __forceinline__ void save_tail(RepairWs const& w, const uint64_t* code_off, const uint64_t* codes, bool in_place) {
    const uint64_t fd_rev = w.ctr->fd_rev;
    if (!fd_rev) return;
    const uint64_t n = w.n_contigs, fd = n - fd_rev, c0 = code_off[fd], nc = in_place ? code_off[n] - c0 : 0;
    const uint64_t tid = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x, stride = uint64_t(gridDim.x) * blockDim.x;
    for (uint64_t i = tid; i <= fd_rev; i += stride) w.tail_off[i] = code_off[fd + i];
    if (!nc) return;
    const uint64_t* src = codes + c0;
    const uint64_t head = tail_shift(src);
    uint64_t* dst = w.tail_codes + head;
    if (head && tid == 0) dst[0] = src[0];
    const uint64_t n2 = (nc - head) / 2;
    const ulonglong2* s2 = reinterpret_cast<const ulonglong2*>(src + head);
    ulonglong2* d2 = reinterpret_cast<ulonglong2*>(dst + head);
    const uint64_t tile = 4 * uint64_t(blockDim.x);
    for (uint64_t t0 = blockIdx.x * tile; t0 < n2; t0 += gridDim.x * tile) {
        ulonglong2 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint64_t q = t0 + u * blockDim.x + threadIdx.x;
            if (q < n2) v[u] = __ldcs(s2 + q);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint64_t q = t0 + u * blockDim.x + threadIdx.x;
            if (q < n2) d2[q] = v[u];
        }
    }
    if ((nc - head) & 1 && tid == 0) dst[nc - 1] = src[nc - 1];
}

struct MaxOp {
    __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};
struct MinOp {
    __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a < b ? a : b; }
};
// per chunk: its spurious flags cleared, where its first ACGT byte and its last non-ACGT byte are; then save_tail
__global__ void __launch_bounds__(kRepThreads, 4) k_rep_prep(const __grid_constant__ RepairWs w, const uint64_t* code_off,
                                                          const uint64_t* codes, bool in_place) {
    using Reduce = cub::BlockReduce<uint32_t, kRepThreads>;
    __shared__ typename Reduce::TempStorage tmp;
    const uint64_t n_chunks = w.ctr->n_chunks;
    for (uint64_t ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
        const ChunkAt r = chunk_at(w, ch);
        uint32_t first = kRepNone, last = 0;  // (last: 1 + the offset)
        for (uint64_t p = r.a + threadIdx.x; p < r.b; p += blockDim.x) {
            w.spur_flag[r.d + p] = 0;
            if (acgt(w.bases, r.start + p)) first = min(first, uint32_t(p - r.a));
            else last = uint32_t(p - r.a) + 1;
        }
        first = Reduce(tmp).Reduce(first, MinOp{});
        __syncthreads();
        last = Reduce(tmp).Reduce(last, MaxOp{});
        if (threadIdx.x == 0) {
            w.chunk_first[ch] = uint16_t(first);
            w.chunk_last_inv[ch] = last ? uint16_t(last - 1) : kRepNone;
        }
        __syncthreads();
    }
    save_tail(w, code_off, codes, in_place);
}

// First i in [lo, hi) with a[i] != kRepNone (hi if none), and the last one (~0 if none): 8 entries per 16-byte load,
// 4 loads in flight, so that an episode crosses a gap of many chunks at 32 chunks (32 Kbases) per step.  Out of line:
// they run once per stretch, and inlined they would push the episode kernel's registers into spills.
__device__ __forceinline__ bool all_none(uint4 v) { return (v.x & v.y & v.z & v.w) == 0xFFFFFFFFu; }
__device__ __noinline__ uint64_t next_some(const uint16_t* a, uint64_t lo, uint64_t hi) {
    for (; lo < hi && (lo & 7); ++lo)
        if (a[lo] != kRepNone) return lo;
    for (; lo + 32 <= hi; lo += 32) {
        const uint4* v = reinterpret_cast<const uint4*>(a + lo);
        const uint4 v0 = v[0], v1 = v[1], v2 = v[2], v3 = v[3];
        if (!all_none(v0) || !all_none(v1) || !all_none(v2) || !all_none(v3)) break;
    }
    for (; lo < hi; ++lo)
        if (a[lo] != kRepNone) return lo;
    return hi;
}
__device__ __noinline__ uint64_t prev_some(const uint16_t* a, uint64_t lo, uint64_t hi) {
    while (hi > lo && (hi & 7))
        if (a[--hi] != kRepNone) return hi;
    for (; hi >= lo + 32; hi -= 32) {
        const uint4* v = reinterpret_cast<const uint4*>(a + hi - 32);
        const uint4 v0 = v[0], v1 = v[1], v2 = v[2], v3 = v[3];
        if (!all_none(v0) || !all_none(v1) || !all_none(v2) || !all_none(v3)) break;
    }
    while (hi > lo)
        if (a[--hi] != kRepNone) return hi;
    return ~uint64_t(0);
}

// One thread per episode: its head is the last byte p of a run of >= k ACGT bytes followed, in the contig, by a
// non-ACGT byte.  The state the run leaves is rebuilt from its tail (from a start a multiple of w bases into the
// run, which keeps the ring's phase, and at least k + w bases before p), then the bytes after p are fed until the
// first byte that would complete a run of k, and every code pushed there is a spurious one, stored at its byte's
// scratch slot.  The bytes are walked one by one inside a chunk; across chunks, the chunk summaries of k_rep_prep
// find the run's start and the end of a stretch of non-ACGT bytes (one invalid() stands for the whole stretch), so a
// long gap costs a few steps per 32 chunks.  (The ring lives in local memory: the 1.1 KB stack frame of this kernel.)
__global__ void __launch_bounds__(kRepThreads) k_rep_episodes(const __grid_constant__ DevImage f,
                                                              const __grid_constant__ RepairWs w) {
    const uint64_t n_chunks = w.ctr->n_chunks;
    const uint32_t k = f.k;
    for (uint64_t ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
        const ChunkAt r = chunk_at(w, ch);
        const char* s = w.bases + r.start;
        for (uint64_t p = r.a + threadIdx.x; p < r.b; p += blockDim.x) {
            if (p + 1 >= r.len || p + 1 < k || !acgt(s, p) || acgt(s, p + 1)) continue;
            // start of p's run: in this chunk, else after the last non-ACGT byte of an earlier chunk
            uint64_t run0 = r.a;
            bool found = false;
            for (uint64_t q = p; q > r.a; --q)
                if (!acgt(s, q - 1)) {
                    run0 = q;
                    found = true;
                    break;
                }
            if (!found) {
                const uint64_t cb = w.list[3 * r.j + 2];
                const uint64_t c2 = prev_some(w.chunk_last_inv, cb, ch);
                run0 = c2 == ~uint64_t(0) ? 0 : (c2 - cb) * kRepairChunk + w.chunk_last_inv[c2] + 1;
            }
            const uint64_t L = p + 1 - run0;
            if (L < k) continue;
            QuirkState st;
            st.init(f);
            auto drop = [](uint64_t) {};
            const uint64_t t0 = L > uint64_t(k + st.w) ? (L - (k + st.w)) / st.w * st.w : 0;
            for (uint64_t i = run0 + t0; i <= p; ++i) st.feed<false>(f, nt4(uint8_t(s[i])), drop);
            for (uint64_t q = p + 1; q < r.len; ++q) {
                const uint32_t code = nt4(uint8_t(s[q]));
                if (code > 3) {  // the stretch of non-ACGT bytes from q: one invalid(), then its next ACGT byte
                    st.invalid();
                    const uint64_t q_end = min((q / kRepairChunk + 1) * kRepairChunk, r.len);
                    uint64_t x = q + 1;
                    while (x < q_end && !acgt(s, x)) ++x;
                    if (x == q_end && x < r.len) {
                        const uint64_t cb = w.list[3 * r.j + 2], c_end = cb + (r.len + kRepairChunk - 1) / kRepairChunk;
                        const uint64_t c2 = next_some(w.chunk_first, cb + x / kRepairChunk, c_end);
                        x = c2 == c_end ? r.len : (c2 - cb) * kRepairChunk + w.chunk_first[c2];
                    }
                    q = x - 1;
                    continue;
                }
                if (st.run + 1 >= k) break;  // the next run of >= k bytes: its windows are valid codes
                st.feed<true>(f, code, [&](uint64_t v) {
                    w.spur_code[r.d + q] = v;
                    w.spur_flag[r.d + q] = 1;
                });
            }
        }
    }
}

// The chunk's bytes [a - kRepLook, a + kRepairChunk) as a bit mask of "not ACGT" (bytes before the contig count as
// not ACGT, so that no window reaches across its start), then the pushes of the 4 bytes of this thread.
__device__ __forceinline__ void chunk_mask(RepairWs const& w, ChunkAt const& r, uint32_t* s_mask) {
    const char* s = w.bases + r.start;
    for (uint32_t t0 = 0; t0 < kRepMask; t0 += kRepThreads) {
        const uint32_t t = t0 + threadIdx.x;
        const int64_t p = int64_t(r.a) - int64_t(kRepLook) + int64_t(t);
        const bool bad = t < kRepMask && (p < 0 || uint64_t(p) >= r.b || !acgt(s, uint64_t(p)));
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, bad);
        if ((threadIdx.x & 31) == 0 && t < kRepMask) s_mask[t >> 5] = bal;
    }
    __syncthreads();
}
__device__ __forceinline__ bool any_bit(const uint32_t* m, uint32_t lo, uint32_t hi) {  // bits [lo, hi]
    for (uint32_t x = lo >> 5; x <= (hi >> 5); ++x) {
        uint32_t bits = m[x];
        if (x == (lo >> 5)) bits &= 0xFFFFFFFFu << (lo & 31);
        if (x == (hi >> 5)) bits &= 0xFFFFFFFFu >> (31 - (hi & 31));
        if (bits) return true;
    }
    return false;
}
// bit i of the result: byte a + 4 * threadIdx.x + i pushes a code; bit 4 + i: that code is spurious
__device__ __forceinline__ uint32_t thread_pushes(RepairWs const& w, ChunkAt const& r, const uint32_t* s_mask, uint32_t k) {
    uint32_t out = 0;
    for (uint32_t i = 0; i < 4; ++i) {
        const uint64_t p = r.a + 4 * threadIdx.x + i;
        if (p >= r.b) break;
        const uint32_t t = uint32_t(p - r.a) + kRepLook;
        if (w.spur_flag[r.d + p]) out |= 0x11u << i;
        else if (!any_bit(s_mask, t + 1 - k, t)) out |= 1u << i;
    }
    return out;
}

// ---- exclusive scan whose length (or whether it runs at all) is known on the device only ----
// Up-sweep: block b of kRepairScanBlocks sums items [b * per, (b + 1) * per), and the last block to finish scans
// the block sums (the spine); down-sweep: block b scans its items again from its sum on, handing item i's exclusive
// sum to out.put(i, .) and the total to out.close(n, .).
struct ScanLen {  // the length, in device memory; nothing to do when it is 0
    const unsigned long long* n_dev;
    __device__ __forceinline__ bool get(uint64_t* n) const {
        *n = *n_dev;
        return *n != 0;
    }
};
constexpr int kSpineItems = kRepairScanBlocks / 256;
// called by every block of an up-sweep (256 threads) once part[blockIdx.x] is written
__device__ __forceinline__ void spine_if_last(uint64_t* part, unsigned long long* done) {
    using Scan = cub::BlockScan<unsigned long long, 256>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(done, 1ull) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    unsigned long long v[kSpineItems], total = 0;
#pragma unroll
    for (int u = 0; u < kSpineItems; ++u) v[u] = __ldcg(part + threadIdx.x * kSpineItems + u);
    Scan(tmp).ExclusiveSum(v, v, total);
#pragma unroll
    for (int u = 0; u < kSpineItems; ++u) part[threadIdx.x * kSpineItems + u] = v[u];
    if (threadIdx.x == 0) part[kRepairScanBlocks] = total;
}
template <class Item>
__global__ void __launch_bounds__(256) k_scan_up(Item it, ScanLen sl, uint64_t* part, unsigned long long* done) {
    using Reduce = cub::BlockReduce<unsigned long long, 256>;
    __shared__ typename Reduce::TempStorage tmp;
    uint64_t n;
    if (!sl.get(&n)) return;
    const uint64_t per = (n + gridDim.x - 1) / gridDim.x, lo = min(n, blockIdx.x * per), hi = min(n, lo + per);
    unsigned long long sum = 0;
    for (uint64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) sum += it(i);
    sum = Reduce(tmp).Sum(sum);
    if (threadIdx.x == 0) part[blockIdx.x] = sum;
    spine_if_last(part, done);
}
template <class Item, class Out>
__global__ void __launch_bounds__(256) k_scan_down(Item it, ScanLen sl, const uint64_t* part, Out out) {
    using Scan = cub::BlockScan<unsigned long long, 256>;
    __shared__ typename Scan::TempStorage tmp;
    uint64_t n;
    if (!sl.get(&n)) return;
    const uint64_t per = (n + gridDim.x - 1) / gridDim.x, lo = min(n, blockIdx.x * per), hi = min(n, lo + per);
    unsigned long long carry = part[blockIdx.x];
    for (uint64_t t0 = lo; t0 < hi; t0 += blockDim.x) {
        const uint64_t i = t0 + threadIdx.x;
        unsigned long long v = i < hi ? it(i) : 0, agg = 0;
        Scan(tmp).ExclusiveSum(v, v, agg);
        if (i < hi) out.put(i, carry + v);
        carry += agg;
        __syncthreads();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) out.close(n, part[kRepairScanBlocks]);
}
// The chunks' up-sweep: block b counts the codes of chunks [b * per, (b + 1) * per) one by one (chunk_cnt) and
// sums them for the spine.
__global__ void __launch_bounds__(kRepThreads) k_rep_count(const __grid_constant__ RepairWs w, uint32_t k) {
    using Reduce = cub::BlockReduce<unsigned long long, kRepThreads>;
    __shared__ typename Reduce::TempStorage tmp;
    __shared__ uint32_t s_mask[kRepMask / 32];
    const uint64_t n_chunks = w.ctr->n_chunks;
    if (!n_chunks) return;
    const uint64_t per = (n_chunks + gridDim.x - 1) / gridDim.x, lo = min(n_chunks, blockIdx.x * per),
                   hi = min(n_chunks, lo + per);
    unsigned long long sum = 0;
    for (uint64_t ch = lo; ch < hi; ++ch) {
        const ChunkAt r = chunk_at(w, ch);
        chunk_mask(w, r, s_mask);
        const unsigned long long n = Reduce(tmp).Sum((unsigned long long)__popc(thread_pushes(w, r, s_mask, k) & 15u));
        if (threadIdx.x == 0) {
            w.chunk_cnt[ch] = n;
            sum += n;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) w.part[blockIdx.x] = sum;
    spine_if_last(w.part, &w.ctr->scan_done[0]);
}

struct ChunkItem {
    const uint64_t* cnt;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return cnt[i]; }
};
struct ChunkOut {
    uint64_t* out;
    __device__ __forceinline__ void put(uint64_t i, uint64_t v) const { out[i] = v; }
    __device__ __forceinline__ void close(uint64_t n, uint64_t t) const { out[n] = t; }
};
// The contigs' scan runs over the contigs from the first dirty one fd on (item i: contig fd + i), from the clean
// offset of fd (tail_off[0]: the contigs before fd keep theirs).
struct ContigItem {  // final codes of contig fd + i
    RepairWs w;
    uint32_t k;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const {
        const uint64_t c = w.n_contigs - w.ctr->fd_rev + i;
        const uint64_t len = w.offsets[c + 1] - w.offsets[c];
        if (!w.dirty[c]) return len >= k ? len - k + 1 : 0;
        const uint64_t cb = w.list[3 * w.slot[c] + 2];
        return w.chunk_out[cb + (len + kRepairChunk - 1) / kRepairChunk] - w.chunk_out[cb];
    }
};

struct CodeOffOut {
    RepairWs w;
    uint64_t* code_off;
    unsigned long long* total_to;
    __device__ __forceinline__ void put(uint64_t i, uint64_t v) const {
        code_off[w.n_contigs - w.ctr->fd_rev + i] = w.tail_off[0] + v;
    }
    __device__ __forceinline__ void close(uint64_t, uint64_t t) const {
        code_off[w.n_contigs] = w.tail_off[0] + t;
        *total_to = w.tail_off[0] + t;
    }
};

// clean code i of contig c >= the first dirty contig fd
struct CleanSrc {
    const uint64_t* base;  // indexed by the clean code offsets
    const uint64_t* tail_off;
    uint64_t fd;
    __device__ __forceinline__ uint64_t operator()(uint64_t c, uint64_t i) const { return base[tail_off[c - fd] + i]; }
};
__device__ __forceinline__ CleanSrc clean_src(RepairWs const& w, const uint64_t* src, bool in_place, uint64_t fd) {
    const uint64_t c0 = w.tail_off[0];
    return CleanSrc{in_place ? w.tail_codes + tail_shift(src + c0) - c0 : src, w.tail_off, fd};
}

// The assemble, one kernel: blocks [0, g_dirty) write the codes of the dirty contigs, a chunk per block step and 4
// bytes per thread; the others the codes of the clean contigs that move (in place: from the first dirty contig on;
// else all), kEmitStep output positions per block step with their contigs bracketed by one search per step and 8
// independent loads in flight per thread.
constexpr int kEmitStep = 2048;
__device__ __forceinline__ uint64_t contig_of(const uint64_t* off, uint64_t lo, uint64_t hi, uint64_t i) {
    while (hi - lo > 1) {  // off[lo] <= i < off[hi]
        const uint64_t mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ void emit_dirty(RepairWs const& w, uint32_t k, const uint64_t* code_off, CleanSrc const& cs,
                                           uint64_t* dst, uint64_t block, uint64_t blocks) {
    using Scan = cub::BlockScan<uint32_t, kRepThreads>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ uint32_t s_mask[kRepMask / 32];
    const uint64_t n_chunks = w.ctr->n_chunks;
    for (uint64_t ch = block; ch < n_chunks; ch += blocks) {
        const ChunkAt r = chunk_at(w, ch);
        chunk_mask(w, r, s_mask);
        const uint32_t pushes = thread_pushes(w, r, s_mask, k);
        uint32_t rank;
        Scan(tmp).ExclusiveSum(uint32_t(__popc(pushes & 15u)), rank);
        uint64_t at = code_off[r.c] + w.chunk_out[ch] - w.chunk_out[w.list[3 * r.j + 2]] + rank;
        for (uint32_t i = 0; i < 4; ++i) {
            if (!((pushes >> i) & 1u)) continue;
            const uint64_t p = r.a + 4 * threadIdx.x + i;
            dst[at++] = (pushes >> (4 + i)) & 1u ? w.spur_code[r.d + p] : cs(r.c, p + 1 - k);
        }
        __syncthreads();
    }
}
__device__ __forceinline__ void emit_clean(RepairWs const& w, const uint64_t* code_off, const uint64_t* src,
                                           CleanSrc const& cs, bool in_place, uint64_t* dst, uint64_t block,
                                           uint64_t blocks) {
    constexpr int kPer = kEmitStep / 256, kTab = 128;
    __shared__ uint64_t s_lo, s_hi, t_off[kTab + 1];
    __shared__ const uint64_t* t_src[kTab];  // where the contig's code i - t_off[t] is; null: a dirty contig
    const uint64_t n = w.n_contigs, fd = cs.fd, c_lo = in_place ? fd : 0;
    const uint64_t o0 = code_off[c_lo], total = code_off[n];
    for (uint64_t b0 = o0 + block * kEmitStep; b0 < total; b0 += blocks * kEmitStep) {
        const uint64_t b1 = min(b0 + kEmitStep, total);
        if (threadIdx.x == 0) {
            s_lo = contig_of(code_off, c_lo, n, b0);
            s_hi = contig_of(code_off, c_lo, n, b1 - 1) + 1;
        }
        __syncthreads();
        const uint64_t lo = s_lo, hi = s_hi;
        const bool tab = hi - lo <= kTab;  // (a step of many empty contigs searches in global memory)
        if (tab && threadIdx.x <= hi - lo) {
            const uint64_t c = lo + threadIdx.x;
            t_off[threadIdx.x] = code_off[c];
            if (c < hi) t_src[threadIdx.x] = w.dirty[c] ? nullptr : c < fd ? src + code_off[c] : cs.base + cs.tail_off[c - fd];
        }
        __syncthreads();
        uint64_t v[kPer];
        bool keep[kPer];
        uint64_t at = 0;
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const uint64_t i = b0 + u * 256 + threadIdx.x;
            keep[u] = false;
            if (i >= b1) continue;
            if (tab) {
                at = contig_of(t_off, at, hi - lo, i);
                const uint64_t* p = t_src[at];
                if (!p) continue;
                v[u] = p[i - t_off[at]];
            } else {
                const uint64_t c = contig_of(code_off, lo, hi, i);
                if (w.dirty[c]) continue;
                v[u] = c < fd ? src[i] : cs(c, i - code_off[c]);
            }
            keep[u] = true;
        }
#pragma unroll
        for (int u = 0; u < kPer; ++u)
            if (keep[u]) dst[b0 + u * 256 + threadIdx.x] = v[u];
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) k_rep_emit(const __grid_constant__ RepairWs w, uint32_t k, const uint64_t* code_off,
                                                  const uint64_t* src, bool in_place, uint64_t* dst, uint32_t g_dirty) {
    const uint64_t fd_rev = w.ctr->fd_rev;
    if (!fd_rev) return;
    const CleanSrc cs = clean_src(w, src, in_place, w.n_contigs - fd_rev);
    if (blockIdx.x < g_dirty) emit_dirty(w, k, code_off, cs, dst, blockIdx.x, g_dirty);
    else emit_clean(w, code_off, src, cs, in_place, dst, blockIdx.x - g_dirty, gridDim.x - g_dirty);
}

unsigned grid_for(uint64_t n, uint64_t per_block, unsigned cap) {
    uint64_t b = (n + per_block - 1) / per_block;
    return unsigned(b < 1 ? 1 : b > cap ? cap : b);
}

unsigned blocks_for(uint64_t n, unsigned cap = 148 * 32) {
    uint64_t b = (n + 255) / 256;
    if (b < 1) b = 1;
    if (b > cap) b = cap;
    return unsigned(b);
}

}  // namespace

uint64_t quirk_tmp_bytes(uint64_t n) {
    size_t a = 0, b = 0;
    cub::CountingInputIterator<uint64_t> cnt(0);
    cub::DeviceSelect::Flagged(nullptr, a, cnt, (const uint8_t*)nullptr, (uint64_t*)nullptr, (unsigned long long*)nullptr, n);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (uint64_t*)nullptr, (uint64_t*)nullptr, n);
    return (a > b ? a : b) + 256;
}

// runs of a batch (build side): voff[0..*n_v] (boundaries, closed with n), vstart[0..n_list] (first run per contig)
void launch_find_runs(const char* d_bases, uint64_t n, const uint64_t* d_starts, uint64_t n_list, uint8_t* d_flag,
                      uint64_t* d_voff, unsigned long long* d_n_v, uint32_t* d_vstart, void* d_tmp, uint64_t tmp_bytes,
                      cudaStream_t stream) {
    cudaMemsetAsync(d_flag, 0, n, stream);
    k_mark_starts<<<unsigned((n_list + 255) / 256), 256, 0, stream>>>(d_starts, n_list, n, d_flag);
    k_run_boundaries<<<blocks_for(n), 256, 0, stream>>>(d_bases, n, d_flag);
    size_t bytes = tmp_bytes;
    cub::CountingInputIterator<uint64_t> cnt(0);
    cub::DeviceSelect::Flagged(d_tmp, bytes, cnt, d_flag, d_voff, d_n_v, n, stream);
    k_close_offsets<<<1, 1, 0, stream>>>(d_voff, d_n_v, n);
    k_first_run<<<unsigned((n_list + 256) / 256), 256, 0, stream>>>(d_voff, d_n_v, d_starts, n_list, n, d_vstart);
}

uint64_t repair_scratch(uint64_t n_contigs, uint64_t span, uint64_t clean_total, bool in_place, char* base, RepairWs* w) {
    const uint64_t max_chunks = span / kRepairChunk + n_contigs + 1;
    uint64_t at = 0;
    auto take = [&](uint64_t bytes) {
        char* p = base ? base + at : nullptr;
        at += (bytes + 255) / 256 * 256;
        return p;
    };
    RepairWs r{};
    r.ctr = reinterpret_cast<RepairCounters*>(take(sizeof(RepairCounters)));
    r.list = reinterpret_cast<uint64_t*>(take(3 * n_contigs * 8));
    r.slot = reinterpret_cast<uint64_t*>(take(n_contigs * 8));
    r.chunk_tab = reinterpret_cast<uint64_t*>(take(max_chunks * 8));
    r.chunk_first = reinterpret_cast<uint16_t*>(take(max_chunks * 2));
    r.chunk_last_inv = reinterpret_cast<uint16_t*>(take(max_chunks * 2));
    r.chunk_cnt = reinterpret_cast<uint64_t*>(take(max_chunks * 8));
    r.chunk_out = reinterpret_cast<uint64_t*>(take((max_chunks + 1) * 8));
    r.spur_flag = reinterpret_cast<uint8_t*>(take(span));
    r.spur_code = reinterpret_cast<uint64_t*>(take(span * 8));
    r.tail_off = reinterpret_cast<uint64_t*>(take((n_contigs + 1) * 8));
    r.tail_codes = reinterpret_cast<uint64_t*>(take(in_place ? clean_total * 8 + 16 : 0));
    r.part = reinterpret_cast<uint64_t*>(take((kRepairScanBlocks + 1) * 8));
    if (w) {
        r.bases = w->bases;
        r.offsets = w->offsets;
        r.n_contigs = w->n_contigs;
        r.dirty = w->dirty;
        *w = r;
    }
    return at;
}

int launch_repair_layout(DevImage const& img, RepairWs const& w, uint64_t* d_code_off, const uint64_t* codes,
                         uint64_t clean_total, bool in_place, unsigned long long* d_total, cudaStream_t stream) {
    const uint64_t n = w.n_contigs;
    if (!n) return 0;
    const unsigned g_chunks = 148 * 8;  // chunk kernels: grid-stride over the listed chunks
    k_rep_list<<<grid_for(n, 256 * 8, 148 * 8), 256, 0, stream>>>(w);
    k_rep_prep<<<std::max(g_chunks, grid_for(in_place ? clean_total : 0, 256 * 4, 148 * 8)), kRepThreads, 0, stream>>>(
        w, d_code_off, codes, in_place);
    k_rep_episodes<<<g_chunks, kRepThreads, 0, stream>>>(img, w);
    k_rep_count<<<kRepairScanBlocks, kRepThreads, 0, stream>>>(w, img.k);
    const ScanLen chunks{&w.ctr->n_chunks};
    k_scan_down<<<kRepairScanBlocks, 256, 0, stream>>>(ChunkItem{w.chunk_cnt}, chunks, w.part, ChunkOut{w.chunk_out});
    const ScanLen contigs{&w.ctr->fd_rev};
    const ContigItem item{w, img.k};
    k_scan_up<<<kRepairScanBlocks, 256, 0, stream>>>(item, contigs, w.part, &w.ctr->scan_done[1]);
    k_scan_down<<<kRepairScanBlocks, 256, 0, stream>>>(item, contigs, w.part, CodeOffOut{w, d_code_off, d_total});
    return 7;
}

int launch_repair_assemble(DevImage const& img, RepairWs const& w, const uint64_t* d_code_off, const uint64_t* src,
                           bool in_place, uint64_t* dst, uint64_t max_total, cudaStream_t stream) {
    if (!w.n_contigs) return 0;
    const unsigned g_dirty = 148 * 8;
    k_rep_emit<<<g_dirty + grid_for(max_total, kEmitStep, 148 * 16), 256, 0, stream>>>(w, img.k, d_code_off, src, in_place,
                                                                                         dst, g_dirty);
    return 1;
}

void launch_shift_starts(const uint64_t* d_offsets, uint64_t n_contigs, uint64_t first, uint64_t* d_starts, cudaStream_t stream) {
    k_shift_starts<<<unsigned((n_contigs + 256) / 256), 256, 0, stream>>>(d_offsets, n_contigs, first, d_starts);
}

// per run: pieces / m-mer ordinals / k-mers, then exclusive sums in place (entry n_v = totals)
void launch_build_run_counts(const char* d_bases, const uint64_t* d_voff, const unsigned long long* d_n_v,
                             const uint32_t* d_vstart, uint64_t n_list, uint64_t n_v_host, uint32_t k, uint32_t m,
                             uint64_t* d_pieces, uint64_t* d_ids, uint64_t* d_kmers, void* d_tmp, uint64_t tmp_bytes,
                             cudaStream_t stream) {
    k_build_run_counts<<<unsigned((n_v_host + 256) / 256), 256, 0, stream>>>(d_bases, d_voff, d_n_v, d_vstart, n_list, k, m,
                                                                             d_pieces, d_ids, d_kmers);
    for (uint64_t* a : {d_pieces, d_ids, d_kmers}) {
        size_t bytes = tmp_bytes;
        cub::DeviceScan::ExclusiveSum(d_tmp, bytes, a, a, n_v_host + 1, stream);
    }
}

void launch_build_pieces(const uint64_t* d_voff, const unsigned long long* d_n_v, uint64_t n_v_host, uint32_t k,
                         const uint64_t* d_pieces, const uint64_t* d_ids, uint64_t mm_count_in, uint64_t n, uint64_t* d_poff,
                         uint64_t* d_pid, cudaStream_t stream) {
    k_build_pieces<<<unsigned((n_v_host + 256) / 256), 256, 0, stream>>>(d_voff, d_n_v, k, d_pieces, d_ids, mm_count_in, n,
                                                                         d_poff, d_pid);
}

}  // namespace lphb
