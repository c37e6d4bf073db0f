// Launchers of the query kernels (query_generic.cu, query_tiled.cu).  All pointers are device
// pointers; all launches are asynchronous on `stream`.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_image.h"

namespace lphb {

// Per-batch device-side description of the contig layout.
struct DevBatch {
    const char* bases;          // concatenated ASCII
    const uint64_t* offsets;    // n_contigs + 1, indexes `bases`
    const uint64_t* code_off;   // n_contigs + 1: exclusive scan of max(0, L - k + 1)
    uint64_t n_contigs;
    uint64_t first_base;        // offsets[0]
    uint64_t end_base;          // offsets[n_contigs]
    uint64_t* codes;            // output
    uint8_t* dirty;             // n_contigs flags: contig contains a non-ACGT byte
    unsigned long long* status; // [0] unused here, [1] += number of dirty contigs
    void* tile_ws;              // scratch for the tiled kernel (query_tiled_ws_bytes), may be null
    uint64_t tile_ws_bytes;
};
uint64_t query_tiled_ws_bytes(uint64_t span_bases);

// code_off[c] = sum_{c' < c} max(0, L_c' - k + 1); status[0] = total.  One launch, any n.
void launch_code_offsets(const uint64_t* d_offsets, uint64_t n_contigs, uint32_t k,
                         uint64_t* d_code_off, unsigned long long* d_status, void* d_tmp,
                         uint64_t tmp_bytes, cudaStream_t stream);
uint64_t code_offsets_tmp_bytes(uint64_t n_contigs);

// Generic kernel: any (k, m); one thread per k-mer, everything recomputed per k-mer.
void launch_query_generic(DevImage const& img, DevBatch const& b, cudaStream_t stream);

// Packed k-mers (lookup_kernels.cu): d_codes[i] = code of the k-mer in the low 2k bits of d_kmers[i], which holds
// img.kmer_bits / 8 little-endian bytes ({lo, hi} for 128 bits, 16-byte aligned then); any (k, m), any n.
void launch_lookup_kmers(DevImage const& img, const void* d_kmers, uint64_t n, uint64_t* d_codes, cudaStream_t stream);

// Tiled kernel for the (k, m) pairs it is instantiated for; returns false if (k, m) is not one
// of them (the caller then uses the generic kernel).
bool launch_query_tiled(DevImage const& img, DevBatch const& b, cudaStream_t stream);

// Build-side form of the tiled kernel (minimizer::from_string): writes the packed 18-byte mm_record_t
// stream of the batch in scan order to d_records (capacity: one record per k-mer start), the stream
// position (relative to b.first_base) of every record's first k-mer to d_start_pos, and the number of
// records to *d_n_records; flags contigs with non-ACGT bytes in b.dirty (their records are then
// meaningless).  d_id_base[c] = m-mer ordinal of contig c's first m-mer.  b.codes / b.code_off are not
// used.  Returns false if (k, m) is not instantiated (the caller then uses the generic scan kernels).
bool launch_scan_records_tiled(uint32_t k, uint32_t m, uint64_t seed, DevBatch const& b, const uint64_t* d_id_base,
                               uint8_t* d_records, uint32_t* d_start_pos, unsigned long long* d_n_records,
                               cudaStream_t stream);
bool scan_tiled_available(uint32_t k, uint32_t m);

// Contigs with non-ACGT bytes (quirk_kernels.cu): the build side's run finder, and the query side's repair.
uint64_t quirk_tmp_bytes(uint64_t n);
void launch_find_runs(const char* d_bases, uint64_t n, const uint64_t* d_starts, uint64_t n_list, uint8_t* d_flag,
                      uint64_t* d_voff, unsigned long long* d_n_v, uint32_t* d_vstart, void* d_tmp, uint64_t tmp_bytes,
                      cudaStream_t stream);

// The repair of a batch after its clean pass (the stateless codes in the clean layout, L-k+1 slots per contig, and
// the dirty flags), all on the device and asynchronous: every count it depends on stays in device memory, and every
// kernel reads it there and exits early when there is nothing to do (a clean batch).  A dirty contig is cut into
// chunks of kRepairChunk bytes; each chunk is one block's work.  Scratch, sized from the host offsets alone
// (repair_scratch): 68 bytes per contig, 9.03 bytes per base (a flag and a code slot per byte of a dirty contig,
// 28 bytes per chunk), 8 bytes per clean code when the clean pass wrote in place, and 12 KB.
constexpr uint32_t kRepairChunk = 1024;
constexpr uint32_t kRepairScanBlocks = 1024;
struct RepairCounters {
    unsigned long long n_list;    // dirty contigs listed
    unsigned long long bytes;     // their bytes (the scratch slots handed out)
    unsigned long long n_chunks;  // their chunks
    unsigned long long fd_rev;    // n_contigs - (first dirty contig); 0: none
    unsigned long long scan_done[2];  // up-sweep blocks finished (the chunks' scan, the contigs')
};
struct RepairWs {
    const char* bases;            // indexed by the offsets
    const uint64_t* offsets;      // n_contigs + 1 (device)
    uint64_t n_contigs;
    const uint8_t* dirty;         // per contig (the clean pass's flags)
    RepairCounters* ctr;          // zeroed by the caller before launch_repair_layout
    uint64_t* list;               // 3 words per listed contig: contig, first scratch slot, first chunk
    uint64_t* slot;               // per contig: its list entry (dirty contigs only)
    uint64_t* chunk_tab;          // per chunk: its list entry
    uint16_t* chunk_first;        // per chunk: offset of its first ACGT byte, 0xFFFF if none
    uint16_t* chunk_last_inv;     // per chunk: offset of its last non-ACGT byte, 0xFFFF if none
    uint64_t* chunk_cnt;          // per chunk: codes it yields
    uint64_t* chunk_out;          // exclusive sums of chunk_cnt (n_chunks + 1)
    uint8_t* spur_flag;           // per scratch slot: a spurious code is pushed at this byte
    uint64_t* spur_code;          // ... and this is it
    uint64_t* tail_off;           // clean code offsets of the contigs from the first dirty one on
    uint64_t* tail_codes;         // in place: the clean codes from the first dirty contig on
    uint64_t* part;               // scan spine (kRepairScanBlocks + 1)
};
// Bytes of scratch for a batch (offsets of the fields above in one allocation, 256-byte aligned): fills `w`'s pointers
// relative to `base` when base is not null.
uint64_t repair_scratch(uint64_t n_contigs, uint64_t span, uint64_t clean_total, bool in_place, char* base, RepairWs* w);
// Layout stage (the caller zeroes w.ctr first, on the same stream): lists the dirty contigs, replays their
// episodes, counts every chunk's codes and writes the final layout to d_code_off (n_contigs + 1, the clean layout on
// entry; rewritten from the first dirty contig on) and its total to *d_total.  `codes` holds the clean pass's
// clean_total codes; when in_place they are saved from the first dirty contig on (the assemble then overwrites
// them).  Returns the launches.
int launch_repair_layout(DevImage const& img, RepairWs const& w, uint64_t* d_code_off, const uint64_t* codes,
                         uint64_t clean_total, bool in_place, unsigned long long* d_total, cudaStream_t stream);
// Assemble stage: the final codes into dst in the layout of d_code_off.  in_place: dst is the clean pass's buffer and
// only codes from the first dirty contig on are written; otherwise src holds the clean codes and every code is
// written.  max_total bounds the final total (grid size).  Returns the launches.
int launch_repair_assemble(DevImage const& img, RepairWs const& w, const uint64_t* d_code_off, const uint64_t* src,
                           bool in_place, uint64_t* dst, uint64_t max_total, cudaStream_t stream);

// Build side (minimizer::from_string over contigs with non-ACGT bytes): launch_find_runs over the whole batch
// (d_starts = contig starts relative to the batch, launch_shift_starts), then per run r the number of pieces the
// scan kernels get it in (1 for a run they must scan; invalid runs and runs of exactly k bases followed by an
// invalid byte are cut into pieces of k-1 bytes, which hold no k-mer), its m-mer ordinals and k-mers - exclusive
// sums in place, entry n_v = totals - and finally the piece offsets (n_pieces + 1, relative to the batch) with the
// m-mer ordinal of every piece's first m-mer.
void launch_shift_starts(const uint64_t* d_offsets, uint64_t n_contigs, uint64_t first, uint64_t* d_starts, cudaStream_t stream);
void launch_build_run_counts(const char* d_bases, const uint64_t* d_voff, const unsigned long long* d_n_v,
                             const uint32_t* d_vstart, uint64_t n_list, uint64_t n_v_host, uint32_t k, uint32_t m,
                             uint64_t* d_pieces, uint64_t* d_ids, uint64_t* d_kmers, void* d_tmp, uint64_t tmp_bytes,
                             cudaStream_t stream);
void launch_build_pieces(const uint64_t* d_voff, const unsigned long long* d_n_v, uint64_t n_v_host, uint32_t k,
                         const uint64_t* d_pieces, const uint64_t* d_ids, uint64_t mm_count_in, uint64_t n, uint64_t* d_poff,
                         uint64_t* d_pid, cudaStream_t stream);

// Run-length form of a code stream on the device (runs_kernels.cu): codes[0..n), n < 2^31 -> 12-byte
// records {u64 first, i32 n} (n > 0 ascending, n < 0 descending), never across a contig start.
uint64_t runs_tmp_bytes(uint64_t n);
void launch_runs(const uint64_t* codes, uint64_t n, const uint64_t* code_off, uint64_t n_contigs, uint64_t o0,
                 uint8_t* d_start, uint8_t* d_head, uint32_t* d_rank, uint32_t* d_head_at, void* d_tmp,
                 uint64_t tmp_bytes, uint8_t* d_runs, unsigned long long* d_n_runs, cudaStream_t stream);

// non-ACGT bytes -> 'A' in place (the reference's non-streaming branch, include/mphf_utils.hpp:108)
void launch_sanitize(char* d_bases, uint64_t n, cudaStream_t stream);

// The same into a copy: d_src[0..n) (any alignment, not modified) -> d_dst + copy_sanitize_at(d_src), which has
// d_src's address mod 16, followed by kCopySanitizePad bytes of 'A'.  d_dst: 16-byte aligned,
// n + 16 + kCopySanitizePad bytes.
constexpr uint32_t kCopySanitizePad = 64;
uint64_t copy_sanitize_at(const char* d_src);
void launch_copy_sanitize(char* d_dst, const char* d_src, uint64_t n, cudaStream_t stream);

// status[1] += number of set flags in dirty[0..n)
void launch_count_dirty(const uint8_t* dirty, uint64_t n, unsigned long long* status,
                        cudaStream_t stream);

}  // namespace lphb
