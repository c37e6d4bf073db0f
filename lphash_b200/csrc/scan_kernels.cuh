// Launchers of the build-side scan kernels (scan_kernels.cu): the data-parallel form of
// minimizer::from_string / get_colliding_kmers (SURVEY.md S2').  Device pointers, asynchronous.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lphb {

struct ScanBatch {
    const char* bases;         // concatenated ASCII (indexable by offsets[])
    const uint64_t* offsets;   // n_contigs + 1
    const uint64_t* code_off;  // n_contigs + 1: exclusive scan of max(0, L - k + 1)  (dense k-mer index)
    const uint64_t* id_base;   // n_contigs + 1: mm_count_in + exclusive scan of max(0, L - m + 1)
    uint64_t n_contigs, first_base, end_base;
    uint64_t n_kmers;          // code_off[n_contigs]
    uint32_t k, m;
    uint64_t seed;
    uint8_t* dirty;            // n_contigs flags
};

// id_base[c] = mm_count_in + sum_{c' < c} max(0, L_c' - m + 1)
void launch_id_base(const uint64_t* d_offsets, uint64_t n_contigs, uint32_t m, uint64_t mm_count_in,
                    uint64_t* d_id_base, void* d_tmp, uint64_t tmp_bytes, cudaStream_t stream);

// Pass 1: head[d] = 1 where k-mer d starts a super-k-mer, pos[d] = offset of its minimizer.
void launch_scan_heads(ScanBatch const& b, uint8_t* head, uint8_t* pos, cudaStream_t stream);

// rank[d] = number of heads before d (exclusive); rank[n_kmers] = number of records.
void launch_head_ranks(const uint8_t* head, uint64_t n_kmers, uint32_t* rank, void* d_tmp,
                       uint64_t tmp_bytes, cudaStream_t stream);
uint64_t head_ranks_tmp_bytes(uint64_t n_kmers);

// Pass 2: write the 18-byte records {itself, id, p1, size} and start_pos[r] = stream position of
// record r's first k-mer, relative to b.first_base.
void launch_scan_emit(ScanBatch const& b, const uint8_t* head, const uint8_t* pos,
                      const uint32_t* rank, uint8_t* records, uint32_t* start_pos, cudaStream_t stream);

// dirty[c] = 1 for every contig holding a byte outside ACGT/acgt/U/u, whatever its length (the scan kernels only
// look at contigs that hold a k-mer)
void launch_flag_invalid_bytes(const char* bases, uint64_t first, uint64_t span, const uint64_t* offsets, uint64_t n_contigs,
                               uint8_t* dirty, cudaStream_t stream);

// get_colliding_kmers: take[r] = (record r's id is in ids) ? size : 0 ...
void launch_colliding_mark(const uint8_t* records, uint64_t n_records, const uint64_t* ids,
                           uint64_t n_ids, uint32_t* take, cudaStream_t stream);
// ... out_off = exclusive scan of take (done with launch_exclusive_u32), then write the k-mers.
void launch_exclusive_u32(const uint32_t* in, uint64_t n, uint64_t* out, void* d_tmp,
                          uint64_t tmp_bytes, cudaStream_t stream);
uint64_t exclusive_u32_tmp_bytes(uint64_t n);
void launch_colliding_emit(ScanBatch const& b, uint64_t n_records, const uint32_t* start_pos,
                           const uint32_t* take, const uint64_t* out_off, int kmer_bits,
                           uint8_t* kmers, cudaStream_t stream);

// minimizer::classify (classify_kernels.cu).  Step 1: sort by minimizer (key_bits = significant bits of a
// minimizer: 2m when the caller knows m, else 64), group flags (bit 0: first of
// its group, bit 1: member of a group of several), output slots; counts[0] = #triplets, counts[1] = #ids.
uint64_t classify_tmp_bytes(uint64_t n);
void launch_classify_groups(const uint8_t* records, uint64_t n, uint64_t* key, uint64_t* key_sorted,
                            uint32_t* idx, uint32_t* idx_sorted, uint8_t* flags, uint32_t* gslot,
                            uint32_t* cslot, unsigned long long* counts, void* d_tmp, uint64_t tmp_bytes,
                            int key_bits, cudaStream_t stream);
// Step 2: 10-byte triplets in ascending minimizer order, colliding ids gathered and sorted ascending.
void launch_classify_emit(const uint8_t* records, const uint64_t* key_sorted, const uint32_t* idx_sorted,
                          const uint8_t* flags, const uint32_t* gslot, const uint32_t* cslot, uint64_t n,
                          uint8_t* triplets, uint64_t* ids_unsorted, uint64_t* ids_sorted, uint64_t n_ids,
                          void* d_tmp, uint64_t tmp_bytes, cudaStream_t stream);
// After step 1: sid[g] = the id of group g's record when the group holds one record, UINT64_MAX otherwise.
void launch_classify_singleton_ids(const uint8_t* records, const uint32_t* idx_sorted, const uint8_t* flags,
                                   const uint32_t* gslot, uint64_t n, uint64_t* sid, cudaStream_t stream);

}  // namespace lphb
