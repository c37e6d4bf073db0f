/*
 * lphash_b200 — C ABI of the B200-native LPHash hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types, no exceptions.
 * The reference (jermp/lphash) has no FFI of its own; its seam for this path is a C++ member
 * function, so each entry point below cites the reference interface it replaces
 * (paths relative to the reference tree; "pthash/" = external/pthash/).  INTEGRATION.md shows
 * the binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - every function returns LPHB_OK (0) or a negative LPHB_E_* code; lphb_last_error() gives the
 *     message of the last failure on the calling thread;
 *   - the caller owns all host buffers; the library owns device memory behind opaque handles;
 *   - one handle = one `.lph` image resident on one GPU; calls on one handle are serialised by
 *     the caller, different handles (different GPUs) may be driven from different host threads;
 *   - "batch" = ASCII bases of n_contigs contigs concatenated without separators + offsets
 *     (n_contigs + 1 entries, offsets[0] need not be 0 but must index `bases`); this is what
 *     kseq hands the reference one record at a time (src/query.cpp:51-52);
 *   - there is NO CPU fallback: every call that computes needs a CUDA device and fails with
 *     LPHB_E_CUDA otherwise.
 */
#ifndef LPHASH_B200_H
#define LPHASH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LPHB_OK 0
#define LPHB_E_ARG (-1)      /* bad argument (null pointer, k/m out of range, ...)            */
#define LPHB_E_IO (-2)       /* cannot open / read the .lph file                              */
#define LPHB_E_FORMAT (-3)   /* not a partitioned-LP-MPHF image (truncated, trailing bytes...) */
#define LPHB_E_CUDA (-4)     /* CUDA error or no device                                       */
#define LPHB_E_CAPACITY (-5) /* output buffer too small; required size reported where possible */
#define LPHB_E_NOMEM (-6)

typedef struct lphb_mphf lphb_mphf; /* device image of one lphash::mphf on one GPU */

/* Header fields of the serialized lphash::mphf (include/partitioned_mphf.hpp:204-211, :42-48). */
typedef struct lphb_info {
    uint32_t k, m;
    uint32_t kmer_bits; /* 64 or 128: the kmer_t the file was built with (compile_constants.tpd) */
    int32_t device;
    uint64_t mm_seed;
    uint64_t nkmers;
    uint64_t distinct_minimizers;
    uint64_t n_maximal;
    uint64_t right_coll_sizes_start;
    uint64_t none_sizes_start;
    uint64_t none_pos_start;
    uint64_t fallback_keys; /* k-mers handled by fallback_kmer_order */
    uint64_t file_bytes;    /* size of the .lph image parsed                                    */
    uint64_t device_bytes;  /* bytes of HBM the device image occupies                           */
    double load_host_ms;    /* load time on the host: structure walk of the image (+ CUDA start-up if this
                               is the process's first CUDA call; + the decode with LPHB_HOST_DECODE=1) */
    double load_h2d_ms;     /* load time on the device: allocation, upload, decode kernels          */
} lphb_info;

const char* lphb_last_error(void);
const char* lphb_version(void);
int lphb_device_count(int* count);

/* ---- loading: replaces essentials::load(hf, file) (src/query.cpp:37) ----------------------
 * Parses the byte-exact essentials visitor image of lphash::mphf
 * (include/partitioned_mphf.hpp:204-219) and builds a flat device image from it.  The host only walks the
 * structure (sizes, ranges: LPHB_E_FORMAT before any CUDA call for a malformed file); the decoding -
 * compact_vector::access, Elias-Fano access, rs_bit_vector::rank, quartet_wtree::rank_of, one word per bucket -
 * runs on the GPU (lphash_b200/csrc/image_decode.cu) and reports what only decoding reveals as
 * LPHB_E_FORMAT too.  kmer_bits selects the fallback hash flavour of include/constants.hpp:56-70 (the
 * file does not record it).                                                                      */
int lphb_mphf_load_file(const char* path, int kmer_bits, int device, lphb_mphf** out);
int lphb_mphf_load_memory(const void* image, uint64_t nbytes, int kmer_bits, int device,
                          lphb_mphf** out);
/* The same for the UNPARTITIONED variant, lphash::mphf_alt (`build-u` / `query-u`: include/
 * unpartitioned_mphf.hpp:198-210 is the file format, src/unpartitioned_mphf.cpp:191-206 the probe).  The
 * handle then serves every query entry point below exactly like a partitioned one: mphf_alt's
 * operator() (include/unpartitioned_mphf.hpp:72-192) is the same streaming loop over another probe.
 * (lphb_info: n_maximal and the *_start fields are 0.)                                              */
int lphb_mphf_alt_load_file(const char* path, int kmer_bits, int device, lphb_mphf** out);
int lphb_mphf_alt_load_memory(const void* image, uint64_t nbytes, int kmer_bits, int device,
                              lphb_mphf** out);
int lphb_mphf_free(lphb_mphf* f);
int lphb_mphf_info(const lphb_mphf* f, lphb_info* info);

/* ---- query-p hot call ----------------------------------------------------------------------
 * Replaces `hf(seq->seq.s, seq->seq.l, true)` = lphash::mphf::operator()(contig, len,
 * streaming=true) (include/partitioned_mphf.hpp:73-184; caller src/query.cpp:52) for a whole
 * batch of contigs.  HOST buffers in, HOST buffers out (H2D / D2H copies happen inside).
 *   codes         receives the hash codes of all contigs, concatenated in contig order
 *   code_offsets  (n_contigs + 1) receives where each contig's codes start; contig c produced
 *                 code_offsets[c+1] - code_offsets[c] codes: L-k+1 for an ACGT-only contig of
 *                 length L >= k, 0 if L < k; contigs with other bytes follow the reference's
 *                 streaming behaviour exactly (its spurious entries included, SURVEY.md Q1)
 *   n_codes       total number of codes (also set when returning LPHB_E_CAPACITY)
 * Workspace: beyond the staging of the batch, a batch with a contig holding a non-ACGT byte grows the handle's
 * repair scratch (the device repair of lphb_query_stream_exact_device_async) to 68 bytes per contig + 9.03 bytes
 * per base of the whole batch + 12 KB, plus 8 bytes per code of the result; it is kept for the next call.  The same
 * holds for lphb_query_stream_runs.                                                                               */
int lphb_query_stream(lphb_mphf* f, const char* bases, const uint64_t* offsets,
                      uint64_t n_contigs, uint64_t* codes, uint64_t codes_capacity,
                      uint64_t* code_offsets, uint64_t* n_codes);

/* The reference's NON-streaming branch, hf(seq, len, false) (include/partitioned_mphf.hpp:185-195;
 * pass 2 of query-p, src/query.cpp:72, and `--check`, include/mphf_utils.hpp:56,85): the stateless
 * evaluation of every window of k bytes, where a non-ACGT byte counts as 'A'
 * (include/mphf_utils.hpp:108).  Same arguments as lphb_query_stream; contig c always yields
 * max(0, L-k+1) codes (the reference itself is undefined for L < k).  On ACGT-only input the two
 * branches return the same codes (SURVEY.md S1).                                                  */
int lphb_query_nonstreaming(lphb_mphf* f, const char* bases, const uint64_t* offsets,
                            uint64_t n_contigs, uint64_t* codes, uint64_t codes_capacity,
                            uint64_t* code_offsets, uint64_t* n_codes);

/* Same call with the codes returned in RUN-LENGTH form: consecutive k-mers of a super-k-mer get
 * consecutive codes (include/partitioned_mphf.hpp:131-145: local_rank +-1 per k-mer), so the vector
 * the reference returns is a sequence of arithmetic runs.  `runs` receives packed 12-byte records
 * {uint64_t first; int32_t n} (little-endian; n > 0: first, first+1, ... n codes; n < 0: first,
 * first-1, ... |n| codes), in stream order and never across a contig start: about 2 bytes per k-mer
 * over PCIe instead of 8.  lphb_expand_runs rebuilds the identical uint64_t vector on the host.
 * Works for any input (non-members, colliding minimizers, non-ACGT contigs: their runs are just
 * shorter).  A batch must hold fewer than 2^31 k-mers.  n_runs is also set when returning
 * LPHB_E_CAPACITY (which is also what runs == NULL returns after reporting n_runs / n_codes /
 * code_offsets).                                                                                  */
int lphb_query_stream_runs(lphb_mphf* f, const char* bases, const uint64_t* offsets,
                           uint64_t n_contigs, void* runs, uint64_t runs_capacity, uint64_t* n_runs,
                           uint64_t* code_offsets, uint64_t* n_codes);

/* Host-only decoding of run records into the codes of lphb_query_stream (same order, same values);
 * `threads` host threads share the work (<= 1: the calling thread).  n_codes is also set when
 * returning LPHB_E_CAPACITY.                                                                       */
int lphb_expand_runs(const void* runs, uint64_t n_runs, uint64_t* codes, uint64_t codes_capacity,
                     uint64_t* n_codes, int threads);

/* Device-resident variant: d_* are device pointers on the handle's GPU, `stream` is a
 * cudaStream_t (NULL = default stream).  Asynchronous.  h_offsets is the host copy of the same
 * offsets (used only for sizes).  Evaluates the stateless definition (one code per window of k
 * ACGT bases, SURVEY.md S1); d_status[0] = number of codes laid out (sum of max(0, L-k+1)),
 * d_status[1] = number of contigs containing a non-ACGT byte.  For such a contig the code slot of
 * every k-mer window that contains a non-ACGT byte is UNSPECIFIED (the slots of its other k-mers hold
 * their codes); lphb_mphf_dirty_flags names those contigs, and lphb_query_stream,
 * lphb_query_stream_exact_device and lphb_query_stream_exact_device_async apply the reference's exact streaming
 * behaviour to them - this call does not.
 * Ordering: a handle owns one device workspace, so consecutive calls on one handle are ordered on
 * the device (each call makes its stream wait for the previous call's kernels), on whatever
 * streams they are issued; they never overlap each other.  Overlap comes from several handles or
 * from the copies of the caller's other streams.                                                  */
int lphb_query_stream_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                             const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                             uint64_t codes_capacity, uint64_t* d_code_offsets,
                             uint64_t* d_status, void* stream);

/* Exact streaming branch on device buffers (include/partitioned_mphf.hpp:73-184, src/query.cpp:52): d_codes and
 * d_code_offsets receive what lphb_query_stream gives for the same batch, the reference's spurious codes of contigs
 * with non-ACGT bytes included (SURVEY.md Q1).  Arguments as in lphb_query_stream_device; n_codes receives the total.
 * SYNCHRONOUS: returns once d_codes / d_code_offsets hold the result.  The work runs on `stream` and is ordered
 * against the handle's other calls as in lphb_query_stream_device; every copy goes on `stream`.  A clean batch costs
 * the stateless form plus one read-back of its 32-byte status; a batch with non-ACGT bytes adds the repair of
 * lphb_query_stream_exact_device_async on the device and one 8-byte read-back of the final total between its layout
 * and its assemble (the capacity check).  lphb_query_stream_exact_device_async is the same without any of these
 * host synchronisations.
 * Capacity: sum of max(0, L-m+1) over the contigs always suffices.  With less than the result needs, the call
 * returns LPHB_E_CAPACITY with *n_codes set; it then writes nothing at or past d_codes + codes_capacity, and the
 * contents of d_codes / d_code_offsets are unspecified.                                                            */
int lphb_query_stream_exact_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                                   const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                                   uint64_t codes_capacity, uint64_t* d_code_offsets,
                                   uint64_t* n_codes, void* stream);

/* The exact streaming branch, ASYNCHRONOUS: d_codes and d_code_offsets receive what lphb_query_stream gives for the
 * batch (spurious codes included, as lphb_query_stream_exact_device), d_status[0] the number of codes and
 * d_status[1] the number of contigs holding a non-ACGT byte (4 words; [2] and [3] are not written).  Arguments as in
 * lphb_query_stream_device.  The call returns once the work is enqueued on `stream`: it makes no host
 * synchronisation, no read-back and no pageable copy, and every kernel whose work depends on a count produced on the
 * device reads that count there.  Ordered against the handle's other calls as lphb_query_stream_device; afterwards
 * lphb_mphf_dirty_flags names the batch's dirty contigs and lphb_mphf_stats reports the launches and the main
 * kernel's time, but its dirty_contigs is 0: the count is in d_status[1].
 * Capacity: codes_capacity must be at least sum of max(0, L-m+1) over the contigs, else LPHB_E_CAPACITY (the bound in
 * the message) before anything is enqueued.  The device never writes at or past d_codes + codes_capacity.
 * Workspace: the repair's scratch grows to 68 bytes per contig + 9.03 bytes per base of the batch + 8 bytes per
 * clean code (those it moves) + 12 KB, sized from h_offsets alone; a call that grows it waits for the
 * device while it frees the old buffer (cudaFree), so a pipeline reaches full asynchrony from its second call on
 * batches no larger than the first.  The repair's work grows with the dirty contigs: a clean batch costs the
 * stateless form plus 8 launches and a 48-byte memset that find nothing to do.                                    */
int lphb_query_stream_exact_device_async(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                                         const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                                         uint64_t codes_capacity, uint64_t* d_code_offsets,
                                         uint64_t* d_status, void* stream);

/* Non-streaming branch on device buffers, hf(seq, len, false) (include/partitioned_mphf.hpp:185-195; a non-ACGT
 * byte counts as 'A', include/mphf_utils.hpp:108): every window of k bytes has its code, max(0, L-k+1) per contig,
 * equal to lphb_query_nonstreaming.  Arguments, d_status and ordering as in lphb_query_stream_device (d_status[1]
 * is 0); asynchronous.  The caller's bases are not modified: the kernels read a sanitized copy in the handle's
 * workspace.                                                                                                      */
int lphb_query_nonstreaming_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets,
                                   const uint64_t* h_offsets, uint64_t n_contigs, uint64_t* d_codes,
                                   uint64_t codes_capacity, uint64_t* d_code_offsets,
                                   uint64_t* d_status, void* stream);

/* ---- lookup of packed k-mers -----------------------------------------------------------------
 * The code of each of n k-mers the caller already holds as integers (from a counter, an earlier GPU stage,
 * lphb_colliding_kmers, ...): codes[i] is what the reference's NON-streaming branch
 * (include/partitioned_mphf.hpp:185-195) returns for the window of k bases that kmers[i] encodes - the
 * integer k-mer of string_to_integer_no_reverse (include/mphf_utils.hpp:110-116), its leftmost-minimum
 * m-mer (compute_minimizer_triplet, include/mphf_utils.hpp:118-137) and mphf::query
 * (src/partitioned_mphf.cpp:292-339; for the unpartitioned handle src/unpartitioned_mphf.cpp:191-206).
 *   kmers   n k-mers in the handle's kmer_t layout, kmer_bits / 8 little-endian bytes each: 8 for a
 *           64-bit handle, 16 ({lo, hi}) for a 128-bit one - the layout lphb_colliding_kmers writes.
 *           The first base sits in the most significant of the 2k used bits, A=0 C=1 G=2 T=3
 *           (include/partitioned_mphf.hpp:106-108); bits at position 2k and above are ignored.
 *   codes   n codes in input order: in [0, nkmers) for a member; for any other k-mer the 64-bit value
 *           mphf::query yields (mod 2^64), as every query entry point gives it.
 * HOST buffers in and out; n == 0 does nothing.  lphb_mphf_dirty_flags reports 0 contigs afterwards.      */
int lphb_lookup_kmers(lphb_mphf* f, const void* kmers, uint64_t n, uint64_t* codes);

/* Device-resident variant: d_kmers / d_codes are device pointers on the handle's GPU, d_kmers aligned to
 * kmer_bits / 8 bytes and d_codes to 8; `stream` is a cudaStream_t (NULL = default stream).  Asynchronous,
 * and ordered against the handle's other calls as lphb_query_stream_device is.                             */
int lphb_lookup_kmers_device(lphb_mphf* f, const void* d_kmers, uint64_t n, uint64_t* d_codes, void* stream);

/* ---- the index self-check: build-p --check ---------------------------------------------------------------------
 * Replaces `check` (include/mphf_utils.hpp:51-100; caller src/build.cpp:36-43), which runs three tests over the
 * index's input, contig by contig: check_collisions (every non-streaming code is in range and was not seen before),
 * check_streaming_correctness (the streaming codes equal the non-streaming ones) and check_perfection (every code of
 * 0..nkmers-1 is hit).  Here one kernel does the first two for every window of k bytes of a batch, and the third
 * runs at the end of a SESSION, which spans any number of batches: a unitig file larger than one batch is checked as
 * a stream.  The report does not depend on how the input is split into batches, nor on host versus device form.
 *
 * Definitions, per window of k bytes of the session's contigs, in session order (the k-mer ORDINAL: the position of
 * the window in the non-streaming layout, sum of max(0, L-k+1) over the contigs before it plus its offset):
 *   - its non-streaming code is that of lphb_query_nonstreaming: a non-ACGT byte counts as 'A'
 *     (include/mphf_utils.hpp:108);
 *   - a contig holding a byte outside ACGT/acgt/U/u is DIRTY, whatever its length.  Its windows are checked for
 *     range and collisions like every other, but left out of the streaming comparison: its streaming slots are
 *     unspecified in the stateless layout (lphb_query_stream_device).  The reference compares the two branches
 *     element by element (include/mphf_utils.hpp:83-100), which the streaming branch's spurious codes on such a
 *     contig would fail; on ACGT-only input the verdicts agree (DESIGN.md 4.11);
 *   - a code >= nkmers is OUT OF RANGE.  (The reference tests hash <= nkmers, include/mphf_utils.hpp:58; with a code
 *     equal to nkmers on the key set some code of [0, nkmers) stays unhit, so its perfection test fails and the
 *     overall verdict is the same.)
 * The bitmap of nkmers bits (nkmers / 8 bytes of HBM, kept by the handle and grown only) lives for the session.   */
typedef struct lphb_check_report {
    uint64_t kmers;              /* windows checked: sum of max(0, L-k+1) over the session's contigs        */
    uint64_t contigs, dirty_contigs;
    uint64_t out_of_range;       /* non-streaming codes >= nkmers                                            */
    uint64_t duplicates;         /* in-range hits on a code already hit (= hits - distinct codes hit)        */
    uint64_t missing;            /* codes of [0, nkmers) never hit                                           */
    uint64_t stream_mismatches;  /* windows of clean contigs whose streaming code != non-streaming code      */
    uint64_t first_out_of_range; /* k-mer ordinal in session order; UINT64_MAX if none                       */
    uint64_t first_mismatch;     /* likewise                                                                 */
    uint64_t min_duplicate_code, min_missing_code; /* UINT64_MAX if none                                     */
    int32_t ok;                  /* 1 iff out_of_range, duplicates, missing and stream_mismatches are all 0  */
} lphb_check_report;

/* (Re)starts the handle's session: clears the bitmap and the counters.  Ordered against the handle's other calls.
 * The bitmap holds nkmers bits: LPHB_E_ARG for nkmers >= 2^64 - 32, LPHB_E_NOMEM (with the size) when the device
 * cannot hold it; either way no session is open afterwards and the handle stays usable.                          */
int lphb_check_begin(lphb_mphf* f);

/* One batch of the session, HOST buffers (as lphb_query_stream takes them).  The bases go up in contig-aligned
 * chunks of LPHB_CHUNK_BASES through the query path's staging; the streaming pass runs on the device and no code
 * comes back.  Returns once the caller's buffers may be reused.  LPHB_E_ARG without an open session.              */
int lphb_check_batch(lphb_mphf* f, const char* bases, const uint64_t* offsets, uint64_t n_contigs);

/* The same for a batch in device buffers (arguments as in lphb_query_stream_device), asynchronous on `stream` and
 * ordered against the handle's other calls: queries may run between the batches of a session.  d_stream_codes is
 * optional: when given, it holds the caller's streaming codes of this batch in the layout lphb_query_stream_device
 * writes, and they are compared instead of the library running the streaming pass itself (so that a pipeline can
 * verify codes it already produced).                                                                           */
int lphb_check_batch_device(lphb_mphf* f, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                            uint64_t n_contigs, const uint64_t* d_stream_codes, void* stream);

/* Ends the session: counts the missing codes, synchronises and fills *report.  LPHB_E_ARG without an open session.
 * After a check call lphb_mphf_stats reports that call, lphb_mphf_dirty_flags the last batch's contigs.          */
int lphb_check_end(lphb_mphf* f, lphb_check_report* report);

/* Diagnostic: the flat device image behind the handle (layout: lphash_b200/csrc/device_image.h), e.g. to compare
 * the GPU-side decode of a load with the host-side one (LPHB_HOST_DECODE=1).  Read it with lphb_copy_to_host.  */
int lphb_mphf_device_image(const lphb_mphf* f, const void** d_image, uint64_t* nbytes);

/* Per-contig flags of the last query call on the handle: *d_flags = DEVICE pointer to *n_contigs
 * bytes, nonzero where the contig contains a non-ACGT byte; valid (in stream order) until the next
 * query call on the handle.                                                                        */
int lphb_mphf_dirty_flags(const lphb_mphf* f, const uint8_t** d_flags, uint64_t* n_contigs);

/* ---- build-p Part 1: minimizer / super-k-mer scan -------------------------------------------
 * Replaces the loop over minimizer::from_string (include/minimizer.hpp:11-170; caller
 * src/partitioned_mphf.cpp:70-77) for a batch of contigs.  records receives packed 18-byte
 * mm_record_t {u64 itself, u64 id, u8 p1, u8 size} (include/constants.hpp:26-33) in scan order;
 * mm_count is the running global m-mer ordinal (in: value before the batch, out: after).
 * Bytes other than ACGT/acgt (U/u) are handled as the reference's loop does (include/minimizer.hpp:
 * 138-151): the open super-k-mer is flushed at the byte and the window restarts, m-mer ordinals advance
 * over valid runs only, and a run of exactly k valid bases that is followed by such a byte counts its
 * k-mer in *n_kmers without ever emitting a record for it.  (Clean batches - the unitig sets lphash is
 * built from - take one kernel; a batch with such bytes is cut at them on the device and scanned again.)
 * A batch must hold fewer than 2^32 k-mers and span fewer than 2^32 bases.                         */
int lphb_scan_superkmers(int device, uint32_t k, uint32_t m, uint64_t seed, const char* bases,
                         const uint64_t* offsets, uint64_t n_contigs, uint64_t* mm_count,
                         void* records, uint64_t records_capacity, uint64_t* n_records,
                         uint64_t* n_kmers);

/* Device-resident variant: d_bases / d_offsets are device pointers on `device` (d_bases indexed by
 * the offsets), h_offsets the host copy of the offsets.  Synchronous.  *d_records receives a DEVICE
 * pointer to the packed records (scan order), owned by the library and valid until the next scan
 * call on the device or lphb_scan_release; *kernel_ms (optional) the CUDA-event time of the
 * record-producing kernels.                                                                        */
int lphb_scan_superkmers_device(int device, uint32_t k, uint32_t m, uint64_t seed, const char* d_bases,
                                const uint64_t* d_offsets, const uint64_t* h_offsets, uint64_t n_contigs,
                                uint64_t* mm_count, const void** d_records, uint64_t* n_records,
                                uint64_t* n_kmers, double* kernel_ms);

/* The two build-side entry points keep their device workspace per device between calls (a caller
 * streaming batches does not pay allocation on every batch); this frees it.                      */
int lphb_scan_release(int device);

/* ---- build-p Part 2: sort by minimizer + classify ----------------------------------------------
 * Replaces the sort of the mm_record_t stream by minimizer (external_memory_vector<mm_record_t>,
 * src/partitioned_mphf.cpp:62-66) and minimizer::classify (src/minimizer.cpp:5-50; caller
 * src/partitioned_mphf.cpp:86).  records = n_records packed 18-byte mm_record_t in any order.
 * triplets receives packed 10-byte mm_triplet_t {u64 itself, u8 p1, u8 size}
 * (include/constants.hpp:35-41), one per distinct minimizer in ascending minimizer order -
 * {itself, p1, size} for a minimizer seen once, {itself, 0, 0} for one seen several times - i.e. the
 * key stream PTHash consumes; ids receives the ids of all occurrences of the latter, ascending.
 * n_triplets / n_ids are also set when returning LPHB_E_CAPACITY.                                 */
int lphb_classify(int device, const void* records, uint64_t n_records, void* triplets,
                  uint64_t triplets_capacity, uint64_t* n_triplets, uint64_t* ids,
                  uint64_t ids_capacity, uint64_t* n_ids);

/* Parts 1 + 2 in one call: lphb_scan_superkmers followed by lphb_classify with the record stream
 * kept on the device (what mphf::build does between src/partitioned_mphf.cpp:62 and :86).        */
int lphb_scan_classify(int device, uint32_t k, uint32_t m, uint64_t seed, const char* bases,
                       const uint64_t* offsets, uint64_t n_contigs, uint64_t* mm_count, void* triplets,
                       uint64_t triplets_capacity, uint64_t* n_triplets, uint64_t* ids,
                       uint64_t ids_capacity, uint64_t* n_ids, uint64_t* n_kmers);

/* ---- build-p Parts 1 + 2 over a stream of batches: the build session ----------------------------
 * lphb_scan_classify over an input of any size, fed batch by batch, with host memory bounded by one batch.
 *   Result   triplets and ids are exactly what lphb_scan_classify returns on the concatenation of the session's
 *            batches started at mm_count = 0, i.e. minimizer::classify (src/minimizer.cpp:5-50) over the whole
 *            record stream: one triplet per distinct minimizer in ascending order, the ascending ids of every
 *            occurrence of a minimizer seen more than once.  They do not depend on how the input is cut into
 *            batches, nor on host versus device form.  A batch holds whole contigs; the per-batch limits of
 *            lphb_scan_superkmers hold (fewer than 2^32 k-mers and 2^32 bases each), session totals are 64-bit.
 *            Each batch is scanned and classified on the device as it comes; the session keeps one summary entry
 *            per distinct minimizer of the batch (18 bytes) and the batch's locally colliding ids (8 bytes each),
 *            and lphb_build_end merges them.  The merge runs in slices of at most LPHB_BUILD_SLICE distinct-minimizer
 *            entries (environment variable; default 2^26, about 5 GB of workspace).
 *   Capacity lphb_build_end with a buffer too small for the result (NULL with capacity 0 asks for the sizes) returns
 *            LPHB_E_CAPACITY with *report filled in; the session stays open and keeps the merged result on the device,
 *            so a second call with the reported sizes only copies it out.  A successful end fills *report, frees the
 *            session's device memory and closes the session.
 *   Errors   a batch or an end on a closed session: LPHB_E_ARG.  An end without a batch: an empty result.  A batch
 *            that cannot get its device memory: LPHB_E_NOMEM with the size in the message; that batch is not added
 *            and the session is unchanged and usable (nothing spills to host memory).  A batch that fails otherwise
 *            is not added either.
 *   Threads  calls on one session are serialised by the caller; a batch takes its turn on the device with the
 *            other build-side calls (lphb_scan_*), an end does not.
 * A batch shares the per-device scan workspace of lphb_scan_superkmers (freed by lphb_scan_release).          */
typedef struct lphb_build lphb_build;
typedef struct lphb_build_report {
    uint64_t batches, contigs, kmers; /* kmers: as lphb_scan_classify's n_kmers, summed                    */
    uint64_t mm_count;                /* m-mer ordinals consumed (the running mm_count)                     */
    uint64_t records;                 /* super-k-mers of Part 1 (the CSV's total_minimizers)                */
    uint64_t n_triplets, n_ids, colliding_minimizers; /* set by lphb_build_end; triplets of size 0 last    */
    uint64_t device_bytes;            /* HBM the session holds (at an end: before it frees it)              */
} lphb_build_report;
/* k, m, seed as for lphb_scan_superkmers.  LPHB_E_ARG for k/m out of range before any CUDA call. */
int lphb_build_begin(int device, uint32_t k, uint32_t m, uint64_t seed, lphb_build** out);
/* One batch in HOST buffers (as lphb_scan_superkmers takes it).  Returns once the batch is in the session. */
int lphb_build_batch(lphb_build* b, const char* bases, const uint64_t* offsets, uint64_t n_contigs);
/* One batch in DEVICE buffers on the session's device (arguments as lphb_scan_superkmers_device).  SYNCHRONOUS:
 * it first waits for `stream` (a cudaStream_t, NULL = default stream), on which the caller wrote the buffers, and
 * returns once the caller's buffers may be reused.                                                               */
int lphb_build_batch_device(lphb_build* b, const char* d_bases, const uint64_t* d_offsets, const uint64_t* h_offsets,
                            uint64_t n_contigs, void* stream);
/* triplets: packed 10-byte mm_triplet_t as lphb_classify writes them; capacities count triplets and ids. */
int lphb_build_end(lphb_build* b, void* triplets, uint64_t triplets_capacity, uint64_t* ids, uint64_t ids_capacity,
                   lphb_build_report* report);
/* Frees the session, open or closed (NULL: nothing to do). */
int lphb_build_free(lphb_build* b);

/* ---- build-p Part 3: the inverted index --------------------------------------------------------
 * Replaces the loop that re-keys every triplet by minimizer_order(itself) and sorts the result
 * (src/partitioned_mphf.cpp:92-106) and mphf::build_inverted_index (src/partitioned_mphf.cpp:163-268):
 * type of every distinct minimizer, the quartet wavelet tree with its rank directories
 * (src/quartet_wtree.cpp:13-53, include/rs_bit_vector.hpp:120-156), the four size / position lists and
 * the Elias-Fano encoding of their prefix sums (include/ef_sequence.hpp:36-75) with its darray1 select
 * index (pthash/include/encoders/darray.hpp:13-48).
 * minimizer_order = the serialized pthash::single_phf built on the distinct minimizers (the bytes
 * essentials::save writes for it; PTHash construction itself stays with the caller); triplets = the
 * packed 10-byte mm_triplet_t of lphb_classify, one per distinct minimizer, in any order.
 * out receives, byte for byte as in the `.lph` file, the image of `wtree` followed by the image of
 * `sizes_and_positions` (include/partitioned_mphf.hpp:213-214); info the four counters stored in front
 * of them.  lphb_inverted_index_bound(n) is a capacity that always suffices; *out_bytes is also set
 * when returning LPHB_E_CAPACITY.  LPHB_E_ARG if minimizer_order is not a bijection of the triplets'
 * minimizers onto [0, n_triplets).                                                                   */
typedef struct lphb_inverted_index {
    uint64_t n_maximal, right_coll_sizes_start, none_sizes_start, none_pos_start; /* include/partitioned_mphf.hpp:208-211 */
    uint64_t colliding_minimizers; /* triplets of size 0 */
    uint64_t universe;             /* last prefix sum (src/partitioned_mphf.cpp:267) */
    uint64_t wtree_bytes, ef_bytes; /* the two images inside out */
    double device_ms;              /* CUDA-event time of the kernels, copies excluded */
} lphb_inverted_index;
uint64_t lphb_inverted_index_bound(uint64_t n_triplets);
int lphb_build_inverted_index(int device, uint32_t k, uint32_t m, const void* minimizer_order,
                              uint64_t minimizer_order_bytes, const void* triplets, uint64_t n_triplets,
                              void* out, uint64_t out_capacity, uint64_t* out_bytes,
                              lphb_inverted_index* info);

/* The same for the unpartitioned variant (build-u, lphash::mphf_alt; src/unpartitioned_mphf.cpp:78-96 re-key and
 * :152-169 build_pos_index / build_size_index): out receives the image of `positions` (Elias-Fano of the prefix sums
 * of p1 in minimizer_order order) followed by the image of `sizes` (include/unpartitioned_mphf.hpp:206-207);
 * lphb_inverted_index_bound(n_triplets) suffices as capacity.                                              */
typedef struct lphb_inverted_index_alt {
    uint64_t num_kmers_in_main_index;      /* last prefix sum of the sizes (src/unpartitioned_mphf.cpp:168) */
    uint64_t positions_bytes, sizes_bytes; /* the two images inside out */
    double device_ms;
} lphb_inverted_index_alt;
int lphb_build_inverted_index_alt(int device, const void* minimizer_order, uint64_t minimizer_order_bytes,
                                  const void* triplets, uint64_t n_triplets, void* out, uint64_t out_capacity,
                                  uint64_t* out_bytes, lphb_inverted_index_alt* info);
int lphb_lph_assemble_alt(uint32_t k, uint32_t m, uint64_t mm_seed, uint64_t nkmers, uint64_t distinct_minimizers,
                          const lphb_inverted_index_alt* index, const void* minimizer_order,
                          uint64_t minimizer_order_bytes, const void* index_body, uint64_t index_body_bytes,
                          const void* fallback_kmer_order, uint64_t fallback_bytes, void* out,
                          uint64_t out_capacity, uint64_t* out_bytes);

/* ---- the `.lph` writer (host only) ------------------------------------------------------------
 * lphb_lph_assemble lays out a complete serialized lphash::mphf in the visitor order of
 * include/partitioned_mphf.hpp:204-219 - what essentials::save(hf, file) writes (src/build.cpp:52) -
 * from the header fields, the two serialized single_phf objects (built by PTHash on the caller's side)
 * and the index body of lphb_build_inverted_index.  The result loads with the reference's
 * essentials::load and with lphb_mphf_load_memory.
 * lphb_lph_sections reports where the parts of an existing image start: minimizer_order, the wavelet
 * tree (alt: positions), sizes_and_positions (alt: sizes), fallback_kmer_order, end of the image.   */
int lphb_lph_assemble(uint32_t k, uint32_t m, uint64_t mm_seed, uint64_t nkmers, uint64_t distinct_minimizers,
                      const lphb_inverted_index* index, const void* minimizer_order,
                      uint64_t minimizer_order_bytes, const void* index_body, uint64_t index_body_bytes,
                      const void* fallback_kmer_order, uint64_t fallback_bytes, void* out,
                      uint64_t out_capacity, uint64_t* out_bytes);
int lphb_lph_sections(const void* image, uint64_t nbytes, int kmer_bits, int alt, uint64_t sections[5]);

/* ---- build-p Part 4: k-mers of colliding minimizers -----------------------------------------
 * Replaces the loop over minimizer::get_colliding_kmers (include/minimizer.hpp:172-319; caller
 * src/partitioned_mphf.cpp:120-129).  ids = ascending minimizer-occurrence ids (classify's second
 * output).  kmers receives kmer_bits/8 little-endian bytes per k-mer, in scan order.            */
int lphb_colliding_kmers(int device, uint32_t k, uint32_t m, uint64_t seed, const char* bases,
                         const uint64_t* offsets, uint64_t n_contigs, uint64_t* mm_count,
                         const uint64_t* ids, uint64_t n_ids, int kmer_bits, void* kmers,
                         uint64_t kmers_capacity, uint64_t* n_kmers);

/* ---- pinned host memory (optional; makes the copies inside lphb_query_stream asynchronous) -- */
int lphb_host_alloc(void** ptr, uint64_t nbytes);
/* synchronous copy of a library-owned device buffer (e.g. *d_records of lphb_scan_superkmers_device) */
int lphb_copy_to_host(int device, void* dst, const void* d_src, uint64_t nbytes);
int lphb_host_free(void* ptr);

/* Counters for the last lphb_query_* or lphb_lookup_kmers* call on the handle (kernel launches, device ms). */
typedef struct lphb_stats {
    uint64_t kernel_launches;
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t dirty_contigs;
    double kernel_ms; /* mean CUDA-event time of the main query kernel over the calls since the last
                         lphb_mphf_stats (most recent 128) */
} lphb_stats;
int lphb_mphf_stats(const lphb_mphf* f, lphb_stats* stats);

#ifdef __cplusplus
}
#endif
#endif /* LPHASH_B200_H */
