// TEST INFRASTRUCTURE — NOT PRODUCT CODE.  The product (lphash_b200/) never links, imports or
// executes anything in oracle/; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
// --impl reference legs do, and only as the checker / the reported CPU baseline.
//
// CPU restatement ("oracle") of the hot path of jermp/lphash @ 9af2242 (pthash @ 561e513):
// the streaming query of the partitioned LP-MPHF and the build-side minimizer / super-k-mer
// scan.  Written from the reference's semantics, not from its text: one flat `.lph` image,
// plain functions, k-mers always held in 128 bits with the fallback-hash flavour chosen at load
// time.  Every function cites the reference lines it restates ("ref:" = /root/reference/,
// "pthash/" = external/pthash/).
//
// PARITY IS PINNED: tests/test_oracle_vs_reference.py checks this file against what the unmodified
// reference (compiled into oracle/_ref/ by oracle/build_ref.sh) returned on its own bundled data
// (BASELINE config 1: se.ust.k31 index k=31 m=16 128-bit, the three bundled query files incl. the
// non-ACGT streaming quirk of ecoli1.fasta and the FASTQ, and the from_string stream; inputs and
// expected outputs committed under tests/golden/config1/ by tools/make_config1.py - the folds are
// those of SURVEY.md section 8c), and tests/test_oracle_golden.py checks it against the committed
// golden fixtures in tests/golden/ (8 (k, m, kmer_t) combinations, generated from the reference by
// tools/make_golden.py), so that the pin also holds on the GPU box where /root/reference does not exist.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

typedef uint64_t u64;
typedef unsigned __int128 u128;

namespace orc {

// ---------------------------------------------------------------------------------------------
// a1  ASCII -> 2-bit.  ref: src/constants.cpp:5-13 (A/a=0 C/c=1 G/g=2 T/t/U/u=3, else 4)
// ---------------------------------------------------------------------------------------------
static inline int nt4(unsigned char ch) {
    switch (ch) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': case 'U': case 'u': return 3;
        default: return 4;
    }
}

// ---------------------------------------------------------------------------------------------
// a3  MurmurHash2-64 of one 8-byte word.  ref: pthash/include/utils/hasher.hpp:46-110 with
//     len == 8 (one block, empty tail), :175-177 (murmurhash2_64::hash(uint64_t)), :112-114
//     (default_hash64).
// ---------------------------------------------------------------------------------------------
static inline u64 murmur64(u64 v, u64 seed) {
    const u64 M = 0xc6a4a7935bd1e995ULL;
    u64 h = seed ^ (8 * M);
    u64 x = v * M;
    x ^= x >> 47;
    x *= M;
    h ^= x;
    h *= M;
    h ^= h >> 47;
    h *= M;
    h ^= h >> 47;
    return h;
}

// fastmod.  ref: pthash/external/fastmod/fastmod.h:56-63 (mul128_u64), :159-162 (fastmod_u64).
static inline u64 fastmod_u64(u64 a, u128 M, u64 d) {
    u128 low = M * a;  // mod 2^128
    u128 bottom = ((low & ~u64(0)) * d) >> 64;
    u128 top = (low >> 64) * d;
    return u64((bottom + top) >> 64);
}

// ---------------------------------------------------------------------------------------------
// Flat views of the serialized containers.  Serialization = essentials visitor: PODs raw
// little-endian, vector<T> = u64 n + n*sizeof(T) bytes.
// ref: pthash/external/essentials/include/essentials.hpp:98-119, 268-306.
// ---------------------------------------------------------------------------------------------
struct Reader {
    const unsigned char* p;
    const unsigned char* end;
    template <class T>
    T pod() {
        if (size_t(end - p) < sizeof(T)) throw std::runtime_error("lph: truncated file");
        T v;
        std::memcpy(&v, p, sizeof(T));
        p += sizeof(T);
        return v;
    }
    template <class T>
    std::vector<T> vec() {
        u64 n = pod<u64>();
        if (n > u64(end - p) / sizeof(T)) throw std::runtime_error("lph: truncated vector");
        std::vector<T> v(n);
        if (n) std::memcpy(v.data(), p, n * sizeof(T));
        p += n * sizeof(T);
        return v;
    }
};

// a8  compact_vector.  ref: pthash/include/encoders/compact_vector.hpp:229-234 (access; the
// unaligned 8-byte load is restated as a two-word funnel, identical for width <= 57), :277-283.
struct CompactVec {
    u64 size = 0, width = 0, mask = 0;
    std::vector<u64> bits;
    void read(Reader& r) {
        size = r.pod<u64>();
        width = r.pod<u64>();
        mask = r.pod<u64>();
        bits = r.vec<u64>();
    }
    u64 get(u64 i) const {
        if (width == 0) return 0;  // E1(i): width-0 low-bits vector is legal; mask == 0
        u64 pos = i * width, wd = pos >> 6, sh = pos & 63;
        u64 v = bits[wd] >> sh;
        if (sh && wd + 1 < bits.size()) v |= bits[wd + 1] << (64 - sh);
        return v & mask;
    }
};

// bit_vector.  ref: pthash/include/encoders/bit_vector.hpp:149-310.
struct BitVec {
    u64 nbits = 0;
    std::vector<u64> w;
    void read(Reader& r) {
        nbits = r.pod<u64>();
        w = r.vec<u64>();
    }
    int bit(u64 i) const { return int(w[i >> 6] >> (i & 63) & 1); }
    // position of the first set bit at or after `pos` (unary_iterator(bv,pos).next(), :235-258)
    u64 next_one(u64 pos) const {
        u64 wd = pos >> 6;
        u64 cur = w[wd] & (~u64(0) << (pos & 63));
        while (cur == 0) cur = w[++wd];
        return (wd << 6) + u64(__builtin_ctzll(cur));
    }
};

// position of the r-th (0-based) set bit of x.  ref: pthash/include/encoders/util.hpp:54-97.
static inline unsigned select_in_word(u64 x, unsigned r) {
    for (unsigned i = 0; i < r; ++i) x &= x - 1;
    return unsigned(__builtin_ctzll(x));
}

// a9  darray1 select.  ref: pthash/include/encoders/darray.hpp:51-76 (block 1024, subblock 32),
// serialized fields :88-94.
struct DArray {
    u64 positions = 0;
    std::vector<int64_t> block_inv;
    std::vector<uint16_t> sub_inv;
    std::vector<u64> overflow;
    void read(Reader& r) {
        positions = r.pod<u64>();
        block_inv = r.vec<int64_t>();
        sub_inv = r.vec<uint16_t>();
        overflow = r.vec<u64>();
    }
    u64 select(BitVec const& bv, u64 idx) const {
        int64_t bp = block_inv[idx / 1024];
        if (bp < 0) return overflow[u64(-bp - 1) + (idx & 1023)];
        u64 start = u64(bp) + sub_inv[idx / 32];
        u64 rem = idx & 31;
        if (rem == 0) return start;
        u64 wd = start >> 6;
        u64 cur = bv.w[wd] & (~u64(0) << (start & 63));
        for (;;) {
            u64 pc = u64(__builtin_popcountll(cur));
            if (rem < pc) break;
            rem -= pc;
            cur = bv.w[++wd];
        }
        return (wd << 6) + select_in_word(cur, unsigned(rem));
    }
};

// a9/a12  Elias-Fano.  Both pthash::ef_sequence<false> (free_slots,
// pthash/include/encoders/ef_sequence.hpp:55-59, 94-99) and lphash::ef_sequence
// (sizes_and_positions, ref: include/ef_sequence.hpp:77-99, 107-112) serialize as
// {high bit_vector, darray1, low compact_vector} and share access(); pair()/diff() exist only
// on the lphash one.
struct EliasFano {
    BitVec high;
    DArray d1;
    CompactVec low;
    void read(Reader& r) {
        high.read(r);
        d1.read(r);
        low.read(r);
    }
    u64 size() const { return low.size; }
    u64 access(u64 i) const { return ((d1.select(high, i) - i) << low.width) | low.get(i); }
    void pair(u64 i, u64& v1, u64& v2) const {
        u64 l = low.width;
        u64 pos = d1.select(high, i);
        u64 nxt = high.next_one(pos + 1);
        v1 = ((pos - i) << l) | low.get(i);
        v2 = ((nxt - i - 1) << l) | low.get(i + 1);
    }
    u64 diff(u64 i) const {
        u64 a, b;
        pair(i, a, b);
        return b - a;
    }
};

// a11  rank9-style bit vector.  ref: include/rs_bit_vector.hpp:27-36 (rank), :101-114
// (sub_block_rank), :91-96 (fields), :24 (num_ones = pairs[size-2]).
struct RankVec {
    BitVec bv;
    std::vector<u64> pairs, hints;
    void read(Reader& r) {
        bv.read(r);
        pairs = r.vec<u64>();
        hints = r.vec<u64>();
    }
    u64 rank1(u64 pos) const {
        if (pos == bv.nbits) return pairs[pairs.size() - 2];
        u64 word = pos / 64, block = word / 8, left = word % 8;
        u64 r = pairs[2 * block] + ((pairs[2 * block + 1] >> ((7 - left) * 9)) & 0x1FF);
        u64 sub = pos % 64;
        if (sub) r += u64(__builtin_popcountll(bv.w[word] << (64 - sub)));
        return r;
    }
    u64 rank(int bit, u64 pos) const { return bit ? rank1(pos) : pos - rank1(pos); }
};

// a7/a13  pthash::single_phf<*, dictionary_dictionary, true> evaluation.
// ref: pthash/include/single_phf.hpp:50-65 (operator(), position), :88-97 (fields);
// pthash/include/utils/bucketers.hpp:17-22, 40-46; pthash/include/encoders/encoders.hpp:167-176
// (dictionary), :268-277 (dual).
struct SinglePhf {
    u64 seed = 0, num_keys = 0, table_size = 0;
    u128 M = 0;
    u64 dense = 0, sparse = 0;
    u128 M_dense = 0, M_sparse = 0;
    CompactVec front_ranks, front_dict, back_ranks, back_dict;
    EliasFano free_slots;
    void read(Reader& r) {
        seed = r.pod<u64>();
        num_keys = r.pod<u64>();
        table_size = r.pod<u64>();
        M = r.pod<u128>();
        dense = r.pod<u64>();
        sparse = r.pod<u64>();
        M_dense = r.pod<u128>();
        M_sparse = r.pod<u128>();
        front_ranks.read(r);
        front_dict.read(r);
        back_ranks.read(r);
        back_dict.read(r);
        free_slots.read(r);
    }
    u64 bucket(u64 h) const {
        // T = (uint64_t)(0.6 * UINT64_MAX) evaluated in double: 0.6*(2^64) rounded to 53 bits
        const u64 T = 0x9999999999999800ULL;
        return h < T ? fastmod_u64(h, M_dense, dense) : dense + fastmod_u64(h, M_sparse, sparse);
    }
    u64 pilot(u64 b) const {
        if (b < front_ranks.size) return front_dict.get(front_ranks.get(b));
        b -= front_ranks.size;
        return back_dict.get(back_ranks.get(b));
    }
    u64 position(u64 h) const {
        u64 hp = murmur64(pilot(bucket(h)), seed);
        u64 p = fastmod_u64(h ^ hp, M, table_size);
        return p < num_keys ? p : free_slots.access(p - num_keys);
    }
};

enum { LEFT = 0, RIGHT_OR_COLLISION = 1, MAXIMAL = 2, NONE = 3, COLLISION = 4 };

// The whole `.lph` file.  Field order ref: include/partitioned_mphf.hpp:204-219,
// include/quartet_wtree.hpp:43-48.
struct Mphf {
    unsigned k = 0, m = 0;
    u64 mm_seed = 0, nkmers = 0, distinct = 0, n_maximal = 0, right_start = 0, none_sizes_start = 0,
        none_pos_start = 0;
    SinglePhf minimizer_order, fallback;
    RankVec root, left_right, max_none;
    EliasFano sp;  // sizes_and_positions
    int kmer_bits = 64;
    u64 file_bytes = 0;

    void parse(const unsigned char* data, u64 n) {
        Reader r{data, data + n};
        k = r.pod<uint8_t>();
        m = r.pod<uint8_t>();
        mm_seed = r.pod<u64>();
        nkmers = r.pod<u64>();
        distinct = r.pod<u64>();
        n_maximal = r.pod<u64>();
        right_start = r.pod<u64>();
        none_sizes_start = r.pod<u64>();
        none_pos_start = r.pod<u64>();
        minimizer_order.read(r);
        root.read(r);
        left_right.read(r);
        max_none.read(r);
        sp.read(r);
        fallback.read(r);
        if (r.p != r.end) throw std::runtime_error("lph: trailing bytes");
        file_bytes = n;
    }

    // a13  fallback_hasher.  ref: include/constants.hpp:56-70.
    u64 fallback_order(u128 kmer) const {
        u64 lo = u64(kmer), hi = u64(kmer >> 64);
        u64 h = kmer_bits == 64 ? murmur64(lo, fallback.seed)
                                : (murmur64(lo, fallback.seed) ^ murmur64(hi, ~fallback.seed));
        return fallback.position(h);
    }

    // a10  quartet_wtree::rank_of.  ref: src/quartet_wtree.cpp:84-99.
    void rank_of(u64 idx, int& type, u64& rank) const {
        int msb = root.bv.bit(idx);
        u64 r = root.rank(msb, idx);
        RankVec const& leaf = msb ? max_none : left_right;
        int lsb = leaf.bv.bit(r);
        rank = leaf.rank(lsb, r);
        type = (msb << 1) | lsb;
    }

    struct Ctx {
        u64 hval = 0, global_rank = 0, local_rank = 0;
        int type = 0;
    };

    // a6  mphf::query.  ref: src/partitioned_mphf.cpp:292-339.  All arithmetic mod 2^64.
    Ctx query(u128 kmer, u64 minimizer, u64 position) const {
        Ctx c;
        u64 w = k - m + 1;
        u64 bucket = minimizer_order.position(murmur64(minimizer, minimizer_order.seed));
        int type;
        u64 rk;
        rank_of(bucket, type, rk);
        u64 maximal_block = w * n_maximal;
        switch (type) {
            case LEFT:
                c.global_rank = sp.access(rk) + maximal_block;
                c.local_rank = position;
                c.type = LEFT;
                break;
            case RIGHT_OR_COLLISION: {
                u64 v1, v2;
                sp.pair(right_start + rk, v1, v2);
                if (v2 - v1 == 0) {
                    c.global_rank = sp.access(none_pos_start) + maximal_block;
                    c.local_rank = fallback_order(kmer);
                    c.type = COLLISION;
                } else {
                    c.global_rank = v1 + maximal_block;
                    c.local_rank = u64(k - m) - position;
                    c.type = RIGHT_OR_COLLISION;
                }
            } break;
            case MAXIMAL:
                c.global_rank = w * rk;
                c.local_rank = position;
                c.type = MAXIMAL;
                break;
            default:  // NONE
                c.global_rank = sp.access(none_sizes_start + rk) + maximal_block;
                c.local_rank = sp.diff(none_pos_start + rk) - position;
                c.type = NONE;
        }
        c.hval = c.global_rank + c.local_rank;
        return c;
    }

    // a2-a5  mphf::operator()(contig, len, streaming=true), INCLUDING the non-ACGT quirk (Q1):
    // on an invalid byte only the run length and the ring cursor are reset, so stale ring
    // entries / stale minimum slot can trigger a rescan and a spurious output while the new run
    // is still shorter than k.  ref: include/partitioned_mphf.hpp:73-184.
    void streaming(const char* s, u64 len, std::vector<u64>& out) const {
        if (len < k) return;
        const u64 w = k - m + 1;
        const u64 mm_mask = (u64(1) << (2 * m)) - 1;
        const u128 km_mask = (u128(1) << (2 * k)) - 1;
        struct Slot {
            u64 mmer = 0, hash = 0;
        };
        std::vector<Slot> ring(w);
        u64 cursor = 0, min_slot = w;  // min_slot == w: "no minimum yet"
        u64 mmer = 0, run = 0;
        u128 kmer = 0;
        u64 p1 = 0;
        Ctx ctx;
        for (u64 i = 0; i < len; ++i) {
            int c = nt4((unsigned char)s[i]);
            if (c > 3) {  // hpp:179-183: nothing else is reset
                run = 0;
                cursor = 0;
                continue;
            }
            mmer = ((mmer << 2) | u64(c)) & mm_mask;
            kmer = ((kmer << 2) | u128(c)) & km_mask;
            ++run;
            if (run < m) continue;
            enum { KEEP, RESCAN, NEWCOMER } action = KEEP;
            if (cursor == min_slot) action = RESCAN;  // the minimum's slot is being overwritten
            ring[cursor].mmer = mmer;
            ring[cursor].hash = murmur64(mmer, mm_seed);
            if (run == k) {
                action = RESCAN;  // first full window
            } else if (run > k && ring[min_slot].hash > ring[cursor].hash) {
                p1 = k - m;
                min_slot = cursor;
                action = NEWCOMER;
            }
            if (action == KEEP) {
                if (run >= k) {  // same super-k-mer: slide by one (hpp:131-145)
                    if (ctx.type == COLLISION) ctx.local_rank = fallback_order(kmer);
                    else if (ctx.type == RIGHT_OR_COLLISION || ctx.type == NONE) ++ctx.local_rank;
                    else --ctx.local_rank;
                    ctx.hval = ctx.global_rank + ctx.local_rank;
                    out.push_back(ctx.hval);
                }
            } else {
                if (action == RESCAN) {
                    // hpp:146-165: candidates visited oldest-first starting after the cursor;
                    // strict '>' keeps the earliest visited on ties.  The second sweep runs up
                    // to and including slot (cursor+2)%w, i.e. it revisits slots (harmless:
                    // a revisited slot can never be strictly smaller than the current best).
                    min_slot = (cursor + 1) % w;
                    p1 = 0;
                    u64 step = 1;
                    for (u64 j = (cursor + 2) % w; j < w; ++j, ++step)
                        if (ring[min_slot].hash > ring[j].hash) min_slot = j, p1 = step;
                    for (u64 j = 0; j <= (cursor + 2) % w; ++j, ++step)
                        if (ring[min_slot].hash > ring[j].hash) min_slot = j, p1 = step;
                }
                ctx = query(kmer, ring[min_slot].mmer, p1);
                out.push_back(ctx.hval);
            }
            cursor = (cursor + 1) % w;
        }
    }

    // S1  the stateless definition the GPU path implements: for every window of k valid bases,
    // code = query(kmer, leftmost-minimum m-mer, its offset).  Equals streaming() on ACGT-only
    // contigs; on contigs with invalid bytes it yields the codes of the valid k-mers only (the
    // reference's output minus its spurious entries).  cf. the reference's own stateless branch,
    // include/partitioned_mphf.hpp:185-195 + include/mphf_utils.hpp:118-137 (rightmost-to-left
    // scan with '<=' == leftmost minimum).
    void stateless(const char* s, u64 len, std::vector<u64>& out, std::vector<u64>* positions) const {
        if (len < k) return;
        const u64 w = k - m + 1;
        const u64 mm_mask = (u64(1) << (2 * m)) - 1;
        for (u64 i = 0; i + k <= len; ++i) {
            u128 kmer = 0;
            bool ok = true;
            for (u64 j = 0; j < k; ++j) {
                int c = nt4((unsigned char)s[i + j]);
                if (c > 3) { ok = false; break; }
                kmer = (kmer << 2) | u128(c);
            }
            if (!ok) continue;
            u64 best_hash = 0, best_mmer = 0, best_pos = 0;
            for (u64 p = 0; p < w; ++p) {
                u64 mmer = u64(kmer >> (2 * (k - m - p))) & mm_mask;
                u64 h = murmur64(mmer, mm_seed);
                if (p == 0 || h < best_hash) best_hash = h, best_mmer = mmer, best_pos = p;
            }
            out.push_back(query(kmer, best_mmer, best_pos).hval);
            if (positions) positions->push_back(i);
        }
    }
};

// ---------------------------------------------------------------------------------------------
// a14  minimizer::from_string, sequential restatement incl. its behaviour around invalid bytes
//      (Q3).  ref: include/minimizer.hpp:11-170.  Record = mm_record_t, ref:
//      include/constants.hpp:26-33 (18 bytes, pack(2)).
// ---------------------------------------------------------------------------------------------
#pragma pack(push, 2)
struct Record {
    u64 itself, id;
    uint8_t p1, size;
};
struct Triplet {
    u64 itself;
    uint8_t p1, size;
};
#pragma pack(pop)
static_assert(sizeof(Record) == 18 && sizeof(Triplet) == 10, "packed layouts");

static u64 from_string(const char* s, u64 len, unsigned k, unsigned m, u64 seed, u64& mm_count,
                       std::vector<Record>& out) {
    const u64 w = k - m + 1;
    const u64 mm_mask = (u64(1) << (2 * m)) - 1;
    struct Slot {
        u64 mmer = 0, hash = 0, id = 0;
    };
    std::vector<Slot> ring(w);
    u64 cursor = 0, min_slot = w, run = 0, mmer = 0, kmers = 0;
    unsigned run_len = 0, p1 = 0;  // run_len = k-mers in the open super-k-mer
    auto emit = [&](Slot const& sl) {
        out.push_back(Record{sl.mmer, sl.id, uint8_t(p1), uint8_t(run_len)});
    };
    auto first_window = [&]() {  // :61-78 / :153-163: '<' keeps the leftmost on ties
        min_slot = 0;
        p1 = 0;
        for (u64 j = 0; j < w; ++j)
            if (ring[j].hash < ring[min_slot].hash) min_slot = j, p1 = unsigned(j);
        run_len = 1;
    };
    for (u64 i = 0; i < len; ++i) {
        int c = nt4((unsigned char)s[i]);
        if (c > 3) {  // :136-151
            run = 0;
            if (min_slot < w) emit(ring[min_slot]);
            run_len = 0;
            min_slot = w;
            cursor = 0;
            continue;
        }
        mmer = ((mmer << 2) | u64(c)) & mm_mask;
        ++run;
        if (run < m) continue;
        Slot cur;
        cur.mmer = mmer;
        cur.hash = murmur64(mmer, seed);
        cur.id = mm_count++;
        bool rescan = false;
        if (run == k) ++kmers;
        if (run == k + 1) first_window();  // the first window is resolved one base late
        if (run >= k + 1) {
            if (cursor % w == min_slot) {  // minimum leaves the window
                emit(ring[min_slot]);
                run_len = 0;
                rescan = true;
            } else if (cur.hash < ring[min_slot].hash) {  // strictly smaller newcomer
                emit(ring[min_slot]);
                run_len = 0;
                p1 = k - m;
                min_slot = cursor;
            }
            ++run_len;
            ++kmers;
        }
        ring[cursor] = cur;
        cursor = (cursor + 1) % w;
        if (rescan) {  // :103-131, oldest-first, strict '>' keeps the leftmost
            min_slot = cursor;
            p1 = 0;
            unsigned step = 1;
            for (u64 j = (cursor + 1) % w; j < w; ++j, ++step)
                if (ring[min_slot].hash > ring[j].hash) min_slot = j, p1 = step;
            for (u64 j = 0; j <= cursor; ++j, ++step)
                if (ring[min_slot].hash > ring[j].hash) min_slot = j, p1 = step;
        }
    }
    if (run == k) first_window();
    if (min_slot < w) emit(ring[min_slot]);
    return kmers;
}

// S2'  the stateless definition of the same stream for ACGT-only contigs (what the GPU scan
// kernel implements): b(i) = leftmost argmin over m-mer offsets i..i+w-1; a record starts
// wherever b(i) != b(i-1).  Contigs are assumed clean (callers check).
static u64 scan_stateless(const char* s, u64 len, unsigned k, unsigned m, u64 seed, u64& mm_count,
                          std::vector<Record>& out) {
    if (len < m) return 0;
    const u64 w = k - m + 1, n_mm = len - m + 1;
    const u64 mm_mask = (u64(1) << (2 * m)) - 1;
    u64 id_base = mm_count;
    mm_count += n_mm;
    if (len < k) return 0;
    std::vector<u64> mmers(n_mm), hashes(n_mm);
    u64 mmer = 0;
    for (u64 i = 0; i < len; ++i) {
        mmer = ((mmer << 2) | u64(nt4((unsigned char)s[i]))) & mm_mask;
        if (i + 1 >= m) mmers[i + 1 - m] = mmer, hashes[i + 1 - m] = murmur64(mmer, seed);
    }
    u64 nk = len - k + 1, prev = ~u64(0);
    for (u64 i = 0; i < nk; ++i) {
        u64 b = i;
        for (u64 j = i + 1; j < i + w; ++j)
            if (hashes[j] < hashes[b]) b = j;
        if (b != prev) {
            out.push_back(Record{mmers[b], id_base + b, uint8_t(b - i), 1});
            prev = b;
        } else {
            ++out.back().size;
        }
    }
    return nk;
}

// a16  minimizer::classify over records sorted by minimizer.  ref: src/minimizer.cpp:5-50.
// Singletons -> {itself,p1,size}; groups -> one {itself,0,0} + all their ids (ascending).
static void classify(std::vector<Record> recs, std::vector<Triplet>& uniq, std::vector<u64>& ids) {
    std::stable_sort(recs.begin(), recs.end(),
                     [](Record const& a, Record const& b) { return a.itself < b.itself; });
    for (size_t i = 0; i < recs.size();) {
        size_t j = i + 1;
        while (j < recs.size() && recs[j].itself == recs[i].itself) ++j;
        if (j - i == 1) {
            uniq.push_back(Triplet{recs[i].itself, recs[i].p1, recs[i].size});
        } else {
            uniq.push_back(Triplet{recs[i].itself, 0, 0});
            for (size_t t = i; t < j; ++t) ids.push_back(recs[t].id);
        }
        i = j;
    }
    std::sort(ids.begin(), ids.end());
}

// a15  get_colliding_kmers, sequential restatement incl. its behaviour around invalid bytes: the same window
// walk as from_string with the k-mers of the open super-k-mer buffered; a super-k-mer is written out when it closes
// and the id of its minimizer occurrence is the next one of the ascending id list (one forward cursor, as the
// reference's `itr`).  ref: include/minimizer.hpp:172-319; caller src/partitioned_mphf.cpp:120-129.
static void colliding_kmers_contig(const char* s, u64 len, unsigned k, unsigned m, u64 seed, const u64* ids, u64 n_ids,
                                   u64& next_id, u64& mm_count, std::vector<u128>& out) {
    const u64 w = k - m + 1;
    const u64 mm_mask = (u64(1) << (2 * m)) - 1;
    const u128 km_mask = (u128(1) << (2 * k)) - 1;
    struct Slot {
        u64 hash = 0, id = 0;
    };
    std::vector<Slot> ring(w);
    std::vector<u128> open;  // k-mers of the open super-k-mer
    u64 cursor = 0, min_slot = w, run = 0, mmer = 0;
    u128 kmer = 0;
    auto close = [&]() {  // :241-246, :287-291, :311-316
        if (next_id < n_ids && ids[next_id] == ring[min_slot].id) {
            out.insert(out.end(), open.begin(), open.end());
            ++next_id;
        }
    };
    auto first_window = [&]() {  // :226-232 / :303-309
        min_slot = 0;
        for (u64 j = 0; j < w; ++j)
            if (ring[j].hash < ring[min_slot].hash) min_slot = j;
    };
    for (u64 i = 0; i < len; ++i) {
        int c = nt4((unsigned char)s[i]);
        if (c > 3) {  // :283-300
            run = 0;
            if (min_slot < w) close();
            open.clear();
            min_slot = w;
            cursor = 0;
            continue;
        }
        mmer = ((mmer << 2) | u64(c)) & mm_mask;
        kmer = ((kmer << 2) | u128(c)) & km_mask;
        ++run;
        if (run < m) continue;
        Slot cur;
        cur.hash = murmur64(mmer, seed);
        cur.id = mm_count++;
        bool rescan = false;
        if (run == k + 1) first_window();
        if (run >= k + 1) {
            if (cursor % w == min_slot || cur.hash < ring[min_slot].hash) {  // :238-256
                close();
                open.clear();
                if (cursor % w == min_slot) rescan = true;
                else min_slot = cursor;
            }
        }
        ring[cursor] = cur;
        cursor = (cursor + 1) % w;
        if (run >= k) open.push_back(kmer);
        if (rescan) {  // :265-276
            min_slot = cursor;
            for (u64 j = (cursor + 1) % w; j < w; ++j)
                if (ring[min_slot].hash > ring[j].hash) min_slot = j;
            for (u64 j = 0; j <= cursor; ++j)
                if (ring[min_slot].hash > ring[j].hash) min_slot = j;
        }
    }
    if (run == k) first_window();
    if (min_slot < w) close();
}

static void colliding_kmers(const char* bases, const u64* offsets, u64 n_contigs, unsigned k,
                            unsigned m, u64 seed, const u64* ids, u64 n_ids,
                            std::vector<u128>& out) {
    u64 mm_count = 0, next_id = 0;
    for (u64 c = 0; c < n_contigs; ++c)
        colliding_kmers_contig(bases + offsets[c], offsets[c + 1] - offsets[c], k, m, seed, ids, n_ids, next_id, mm_count,
                               out);
}

}  // namespace orc

// ---------------------------------------------------------------------------------------------
// C entry points (ctypes binding: oracle/oracle.py)
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_err;

extern "C" {

const char* orc_last_error() { return g_err.c_str(); }

void* orc_load(const char* path, int kmer_bits) {
    try {
        FILE* f = std::fopen(path, "rb");
        if (!f) throw std::runtime_error(std::string("cannot open ") + path);
        std::fseek(f, 0, SEEK_END);
        long n = std::ftell(f);
        std::fseek(f, 0, SEEK_SET);
        std::vector<unsigned char> buf(n);
        if (n && std::fread(buf.data(), 1, n, f) != size_t(n)) {
            std::fclose(f);
            throw std::runtime_error("short read");
        }
        std::fclose(f);
        auto* h = new orc::Mphf();
        h->kmer_bits = kmer_bits;
        h->parse(buf.data(), buf.size());
        return h;
    } catch (std::exception const& e) {
        g_err = e.what();
        return nullptr;
    }
}
void orc_free(void* h) { delete static_cast<orc::Mphf*>(h); }

// info[0..]: k, m, mm_seed, nkmers, distinct, n_maximal, right_start, none_sizes_start,
// none_pos_start, mo.num_keys, mo.table_size, mo.dense, mo.sparse, fb.num_keys, fb.table_size,
// file_bytes, sp.size, sp.low.width
void orc_info(void* h, u64* info) {
    auto& f = *static_cast<orc::Mphf*>(h);
    u64 v[] = {f.k, f.m, f.mm_seed, f.nkmers, f.distinct, f.n_maximal, f.right_start,
               f.none_sizes_start, f.none_pos_start, f.minimizer_order.num_keys,
               f.minimizer_order.table_size, f.minimizer_order.dense, f.minimizer_order.sparse,
               f.fallback.num_keys, f.fallback.table_size, f.file_bytes, f.sp.size(),
               f.sp.low.width};
    std::memcpy(info, v, sizeof(v));
}

static int64_t emit(std::vector<u64> const& v, u64* out, u64 cap) {
    u64 n = v.size() < cap ? v.size() : cap;
    if (out && n) std::memcpy(out, v.data(), n * 8);
    return int64_t(v.size());
}

int64_t orc_query_streaming(void* h, const char* s, u64 len, u64* out, u64 cap) {
    std::vector<u64> v;
    static_cast<orc::Mphf*>(h)->streaming(s, len, v);
    return emit(v, out, cap);
}
int64_t orc_query_stateless(void* h, const char* s, u64 len, u64* out, u64 cap) {
    std::vector<u64> v;
    static_cast<orc::Mphf*>(h)->stateless(s, len, v, nullptr);
    return emit(v, out, cap);
}
// Batch streaming query: codes concatenated in contig order, out_offsets[n_contigs+1] filled.
int64_t orc_query_batch(void* h, const char* bases, const u64* offsets, u64 n_contigs, u64* out,
                        u64 cap, u64* out_offsets) {
    auto& f = *static_cast<orc::Mphf*>(h);
    std::vector<u64> v;
    u64 total = 0;
    for (u64 c = 0; c < n_contigs; ++c) {
        v.clear();
        f.streaming(bases + offsets[c], offsets[c + 1] - offsets[c], v);
        if (out_offsets) out_offsets[c] = total;
        for (u64 x : v) {
            if (total < cap && out) out[total] = x;
            ++total;
        }
    }
    if (out_offsets) out_offsets[n_contigs] = total;
    return int64_t(total);
}

// read-side primitives, for unit tests of the device primitives
u64 orc_murmur64(u64 v, u64 seed) { return orc::murmur64(v, seed); }
u64 orc_fastmod(u64 a, u64 d) {
    u128 M = ~u128(0) / d + 1;  // fastmod.h:126-132 computeM_u64
    return orc::fastmod_u64(a, M, d);
}
u64 orc_minimizer_order(void* h, u64 mmer) {
    auto& f = *static_cast<orc::Mphf*>(h);
    return f.minimizer_order.position(orc::murmur64(mmer, f.minimizer_order.seed));
}
// minimizer_order(keys[i]) through a serialized single_phf on its own (build-p Part 3 re-keys the triplets with
// it, ref src/partitioned_mphf.cpp:96-100)
int orc_phf_positions(const unsigned char* phf, u64 nbytes, const u64* keys, u64 n, u64* out) {
    try {
        orc::Reader r{phf, phf + nbytes};
        orc::SinglePhf f;
        f.read(r);
        if (r.p != r.end) throw std::runtime_error("trailing bytes after the single_phf");
        for (u64 i = 0; i < n; ++i) out[i] = f.position(orc::murmur64(keys[i], f.seed));
        return 0;
    } catch (std::exception const& e) {
        g_err = e.what();
        return -1;
    }
}
// Pilot search of a single_phf over pre-hashed keys, for indexes made without the reference's PTHash (oracle/phf.py).
// Same bucketer, position function and search order as pthash (buckets by size, largest first; smallest pilot whose
// positions are all free), so the result is a valid single_phf; it is not bit-identical to pthash's own builder.
// taken[table_size] comes back with the occupied positions set.  Returns 0, -1 when two keys share a hash, -2 when a
// bucket holds more than 256 keys.
int orc_phf_search(const u64* hashes, u64 n, u64 seed, u64 dense, u64 sparse, u64 table_size, u64* pilots,
                   unsigned char* taken) {
    orc::SinglePhf f;
    f.dense = dense;
    f.sparse = sparse;
    f.M_dense = ~u128(0) / dense + 1;
    f.M_sparse = ~u128(0) / sparse + 1;
    const u128 M = ~u128(0) / table_size + 1;
    const u64 nb = dense + sparse;
    std::vector<u64> start(nb + 1, 0), bucket(n);
    for (u64 i = 0; i < n; ++i) ++start[(bucket[i] = f.bucket(hashes[i])) + 1];
    for (u64 b = 0; b < nb; ++b) start[b + 1] += start[b];
    std::vector<u64> keys(n), fill(start.begin(), start.end() - 1);
    for (u64 i = 0; i < n; ++i) keys[fill[bucket[i]]++] = hashes[i];
    std::vector<u64> order(nb);
    for (u64 b = 0; b < nb; ++b) order[b] = b;
    std::stable_sort(order.begin(), order.end(),
                     [&](u64 a, u64 b) { return start[a + 1] - start[a] > start[b + 1] - start[b]; });
    std::vector<u64> used((table_size + 63) / 64, 0);  // a bit per slot: stays in cache where a byte map would not
    auto is_used = [&](u64 q) { return (used[q >> 6] >> (q & 63)) & 1; };
    // pilot p fits when every key lands on a free slot and no two keys of the bucket share one
    auto fits = [&](const u64* k0, u64 s, u64 p) {
        const u64 hp = orc::murmur64(p, seed);
        u64 q[256];
        for (u64 i = 0; i < s; ++i) {
            q[i] = orc::fastmod_u64(k0[i] ^ hp, M, table_size);
            if (is_used(q[i])) return false;
            for (u64 j = 0; j < i; ++j)
                if (q[j] == q[i]) return false;
        }
        return true;
    };
    for (u64 b = 0; b < nb; ++b) {
        u64* k0 = keys.data() + start[b];
        const u64 s = start[b + 1] - start[b];
        if (s > 256) return -2;
        std::sort(k0, k0 + s);
        for (u64 i = 1; i < s; ++i)
            if (k0[i] == k0[i - 1]) return -1;
    }
    // Buckets are searched a batch at a time on every core against the slots taken before the batch, then committed
    // in order.  A pilot found that way is the smallest fitting a subset of the slots taken at commit time, so when
    // it still fits it is the pilot the one-bucket-at-a-time search finds; when it does not, the search goes on
    // from there.  The result does not depend on the number of threads.
    const unsigned nt = std::max(1u, std::thread::hardware_concurrency());
    const u64 batch = 1024 * nt;
    std::vector<u64> spec(batch);
    for (u64 b0 = 0; b0 < nb; b0 += batch) {
        const u64 b1 = std::min(nb, b0 + batch);
        auto work = [&](unsigned t) {
            for (u64 i = b0 + t; i < b1; i += nt) {
                const u64 b = order[i], s = start[b + 1] - start[b];
                u64 p = 0;
                while (s && !fits(keys.data() + start[b], s, p)) ++p;
                spec[i - b0] = p;
            }
        };
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < nt; ++t) pool.emplace_back(work, t);
        work(0);
        for (auto& th : pool) th.join();
        for (u64 i = b0; i < b1; ++i) {
            const u64 b = order[i], s = start[b + 1] - start[b];
            const u64* k0 = keys.data() + start[b];
            u64 p = spec[i - b0];
            pilots[b] = 0;
            if (s == 0) continue;
            while (!fits(k0, s, p)) ++p;
            pilots[b] = p;
            const u64 hp = orc::murmur64(p, seed);
            for (u64 j = 0; j < s; ++j) {
                const u64 q = orc::fastmod_u64(k0[j] ^ hp, M, table_size);
                used[q >> 6] |= u64(1) << (q & 63);
            }
        }
    }
    for (u64 q = 0; q < table_size; ++q) taken[q] = is_used(q);
    return 0;
}
u64 orc_fallback_order(void* h, u64 lo, u64 hi) {
    return static_cast<orc::Mphf*>(h)->fallback_order((u128(hi) << 64) | lo);
}
void orc_rank_of(void* h, u64 idx, int* type, u64* rank) {
    static_cast<orc::Mphf*>(h)->rank_of(idx, *type, *rank);
}
u64 orc_sp_access(void* h, u64 i) { return static_cast<orc::Mphf*>(h)->sp.access(i); }
void orc_sp_pair(void* h, u64 i, u64* a, u64* b) { static_cast<orc::Mphf*>(h)->sp.pair(i, *a, *b); }
// mphf::query on an explicit (kmer, minimizer, position) triple; returns hval, *type gets 0..4
u64 orc_query_triple(void* h, u64 lo, u64 hi, u64 mmer, u64 pos, int* type) {
    auto c = static_cast<orc::Mphf*>(h)->query((u128(hi) << 64) | lo, mmer, pos);
    if (type) *type = c.type;
    return c.hval;
}

// build-side scan over a batch (mm_count carried across contigs; starts at *mm_count).
// mode 0 = sequential restatement of from_string, 1 = stateless definition (clean input).
int64_t orc_scan(const char* bases, const u64* offsets, u64 n_contigs, unsigned k, unsigned m,
                 u64 seed, int mode, u64* mm_count, void* records, u64 cap, u64* n_kmers) {
    std::vector<orc::Record> recs;
    u64 nk = 0;
    for (u64 c = 0; c < n_contigs; ++c) {
        const char* s = bases + offsets[c];
        u64 len = offsets[c + 1] - offsets[c];
        nk += mode == 0 ? orc::from_string(s, len, k, m, seed, *mm_count, recs)
                        : orc::scan_stateless(s, len, k, m, seed, *mm_count, recs);
    }
    u64 n = recs.size() < cap ? recs.size() : cap;
    if (records && n) std::memcpy(records, recs.data(), n * sizeof(orc::Record));
    if (n_kmers) *n_kmers = nk;
    return int64_t(recs.size());
}

// classify: in = records (any order), out = unique triplets in ascending minimizer order and
// ascending colliding ids.
void orc_classify(const void* records, u64 n, void* triplets, u64* n_triplets, u64* ids, u64* n_ids) {
    std::vector<orc::Record> recs(n);
    if (n) std::memcpy(recs.data(), records, n * sizeof(orc::Record));
    std::vector<orc::Triplet> uniq;
    std::vector<u64> idv;
    orc::classify(std::move(recs), uniq, idv);
    if (triplets && !uniq.empty()) std::memcpy(triplets, uniq.data(), uniq.size() * sizeof(orc::Triplet));
    if (ids && !idv.empty()) std::memcpy(ids, idv.data(), idv.size() * 8);
    *n_triplets = uniq.size();
    *n_ids = idv.size();
}

// colliding k-mers; each k-mer written as kmer_bits/8 little-endian bytes.
int64_t orc_colliding_kmers(const char* bases, const u64* offsets, u64 n_contigs, unsigned k,
                            unsigned m, u64 seed, const u64* ids, u64 n_ids, int kmer_bits,
                            void* out, u64 cap) {
    std::vector<u128> v;
    orc::colliding_kmers(bases, offsets, n_contigs, k, m, seed, ids, n_ids, v);
    u64 n = v.size() < cap ? v.size() : cap;
    auto* dst = static_cast<unsigned char*>(out);
    for (u64 i = 0; i < n; ++i) std::memcpy(dst + i * (kmer_bits / 8), &v[i], kmer_bits / 8);
    return int64_t(v.size());
}

}  // extern "C"
