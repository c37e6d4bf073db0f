#include "lph_image.h"

#include <cstdlib>
#include <cstring>
#include <exception>
#include <thread>

namespace lphb {

namespace {

// Load-time decoding is embarrassingly parallel once the running counters are turned into ranks: the loops
// over buckets / Elias-Fano values below are cut into contiguous slices, one per host thread (LPHB_LOAD_THREADS,
// default = hardware threads, at most 32).  An exception in a slice is rethrown on the calling thread.
unsigned load_threads() {
    if (const char* e = getenv("LPHB_LOAD_THREADS")) {
        long v = strtol(e, nullptr, 10);
        if (v >= 1) return unsigned(v > 64 ? 64 : v);
    }
    unsigned hw = std::thread::hardware_concurrency();
    return hw == 0 ? 1 : (hw > 32 ? 32 : hw);
}
template <class F>
void parallel_for(uint64_t n, uint64_t min_per_thread, F&& body) {  // body(begin, end, slice)
    unsigned t = load_threads();
    if (n / (min_per_thread ? min_per_thread : 1) < t) t = unsigned(n / (min_per_thread ? min_per_thread : 1));
    if (t <= 1) {
        body(uint64_t(0), n, 0u);
        return;
    }
    std::vector<std::thread> pool;
    std::vector<std::exception_ptr> err(t);
    for (unsigned i = 0; i < t; ++i)
        pool.emplace_back([&, i] {
            try {
                body(n * i / t, n * (i + 1) / t, i);
            } catch (...) {
                err[i] = std::current_exception();
            }
        });
    for (auto& th : pool) th.join();
    for (auto& e : err)
        if (e) std::rethrow_exception(e);
}

// MurmurHash2-64 of one 8-byte word (pthash hasher.hpp:46-110 with len == 8); used at load time
// only, to pre-hash the pilot dictionaries.
inline uint64_t murmur64_host(uint64_t v, uint64_t seed) {
    const uint64_t M = 0xc6a4a7935bd1e995ULL;
    uint64_t h = seed ^ (8 * M);
    uint64_t x = v * M;
    x ^= x >> 47;
    x *= M;
    h = (h ^ x) * M;
    h ^= h >> 47;
    h *= M;
    h ^= h >> 47;
    return h;
}

// A compact_vector still inside the file buffer (its words may be unaligned there).
struct FileCompact {
    uint64_t size = 0, width = 0, mask = 0, nwords = 0;
    const uint8_t* words = nullptr;
    uint64_t word(uint64_t i) const {
        uint64_t v;
        std::memcpy(&v, words + 8 * i, 8);
        return v;
    }
    uint64_t get(uint64_t i) const {
        if (width == 0) return 0;
        uint64_t pos = i * width, wd = pos >> 6, sh = pos & 63;
        uint64_t v = word(wd) >> sh;
        if (sh && wd + 1 < nwords) v |= word(wd + 1) << (64 - sh);
        return v & mask;
    }
};

}  // namespace

struct ImageBuilder::Cursor {
    const uint8_t* p;
    const uint8_t* end;
    template <class T>
    T pod() {
        if (uint64_t(end - p) < sizeof(T)) throw FormatError("truncated .lph image");
        T v;
        std::memcpy(&v, p, sizeof(T));
        p += sizeof(T);
        return v;
    }
    // vector<T>: returns pointer into the file buffer (possibly unaligned) and its length
    template <class T>
    const uint8_t* vec(uint64_t& n) {
        n = pod<uint64_t>();
        if (n > uint64_t(end - p) / sizeof(T)) throw FormatError("truncated vector in .lph image");
        const uint8_t* q = p;
        p += n * sizeof(T);
        return q;
    }
    FileCompact compact() {
        FileCompact c;
        c.size = pod<uint64_t>();
        c.width = pod<uint64_t>();
        c.mask = pod<uint64_t>();
        c.words = vec<uint64_t>(c.nwords);
        if (c.width > 57) throw FormatError("compact_vector width > 57 unsupported");
        uint64_t expect = c.width ? ((uint64_t(1) << c.width) - 1) : 0;
        if (c.mask != expect) throw FormatError("compact_vector mask/width mismatch");
        if (c.width && (c.size * c.width + 63) / 64 > c.nwords)
            throw FormatError("compact_vector shorter than size*width");
        return c;
    }
};

template <class T>
const T* ImageBuilder::append(const T* src, uint64_t n, uint64_t pad_elems) {
    uint64_t off = (arena_.size() + 255) & ~uint64_t(255);
    arena_.resize(off + (n + pad_elems) * sizeof(T), 0);
    if (n) std::memcpy(arena_.data() + off, src, n * sizeof(T));
    return reinterpret_cast<const T*>(uintptr_t(off));
}

std::vector<uint64_t> ImageBuilder::read_ef(Cursor& c) {
    // pthash ef_sequence / lphash ef_sequence share one layout: {bit_vector high; darray1;
    // compact_vector low} (include/ef_sequence.hpp:107-112, pthash darray.hpp:88-94).
    // value i = ((position of the i-th set high bit) - i) << l | low[i]  (ef_sequence.hpp:77-81)
    uint64_t nbits = c.pod<uint64_t>();
    uint64_t nw;
    const uint8_t* hw = c.vec<uint64_t>(nw);
    if ((nbits + 63) / 64 > nw) throw FormatError("EF high bits shorter than declared");
    uint64_t positions = c.pod<uint64_t>();
    uint64_t nb, ns, no;
    c.vec<int64_t>(nb);   // darray block inventory: select is not needed once decoded
    c.vec<uint16_t>(ns);  // subblock inventory
    c.vec<uint64_t>(no);  // overflow positions
    FileCompact low = c.compact();
    if (low.size != positions) throw FormatError("EF: darray positions != number of values");
    // set high bits before every slice of words (only bits below nbits count), then every slice decodes its own
    auto word_at = [&](uint64_t wi) {
        uint64_t wv;
        std::memcpy(&wv, hw + 8 * wi, 8);
        if ((wi + 1) * 64 > nbits) wv &= nbits > wi * 64 ? ((uint64_t(1) << (nbits - wi * 64)) - 1) : 0;
        return wv;
    };
    const unsigned slices = load_threads();
    std::vector<uint64_t> before(slices + 1, 0);
    parallel_for(slices, 1, [&](uint64_t s0, uint64_t s1, unsigned) {
        for (uint64_t sl = s0; sl < s1; ++sl) {
            uint64_t cnt = 0;
            for (uint64_t wi = nw * sl / slices; wi < nw * (sl + 1) / slices; ++wi) cnt += uint64_t(__builtin_popcountll(word_at(wi)));
            before[sl + 1] = cnt;
        }
    });
    for (unsigned sl = 0; sl < slices; ++sl) before[sl + 1] += before[sl];
    if (before[slices] < positions) throw FormatError("EF: fewer set bits than values");
    std::vector<uint64_t> vals(positions);
    parallel_for(slices, 1, [&](uint64_t s0, uint64_t s1, unsigned) {
        for (uint64_t sl = s0; sl < s1; ++sl) {
            uint64_t i = before[sl];
            for (uint64_t wi = nw * sl / slices; wi < nw * (sl + 1) / slices && i < positions; ++wi) {
                uint64_t wv = word_at(wi);
                while (wv && i < positions) {
                    const uint64_t pos = wi * 64 + uint64_t(__builtin_ctzll(wv));
                    wv &= wv - 1;
                    vals[i] = ((pos - i) << low.width) | low.get(i);
                    ++i;
                }
            }
        }
    });
    return vals;
}

ImageBuilder::Bits ImageBuilder::read_bits(Cursor& c) {
    // rs_bit_vector = {u64 nbits; vec<u64> bits; vec<u64> block_rank_pairs; vec<u64> select_hints}
    // (include/rs_bit_vector.hpp:91-96)
    Bits out;
    out.nbits = c.pod<uint64_t>();
    uint64_t nw, np, nh;
    const uint8_t* bw = c.vec<uint64_t>(nw);
    c.vec<uint64_t>(np);  // rank directory: ranks are recomputed while the buckets are walked
    c.vec<uint64_t>(nh);  // select hints: never built by the reference (quartet_wtree.cpp:51-53)
    if ((out.nbits + 63) / 64 > nw) throw FormatError("bit vector shorter than declared");
    out.words.resize(nw + 1, 0);
    if (nw) std::memcpy(out.words.data(), bw, nw * 8);
    return out;
}

// One word per bucket id: what mphf::query computes from the bucket alone
// (src/partitioned_mphf.cpp:292-339).  Buckets are walked in id order, so the ranks that
// quartet_wtree::rank_of (src/quartet_wtree.cpp:84-99) obtains from its rank directories are
// plain running counters here.  `sp` = decoded sizes_and_positions prefix sums.
void ImageBuilder::build_buckets(Bits const& root, Bits const& left_right, Bits const& max_none,
                                 std::vector<uint64_t> const& sp, std::vector<uint32_t> const& free_slots) {
    const uint64_t D = img_.distinct_minimizers;
    const uint64_t w = img_.w, maxblock = w * img_.n_maximal;
    const uint64_t rs = img_.right_start, ns = img_.none_sizes_start, np = img_.none_pos_start;
    auto S = [&](uint64_t i) -> uint64_t {
        if (i >= sp.size()) throw FormatError("sizes_and_positions index out of range");
        return sp[i];
    };
    img_.collision_base = S(np) + maxblock;  // partitioned_mphf.cpp:308-311
    // The table is indexed by the PTHash table slot BEFORE the minimal remap: slots >= num_keys
    // repeat the word of the key position free_slots sends them to (single_phf.hpp:61-63), so the
    // query needs no free-slot lookup.
    const uint64_t T = D + free_slots.size();
    BucketWriter e = begin_buckets(T);
    if (left_right.nbits + max_none.nbits != D) throw FormatError("wavelet tree: leaves do not add up to the root");
    // ones before every 64-bit word of the three bit vectors: the counters of a slice's first bucket are ranks
    auto prefix_ones = [](Bits const& bv) {
        const uint64_t nw = (bv.nbits + 63) / 64;
        std::vector<uint64_t> cum(nw + 1, 0);
        for (uint64_t w = 0; w < nw; ++w) {
            uint64_t x = bv.words[w];
            if ((w + 1) * 64 > bv.nbits) x &= (uint64_t(1) << (bv.nbits - w * 64)) - 1;
            cum[w + 1] = cum[w] + uint64_t(__builtin_popcountll(x));
        }
        return cum;
    };
    auto rank1 = [](Bits const& bv, std::vector<uint64_t> const& cum, uint64_t pos) {  // ones in [0, pos), pos <= nbits
        const uint64_t w = pos >> 6, r = pos & 63;
        return cum[w] + (r ? uint64_t(__builtin_popcountll(bv.words[w] & ((uint64_t(1) << r) - 1))) : 0);
    };
    const std::vector<uint64_t> cum_root = prefix_ones(root), cum_lr = prefix_ones(left_right), cum_mn = prefix_ones(max_none);
    if (rank1(root, cum_root, D) != max_none.nbits) throw FormatError("wavelet tree: root ones != size of the max/none leaf");
    std::vector<uint64_t> slice_max(64, 0);
    parallel_for(D, 1 << 16, [&](uint64_t b0, uint64_t b1, unsigned slice) {
        uint64_t n1 = rank1(root, cum_root, b0), n0 = b0 - n1;  // ones / zeros of root before the slice
        uint64_t r_right = rank1(left_right, cum_lr, n0), r_left = n0 - r_right;
        uint64_t r_none = rank1(max_none, cum_mn, n1), r_max = n1 - r_none;
        uint64_t max_base = 0;
        for (uint64_t b = b0; b < b1; ++b) {
            bool msb = root.get(b);
            uint64_t base = 0, kind = 0;
            if (!msb) {
                bool lsb = left_right.get(n0++);
                if (!lsb) {  // LEFT: g = EF[rank] + w*n_max, l = p
                    base = S(r_left++) + maxblock;
                    kind = 1;
                } else {     // RIGHT or collision (size 0)
                    uint64_t v1 = S(rs + r_right), v2 = S(rs + r_right + 1);
                    ++r_right;
                    if (v2 == v1) {
                        kind = 0;
                    } else {  // g = v1 + w*n_max, l = (k-m) - p
                        base = v1 + maxblock + uint64_t(img_.k - img_.m);
                        kind = 2;
                    }
                }
            } else {
                bool lsb = max_none.get(n1++);
                if (!lsb) {  // MAXIMAL: g = w*rank, l = p
                    base = w * r_max++;
                    kind = 1;
                } else {     // NONE: g = EF[none_sizes_start+rank] + w*n_max, l = diff(none_pos) - p
                    base = S(ns + r_none) + maxblock + (S(np + r_none + 1) - S(np + r_none));
                    ++r_none;
                    kind = 2;
                }
            }
            if (base >> 62) throw FormatError("bucket base does not fit 62 bits");
            if (base > max_base) max_base = base;
            // slope +1 (else -1) | colliding minimizer | base
            e.set(b, kind == 1, kind == 0, base);
        }
        slice_max[slice] = max_base;
    });
    uint64_t max_base = 0;
    for (uint64_t v : slice_max) max_base = v > max_base ? v : max_base;
    finish_buckets(e, D, max_base, free_slots);
}

// The bucket table is written straight into the arena (at config-3 scale it is 3.3 GB: no temporary copy).
// 32-bit entries when every base is sure to fit 30 bits - every base is a code of the function plus at
// most k, so nkmers decides - else 64-bit; LPHB_FORCE_WIDE_BUCKETS=1 (test hook) keeps the 64-bit form, which
// only indexes of about 2^30 k-mers or more would otherwise exercise.
ImageBuilder::BucketWriter ImageBuilder::begin_buckets(uint64_t T) {
    const char* fw = getenv("LPHB_FORCE_WIDE_BUCKETS");
    const bool force_wide = fw && fw[0] && fw[0] != '0';
    BucketWriter wtr;
    wtr.wide = force_wide || img_.nkmers >= (1ull << 30) - 256;  // not nkmers + 256: the header's nkmers is unbounded
    const uint64_t off = (arena_.size() + 255) & ~uint64_t(255);
    arena_.resize(off + (wtr.wide ? (T + 4) * 8 : (T + 8) * 4), 0);
    wtr.p = arena_.data() + off;
    img_.buckets.n = T;
    img_.buckets.wide = wtr.wide ? 1 : 0;
    img_.buckets.entries = reinterpret_cast<const void*>(uintptr_t(off));
    return wtr;
}

// free slots repeat the word of the key position they map to
void ImageBuilder::finish_buckets(BucketWriter& e, uint64_t D, uint64_t max_base, std::vector<uint32_t> const& free_slots) {
    if (!e.wide && max_base >= (1ull << 30)) throw FormatError("bucket base beyond the number of k-mers");
    parallel_for(free_slots.size(), 1 << 16, [&](uint64_t i0, uint64_t i1, unsigned) {
        for (uint64_t i = i0; i < i1; ++i) {
            if (free_slots[i] >= D) throw FormatError("single_phf: free slot outside [0, num_keys)");
            e.copy(D + i, free_slots[i]);
        }
    });
}

void reciprocal64(uint64_t d, uint32_t out[2]) {
    // M = floor(2^64 / d); d == 1 uses 2^64 - 1 (mod_small still returns 0)
    unsigned __int128 M = d > 1 ? ((((unsigned __int128)1) << 64) / d) : ((((unsigned __int128)1) << 64) - 1);
    out[0] = uint32_t(M);
    out[1] = uint32_t(M >> 32);
}

void ImageBuilder::read_phf(Cursor& c, DevPhf& out) {
    out.seed = c.pod<uint64_t>();
    out.num_keys = c.pod<uint64_t>();
    out.table_size = c.pod<uint64_t>();
    c.pod<unsigned __int128>();  // M: a % d is computed exactly on the device without it
    out.dense = c.pod<uint64_t>();
    out.sparse = c.pod<uint64_t>();
    c.pod<unsigned __int128>();
    c.pod<unsigned __int128>();
    FileCompact fr = c.compact(), fd = c.compact(), br = c.compact(), bd = c.compact();
    uint64_t nbuckets = fr.size + br.size, ndict = fd.size + bd.size;
    if (nbuckets != out.dense + out.sparse) throw FormatError("pilot count != bucket count");
    if (out.table_size == 0 || out.table_size < out.num_keys)
        throw FormatError("single_phf: bad table size");
    if (out.dense == 0 || out.sparse == 0) throw FormatError("single_phf: empty bucket class");
    // one word per bucket: default_hash64(pilot of the bucket, seed) (single_phf.hpp:57-58), the
    // dictionary indirection of dual<dictionary, dictionary> resolved here
    std::vector<uint64_t> hp(ndict);
    for (uint64_t i = 0; i < fd.size; ++i) hp[i] = murmur64_host(fd.get(i), out.seed);
    for (uint64_t i = 0; i < bd.size; ++i) hp[fd.size + i] = murmur64_host(bd.get(i), out.seed);
    std::vector<uint64_t> per_bucket(nbuckets);
    parallel_for(nbuckets, 1 << 16, [&](uint64_t b0, uint64_t b1, unsigned) {
        for (uint64_t b = b0; b < b1; ++b) {
            uint64_t r;
            if (b < fr.size) {
                r = fr.get(b);
                if (r >= fd.size) throw FormatError("pilot rank outside dictionary");
            } else {
                r = br.get(b - fr.size);
                if (r >= bd.size) throw FormatError("pilot rank outside dictionary");
                r += fd.size;
            }
            per_bucket[b] = hp[r];
        }
    });
    out.pilot_hash = append(per_bucket.data(), nbuckets, 2);
    // 64-bit PTHash hashes cap num_keys at 2^30 (hasher.hpp:27-31), so table_size = num_keys/alpha
    // stays below 2^31, which the device-side exact modulo relies on
    if (out.table_size >= (1ull << 31) || out.dense >= (1ull << 31) || out.sparse >= (1ull << 31))
        throw FormatError("single_phf: table larger than 2^31 (impossible with 64-bit PTHash hashes)");
    reciprocal64(out.table_size, out.m_table);
    reciprocal64(out.dense, out.m_dense);
    reciprocal64(out.sparse, out.m_sparse);
    // minimal remap as a plain array: one load instead of an Elias-Fano select
    std::vector<uint64_t> free_vals = read_ef(c);
    if (free_vals.size() != out.table_size - out.num_keys)
        throw FormatError("single_phf: free-slot count mismatch");
    std::vector<uint32_t> f32(free_vals.size());
    parallel_for(free_vals.size(), 1 << 16, [&](uint64_t i0, uint64_t i1, unsigned) {
        for (uint64_t i = i0; i < i1; ++i) {
            if (free_vals[i] >= out.table_size) throw FormatError("single_phf: free slot outside the table");
            f32[i] = uint32_t(free_vals[i]);
        }
    });
    out.free32 = append(f32.data(), f32.size(), 4);
    last_free_ = std::move(f32);
}

void ImageBuilder::parse(const uint8_t* data, uint64_t n, int kmer_bits) {
    if (kmer_bits != 64 && kmer_bits != 128) throw FormatError("kmer_bits must be 64 or 128");
    arena_.clear();
    img_ = DevImage{};
    Cursor c{data, data + n};
    img_.k = c.pod<uint8_t>();
    img_.m = c.pod<uint8_t>();
    img_.kmer_bits = uint32_t(kmer_bits);
    img_.mm_seed = c.pod<uint64_t>();
    img_.nkmers = c.pod<uint64_t>();
    img_.distinct_minimizers = c.pod<uint64_t>();
    img_.n_maximal = c.pod<uint64_t>();
    img_.right_start = c.pod<uint64_t>();
    img_.none_sizes_start = c.pod<uint64_t>();
    img_.none_pos_start = c.pod<uint64_t>();
    if (img_.m == 0 || img_.m > 31 || img_.k < img_.m || img_.k > uint32_t(kmer_bits / 2 - 1))
        throw FormatError("k/m out of range for this kmer_t");
    img_.w = img_.k - img_.m + 1;
    sections_[0] = uint64_t(c.p - data);
    read_phf(c, img_.minimizer_order);
    std::vector<uint32_t> mo_free = std::move(last_free_);
    sections_[1] = uint64_t(c.p - data);
    Bits root = read_bits(c), left_right = read_bits(c), max_none = read_bits(c);
    sections_[2] = uint64_t(c.p - data);
    std::vector<uint64_t> sp = read_ef(c);
    sections_[3] = uint64_t(c.p - data);
    read_phf(c, img_.fallback);
    sections_[4] = uint64_t(c.p - data);
    if (c.p != c.end) throw FormatError("trailing bytes after the .lph image");
    if (img_.minimizer_order.num_keys != img_.distinct_minimizers ||
        root.nbits != img_.distinct_minimizers ||
        left_right.nbits + max_none.nbits != img_.distinct_minimizers)
        throw FormatError("inconsistent minimizer counts");
    if (!(img_.right_start <= img_.none_sizes_start && img_.none_sizes_start <= img_.none_pos_start &&
          img_.none_pos_start < sp.size()))
        throw FormatError("inconsistent sizes_and_positions partition");
    build_buckets(root, left_right, max_none, sp, mo_free);
    fallback_keys_ = img_.fallback.num_keys;
    file_bytes_ = n;
    arena_.resize((arena_.size() + 255) & ~uint64_t(255), 0);
}

void ImageBuilder::parse_alt(const uint8_t* data, uint64_t n, int kmer_bits) {
    if (kmer_bits != 64 && kmer_bits != 128) throw FormatError("kmer_bits must be 64 or 128");
    arena_.clear();
    img_ = DevImage{};
    Cursor c{data, data + n};
    img_.k = c.pod<uint8_t>();
    img_.m = c.pod<uint8_t>();
    img_.kmer_bits = uint32_t(kmer_bits);
    img_.mm_seed = c.pod<uint64_t>();
    img_.nkmers = c.pod<uint64_t>();
    img_.distinct_minimizers = c.pod<uint64_t>();
    const uint64_t main_kmers = c.pod<uint64_t>();  // num_kmers_in_main_index
    if (img_.m == 0 || img_.m > 31 || img_.k < img_.m || img_.k > uint32_t(kmer_bits / 2 - 1))
        throw FormatError("k/m out of range for this kmer_t");
    img_.w = img_.k - img_.m + 1;
    sections_[0] = uint64_t(c.p - data);
    read_phf(c, img_.minimizer_order);
    std::vector<uint32_t> mo_free = std::move(last_free_);
    sections_[1] = uint64_t(c.p - data);
    std::vector<uint64_t> positions = read_ef(c);
    sections_[2] = uint64_t(c.p - data);
    std::vector<uint64_t> sizes = read_ef(c);
    sections_[3] = uint64_t(c.p - data);
    read_phf(c, img_.fallback);
    sections_[4] = uint64_t(c.p - data);
    if (c.p != c.end) throw FormatError("trailing bytes after the .lph image");
    const uint64_t D = img_.distinct_minimizers;
    if (img_.minimizer_order.num_keys != D || positions.size() != D + 1 || sizes.size() != D + 1)
        throw FormatError("inconsistent minimizer counts");
    img_.collision_base = main_kmers;  // unpartitioned_mphf.cpp:198
    // one word per bucket: hval(k-mer) = base - p, base = sizes[i] + positions.diff(i)
    // (unpartitioned_mphf.cpp:193-203); size 0 = colliding minimizer
    BucketWriter e = begin_buckets(D + mo_free.size());
    std::vector<uint64_t> slice_max(64, 0);
    parallel_for(D, 1 << 16, [&](uint64_t b0, uint64_t b1, unsigned slice) {
        uint64_t max_base = 0;
        for (uint64_t b = b0; b < b1; ++b) {
            if (sizes[b + 1] == sizes[b]) {
                e.set(b, false, true, 0);
            } else {
                const uint64_t base = sizes[b] + (positions[b + 1] - positions[b]);
                if (base >> 62) throw FormatError("bucket base does not fit 62 bits");
                if (base > max_base) max_base = base;
                e.set(b, false, false, base);  // slope -1
            }
        }
        slice_max[slice] = max_base;
    });
    uint64_t max_base = 0;
    for (uint64_t v : slice_max) max_base = v > max_base ? v : max_base;
    finish_buckets(e, D, max_base, mo_free);
    fallback_keys_ = img_.fallback.num_keys;
    file_bytes_ = n;
    arena_.resize((arena_.size() + 255) & ~uint64_t(255), 0);
}

void ImageBuilder::parse_phf(const uint8_t* data, uint64_t n) {
    arena_.clear();
    img_ = DevImage{};
    Cursor c{data, data + n};
    read_phf(c, img_.minimizer_order);
    if (c.p != c.end) throw FormatError("trailing bytes after the serialized single_phf");
    file_bytes_ = n;
    arena_.resize((arena_.size() + 255) & ~uint64_t(255), 0);
}

// ---- structure walk for the device-side loader -------------------------------------------------------------------
namespace {
struct Layout {  // the arena offsets ImageBuilder::append would hand out
    uint64_t size = 0;
    uint64_t take(uint64_t bytes) {
        const uint64_t off = (size + 255) & ~uint64_t(255);
        size = off + bytes;
        return off;
    }
};
}  // namespace

void ImageBuilder::walk_compact(Cursor& c, CompactRef& r) {
    FileCompact f = c.compact();
    r.size = f.size;
    r.width = f.width;
    r.words = VecRef{f.words, f.nwords};
}
void ImageBuilder::walk_ef(Cursor& c, EfRef& r) {
    r.nbits = c.pod<uint64_t>();
    r.high.p = c.vec<uint64_t>(r.high.n);
    if ((r.nbits + 63) / 64 > r.high.n) throw FormatError("EF high bits shorter than declared");
    r.positions = c.pod<uint64_t>();
    uint64_t nb, ns, no;
    c.vec<int64_t>(nb);
    c.vec<uint16_t>(ns);
    c.vec<uint64_t>(no);
    walk_compact(c, r.low);
    if (r.low.size != r.positions) throw FormatError("EF: darray positions != number of values");
}
void ImageBuilder::walk_phf(Cursor& c, PhfRef& r, DevPhf& out) {
    out.seed = c.pod<uint64_t>();
    out.num_keys = c.pod<uint64_t>();
    out.table_size = c.pod<uint64_t>();
    c.pod<unsigned __int128>();
    out.dense = c.pod<uint64_t>();
    out.sparse = c.pod<uint64_t>();
    c.pod<unsigned __int128>();
    c.pod<unsigned __int128>();
    walk_compact(c, r.front_ranks);
    walk_compact(c, r.front_dict);
    walk_compact(c, r.back_ranks);
    walk_compact(c, r.back_dict);
    r.n_buckets = r.front_ranks.size + r.back_ranks.size;
    if (r.n_buckets != out.dense + out.sparse) throw FormatError("pilot count != bucket count");
    if (out.table_size == 0 || out.table_size < out.num_keys) throw FormatError("single_phf: bad table size");
    if (out.dense == 0 || out.sparse == 0) throw FormatError("single_phf: empty bucket class");
    if (out.table_size >= (1ull << 31) || out.dense >= (1ull << 31) || out.sparse >= (1ull << 31))
        throw FormatError("single_phf: table larger than 2^31 (impossible with 64-bit PTHash hashes)");
    reciprocal64(out.table_size, out.m_table);
    reciprocal64(out.dense, out.m_dense);
    reciprocal64(out.sparse, out.m_sparse);
    walk_ef(c, r.free_slots);
    r.n_free = out.table_size - out.num_keys;
    if (r.free_slots.positions != r.n_free) throw FormatError("single_phf: free-slot count mismatch");
}

ImagePlan ImageBuilder::plan_phf(const uint8_t* data, uint64_t n) {
    // a serialized single_phf on its own: wrap it in a throw-away plan (walk_phf below is shared with plan())
    ImagePlan P;
    Cursor c{data, data + n};
    walk_phf(c, P.minimizer_order, P.img.minimizer_order);
    if (c.p != c.end) throw FormatError("trailing bytes after the serialized single_phf");
    Layout L;
    P.img.minimizer_order.pilot_hash = reinterpret_cast<const uint64_t*>(uintptr_t(L.take((P.minimizer_order.n_buckets + 2) * 8)));
    P.img.minimizer_order.free32 = reinterpret_cast<const uint32_t*>(uintptr_t(L.take((P.minimizer_order.n_free + 4) * 4)));
    P.arena_bytes = (L.size + 255) & ~uint64_t(255);
    P.file_bytes = n;
    return P;
}

ImagePlan ImageBuilder::plan(const uint8_t* data, uint64_t n, int kmer_bits, bool alt) {
    if (kmer_bits != 64 && kmer_bits != 128) throw FormatError("kmer_bits must be 64 or 128");
    ImagePlan P;
    P.alt = alt;
    DevImage& img = P.img;
    Cursor c{data, data + n};
    img.k = c.pod<uint8_t>();
    img.m = c.pod<uint8_t>();
    img.kmer_bits = uint32_t(kmer_bits);
    img.mm_seed = c.pod<uint64_t>();
    img.nkmers = c.pod<uint64_t>();
    img.distinct_minimizers = c.pod<uint64_t>();
    uint64_t main_kmers = 0;
    if (alt) {
        main_kmers = c.pod<uint64_t>();
    } else {
        img.n_maximal = c.pod<uint64_t>();
        img.right_start = c.pod<uint64_t>();
        img.none_sizes_start = c.pod<uint64_t>();
        img.none_pos_start = c.pod<uint64_t>();
    }
    if (img.m == 0 || img.m > 31 || img.k < img.m || img.k > uint32_t(kmer_bits / 2 - 1))
        throw FormatError("k/m out of range for this kmer_t");
    img.w = img.k - img.m + 1;
    auto ef = [&](EfRef& r) { walk_ef(c, r); };
    auto bits = [&](BitsRef& r) {
        r.nbits = c.pod<uint64_t>();
        r.words.p = c.vec<uint64_t>(r.words.n);
        uint64_t np, nh;
        c.vec<uint64_t>(np);
        c.vec<uint64_t>(nh);
        if ((r.nbits + 63) / 64 > r.words.n) throw FormatError("bit vector shorter than declared");
    };
    auto phf = [&](PhfRef& r, DevPhf& out) { walk_phf(c, r, out); };
    P.sections[0] = uint64_t(c.p - data);
    phf(P.minimizer_order, img.minimizer_order);
    P.sections[1] = uint64_t(c.p - data);
    if (alt) {
        ef(P.positions);
        P.sections[2] = uint64_t(c.p - data);
        ef(P.sizes);
    } else {
        bits(P.root);
        bits(P.left_right);
        bits(P.max_none);
        P.sections[2] = uint64_t(c.p - data);
        ef(P.sizes_and_positions);
    }
    P.sections[3] = uint64_t(c.p - data);
    phf(P.fallback, img.fallback);
    P.sections[4] = uint64_t(c.p - data);
    if (c.p != c.end) throw FormatError("trailing bytes after the .lph image");
    const uint64_t D = img.distinct_minimizers;
    if (img.minimizer_order.num_keys != D) throw FormatError("inconsistent minimizer counts");
    if (alt) {
        if (P.positions.positions != D + 1 || P.sizes.positions != D + 1) throw FormatError("inconsistent minimizer counts");
        img.collision_base = main_kmers;
    } else {
        if (P.root.nbits != D || P.left_right.nbits + P.max_none.nbits != D) throw FormatError("inconsistent minimizer counts");
        if (!(img.right_start <= img.none_sizes_start && img.none_sizes_start <= img.none_pos_start &&
              img.none_pos_start < P.sizes_and_positions.positions))
            throw FormatError("inconsistent sizes_and_positions partition");
    }
    // the arena layout of parse / parse_alt: mo.pilot_hash, mo.free32, fb.pilot_hash, fb.free32, bucket table
    Layout L;
    auto place_phf = [&](PhfRef const& r, DevPhf& out) {
        out.pilot_hash = reinterpret_cast<const uint64_t*>(uintptr_t(L.take((r.n_buckets + 2) * 8)));
        out.free32 = reinterpret_cast<const uint32_t*>(uintptr_t(L.take((r.n_free + 4) * 4)));
    };
    place_phf(P.minimizer_order, img.minimizer_order);
    place_phf(P.fallback, img.fallback);
    const char* fw = getenv("LPHB_FORCE_WIDE_BUCKETS");
    const bool wide = (fw && fw[0] && fw[0] != '0') || img.nkmers >= (1ull << 30) - 256;  // as begin_buckets
    const uint64_t T = D + P.minimizer_order.n_free;
    img.buckets.n = T;
    img.buckets.wide = wide ? 1 : 0;
    img.buckets.entries = reinterpret_cast<const void*>(uintptr_t(L.take(wide ? (T + 4) * 8 : (T + 8) * 4)));
    P.arena_bytes = (L.size + 255) & ~uint64_t(255);
    P.fallback_keys = img.fallback.num_keys;
    P.file_bytes = n;
    return P;
}

DevImage ImageBuilder::rebased(const void* device_base) const {
    DevImage d = img_;
    auto* base = static_cast<const uint8_t*>(device_base);
    for (DevPhf* p : {&d.minimizer_order, &d.fallback}) {
        p->free32 = reinterpret_cast<const uint32_t*>(base + uintptr_t(p->free32));
        p->pilot_hash = reinterpret_cast<const uint64_t*>(base + uintptr_t(p->pilot_hash));
    }
    d.buckets.entries = base + uintptr_t(d.buckets.entries);
    return d;
}

}  // namespace lphb
