// Device-side read primitives over the flat image (device_image.h): MurmurHash2-64, exact
// modulo by invariant divisors, PTHash evaluation and the per-super-k-mer probe `mphf::query`.
// Every function cites the reference code whose RESULT it reproduces bit for bit
// ("ref" = reference tree, "pthash/" = external/pthash/).
#pragma once
#include <stdint.h>

#include "device_image.h"

namespace lphb {

#define LPHB_DEV __device__ __forceinline__

constexpr uint64_t kMurmurM = 0xc6a4a7935bd1e995ULL;

// MurmurHash2-64 of one 8-byte word.  ref: pthash/include/utils/hasher.hpp:46-110 (len == 8:
// one block, empty tail); murmurhash2_64::hash(uint64_t) :175-177; default_hash64 :112-114.
LPHB_DEV uint64_t murmur64(uint64_t v, uint64_t seed) {
    const uint64_t M = kMurmurM;
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

// a % d for 64-bit a and d < 2^31, with M = floor(2^64 / d) as two 32-bit limbs.
// q' = floor(a * M / 2^64) is floor(a / d) or one less (a * M / 2^64 lies in (a/d - 1, a/d]), so
// a - q' * d lies in [0, 2d) and fits 32 bits: only the low word of q' is needed, hence only bits
// 32..63 of the middle partial products (their wrap-around past 2^64 is irrelevant), and one
// unsigned min folds the remainder.  The reference computes fastmod_u64(a, ceil(2^128/d), d)
// (pthash/external/fastmod/fastmod.h:56-63, 159-162), which is a % d exactly; so is this.
LPHB_DEV uint32_t mod_small(uint64_t a, uint32_t M0, uint32_t M1, uint32_t d) {
    const uint32_t a0 = uint32_t(a), a1 = uint32_t(a >> 32);
    uint64_t s = uint64_t(a1) * M0 + __umulhi(a0, M0);
    s += uint64_t(a0) * M1;
    const uint32_t q = a1 * M1 + uint32_t(s >> 32);
    const uint32_t r = a0 - q * d;
    return min(r, r - d);
}

// Gathers from the image carry an L2 evict_last policy: the image (a few bytes per minimizer,
// read at random by every SM) should stay resident in the 126 MB L2 while the base stream and the
// codes (read/written once, evict-first) flow through it.
LPHB_DEV uint64_t l2_keep_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
#ifdef LPHB_NOHINT  // tuning experiment: plain read-only loads without the L2 policy
LPHB_DEV uint32_t ldg_keep(const uint32_t* p, uint64_t) { return __ldg(p); }
LPHB_DEV uint32_t ldg_keep(const uint16_t* p, uint64_t) { return __ldg(p); }
LPHB_DEV uint64_t ldg_keep(const uint64_t* p, uint64_t) { return __ldg(reinterpret_cast<const unsigned long long*>(p)); }
#else
LPHB_DEV uint32_t ldg_keep(const uint32_t* p, uint64_t pol) {
    uint32_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
LPHB_DEV uint32_t ldg_keep(const uint16_t* p, uint64_t pol) {
    uint16_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u16 %0, [%1], %2;" : "=h"(v) : "l"(p), "l"(pol));
    return v;
}
LPHB_DEV uint64_t ldg_keep(const uint64_t* p, uint64_t pol) {
    uint64_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
    return v;
}
#endif

// pthash::single_phf::position, in the stages a caller may interleave across several keys.
// ref: pthash/include/single_phf.hpp:55-65; skew_bucketer::bucket pthash/include/utils/
// bucketers.hpp:17-22 (T = (uint64_t)(0.6*UINT64_MAX) evaluated in double = 0x9999999999999800);
// dual/dictionary access encoders.hpp:167-170,268-271.
LPHB_DEV uint32_t phf_bucket(DevPhf const& p, uint64_t h) {
    const uint64_t T = 0x9999999999999800ULL;
    // one modulo with the divisor selected first (no divergence between dense and sparse buckets)
    const bool dn = h < T;
    const uint32_t d = dn ? uint32_t(p.dense) : uint32_t(p.sparse);
    const uint32_t r0 = dn ? p.m_dense[0] : p.m_sparse[0];
    const uint32_t r1 = dn ? p.m_dense[1] : p.m_sparse[1];
    return mod_small(h, r0, r1, d) + (dn ? 0u : uint32_t(p.dense));
}
LPHB_DEV uint32_t phf_table_slot(DevPhf const& p, uint64_t h_xor_pilot) {
    return mod_small(h_xor_pilot, p.m_table[0], p.m_table[1], uint32_t(p.table_size));
}
LPHB_DEV uint64_t phf_position(DevPhf const& p, uint64_t h) {
    const uint32_t pos = phf_table_slot(p, h ^ __ldg(p.pilot_hash + phf_bucket(p, h)));
    if (pos < p.num_keys) return pos;
    return __ldg(p.free32 + (pos - uint32_t(p.num_keys)));  // minimal remap, single_phf.hpp:61-63
}

// fallback_kmer_order(kmer).  ref: include/constants.hpp:56-70 (fallback_hasher: 64-bit kmer_t
// hashes the single word; 128-bit kmer_t xors murmur(lo, seed) with murmur(hi, ~seed)).
LPHB_DEV uint64_t fallback_order(DevImage const& f, uint64_t lo, uint64_t hi) {
    uint64_t h = murmur64(lo, f.fallback.seed);
    if (f.kmer_bits == 128) h ^= murmur64(hi, ~f.fallback.seed);
    return phf_position(f.fallback, h);
}

// What one super-k-mer probe yields: hval of a k-mer whose minimizer sits at offset p is
// base + slope * p (mod 2^64) for the four regular types; colliding minimizers send every k-mer
// through fallback_order instead (hval = base + fallback).
//   LEFT     g = EF[rank] + w*n_max,                  l = p            -> slope +1
//   RIGHT    (v1,v2) = EF.pair(right_start+rank), v2>v1: g = v1 + w*n_max, l = (k-m) - p  -> -1
//   COLL     v2 == v1: g = EF[none_pos_start] + w*n_max, l = fallback(kmer)                -> 0
//   MAXIMAL  g = w*rank,                              l = p            -> +1
//   NONE     g = EF[none_sizes_start+rank] + w*n_max, l = EF.diff(none_pos_start+rank) - p -> -1
// (ref: src/partitioned_mphf.cpp:292-339; evaluated per bucket at load time, lph_image.cpp)
struct Probe {
    uint64_t base;
    int32_t slope;  // +1, -1, or 0 for a colliding minimizer
};

// one bucket word as loaded (a uint32_t entry zero-extended when the table is narrow)
LPHB_DEV Probe probe_decode(DevImage const& f, uint64_t e) {
    Probe out;
    uint32_t flags;
    if (f.buckets.wide) {
        flags = uint32_t(e >> 62);
        out.base = e & 0x3FFFFFFFFFFFFFFFull;
    } else {
        flags = uint32_t(e) >> 30;
        out.base = e & 0x3FFFFFFFu;
    }
    out.slope = (flags & 1u) ? 0 : ((flags & 2u) ? 1 : -1);
    if (flags & 1u) out.base = f.collision_base;
    return out;
}

LPHB_DEV Probe probe_bucket(DevImage const& f, uint64_t bucket) {
    if (f.buckets.wide) return probe_decode(f, __ldg(reinterpret_cast<const uint64_t*>(f.buckets.entries) + bucket));
    return probe_decode(f, __ldg(reinterpret_cast<const uint32_t*>(f.buckets.entries) + bucket));
}

LPHB_DEV Probe probe_minimizer(DevImage const& f, uint64_t minimizer) {
    return probe_bucket(f, phf_position(f.minimizer_order, murmur64(minimizer, f.minimizer_order.seed)));
}

LPHB_DEV uint64_t probe_hval(Probe const& pr, uint32_t p) {
    return pr.slope > 0 ? pr.base + p : pr.base - p;
}

// Leftmost-minimum m-mer of the k-mer {lo, hi} (first base in the most significant of its 2k bits) and its offset
// p in [0, k - m]: the strict '<' keeps the leftmost on ties.  ref: compute_minimizer_triplet,
// include/mphf_utils.hpp:118-137.
struct Minimizer {
    uint64_t mmer;
    uint32_t pos;
};
LPHB_DEV Minimizer kmer_minimizer(uint32_t k, uint32_t m, uint64_t mm_seed, uint64_t lo, uint64_t hi) {
    const uint64_t mm_mask = (uint64_t(1) << (2 * m)) - 1;
    const uint32_t w = k - m + 1;
    uint64_t best_h = 0;
    Minimizer out{0, 0};
    for (uint32_t p = 0; p < w; ++p) {
        uint32_t sh = 2 * (k - m - p);
        uint64_t mm = sh == 0 ? lo : (sh < 64 ? ((lo >> sh) | (hi << (64 - sh))) : (hi >> (sh - 64)));
        mm &= mm_mask;
        uint64_t h = murmur64(mm, mm_seed);
        if (p == 0 || h < best_h) { best_h = h; out.mmer = mm; out.pos = p; }
    }
    return out;
}

// ASCII -> 2-bit code, 4 = invalid.  ref: src/constants.cpp:5-13.
LPHB_DEV uint32_t nt4(uint32_t ch) {
    uint32_t u = ch & 0xDFu;  // fold case
    uint32_t code = ((ch >> 1) ^ (ch >> 2)) & 3u;  // A0 C1 G2 T/U3
    bool ok = (u == 'A') | (u == 'C') | (u == 'G') | (u == 'T') | (u == 'U');
    return ok ? code : 4u;
}

}  // namespace lphb
