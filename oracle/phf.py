"""TEST INFRASTRUCTURE — `.lph` indexes made without the reference's build-p.

The reference's PTHash construction is out of scope of the GPU path, and its build-p is not always at hand.  This
module makes a valid `.lph` image from the project's own parts: Part 1, 2 and 4 scans and Part 3 through the CUDA
library (lphash_b200.api), and the two `pthash::single_phf<murmurhash2_64, dictionary_dictionary, minimal>` objects
from a plain pilot search (orc_phf_search in lphash_oracle.cpp) serialized in pthash's layout.  Every hash code the
index yields is as valid as the reference's (a minimal perfect hash of the k-mers), but the pilots, hence the codes,
are not the ones pthash's builder would pick.  Used by bench.py to prepare its input.
"""
from __future__ import annotations

import math
import struct

import numpy as np

from oracle import invindex, oracle

PTHASH_SEED = 1  # constants::default_pthash_seed, the seed in the reference's files (tests/golden/*.lph)
MURMUR_M = np.uint64(0xC6A4A7935BD1E995)


def murmur64(values, seed: int) -> np.ndarray:
    """MurmurHash2-64 of each 8-byte word (lphash_oracle.cpp murmur64), vectorised."""
    v = np.ascontiguousarray(values, dtype=np.uint64)
    s47 = np.uint64(47)
    h = np.full(v.shape, (seed ^ (8 * int(MURMUR_M))) & (2**64 - 1), dtype=np.uint64)
    x = v * MURMUR_M
    x ^= x >> s47
    x *= MURMUR_M
    h = (h ^ x) * MURMUR_M
    h ^= h >> s47
    h *= MURMUR_M
    h ^= h >> s47
    return h


def _u128(v: int) -> bytes:
    return int(v).to_bytes(16, "little")


def _fastmod_m(d: int) -> int:
    return ((2**128 - 1) // d + 1) & (2**128 - 1)  # fastmod computeM_u64 (wraps to 0 for d = 1)


def _compact(values, width: int | None = None) -> bytes:
    """pthash compact_vector: {size, width, mask, vector<u64> words}"""
    v = np.ascontiguousarray(values, dtype=np.uint64)
    if width is None:
        width = max(1, int(v.max()).bit_length()) if len(v) else 0
    bits = np.zeros(0, dtype=np.uint8)
    if width and len(v):
        bits = ((v[:, None] >> np.arange(width, dtype=np.uint64)) & np.uint64(1)).astype(np.uint8).reshape(-1)
    words = invindex._bits_to_words(bits) if len(bits) else np.zeros(0, dtype="<u8")
    words = np.concatenate([words, np.zeros(1, dtype="<u8")])
    return struct.pack("<QQQ", len(v), width, (1 << width) - 1) + invindex._vec(words)


def _dictionary(values) -> bytes:
    """pthash dictionary encoder: {ranks, dict} (compact vectors)"""
    dict_, ranks = np.unique(np.asarray(values, dtype=np.uint64), return_inverse=True)
    return _compact(ranks) + _compact(dict_)


def _ef(values) -> bytes:
    """pthash ef_sequence<false>::encode(begin, n), universe = the last value: {high bits, darray1, low bits}"""
    v = np.ascontiguousarray(values, dtype=np.uint64)
    n = len(v)
    if n == 0:
        return invindex._u64(0) + invindex._vec([]) + invindex.darray1_image([]) + _compact([], 0)
    u = int(v[-1])
    l = (u // n).bit_length() - 1 if u // n else 0
    ones = (v >> np.uint64(l)) + np.arange(n, dtype=np.uint64)
    high = np.zeros(n + (u >> l) + 1, dtype=np.uint8)
    high[ones] = 1
    out = invindex._u64(len(high)) + invindex._vec(invindex._bits_to_words(high))
    out += invindex.darray1_image(ones.tolist())
    return out + _compact(v & np.uint64((1 << l) - 1), l)


def single_phf(hashes, seed: int = PTHASH_SEED, c: float = 3.0, alpha: float = 0.94) -> bytes:
    """A serialized minimal single_phf over keys whose murmur64(key, seed) hashes are given (all distinct)."""
    h = np.ascontiguousarray(hashes, dtype=np.uint64)
    n = len(h)
    if n == 0:
        raise ValueError("single_phf needs at least one key")
    num_buckets = max(2, math.ceil(c * n / max(math.log2(n), 1.0)))  # pthash: ceil(c n / log2 n)
    dense = max(1, int(0.3 * num_buckets))  # skew_bucketer: 60 % of the keys into 30 % of the buckets
    sparse = num_buckets - dense
    table_size = max(n, int(n / alpha))
    if table_size & (table_size - 1) == 0:
        table_size += 1
    pilots = np.empty(num_buckets, dtype=np.uint64)
    taken = np.empty(table_size, dtype=np.uint8)
    rc = oracle.lib().orc_phf_search(h.ctypes.data, n, seed, dense, sparse, table_size, pilots.ctypes.data,
                                     taken.ctypes.data)
    if rc != 0:
        raise ValueError("two keys share a 64-bit hash" if rc == -1 else "a bucket holds more than 256 keys")
    # minimal remap: occupied slot n + j -> the j-th free slot below n; unoccupied ones repeat the next value so the
    # sequence stays non-decreasing for Elias-Fano
    free = np.flatnonzero(taken[:n] == 0).astype(np.uint64)
    tail = taken[n:].astype(np.int64)
    before = np.cumsum(tail) - tail  # occupied slots in [n, pos)
    free_slots = free[np.minimum(before, max(len(free) - 1, 0))] if len(free) else np.zeros(len(tail), np.uint64)
    out = struct.pack("<QQQ", seed, n, table_size) + _u128(_fastmod_m(table_size))
    out += struct.pack("<QQ", dense, sparse) + _u128(_fastmod_m(dense)) + _u128(_fastmod_m(sparse))
    out += _dictionary(pilots[:dense]) + _dictionary(pilots[dense:])
    return out + _ef(free_slots)


def build_lph(bases, offsets, k: int, m: int, kmer_bits: int = 64, mm_seed: int = 42, device: int = 0) -> bytes:
    """A complete `.lph` image of the contigs (build-p with c = 3.0, alpha = 0.94); needs a GPU."""
    from lphash_b200 import api

    trip, ids, nkmers, _ = api.scan_classify(bases, offsets, k, m, seed=mm_seed, device=device)
    mo = single_phf(murmur64(trip["itself"], PTHASH_SEED))
    info, body = api.build_inverted_index(k, m, mo, trip, device=device)
    kmers = api.colliding_kmers(bases, offsets, k, m, ids, seed=mm_seed, kmer_bits=kmer_bits, device=device)
    fh = murmur64(kmers[:, 0], PTHASH_SEED)
    if kmer_bits == 128:  # constants.hpp fallback_hasher: murmur(lo, seed) ^ murmur(hi, ~seed)
        fh ^= murmur64(kmers[:, 1], ~PTHASH_SEED & (2**64 - 1))
    fb = single_phf(fh)
    return api.lph_assemble(k, m, mm_seed, nkmers, len(trip), info, mo, body, fb)
