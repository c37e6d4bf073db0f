"""TEST INFRASTRUCTURE — ctypes binding of oracle/liboracle.so (oracle/lphash_oracle.cpp), the CPU
restatement of the reference's hot path.  Checker only: imported by tests/, smoke() and bench.py's
cpu_baseline leg; never by the product package."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "liboracle.so")

RECORD_DTYPE = np.dtype([("itself", "<u8"), ("id", "<u8"), ("p1", "u1"), ("size", "u1")])
TRIPLET_DTYPE = np.dtype([("itself", "<u8"), ("p1", "u1"), ("size", "u1")])

TYPE_NAMES = ["LEFT", "RIGHT", "MAXIMAL", "NONE", "COLLISION"]


def build(force: bool = False) -> str:
    src = os.path.join(HERE, "lphash_oracle.cpp")
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", HERE, "liboracle.so"])
    return LIB


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build())
    u64, p, i64 = C.c_uint64, C.c_void_p, C.c_int64
    L.orc_last_error.restype = C.c_char_p
    L.orc_load.restype = p
    L.orc_load.argtypes = [C.c_char_p, C.c_int]
    L.orc_free.argtypes = [p]
    L.orc_info.argtypes = [p, p]
    L.orc_query_streaming.restype = i64
    L.orc_query_streaming.argtypes = [p, C.c_char_p, u64, p, u64]
    L.orc_query_stateless.restype = i64
    L.orc_query_stateless.argtypes = [p, C.c_char_p, u64, p, u64]
    L.orc_query_batch.restype = i64
    L.orc_query_batch.argtypes = [p, p, p, u64, p, u64, p]
    L.orc_murmur64.restype = u64
    L.orc_murmur64.argtypes = [u64, u64]
    L.orc_fastmod.restype = u64
    L.orc_fastmod.argtypes = [u64, u64]
    L.orc_minimizer_order.restype = u64
    L.orc_minimizer_order.argtypes = [p, u64]
    L.orc_phf_positions.restype = C.c_int
    L.orc_phf_positions.argtypes = [p, u64, p, u64, p]
    L.orc_phf_search.restype = C.c_int
    L.orc_phf_search.argtypes = [p, u64, u64, u64, u64, u64, p, p]
    L.orc_fallback_order.restype = u64
    L.orc_fallback_order.argtypes = [p, u64, u64]
    L.orc_rank_of.argtypes = [p, u64, C.POINTER(C.c_int), C.POINTER(u64)]
    L.orc_sp_access.restype = u64
    L.orc_sp_access.argtypes = [p, u64]
    L.orc_sp_pair.argtypes = [p, u64, C.POINTER(u64), C.POINTER(u64)]
    L.orc_query_triple.restype = u64
    L.orc_query_triple.argtypes = [p, u64, u64, u64, u64, C.POINTER(C.c_int)]
    L.orc_scan.restype = i64
    L.orc_scan.argtypes = [p, p, u64, C.c_uint, C.c_uint, u64, C.c_int, C.POINTER(u64), p, u64,
                           C.POINTER(u64)]
    L.orc_classify.argtypes = [p, u64, p, C.POINTER(u64), p, C.POINTER(u64)]
    L.orc_colliding_kmers.restype = i64
    L.orc_colliding_kmers.argtypes = [p, p, u64, C.c_uint, C.c_uint, u64, p, u64, C.c_int, p, u64]
    _lib = L
    return L


INFO_FIELDS = ["k", "m", "mm_seed", "nkmers", "distinct_minimizers", "n_maximal",
               "right_coll_sizes_start", "none_sizes_start", "none_pos_start", "mo_num_keys",
               "mo_table_size", "mo_dense", "mo_sparse", "fb_num_keys", "fb_table_size",
               "file_bytes", "sp_size", "sp_low_width"]


class OracleMphf:
    def __init__(self, path: str, kmer_bits: int = 64):
        self.L = lib()
        self.h = self.L.orc_load(path.encode(), kmer_bits)
        if not self.h:
            raise RuntimeError("oracle load failed: " + self.L.orc_last_error().decode())
        info = np.zeros(len(INFO_FIELDS), dtype=np.uint64)
        self.L.orc_info(self.h, info.ctypes.data)
        self.info = {k: int(v) for k, v in zip(INFO_FIELDS, info)}
        self.k, self.m = self.info["k"], self.info["m"]

    def close(self):
        if getattr(self, "h", None):
            self.L.orc_free(self.h)
            self.h = None

    __del__ = close

    def _run(self, fn, contig: bytes) -> np.ndarray:
        cap = max(len(contig), 1)
        out = np.empty(cap, dtype=np.uint64)
        n = fn(self.h, contig, len(contig), out.ctypes.data, cap)
        assert 0 <= n <= cap
        return out[:n].copy()

    def query(self, contig: bytes) -> np.ndarray:
        """operator()(contig, len, streaming=true), quirk included."""
        return self._run(self.L.orc_query_streaming, contig)

    def query_stateless(self, contig: bytes) -> np.ndarray:
        return self._run(self.L.orc_query_stateless, contig)

    def query_batch(self, bases: np.ndarray, offsets: np.ndarray):
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        cap = max(int(offsets[-1] - offsets[0]), 1)
        out = np.empty(cap, dtype=np.uint64)
        out_off = np.zeros(n + 1, dtype=np.uint64)
        tot = self.L.orc_query_batch(self.h, bases.ctypes.data, offsets.ctypes.data, n,
                                     out.ctypes.data, cap, out_off.ctypes.data)
        assert 0 <= tot <= cap
        return out[:tot].copy(), out_off

    def minimizer_order(self, mmer: int) -> int:
        return self.L.orc_minimizer_order(self.h, mmer)

    def fallback_order(self, lo: int, hi: int = 0) -> int:
        return self.L.orc_fallback_order(self.h, lo, hi)

    def rank_of(self, idx: int):
        t, r = C.c_int(0), C.c_uint64(0)
        self.L.orc_rank_of(self.h, idx, C.byref(t), C.byref(r))
        return t.value, r.value

    def sp_access(self, i: int) -> int:
        return self.L.orc_sp_access(self.h, i)

    def sp_pair(self, i: int):
        a, b = C.c_uint64(0), C.c_uint64(0)
        self.L.orc_sp_pair(self.h, i, C.byref(a), C.byref(b))
        return a.value, b.value

    def query_triple(self, kmer: int, mmer: int, pos: int):
        t = C.c_int(0)
        h = self.L.orc_query_triple(self.h, kmer & (2**64 - 1), kmer >> 64, mmer, pos, C.byref(t))
        return h, t.value


def murmur64(v: int, seed: int) -> int:
    return lib().orc_murmur64(v, seed)


def phf_positions(phf: bytes, keys: np.ndarray) -> np.ndarray:
    """single_phf(keys[i]) for a serialized pthash::single_phf over u64 keys (minimizer_order on its own)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    buf = np.frombuffer(phf, dtype=np.uint8)
    out = np.empty(len(keys), dtype=np.uint64)
    if lib().orc_phf_positions(buf.ctypes.data, len(buf), keys.ctypes.data, len(keys), out.ctypes.data) != 0:
        raise RuntimeError(lib().orc_last_error().decode())
    return out


def fastmod(a: int, d: int) -> int:
    return lib().orc_fastmod(a, d)


def scan(bases: np.ndarray, offsets: np.ndarray, k: int, m: int, seed: int = 42, mode: int = 0,
         mm_count: int = 0):
    """Build-side scan.  mode 0: sequential restatement of from_string; 1: stateless definition.
    Returns (records, n_kmers, mm_count_out)."""
    L = lib()
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    cap = max(int(offsets[-1] - offsets[0]), 1)
    rec = np.empty(cap, dtype=RECORD_DTYPE)
    mm = C.c_uint64(mm_count)
    nk = C.c_uint64(0)
    n = L.orc_scan(bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1, k, m, seed, mode,
                   C.byref(mm), rec.ctypes.data, cap, C.byref(nk))
    assert 0 <= n <= cap
    return rec[:n].copy(), nk.value, mm.value


def classify(records: np.ndarray):
    L = lib()
    records = np.ascontiguousarray(records)
    n = len(records)
    trip = np.empty(max(n, 1), dtype=TRIPLET_DTYPE)
    ids = np.empty(max(n, 1), dtype=np.uint64)
    nt, ni = C.c_uint64(0), C.c_uint64(0)
    L.orc_classify(records.ctypes.data, n, trip.ctypes.data, C.byref(nt), ids.ctypes.data, C.byref(ni))
    return trip[: nt.value].copy(), ids[: ni.value].copy()


def colliding_kmers(bases, offsets, k, m, ids, seed: int = 42, kmer_bits: int = 64) -> np.ndarray:
    L = lib()
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    words = kmer_bits // 64
    cap = max(int(np.maximum(np.diff(offsets).astype(np.int64) - k + 1, 0).sum()), 1)
    out = np.empty((cap, words), dtype=np.uint64)
    n = L.orc_colliding_kmers(bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1, k, m, seed,
                              ids.ctypes.data, len(ids), kmer_bits, out.ctypes.data, cap)
    assert 0 <= n <= cap
    return out[:n].copy()
