"""TEST INFRASTRUCTURE — ctypes binding of oracle/_ref/libref{64,128}.so.

That library is the UNMODIFIED reference (jermp/lphash) compiled by oracle/build_ref.sh plus the
extern "C" harness oracle/ref_harness.cpp.  It is used to (a) pin the CPU restatement
(oracle/lphash_oracle.cpp), (b) generate the golden fixtures under tests/golden/, (c) produce
`.lph` index files (the reference's build-p is their only producer) and (d) time the CPU
baseline in bench.py.  Never imported by the product package.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")

RECORD_DTYPE = np.dtype([("itself", "<u8"), ("id", "<u8"), ("p1", "u1"), ("size", "u1")])  # 18 B
TRIPLET_DTYPE = np.dtype([("itself", "<u8"), ("p1", "u1"), ("size", "u1")])  # 10 B
assert RECORD_DTYPE.itemsize == 18 and TRIPLET_DTYPE.itemsize == 10


def available(bits: int = 64) -> bool:
    return os.path.exists(os.path.join(REF_DIR, f"libref{bits}.so"))


def cli_path(bits: int = 64) -> str:
    return os.path.join(REF_DIR, f"lphash{bits}")


_libs: dict[int, C.CDLL] = {}


def lib(bits: int) -> C.CDLL:
    if bits in _libs:
        return _libs[bits]
    path = os.path.join(REF_DIR, f"libref{bits}.so")
    if not os.path.exists(path):
        raise FileNotFoundError(f"{path} missing: build it with oracle/build_ref.sh (LPHASH_REF_DIR = the reference's "
                                "source tree)")
    L = C.CDLL(path)
    u64, p = C.c_uint64, C.c_void_p
    L.ref_last_error.restype = C.c_char_p
    L.ref_kmer_bits.restype = C.c_int
    L.ref_build.restype = C.c_int
    L.ref_build.argtypes = [C.c_char_p, C.c_int, C.c_int, u64, C.c_double, C.c_int, C.c_int,
                            C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, u64]
    L.ref_load.restype = p
    L.ref_load.argtypes = [C.c_char_p]
    L.ref_free.argtypes = [p]
    L.ref_kmer_count.restype = u64
    L.ref_kmer_count.argtypes = [p]
    L.ref_minimizer_count.restype = u64
    L.ref_minimizer_count.argtypes = [p]
    L.ref_query.restype = C.c_int64
    L.ref_query.argtypes = [p, C.c_char_p, u64, C.c_int, p, u64]
    L.ref_query_batch.restype = C.c_double
    L.ref_query_batch.argtypes = [p, p, p, u64, C.c_int, p, p, C.POINTER(u64)]
    L.ref_scan_new.restype = p
    L.ref_scan_new.argtypes = [C.c_char_p, C.c_int]
    L.ref_scan_free.argtypes = [p]
    L.ref_from_string.restype = u64
    L.ref_from_string.argtypes = [p, C.c_char_p, u64, C.c_uint32, C.c_uint32, u64, C.POINTER(u64)]
    L.ref_scan_size.restype = u64
    L.ref_scan_size.argtypes = [p]
    L.ref_scan_dump.restype = u64
    L.ref_scan_dump.argtypes = [p, p, u64]
    L.ref_classify.restype = C.c_int
    L.ref_classify.argtypes = [p, C.c_char_p, p, u64, C.POINTER(u64), p, u64, C.POINTER(u64)]
    L.ref_colliding_kmers.restype = C.c_int64
    L.ref_colliding_kmers.argtypes = [p, p, u64, C.c_uint32, C.c_uint32, u64, p, u64, C.c_char_p, p, u64]
    L.ref_scan_batch.restype = C.c_double
    L.ref_scan_batch.argtypes = [p, p, u64, C.c_uint32, C.c_uint32, u64, C.c_int, C.c_char_p,
                                 C.POINTER(u64), C.POINTER(u64)]
    L.ref_build_alt.restype = C.c_int
    L.ref_build_alt.argtypes = [C.c_char_p, C.c_int, C.c_int, u64, C.c_double, C.c_int, C.c_int, C.c_char_p, C.c_char_p,
                                C.c_char_p, u64]
    L.ref_load_alt.restype = p
    L.ref_load_alt.argtypes = [C.c_char_p]
    L.ref_free_alt.argtypes = [p]
    L.ref_kmer_count_alt.restype = u64
    L.ref_kmer_count_alt.argtypes = [p]
    L.ref_query_alt.restype = C.c_int64
    L.ref_query_alt.argtypes = [p, C.c_char_p, u64, C.c_int, p, u64]
    L.ref_build_minimizer_phf.restype = C.c_int
    L.ref_build_minimizer_phf.argtypes = [p, u64, C.c_double, C.c_int, C.c_char_p, C.c_char_p]
    L.ref_ef_sequence.restype = C.c_int
    L.ref_ef_sequence.argtypes = [p, u64, u64, C.c_char_p]
    assert L.ref_kmer_bits() == bits
    _libs[bits] = L
    return L


def _tmp() -> str:
    return tempfile.mkdtemp(prefix="lphref_")


def build(input_path: str, k: int, m: int, output: str, *, bits: int = 64, seed: int = 42,
          c: float = 3.0, threads: int = 1, max_memory_gb: int = 8, tmp_dir: str | None = None) -> str:
    """build-p through the reference's own mphf::build + essentials::save; returns its CSV line."""
    L = lib(bits)
    tmp = tmp_dir or _tmp()
    buf = C.create_string_buffer(4096)
    rc = L.ref_build(input_path.encode(), k, m, seed, c, threads, max_memory_gb, tmp.encode(),
                     output.encode(), 0, buf, 4096)
    if rc != 0:
        raise RuntimeError("reference build failed: " + L.ref_last_error().decode())
    return buf.value.decode().strip()


def build_alt(input_path: str, k: int, m: int, output: str, *, bits: int = 64, seed: int = 42,
              c: float = 3.0, threads: int = 1, max_memory_gb: int = 8, tmp_dir: str | None = None) -> str:
    """build-u through the reference's own mphf_alt::build + essentials::save; returns its CSV line."""
    L = lib(bits)
    tmp = tmp_dir or _tmp()
    buf = C.create_string_buffer(4096)
    rc = L.ref_build_alt(input_path.encode(), k, m, seed, c, threads, max_memory_gb, tmp.encode(),
                         output.encode(), buf, 4096)
    if rc != 0:
        raise RuntimeError("reference build-u failed: " + L.ref_last_error().decode())
    return buf.value.decode().strip()


class RefMphfAlt:
    """A loaded reference `lphash::mphf_alt` (the unpartitioned variant, build-u / query-u)."""

    def __init__(self, path: str, bits: int = 64):
        self.L = lib(bits)
        self.h = self.L.ref_load_alt(path.encode())
        if not self.h:
            raise RuntimeError(self.L.ref_last_error().decode())

    def close(self):
        if self.h:
            self.L.ref_free_alt(self.h)
            self.h = None

    @property
    def kmer_count(self) -> int:
        return self.L.ref_kmer_count_alt(self.h)

    def query(self, contig: bytes, streaming: bool = True) -> np.ndarray:
        cap = max(len(contig), 1)
        out = np.empty(cap, dtype=np.uint64)
        n = self.L.ref_query_alt(self.h, contig, len(contig), 1 if streaming else 0, out.ctypes.data, cap)
        if n < 0:
            raise RuntimeError(self.L.ref_last_error().decode())
        assert n <= cap
        return out[:n].copy()


class RefMphf:
    """A loaded reference `lphash::mphf`."""

    def __init__(self, path: str, bits: int = 64):
        self.L = lib(bits)
        self.bits = bits
        self.h = self.L.ref_load(path.encode())
        if not self.h:
            raise RuntimeError("reference load failed: " + self.L.ref_last_error().decode())

    def close(self):
        if getattr(self, "h", None):  # absent when the library failed to load
            self.L.ref_free(self.h)
            self.h = None

    __del__ = close

    @property
    def kmer_count(self) -> int:
        return self.L.ref_kmer_count(self.h)

    def query(self, contig: bytes, streaming: bool = True) -> np.ndarray:
        """hf(contig, len, streaming) — include/partitioned_mphf.hpp:73-197."""
        cap = max(len(contig), 1)
        out = np.empty(cap, dtype=np.uint64)
        n = self.L.ref_query(self.h, contig, len(contig), int(streaming), out.ctypes.data, cap)
        if n < 0:
            raise RuntimeError(self.L.ref_last_error().decode())
        assert n <= cap
        return out[:n].copy()

    def query_batch(self, bases: np.ndarray, offsets: np.ndarray, threads: int = 1,
                    want_codes: bool = True, k: int | None = None):
        """Multi-thread streaming query over concatenated contigs (clean input when want_codes)."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        total = C.c_uint64(0)
        out = out_off = None
        if want_codes:
            assert k is not None
            lens = np.diff(offsets).astype(np.int64)
            cnt = np.maximum(lens - k + 1, 0).astype(np.uint64)
            out_off = np.zeros(n + 1, dtype=np.uint64)
            np.cumsum(cnt, out=out_off[1:])
            out = np.empty(int(out_off[-1]), dtype=np.uint64)
        secs = self.L.ref_query_batch(self.h, bases.ctypes.data, offsets.ctypes.data, n, threads,
                                      out.ctypes.data if out is not None else None,
                                      out_off.ctypes.data if out_off is not None else None,
                                      C.byref(total))
        return secs, total.value, out, out_off


def scan(bases: np.ndarray, offsets: np.ndarray, k: int, m: int, seed: int = 42, bits: int = 64,
         by_minimizer: bool = False):
    """minimizer::from_string over all contigs (mm_count carried across, as mphf::build Part 1).
    Returns (records[RECORD_DTYPE] in scan order (or minimizer order), n_kmers, mm_count)."""
    L = lib(bits)
    tmp = _tmp()
    acc = L.ref_scan_new(tmp.encode(), int(by_minimizer))
    try:
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        mm = C.c_uint64(0)
        nk = 0
        raw = bases.tobytes()
        for c in range(len(offsets) - 1):
            s, e = int(offsets[c]), int(offsets[c + 1])
            nk += L.ref_from_string(acc, raw[s:e], e - s, k, m, seed, C.byref(mm))
        n = L.ref_scan_size(acc)
        rec = np.empty(n, dtype=RECORD_DTYPE)
        got = L.ref_scan_dump(acc, rec.ctypes.data, n)
        assert got == n
        return rec, nk, mm.value
    finally:
        L.ref_scan_free(acc)


def classify(bases: np.ndarray, offsets: np.ndarray, k: int, m: int, seed: int = 42, bits: int = 64):
    """from_string → (sorted by minimizer) → classify.  Returns (triplets, colliding ids)."""
    L = lib(bits)
    tmp = _tmp()
    acc = L.ref_scan_new(tmp.encode(), 1)
    try:
        raw = np.ascontiguousarray(bases, dtype=np.uint8).tobytes()
        mm = C.c_uint64(0)
        for c in range(len(offsets) - 1):
            s, e = int(offsets[c]), int(offsets[c + 1])
            L.ref_from_string(acc, raw[s:e], e - s, k, m, seed, C.byref(mm))
        n = L.ref_scan_size(acc)
        trip = np.empty(n, dtype=TRIPLET_DTYPE)
        ids = np.empty(n, dtype=np.uint64)
        nt, ni = C.c_uint64(0), C.c_uint64(0)
        rc = L.ref_classify(acc, tmp.encode(), trip.ctypes.data, n, C.byref(nt), ids.ctypes.data, n,
                            C.byref(ni))
        if rc != 0:
            raise RuntimeError(L.ref_last_error().decode())
        return trip[: nt.value].copy(), ids[: ni.value].copy()
    finally:
        L.ref_scan_free(acc)


def colliding_kmers(bases: np.ndarray, offsets: np.ndarray, k: int, m: int, ids: np.ndarray,
                    seed: int = 42, bits: int = 64) -> np.ndarray:
    """minimizer::get_colliding_kmers over all contigs; returns raw little-endian k-mers as a
    (n, bits//64) uint64 array (column 0 = low word)."""
    L = lib(bits)
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    words = bits // 64
    cap = int(np.maximum(np.diff(offsets).astype(np.int64) - k + 1, 0).sum())
    out = np.empty((max(cap, 1), words), dtype=np.uint64)
    n = L.ref_colliding_kmers(bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1, k, m, seed,
                              ids.ctypes.data, len(ids), _tmp().encode(), out.ctypes.data, cap)
    if n < 0:
        raise RuntimeError(L.ref_last_error().decode())
    return out[:n].copy()


def build_minimizer_phf(keys: np.ndarray, c: float = 3.0, threads: int = 1) -> bytes:
    """The serialized minimizer_order the reference builds on `keys` (src/partitioned_mphf.cpp:45-52, 147-153)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    d = _tmp()
    try:
        out = os.path.join(d, "phf.bin")
        if lib(64).ref_build_minimizer_phf(keys.ctypes.data, len(keys), c, threads, d.encode(), out.encode()) != 0:
            raise RuntimeError(lib(64).ref_last_error().decode())
        return open(out, "rb").read()
    finally:
        shutil.rmtree(d, ignore_errors=True)


def ef_sequence(values: np.ndarray, universe: int) -> bytes:
    """essentials::save of ef_sequence::encode(values, n, universe) (include/ef_sequence.hpp:36-75)."""
    values = np.ascontiguousarray(values, dtype=np.uint64)
    d = _tmp()
    try:
        out = os.path.join(d, "ef.bin")
        if lib(64).ref_ef_sequence(values.ctypes.data, len(values), universe, out.encode()) != 0:
            raise RuntimeError(lib(64).ref_last_error().decode())
        return open(out, "rb").read()
    finally:
        shutil.rmtree(d, ignore_errors=True)
