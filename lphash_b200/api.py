"""Host-side mirror of the reference's `lphash::mphf` query interface on top of the C ABI
(include/lphash_b200.h, built into lphash_b200/liblphash_b200.so).

Reference interface mirrored (/root/reference/include/partitioned_mphf.hpp:13-39):
    hf = mphf(); essentials::load(hf, file)        ->  hf = Mphf.load(file, kmer_bits)
    hf(contig, len, streaming=true)                 ->  hf(contig)            (np.uint64 array)
    hf.get_kmer_count(), hf.get_minimizer_L0()      ->  same names
Batch entry points (`query_batch`, `query_device`) are what a driver that wants throughput calls:
one C-ABI call for many contigs.

There is no CPU implementation behind this module: if the CUDA library is missing or no GPU is
visible, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# LPHASH_B200_LIB selects a tuning variant of the same library (csrc/Makefile: `make variant`)
LIB_PATH = os.environ.get("LPHASH_B200_LIB") or os.path.join(HERE, "liblphash_b200.so")

RECORD_DTYPE = np.dtype([("itself", "<u8"), ("id", "<u8"), ("p1", "u1"), ("size", "u1")])  # mm_record_t

OK, E_ARG, E_IO, E_FORMAT, E_CUDA, E_CAPACITY, E_NOMEM = 0, -1, -2, -3, -4, -5, -6


class LphashError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"lphash_b200 error {code}: {msg}")
        self.code = code


class CapacityError(LphashError):
    """LPHB_E_CAPACITY of a call that reports the size it needed (n_codes)"""

    def __init__(self, code: int, msg: str, n_codes: int):
        super().__init__(code, msg)
        self.n_codes = n_codes


class Info(C.Structure):
    _fields_ = [("k", C.c_uint32), ("m", C.c_uint32), ("kmer_bits", C.c_uint32), ("device", C.c_int32),
                ("mm_seed", C.c_uint64), ("nkmers", C.c_uint64), ("distinct_minimizers", C.c_uint64),
                ("n_maximal", C.c_uint64), ("right_coll_sizes_start", C.c_uint64),
                ("none_sizes_start", C.c_uint64), ("none_pos_start", C.c_uint64),
                ("fallback_keys", C.c_uint64), ("file_bytes", C.c_uint64), ("device_bytes", C.c_uint64),
                ("load_host_ms", C.c_double), ("load_h2d_ms", C.c_double)]


class InvertedIndex(C.Structure):
    _fields_ = [("n_maximal", C.c_uint64), ("right_coll_sizes_start", C.c_uint64), ("none_sizes_start", C.c_uint64),
                ("none_pos_start", C.c_uint64), ("colliding_minimizers", C.c_uint64), ("universe", C.c_uint64),
                ("wtree_bytes", C.c_uint64), ("ef_bytes", C.c_uint64), ("device_ms", C.c_double)]


class InvertedIndexAlt(C.Structure):
    _fields_ = [("num_kmers_in_main_index", C.c_uint64), ("positions_bytes", C.c_uint64), ("sizes_bytes", C.c_uint64),
                ("device_ms", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("dirty_contigs", C.c_uint64), ("kernel_ms", C.c_double)]


class CheckReport(C.Structure):
    """lphb_check_report: the verdict of a check session (lphb_check_begin .. lphb_check_end).  first_out_of_range and
    first_mismatch are k-mer ordinals in session order; they and the two code fields are 2^64 - 1 when there is none."""
    _fields_ = [("kmers", C.c_uint64), ("contigs", C.c_uint64), ("dirty_contigs", C.c_uint64),
                ("out_of_range", C.c_uint64), ("duplicates", C.c_uint64), ("missing", C.c_uint64),
                ("stream_mismatches", C.c_uint64), ("first_out_of_range", C.c_uint64), ("first_mismatch", C.c_uint64),
                ("min_duplicate_code", C.c_uint64), ("min_missing_code", C.c_uint64), ("ok", C.c_int32)]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


class BuildReport(C.Structure):
    """lphb_build_report: totals of a build session (n_triplets, n_ids, colliding_minimizers are set by its end)"""
    _fields_ = [("batches", C.c_uint64), ("contigs", C.c_uint64), ("kmers", C.c_uint64), ("mm_count", C.c_uint64),
                ("records", C.c_uint64), ("n_triplets", C.c_uint64), ("n_ids", C.c_uint64),
                ("colliding_minimizers", C.c_uint64), ("device_bytes", C.c_uint64)]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


# every symbol include/lphash_b200.h declares (tests check the library exports all of them)
EXPORTS = ["lphb_last_error", "lphb_version", "lphb_device_count", "lphb_mphf_load_file",
           "lphb_mphf_load_memory", "lphb_mphf_free", "lphb_mphf_info", "lphb_query_stream",
           "lphb_query_stream_device", "lphb_scan_superkmers", "lphb_colliding_kmers",
           "lphb_host_alloc", "lphb_host_free", "lphb_mphf_stats", "lphb_scan_release", "lphb_classify", "lphb_scan_classify",
           "lphb_query_stream_runs", "lphb_expand_runs", "lphb_mphf_dirty_flags",
           "lphb_scan_superkmers_device", "lphb_copy_to_host", "lphb_query_nonstreaming",
           "lphb_mphf_alt_load_file", "lphb_mphf_alt_load_memory", "lphb_inverted_index_bound",
           "lphb_build_inverted_index", "lphb_lph_assemble", "lphb_lph_sections", "lphb_build_inverted_index_alt",
           "lphb_lph_assemble_alt", "lphb_mphf_device_image", "lphb_lookup_kmers", "lphb_lookup_kmers_device",
           "lphb_query_stream_exact_device", "lphb_query_stream_exact_device_async", "lphb_query_nonstreaming_device",
           "lphb_check_begin", "lphb_check_batch",
           "lphb_check_batch_device", "lphb_check_end", "lphb_build_begin", "lphb_build_batch",
           "lphb_build_batch_device", "lphb_build_end", "lphb_build_free"]

_lib = None


def lib() -> C.CDLL:
    """Loads the CUDA extension.  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`"
                          " (or make -C lphash_b200/csrc)")
    L = C.CDLL(LIB_PATH)
    u64, p, i32 = C.c_uint64, C.c_void_p, C.c_int
    L.lphb_last_error.restype = C.c_char_p
    L.lphb_version.restype = C.c_char_p
    L.lphb_device_count.argtypes = [C.POINTER(C.c_int)]
    L.lphb_mphf_load_file.argtypes = [C.c_char_p, i32, i32, C.POINTER(p)]
    L.lphb_mphf_load_memory.argtypes = [p, u64, i32, i32, C.POINTER(p)]
    L.lphb_mphf_alt_load_file.argtypes = [C.c_char_p, i32, i32, C.POINTER(p)]
    L.lphb_mphf_alt_load_memory.argtypes = [p, u64, i32, i32, C.POINTER(p)]
    L.lphb_mphf_free.argtypes = [p]
    L.lphb_mphf_info.argtypes = [p, C.POINTER(Info)]
    L.lphb_mphf_stats.argtypes = [p, C.POINTER(Stats)]
    L.lphb_query_stream.argtypes = [p, p, p, u64, p, u64, p, C.POINTER(u64)]
    L.lphb_query_nonstreaming.argtypes = [p, p, p, u64, p, u64, p, C.POINTER(u64)]
    L.lphb_query_stream_device.argtypes = [p, p, p, p, u64, p, u64, p, p, p]
    L.lphb_query_stream_exact_device.argtypes = [p, p, p, p, u64, p, u64, p, C.POINTER(u64), p]
    L.lphb_query_stream_exact_device_async.argtypes = [p, p, p, p, u64, p, u64, p, p, p]
    L.lphb_query_nonstreaming_device.argtypes = [p, p, p, p, u64, p, u64, p, p, p]
    L.lphb_lookup_kmers.argtypes = [p, p, u64, p]
    L.lphb_lookup_kmers_device.argtypes = [p, p, u64, p, p]
    L.lphb_check_begin.argtypes = [p]
    L.lphb_check_batch.argtypes = [p, p, p, u64]
    L.lphb_check_batch_device.argtypes = [p, p, p, p, u64, p, p]
    L.lphb_check_end.argtypes = [p, C.POINTER(CheckReport)]
    L.lphb_query_stream_runs.argtypes = [p, p, p, u64, p, u64, C.POINTER(u64), p, C.POINTER(u64)]
    L.lphb_expand_runs.argtypes = [p, u64, p, u64, C.POINTER(u64), i32]
    L.lphb_mphf_dirty_flags.argtypes = [p, C.POINTER(p), C.POINTER(u64)]
    L.lphb_scan_superkmers.argtypes = [i32, C.c_uint32, C.c_uint32, u64, p, p, u64, C.POINTER(u64), p,
                                       u64, C.POINTER(u64), C.POINTER(u64)]
    L.lphb_colliding_kmers.argtypes = [i32, C.c_uint32, C.c_uint32, u64, p, p, u64, C.POINTER(u64), p,
                                       u64, i32, p, u64, C.POINTER(u64)]
    L.lphb_scan_superkmers_device.argtypes = [i32, C.c_uint32, C.c_uint32, u64, p, p, p, u64, C.POINTER(u64), C.POINTER(p),
                                              C.POINTER(u64), C.POINTER(u64), C.POINTER(C.c_double)]
    L.lphb_classify.argtypes = [i32, p, u64, p, u64, C.POINTER(u64), p, u64, C.POINTER(u64)]
    L.lphb_scan_release.argtypes = [i32]
    L.lphb_scan_classify.argtypes = [i32, C.c_uint32, C.c_uint32, u64, p, p, u64, C.POINTER(u64), p, u64,
                                     C.POINTER(u64), p, u64, C.POINTER(u64), C.POINTER(u64)]
    L.lphb_copy_to_host.argtypes = [i32, p, p, u64]
    L.lphb_host_alloc.argtypes = [C.POINTER(p), u64]
    L.lphb_mphf_device_image.argtypes = [p, C.POINTER(p), C.POINTER(u64)]
    L.lphb_inverted_index_bound.argtypes = [u64]
    L.lphb_inverted_index_bound.restype = u64
    L.lphb_build_inverted_index.argtypes = [i32, C.c_uint32, C.c_uint32, p, u64, p, u64, p, u64, C.POINTER(u64),
                                            C.POINTER(InvertedIndex)]
    L.lphb_lph_assemble.argtypes = [C.c_uint32, C.c_uint32, u64, u64, u64, C.POINTER(InvertedIndex), p, u64, p, u64, p,
                                    u64, p, u64, C.POINTER(u64)]
    L.lphb_lph_sections.argtypes = [p, u64, i32, i32, C.POINTER(u64)]
    L.lphb_build_inverted_index_alt.argtypes = [i32, p, u64, p, u64, p, u64, C.POINTER(u64), C.POINTER(InvertedIndexAlt)]
    L.lphb_lph_assemble_alt.argtypes = [C.c_uint32, C.c_uint32, u64, u64, u64, C.POINTER(InvertedIndexAlt), p, u64, p, u64,
                                        p, u64, p, u64, C.POINTER(u64)]
    L.lphb_host_free.argtypes = [p]
    L.lphb_build_begin.argtypes = [i32, C.c_uint32, C.c_uint32, u64, C.POINTER(p)]
    L.lphb_build_batch.argtypes = [p, p, p, u64]
    L.lphb_build_batch_device.argtypes = [p, p, p, p, u64, p]
    L.lphb_build_end.argtypes = [p, p, u64, p, u64, C.POINTER(BuildReport)]
    L.lphb_build_free.argtypes = [p]
    for name in EXPORTS:
        if getattr(L, name).restype is C.c_int:
            pass
    _lib = L
    return L


def _check(rc: int):
    if rc != OK:
        raise LphashError(rc, lib().lphb_last_error().decode())


def device_count() -> int:
    n = C.c_int(0)
    _check(lib().lphb_device_count(C.byref(n)))
    return n.value


def _as_batch(bases, offsets):
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    if offsets.ndim != 1 or len(offsets) < 1:
        raise ValueError("offsets must have n_contigs + 1 entries")
    return bases, offsets


class Mphf:
    """A partitioned LP-MPHF resident on one GPU (the reference's `lphash::mphf`, query side)."""

    def __init__(self, handle: int):
        self._h = C.c_void_p(handle)
        info = Info()
        _check(lib().lphb_mphf_info(self._h, C.byref(info)))
        self.info = info
        self.k, self.m, self.kmer_bits, self.device = info.k, info.m, info.kmer_bits, info.device

    # -- construction ------------------------------------------------------------------------
    @classmethod
    def load(cls, path: str, kmer_bits: int = 64, device: int = 0) -> "Mphf":
        """essentials::load(hf, path) (/root/reference/src/query.cpp:37)."""
        h = C.c_void_p()
        _check(lib().lphb_mphf_load_file(os.fsencode(path), kmer_bits, device, C.byref(h)))
        return cls(h.value)

    @classmethod
    def load_alt(cls, path: str, kmer_bits: int = 64, device: int = 0) -> "Mphf":
        """An unpartitioned LP-MPHF (the reference's `lphash::mphf_alt`, build-u / query-u)."""
        h = C.c_void_p()
        _check(lib().lphb_mphf_alt_load_file(os.fsencode(path), kmer_bits, device, C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_bytes(cls, image: bytes, kmer_bits: int = 64, device: int = 0) -> "Mphf":
        h = C.c_void_p()
        buf = (C.c_char * len(image)).from_buffer_copy(image)
        _check(lib().lphb_mphf_load_memory(C.addressof(buf), len(image), kmer_bits, device, C.byref(h)))
        return cls(h.value)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().lphb_mphf_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference-named accessors -----------------------------------------------------------
    def get_kmer_count(self) -> int:
        return self.info.nkmers

    def get_minimizer_L0(self) -> int:
        return self.info.distinct_minimizers

    def device_image(self) -> bytes:
        """the flat device image behind the handle, copied to the host (diagnostic)"""
        ptr, n = C.c_void_p(), C.c_uint64(0)
        _check(lib().lphb_mphf_device_image(self._h, C.byref(ptr), C.byref(n)))
        out = np.empty(n.value, dtype=np.uint8)
        _check(lib().lphb_copy_to_host(self.info.device, out.ctypes.data, ptr, n.value))
        return out.tobytes()

    def dirty_flags(self) -> np.ndarray:
        """per contig of the last query call: nonzero where the contig holds a byte outside ACGT/acgt/U/u"""
        ptr, n = C.c_void_p(), C.c_uint64(0)
        _check(lib().lphb_mphf_dirty_flags(self._h, C.byref(ptr), C.byref(n)))
        out = np.zeros(n.value, dtype=np.uint8)
        if n.value:
            _check(lib().lphb_copy_to_host(self.info.device, out.ctypes.data, ptr, n.value))
        return out

    def stats(self) -> Stats:
        s = Stats()
        _check(lib().lphb_mphf_stats(self._h, C.byref(s)))
        return s

    # -- queries -----------------------------------------------------------------------------
    def __call__(self, contig, streaming: bool = True) -> np.ndarray:
        """hf(contig, len, streaming): hash codes of the contig's k-mers.  The two modes of the
        reference agree on ACGT-only input (SURVEY.md S1); `streaming=False` is the reference's
        non-streaming branch, where a non-ACGT byte counts as 'A' (lphb_query_nonstreaming)."""
        if isinstance(contig, str):
            contig = contig.encode()
        bases = np.frombuffer(bytes(contig), dtype=np.uint8)
        offsets = np.array([0, len(bases)], dtype=np.uint64)
        codes, _ = self.query_batch(bases, offsets, streaming=streaming)
        return codes

    def query_batch(self, bases, offsets, out: np.ndarray | None = None, streaming: bool = True):
        """One C-ABI call for a batch: returns (codes, code_offsets) with HOST arrays in and out.
        streaming=False: the reference's non-streaming branch (non-ACGT bytes count as 'A')."""
        bases, offsets = _as_batch(bases, offsets)
        n = len(offsets) - 1
        lens = np.diff(offsets).astype(np.int64)
        if (lens < 0).any():
            raise ValueError("offsets must be non-decreasing")
        if len(offsets) and int(offsets[-1]) > len(bases):
            raise ValueError("offsets index past the end of bases")
        # capacity: clean contigs give L-k+1; contigs with non-ACGT bytes can give up to L-m+1
        cap = int(np.maximum(lens - self.m + 1, 0).sum()) if out is None else len(out)
        codes = np.empty(max(cap, 1), dtype=np.uint64) if out is None else out
        code_off = np.empty(n + 1, dtype=np.uint64)
        total = C.c_uint64(0)
        fn = lib().lphb_query_stream if streaming else lib().lphb_query_nonstreaming
        _check(fn(self._h, bases.ctypes.data, offsets.ctypes.data, n,
                  codes.ctypes.data, cap, code_off.ctypes.data, C.byref(total)))
        return codes[: total.value], code_off

    def query_batch_runs(self, bases, offsets, out: np.ndarray | None = None):
        """lphb_query_stream_runs: the codes of a batch in run-length form (RUN_DTYPE records, about
        2 bytes per k-mer over PCIe instead of 8).  Returns (runs, code_offsets, n_codes)."""
        bases, offsets = _as_batch(bases, offsets)
        n = len(offsets) - 1
        lens = np.diff(offsets).astype(np.int64)
        cap = int(np.maximum(lens - self.m + 1, 0).sum()) if out is None else len(out)
        runs = np.empty(max(cap, 1), dtype=RUN_DTYPE) if out is None else out
        code_off = np.empty(n + 1, dtype=np.uint64)
        n_runs, total = C.c_uint64(0), C.c_uint64(0)
        _check(lib().lphb_query_stream_runs(self._h, bases.ctypes.data, offsets.ctypes.data, n, runs.ctypes.data,
                                            cap, C.byref(n_runs), code_off.ctypes.data, C.byref(total)))
        return runs[: n_runs.value], code_off, total.value

    def query_device(self, d_bases: int, d_offsets: int, h_offsets: np.ndarray, d_codes: int,
                     capacity: int, d_code_offsets: int, d_status: int, stream: int = 0) -> None:
        """Device-resident asynchronous variant; arguments are raw device pointers (ints), e.g.
        torch_tensor.data_ptr(), and a cudaStream_t handle."""
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint64)
        _check(lib().lphb_query_stream_device(self._h, d_bases, d_offsets, h_offsets.ctypes.data,
                                              len(h_offsets) - 1, d_codes, capacity, d_code_offsets,
                                              d_status, stream))

    def query_device_exact(self, d_bases: int, d_offsets: int, h_offsets: np.ndarray, d_codes: int,
                           capacity: int, d_code_offsets: int, stream: int = 0) -> int:
        """lphb_query_stream_exact_device: the codes lphb_query_stream gives (non-ACGT quirk included) for a batch in
        device buffers; raw device pointers (ints) and a cudaStream_t handle as in query_device.  Synchronous: returns
        the number of codes once d_codes / d_code_offsets hold them.  sum(max(0, L-m+1)) is always enough capacity."""
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint64)
        n = C.c_uint64(0)
        rc = lib().lphb_query_stream_exact_device(self._h, d_bases, d_offsets, h_offsets.ctypes.data,
                                                  len(h_offsets) - 1, d_codes, capacity, d_code_offsets,
                                                  C.byref(n), stream)
        if rc == E_CAPACITY:
            raise CapacityError(rc, lib().lphb_last_error().decode(), n.value)
        _check(rc)
        return n.value

    def query_device_exact_async(self, d_bases: int, d_offsets: int, h_offsets: np.ndarray, d_codes: int,
                                 capacity: int, d_code_offsets: int, d_status: int, stream: int = 0) -> None:
        """lphb_query_stream_exact_device_async: the codes of query_device_exact, enqueued on the stream with no host
        synchronisation; d_status (4 int64 words) receives the number of codes and of contigs with non-ACGT bytes.
        capacity must be at least sum(max(0, L-m+1)), else CapacityError (n_codes = that bound) before anything runs."""
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint64)
        rc = lib().lphb_query_stream_exact_device_async(self._h, d_bases, d_offsets, h_offsets.ctypes.data,
                                                        len(h_offsets) - 1, d_codes, capacity, d_code_offsets,
                                                        d_status, stream)
        if rc == E_CAPACITY:
            lens = np.diff(h_offsets.astype(np.int64))
            raise CapacityError(rc, lib().lphb_last_error().decode(), int(np.maximum(lens - self.m + 1, 0).sum()))
        _check(rc)

    def query_device_nonstreaming(self, d_bases: int, d_offsets: int, h_offsets: np.ndarray, d_codes: int,
                                  capacity: int, d_code_offsets: int, d_status: int, stream: int = 0) -> None:
        """lphb_query_nonstreaming_device: the reference's non-streaming branch (a non-ACGT byte counts as 'A') for a
        batch in device buffers, asynchronous like query_device; the caller's bases are left as they are."""
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint64)
        _check(lib().lphb_query_nonstreaming_device(self._h, d_bases, d_offsets, h_offsets.ctypes.data,
                                                    len(h_offsets) - 1, d_codes, capacity, d_code_offsets,
                                                    d_status, stream))

    def lookup(self, kmers, out: np.ndarray | None = None) -> np.ndarray:
        """lphb_lookup_kmers: the codes of packed k-mers (seqio.pack_kmers), in input order.  kmers is a uint64 array
        of shape (n,) for a 64-bit handle, (n, 2) = [lo, hi] for a 128-bit one; the first base sits in the most
        significant of the 2k used bits (A=0 C=1 G=2 T=3), higher bits are ignored.  codes[i] is what the reference's
        non-streaming branch gives for the window kmers[i] encodes.  Returns a uint64 (n,) array (`out` if given)."""
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
        shape = "(n,)" if self.kmer_bits == 64 else "(n, 2)"
        if kmers.ndim != (1 if self.kmer_bits == 64 else 2) or (kmers.ndim == 2 and kmers.shape[1] != 2):
            raise ValueError(f"a {self.kmer_bits}-bit handle takes k-mers of shape {shape}, got {kmers.shape}")
        n = kmers.shape[0]
        codes = np.empty(max(n, 1), dtype=np.uint64) if out is None else out
        if len(codes) < n or codes.dtype != np.uint64 or not codes.flags.c_contiguous:
            raise ValueError("out must be a contiguous uint64 array of at least n entries")
        _check(lib().lphb_lookup_kmers(self._h, kmers.ctypes.data, n, codes.ctypes.data))
        return codes[:n]

    def lookup_device(self, d_kmers: int, n: int, d_codes: int, stream: int = 0) -> None:
        """lphb_lookup_kmers_device: asynchronous on `stream`; raw device pointers (ints), e.g. tensor.data_ptr(),
        d_kmers holding n k-mers of kmer_bits / 8 bytes each."""
        _check(lib().lphb_lookup_kmers_device(self._h, d_kmers, n, d_codes, stream))

    # -- the index self-check (build-p --check) ---------------------------------------------------------------------
    def check_begin(self) -> None:
        """lphb_check_begin: (re)starts the handle's check session"""
        _check(lib().lphb_check_begin(self._h))

    def check_batch(self, bases, offsets) -> None:
        """lphb_check_batch: one batch of the session, host arrays as query_batch takes them"""
        bases, offsets = _as_batch(bases, offsets)
        if np.any(np.diff(offsets.astype(np.int64)) < 0):
            raise ValueError("offsets must be non-decreasing")
        if int(offsets[-1]) > len(bases):
            raise ValueError("offsets index past the end of bases")
        _check(lib().lphb_check_batch(self._h, bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1))

    def check_batch_device(self, d_bases: int, d_offsets: int, h_offsets: np.ndarray, d_stream_codes: int = 0,
                           stream: int = 0) -> None:
        """lphb_check_batch_device: raw device pointers (ints) as in query_device; d_stream_codes (0: none) holds the
        caller's streaming codes of the batch in query_device's layout.  Asynchronous on `stream`."""
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint64)
        _check(lib().lphb_check_batch_device(self._h, d_bases, d_offsets, h_offsets.ctypes.data, len(h_offsets) - 1,
                                             d_stream_codes or None, stream))

    def check_end(self) -> CheckReport:
        """lphb_check_end: closes the session and returns its report"""
        r = CheckReport()
        _check(lib().lphb_check_end(self._h, C.byref(r)))
        return r

    def check(self, bases, offsets) -> CheckReport:
        """one-batch session: is this handle a minimal perfect hash of these contigs' k-mers, and do its streaming
        and non-streaming codes agree on them?"""
        self.check_begin()
        self.check_batch(bases, offsets)
        return self.check_end()


RUN_DTYPE = np.dtype([("first", "<u8"), ("n", "<i4")])  # 12 bytes packed: lphb_query_stream_runs records


def expand_runs(runs, threads: int = 1) -> np.ndarray:
    """lphb_expand_runs: run records -> the uint64 codes lphb_query_stream returns (host only)."""
    runs = np.ascontiguousarray(runs, dtype=RUN_DTYPE)
    total = int(np.abs(runs["n"].astype(np.int64)).sum())
    codes = np.empty(max(total, 1), dtype=np.uint64)
    n = C.c_uint64(0)
    _check(lib().lphb_expand_runs(runs.ctypes.data, len(runs), codes.ctypes.data, total, C.byref(n), threads))
    return codes[: n.value]


# ---- build-side scan (module-level like the reference's free functions in namespace minimizer) --

def scan_superkmers(bases, offsets, k: int, m: int, seed: int = 42, mm_count: int = 0, device: int = 0):
    """minimizer::from_string over a batch (/root/reference/include/minimizer.hpp:11-170).
    Returns (records[RECORD_DTYPE] in scan order, n_kmers, mm_count_out)."""
    bases, offsets = _as_batch(bases, offsets)
    n = len(offsets) - 1
    lens = np.diff(offsets).astype(np.int64)
    cap = int(np.maximum(lens - k + 1, 0).sum()) + n + 1
    rec = np.empty(max(cap, 1), dtype=RECORD_DTYPE)
    mm = C.c_uint64(mm_count)
    nrec, nk = C.c_uint64(0), C.c_uint64(0)
    _check(lib().lphb_scan_superkmers(device, k, m, seed, bases.ctypes.data, offsets.ctypes.data, n,
                                      C.byref(mm), rec.ctypes.data, cap, C.byref(nrec), C.byref(nk)))
    return rec[: nrec.value], nk.value, mm.value


def scan_superkmers_device(d_bases: int, d_offsets: int, h_offsets, k: int, m: int, seed: int = 42,
                           mm_count: int = 0, device: int = 0, fetch: bool = True):
    """lphb_scan_superkmers_device: bases / offsets already on the device (raw pointers).  Returns
    (records or None, n_records, n_kmers, mm_count_out, kernel_ms)."""
    h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint64)
    mm = C.c_uint64(mm_count)
    ptr = C.c_void_p()
    nrec, nk, ms = C.c_uint64(0), C.c_uint64(0), C.c_double(0)
    _check(lib().lphb_scan_superkmers_device(device, k, m, seed, d_bases, d_offsets, h_offsets.ctypes.data,
                                             len(h_offsets) - 1, C.byref(mm), C.byref(ptr), C.byref(nrec), C.byref(nk),
                                             C.byref(ms)))
    rec = None
    if fetch:
        rec = np.empty(nrec.value, dtype=RECORD_DTYPE)
        if nrec.value:
            _check(lib().lphb_copy_to_host(device, rec.ctypes.data, ptr, nrec.value * 18))
    return rec, nrec.value, nk.value, mm.value, ms.value


TRIPLET_DTYPE = np.dtype([("itself", "<u8"), ("p1", "u1"), ("size", "u1")])  # mm_triplet_t


def classify(records, device: int = 0):
    """Sort by minimizer + minimizer::classify (/root/reference/src/minimizer.cpp:5-50).
    Returns (triplets[TRIPLET_DTYPE] in ascending minimizer order, ascending colliding ids)."""
    records = np.ascontiguousarray(records, dtype=RECORD_DTYPE)
    n = len(records)
    trip = np.empty(max(n, 1), dtype=TRIPLET_DTYPE)
    ids = np.empty(max(n, 1), dtype=np.uint64)
    nt, ni = C.c_uint64(0), C.c_uint64(0)
    _check(lib().lphb_classify(device, records.ctypes.data, n, trip.ctypes.data, n, C.byref(nt),
                               ids.ctypes.data, n, C.byref(ni)))
    return trip[: nt.value].copy(), ids[: ni.value].copy()


def scan_classify(bases, offsets, k: int, m: int, seed: int = 42, mm_count: int = 0, device: int = 0):
    """from_string over the batch + sort + classify with the records kept on the device.
    Returns (triplets, colliding ids, n_kmers, mm_count_out)."""
    bases, offsets = _as_batch(bases, offsets)
    n = len(offsets) - 1
    cap = int(np.maximum(np.diff(offsets).astype(np.int64) - k + 1, 0).sum()) + 1
    trip = np.empty(cap, dtype=TRIPLET_DTYPE)
    ids = np.empty(cap, dtype=np.uint64)
    mm = C.c_uint64(mm_count)
    nt, ni, nk = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    _check(lib().lphb_scan_classify(device, k, m, seed, bases.ctypes.data, offsets.ctypes.data, n, C.byref(mm),
                                    trip.ctypes.data, cap, C.byref(nt), ids.ctypes.data, cap, C.byref(ni),
                                    C.byref(nk)))
    return trip[: nt.value].copy(), ids[: ni.value].copy(), nk.value, mm.value


class BuildSession:
    """lphb_build_*: Parts 1 + 2 of build-p over an input fed batch by batch.  end() returns what scan_classify returns
    on the concatenation of the batches (mm_count = 0): (triplets, colliding ids, BuildReport).

        with BuildSession(k, m, seed) as s:
            for bases, offsets in batches:
                s.batch(bases, offsets)
            triplets, ids, report = s.end()
    """

    def __init__(self, k: int, m: int, seed: int = 42, device: int = 0):
        self.k, self.m, self.seed, self.device = k, m, seed, device
        h = C.c_void_p()
        _check(lib().lphb_build_begin(device, k, m, seed, C.byref(h)))
        self._h = h

    def batch(self, bases, offsets) -> None:
        """one batch of whole contigs in host arrays (as scan_classify takes them)"""
        bases, offsets = _as_batch(bases, offsets)
        _check(lib().lphb_build_batch(self._h, bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1))

    def batch_device(self, d_bases: int, d_offsets: int, h_offsets, stream: int = 0) -> None:
        """one batch in device buffers: raw pointers (ints), e.g. tensor.data_ptr(), d_bases indexed by the offsets,
        h_offsets their host copy; waits for `stream` (a cudaStream_t) first.  Synchronous."""
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint64)
        _check(lib().lphb_build_batch_device(self._h, d_bases, d_offsets, h_offsets.ctypes.data, len(h_offsets) - 1,
                                             stream))

    def end(self):
        """merges the batches and closes the session: (triplets[TRIPLET_DTYPE] ascending, ids ascending, BuildReport).
        The first call asks for the sizes, the second copies the result out."""
        L = lib()
        r = BuildReport()
        rc = L.lphb_build_end(self._h, None, 0, None, 0, C.byref(r))
        if rc == OK:
            return np.empty(0, dtype=TRIPLET_DTYPE), np.empty(0, dtype=np.uint64), r
        if rc != E_CAPACITY:
            _check(rc)
        trip = np.empty(r.n_triplets, dtype=TRIPLET_DTYPE)
        ids = np.empty(r.n_ids, dtype=np.uint64)
        _check(L.lphb_build_end(self._h, trip.ctypes.data, len(trip), ids.ctypes.data, len(ids), C.byref(r)))
        return trip, ids, r

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().lphb_build_free(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def colliding_kmers(bases, offsets, k: int, m: int, ids, seed: int = 42, kmer_bits: int = 64,
                    mm_count: int = 0, device: int = 0) -> np.ndarray:
    """minimizer::get_colliding_kmers over a batch (/root/reference/include/minimizer.hpp:172-319).
    Returns an (n, kmer_bits // 64) uint64 array, column 0 = low word."""
    bases, offsets = _as_batch(bases, offsets)
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    n = len(offsets) - 1
    words = kmer_bits // 64
    cap = int(np.maximum(np.diff(offsets).astype(np.int64) - k + 1, 0).sum())
    out = np.empty((max(cap, 1), words), dtype=np.uint64)
    mm = C.c_uint64(mm_count)
    nk = C.c_uint64(0)
    _check(lib().lphb_colliding_kmers(device, k, m, seed, bases.ctypes.data, offsets.ctypes.data, n,
                                      C.byref(mm), ids.ctypes.data, len(ids), kmer_bits,
                                      out.ctypes.data, cap, C.byref(nk)))
    return out[: nk.value]


def build_inverted_index(k: int, m: int, minimizer_order: bytes, triplets, device: int = 0, capacity: int | None = None):
    """build-p Part 3 (re-key by minimizer_order + mphf::build_inverted_index, /root/reference/src/
    partitioned_mphf.cpp:92-106, 163-268).  minimizer_order = serialized single_phf; triplets = TRIPLET_DTYPE array.
    Returns (InvertedIndex, body bytes = image of wtree + image of sizes_and_positions)."""
    trip = np.ascontiguousarray(triplets, dtype=TRIPLET_DTYPE)
    phf = np.frombuffer(minimizer_order, dtype=np.uint8)
    cap = lib().lphb_inverted_index_bound(len(trip)) if capacity is None else capacity
    out = np.empty(max(cap, 1), dtype=np.uint8)
    info = InvertedIndex()
    nb = C.c_uint64(0)
    _check(lib().lphb_build_inverted_index(device, k, m, phf.ctypes.data, len(phf), trip.ctypes.data, len(trip),
                                           out.ctypes.data, cap, C.byref(nb), C.byref(info)))
    return info, out[: nb.value].tobytes()


def lph_sections(image: bytes, kmer_bits: int = 64, alt: bool = False) -> list[int]:
    """Start of minimizer_order, of the wavelet tree (alt: positions), of sizes_and_positions (alt: sizes), of
    fallback_kmer_order, and the end of a serialized index.  Host only."""
    buf = np.frombuffer(image, dtype=np.uint8)
    sec = (C.c_uint64 * 5)()
    _check(lib().lphb_lph_sections(buf.ctypes.data, len(buf), kmer_bits, int(alt), sec))
    return [int(v) for v in sec]


def lph_assemble(k: int, m: int, mm_seed: int, nkmers: int, distinct_minimizers: int, index: InvertedIndex,
                 minimizer_order: bytes, index_body: bytes, fallback_kmer_order: bytes) -> bytes:
    """A complete `.lph` image (what essentials::save writes, /root/reference/src/build.cpp:52) from its parts.  Host only."""
    mo = np.frombuffer(minimizer_order, dtype=np.uint8)
    body = np.frombuffer(index_body, dtype=np.uint8)
    fb = np.frombuffer(fallback_kmer_order, dtype=np.uint8)
    cap = 58 + len(mo) + len(body) + len(fb)
    out = np.empty(cap, dtype=np.uint8)
    nb = C.c_uint64(0)
    _check(lib().lphb_lph_assemble(k, m, mm_seed, nkmers, distinct_minimizers, C.byref(index), mo.ctypes.data, len(mo),
                                   body.ctypes.data, len(body), fb.ctypes.data, len(fb), out.ctypes.data, cap, C.byref(nb)))
    return out[: nb.value].tobytes()


def build_inverted_index_alt(minimizer_order: bytes, triplets, device: int = 0):
    """build-u Part 3 (mphf_alt: /root/reference/src/unpartitioned_mphf.cpp:78-96, 152-169).
    Returns (InvertedIndexAlt, body bytes = image of positions + image of sizes)."""
    trip = np.ascontiguousarray(triplets, dtype=TRIPLET_DTYPE)
    phf = np.frombuffer(minimizer_order, dtype=np.uint8)
    cap = lib().lphb_inverted_index_bound(len(trip))
    out = np.empty(max(cap, 1), dtype=np.uint8)
    info = InvertedIndexAlt()
    nb = C.c_uint64(0)
    _check(lib().lphb_build_inverted_index_alt(device, phf.ctypes.data, len(phf), trip.ctypes.data, len(trip),
                                               out.ctypes.data, cap, C.byref(nb), C.byref(info)))
    return info, out[: nb.value].tobytes()


def lph_assemble_alt(k: int, m: int, mm_seed: int, nkmers: int, distinct_minimizers: int, index: InvertedIndexAlt,
                     minimizer_order: bytes, index_body: bytes, fallback_kmer_order: bytes) -> bytes:
    """A complete serialized lphash::mphf_alt (what build-u saves) from its parts.  Host only."""
    mo = np.frombuffer(minimizer_order, dtype=np.uint8)
    body = np.frombuffer(index_body, dtype=np.uint8)
    fb = np.frombuffer(fallback_kmer_order, dtype=np.uint8)
    cap = 34 + len(mo) + len(body) + len(fb)
    out = np.empty(cap, dtype=np.uint8)
    nb = C.c_uint64(0)
    _check(lib().lphb_lph_assemble_alt(k, m, mm_seed, nkmers, distinct_minimizers, C.byref(index), mo.ctypes.data, len(mo),
                                       body.ctypes.data, len(body), fb.ctypes.data, len(fb), out.ctypes.data, cap,
                                       C.byref(nb)))
    return out[: nb.value].tobytes()
