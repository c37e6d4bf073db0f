"""FASTA / FASTQ (optionally gzip) reader producing the batch layout the C ABI consumes:
one uint8 array of concatenated bases + a uint64 offsets array (n_contigs + 1).

Mirrors what kseq.h hands to `mphf::operator()` in the reference driver
(/root/reference/src/query.cpp:51-52): `seq->seq.s` is the record's sequence with line breaks
removed (multi-line FASTA is joined), nothing else is altered (case, N, ... are preserved).
"""
from __future__ import annotations

import gzip

import numpy as np


def _open(path: str):
    with open(path, "rb") as f:
        magic = f.read(2)
    return gzip.open(path, "rb") if magic == b"\x1f\x8b" else open(path, "rb")


def read_records(path: str) -> list[bytes]:
    """Sequences of a FASTA/FASTQ file in file order."""
    out: list[bytes] = []
    with _open(path) as f:
        data = f.read()
    lines = data.split(b"\n")
    i, n = 0, len(lines)
    while i < n:
        ln = lines[i]
        if ln.startswith(b">"):
            i += 1
            parts = []
            while i < n and not lines[i].startswith(b">"):
                parts.append(lines[i].rstrip(b"\r"))
                i += 1
            out.append(b"".join(parts))
        elif ln.startswith(b"@"):
            # FASTQ (4-line records, as produced by every modern tool)
            seq = lines[i + 1].rstrip(b"\r") if i + 1 < n else b""
            out.append(seq)
            i += 4
        else:
            i += 1
    return out


def concat(records: list[bytes]) -> tuple[np.ndarray, np.ndarray]:
    lens = np.fromiter((len(r) for r in records), dtype=np.uint64, count=len(records))
    offsets = np.zeros(len(records) + 1, dtype=np.uint64)
    np.cumsum(lens, out=offsets[1:])
    bases = np.frombuffer(b"".join(records), dtype=np.uint8).copy()
    return bases, offsets


def read_batch(path: str) -> tuple[np.ndarray, np.ndarray]:
    return concat(read_records(path))


# 2-bit code of every byte as the reference's non-streaming branch reads it: A=0 C=1 G=2 T/U=3 in either case, any
# other byte 0 = 'A' (include/constants.hpp seq_nt4_table & 3, include/mphf_utils.hpp:108)
_NT4 = np.zeros(256, dtype=np.uint8)
for _ch, _v in zip(b"ACGTUacgtu", (0, 1, 2, 3, 3, 0, 1, 2, 3, 3)):
    _NT4[_ch] = _v


def pack_kmers(bases, offsets, k: int, kmer_bits: int = 64) -> np.ndarray:
    """Every window of k bases of every contig, in contig order, as the packed k-mers Mphf.lookup takes: the first
    base in the most significant of the 2k used bits (include/partitioned_mphf.hpp:106-108), non-ACGT bytes as 'A'.
    Returns uint64 (n,) for kmer_bits = 64, (n, 2) = [lo, hi] for 128."""
    if kmer_bits not in (64, 128) or not 1 <= k <= kmer_bits // 2 - 1:
        raise ValueError(f"k = {k} does not fit a {kmer_bits}-bit k-mer")
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64).astype(np.int64)
    nk = np.maximum(np.diff(offsets) - k + 1, 0)
    total = int(nk.sum())
    words = kmer_bits // 64
    if total == 0:
        return np.zeros((0,) if words == 1 else (0, 2), dtype=np.uint64)
    o0, o1 = int(offsets[0]), int(offsets[-1])
    codes = _NT4[bases[o0:o1]]
    w = o1 - o0 - k + 1  # windows of the concatenation; the ones that cross a contig boundary are dropped below
    n_hi = max(k - 32, 0)  # bases in the high word (128 bits): the first k - 32; the last 32 fill the low word

    def pack(first, count):
        acc = np.zeros(w, dtype=np.uint64)
        for j in range(first, first + count):
            np.left_shift(acc, np.uint64(2), out=acc)
            np.bitwise_or(acc, codes[j:j + w], out=acc)
        return acc

    lo = pack(n_hi, k - n_hi)
    hi = pack(0, n_hi) if words == 2 else None
    del codes
    first = np.concatenate([[0], np.cumsum(nk)[:-1]])
    starts = np.repeat(offsets[:-1] - o0 - first, nk) + np.arange(total, dtype=np.int64)
    if hi is None:
        return lo[starts]
    return np.stack([lo[starts], hi[starts]], axis=1)
