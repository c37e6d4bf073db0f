"""Lookup of packed k-mers, the parts that need no GPU: argument checks of the two C entry points and the packing
helper the tests and the lookup bench share (seqio.pack_kmers)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from lphash_b200 import api, seqio


def test_null_handle_and_null_pointers_are_argument_errors():
    L = api.lib()
    buf = np.zeros(8, dtype=np.uint64)
    p = buf.ctypes.data
    for n in (0, 1, 5):
        assert L.lphb_lookup_kmers(None, p, n, p) == api.E_ARG
        assert L.lphb_lookup_kmers(None, None, n, None) == api.E_ARG
        assert L.lphb_lookup_kmers_device(None, p, n, p, None) == api.E_ARG
        assert L.lphb_lookup_kmers_device(None, None, n, None, None) == api.E_ARG
    assert b"null" in L.lphb_last_error()


def _reference_pack(contigs, k):
    """the reference's string_to_integer_no_reverse over every window (include/mphf_utils.hpp:108-116)"""
    code = {ord(c): v for c, v in zip("ACGTUacgtu", (0, 1, 2, 3, 3, 0, 1, 2, 3, 3))}
    out = []
    for seq in contigs:
        for s in range(len(seq) - k + 1):
            x = 0
            for ch in seq[s:s + k]:
                x = (x << 2) | code.get(ch, 0)
            out.append(x)
    return out


@pytest.mark.parametrize("k,bits", [(1, 64), (15, 64), (31, 64), (31, 128), (32, 128), (47, 128), (63, 128)])
def test_pack_kmers_matches_the_reference_encoding(k, bits):
    rng = np.random.default_rng(k * 1000 + bits)
    contigs = [bytes(rng.choice(list(b"ACGTUacgtuN-n"), size=int(n)).tolist()) for n in rng.integers(0, 3 * k, 60)]
    contigs.append(b"")
    bases, offsets = seqio.concat(contigs)
    got = seqio.pack_kmers(bases, offsets, k, bits)
    want = _reference_pack(contigs, k)
    if bits == 64:
        assert got.shape == (len(want),) and got.tolist() == want
    else:
        assert got.shape == (len(want), 2)
        assert [lo | (hi << 64) for lo, hi in got.tolist()] == want


def test_pack_kmers_edges():
    bases, offsets = seqio.concat([b"ACG", b"T"])
    assert seqio.pack_kmers(bases, offsets, 4, 64).shape == (0,)
    assert seqio.pack_kmers(bases, offsets, 4, 128).shape == (0, 2)
    assert seqio.pack_kmers(bases, offsets[:1], 3, 64).shape == (0,)
    # offsets need not start at 0
    assert seqio.pack_kmers(np.frombuffer(b"xxTTTT", dtype=np.uint8), np.array([2, 6], dtype=np.uint64), 4, 64).tolist() \
        == [0xFF]
    for k, bits in ((32, 64), (64, 128), (0, 64)):
        with pytest.raises(ValueError):
            seqio.pack_kmers(bases, offsets, k, bits)


@pytest.mark.parametrize("bits", [64, 128])
def test_cpp_lookup_mirror_compiles_and_fails_loudly_without_gpu(tmp_path, bits):
    exe = str(tmp_path / "lookup_check")
    libdir = os.path.join(ROOT, "lphash_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", f"-DLPHASH_B200_KMER_BITS={bits}",
                           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "lookup_check.cpp"),
                           "-o", exe, "-L", libdir, "-llphash_b200", f"-Wl,-rpath,{libdir}"])
    n = C.c_int(-1)
    if api.lib().lphb_device_count(C.byref(n)) == api.OK and n.value > 0:
        pytest.skip("a GPU is present")
    (tmp_path / "kmers.bin").write_bytes(np.uint64(1).tobytes() + bytes(bits // 8))
    lph = os.path.join(ROOT, "tests", "golden", "k31_m20_u64.lph" if bits == 64 else "k31_m16_u128.lph")
    r = subprocess.run([exe, lph, str(tmp_path / "kmers.bin"), str(tmp_path / "codes.bin")],
                       capture_output=True, text=True)
    assert r.returncode == 3 and "CUDA" in r.stderr
