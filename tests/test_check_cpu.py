"""The index self-check (lphb_check_*), the parts that need no GPU: argument errors, the ctypes mirror of the report
against the C struct, and the C++ mirror and example tool building and failing loudly without a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT
from lphash_b200 import api

LIBDIR = os.path.join(ROOT, "lphash_b200")


def have_gpu():
    n = C.c_int(-1)
    return api.lib().lphb_device_count(C.byref(n)) == api.OK and n.value > 0


def test_null_handle_and_null_pointers_are_argument_errors():
    L = api.lib()
    buf = np.zeros(8, dtype=np.uint64)
    p = buf.ctypes.data
    assert L.lphb_check_begin(None) == api.E_ARG
    for n in (0, 1, 3):
        assert L.lphb_check_batch(None, p, p, n) == api.E_ARG
        assert L.lphb_check_batch(None, None, None, n) == api.E_ARG
        assert L.lphb_check_batch_device(None, p, p, p, n, p, None) == api.E_ARG
        assert L.lphb_check_batch_device(None, p, None, None, n, None, None) == api.E_ARG
    assert L.lphb_check_end(None, C.byref(api.CheckReport())) == api.E_ARG
    assert L.lphb_check_end(None, None) == api.E_ARG
    assert b"null" in L.lphb_last_error()


PROBE = r"""
#include <cstddef>
#include <cstdio>
#include "lphash_b200.h"
#define F(x) std::printf("%s %zu\n", #x, offsetof(lphb_check_report, x));
int main() {
    std::printf("sizeof %zu\n", sizeof(lphb_check_report));
    F(kmers) F(contigs) F(dirty_contigs) F(out_of_range) F(duplicates) F(missing) F(stream_mismatches)
    F(first_out_of_range) F(first_mismatch) F(min_duplicate_code) F(min_missing_code) F(ok)
}
"""


def test_ctypes_report_matches_the_c_struct(tmp_path):
    src = tmp_path / "probe.cpp"
    src.write_text(PROBE)
    exe = str(tmp_path / "probe")
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    got = dict(line.split() for line in subprocess.check_output([exe], text=True).splitlines())
    assert int(got.pop("sizeof")) == C.sizeof(api.CheckReport)
    assert list(got) == [name for name, _ in api.CheckReport._fields_]
    for name, off in got.items():
        assert getattr(api.CheckReport, name).offset == int(off), name


@pytest.mark.parametrize("bits", [64, 128])
def test_cpp_check_mirror_compiles_and_fails_loudly_without_gpu(tmp_path, bits):
    exe = str(tmp_path / "check_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", f"-DLPHASH_B200_KMER_BITS={bits}",
                           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "check_mirror.cpp"),
                           "-o", exe, "-L", LIBDIR, "-llphash_b200", f"-Wl,-rpath,{LIBDIR}"])
    if have_gpu():
        pytest.skip("a GPU is present")
    (tmp_path / "batch.bin").write_bytes(np.array([1, 0, 4], dtype="<u8").tobytes() + b"ACGT")
    lph = os.path.join(GOLDEN_DIR, "k31_m20_u64.lph" if bits == 64 else "k31_m16_u128.lph")
    r = subprocess.run([exe, lph, str(tmp_path / "batch.bin"), "1"], capture_output=True, text=True)
    assert r.returncode == 3 and "CUDA" in r.stderr


def build_check_tool(out_dir) -> str:
    exe = os.path.join(str(out_dir), "lphb_check")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-DLPHASH_B200_WITH_ZLIB",
                           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "lphb_check.cpp"),
                           "-o", exe, "-L", LIBDIR, "-llphash_b200", f"-Wl,-rpath,{LIBDIR}", "-lz", "-pthread"])
    return exe


def test_check_tool_compiles_and_fails_loudly_without_gpu(tmp_path):
    exe = build_check_tool(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode != 0 and "usage" in r.stderr
    if have_gpu():
        pytest.skip("a GPU is present")
    cfg1 = os.path.join(GOLDEN_DIR, "config1")
    r = subprocess.run([exe, os.path.join(cfg1, "se.ust.k31_m16_u128.lph"), "128", os.path.join(cfg1, "se.ust.k31.fa.gz")],
                       capture_output=True, text=True)
    assert r.returncode == 2 and "CUDA" in r.stderr and "Everything is ok" not in r.stdout
