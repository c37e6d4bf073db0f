"""The device forms of the exact streaming and the non-streaming query, the parts that need no GPU: argument checks of
the two C entry points and of their C++ mirror."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from lphash_b200 import api


def test_null_handle_and_null_pointers_are_argument_errors():
    L = api.lib()
    buf = np.zeros(8, dtype=np.uint64)
    p = buf.ctypes.data
    n = C.c_uint64(7)
    for n_contigs in (0, 1, 3):
        # null handle, then each required pointer null in turn
        assert L.lphb_query_stream_exact_device(None, p, p, p, n_contigs, p, 8, p, C.byref(n), None) == api.E_ARG
        assert L.lphb_query_nonstreaming_device(None, p, p, p, n_contigs, p, 8, p, p, None) == api.E_ARG
        for i in (1, 2, 6, 7):  # d_offsets, h_offsets, d_code_offsets, d_status / n_codes
            args = [p, p, p, n_contigs, p, 8, p, p]
            args[i] = None
            assert L.lphb_query_nonstreaming_device(None, *args, None) == api.E_ARG
            args[7] = None if i == 7 else C.byref(n)
            assert L.lphb_query_stream_exact_device(None, *args, None) == api.E_ARG
        assert L.lphb_query_stream_exact_device(None, p, p, p, n_contigs, p, 8, p, None, None) == api.E_ARG
        assert L.lphb_query_nonstreaming_device(None, p, p, p, n_contigs, p, 8, p, None, None) == api.E_ARG
    assert b"null" in L.lphb_last_error()


def test_cpp_device_mirror_compiles_and_fails_loudly_without_gpu(tmp_path):
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    if not os.path.exists(os.path.join(cuda, "include", "cuda_runtime.h")):
        pytest.skip("no CUDA toolkit headers")
    exe = str(tmp_path / "device_exact_check")
    libdir = os.path.join(ROOT, "lphash_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-DLPHASH_B200_KMER_BITS=64",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           os.path.join(ROOT, "tests", "cpp", "device_exact_check.cpp"), "-o", exe,
                           "-L", libdir, "-llphash_b200", f"-Wl,-rpath,{libdir}",
                           "-L", os.path.join(cuda, "lib64"), "-lcudart", f"-Wl,-rpath,{os.path.join(cuda, 'lib64')}"])
    n = C.c_int(-1)
    if api.lib().lphb_device_count(C.byref(n)) == api.OK and n.value > 0:
        pytest.skip("a GPU is present")
    (tmp_path / "batch.bin").write_bytes(np.array([1, 0, 4], dtype="<u8").tobytes() + b"ACGT")
    lph = os.path.join(ROOT, "tests", "golden", "k31_m20_u64.lph")
    r = subprocess.run([exe, lph, str(tmp_path / "batch.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert r.returncode == 3 and "CUDA" in r.stderr
