"""lphb_query_stream_exact_device_async, the parts that need no GPU: argument checks of the C entry point and of its
Python binding, and the C++ mirror, which compiles and fails loudly without a device."""
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
    # a handle that is not null but is never dereferenced: each null pointer alone must be refused before it is
    fake = np.zeros(64, dtype=np.uint64).ctypes.data
    for n_contigs in (0, 1, 3):
        args = [p, p, p, n_contigs, p, 8, p, p]
        assert L.lphb_query_stream_exact_device_async(None, *args, None) == api.E_ARG
        assert b"null" in L.lphb_last_error()
        for i in (1, 2, 6, 7):  # d_offsets, h_offsets, d_code_offsets, d_status
            a = list(args)
            a[i] = None
            assert L.lphb_query_stream_exact_device_async(fake, *a, None) == api.E_ARG
            assert b"null" in L.lphb_last_error()
    assert buf.tolist() == [0] * 8  # nothing was written


def exe_path(tmp_path):
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    if not os.path.exists(os.path.join(cuda, "include", "cuda_runtime.h")):
        pytest.skip("no CUDA toolkit headers")
    exe = str(tmp_path / "exact_async_check")
    libdir = os.path.join(ROOT, "lphash_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-DLPHASH_B200_KMER_BITS=64",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           os.path.join(ROOT, "tests", "cpp", "exact_async_check.cpp"), "-o", exe,
                           "-L", libdir, "-llphash_b200", f"-Wl,-rpath,{libdir}",
                           "-L", os.path.join(cuda, "lib64"), "-lcudart", f"-Wl,-rpath,{os.path.join(cuda, 'lib64')}"])
    return exe


def test_cpp_mirror_compiles_and_fails_loudly_without_gpu(tmp_path):
    exe = exe_path(tmp_path)
    n = C.c_int(-1)
    if api.lib().lphb_device_count(C.byref(n)) == api.OK and n.value > 0:
        pytest.skip("a GPU is present")
    (tmp_path / "batch.bin").write_bytes(np.array([1, 0, 4], dtype="<u8").tobytes() + b"ACGT")
    lph = os.path.join(ROOT, "tests", "golden", "k31_m20_u64.lph")
    r = subprocess.run([exe, lph, str(tmp_path / "batch.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert r.returncode == 3 and "CUDA" in r.stderr
