"""lphash_b200::build_session, the C++ wrapper of the build session (include/lphash_b200.hpp), compiled with g++
against the C-ABI library: one contig per batch gives the golden triplets and ids."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden

SRC = os.path.join(ROOT, "tests", "cpp", "build_session_check.cpp")
LIBDIR = os.path.join(ROOT, "lphash_b200")


def build(tmp):
    exe = os.path.join(tmp, "build_session_check")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), SRC,
                           "-o", exe, "-L", LIBDIR, "-llphash_b200", f"-Wl,-rpath,{LIBDIR}"])
    return exe


def run(tmp_path, g):
    exe = build(str(tmp_path))
    with open(tmp_path / "batch.bin", "wb") as f:
        n = len(g.index_offsets) - 1
        f.write(np.array([g.k, g.m, n], dtype="<u8").tobytes() + g.index_offsets.astype("<u8").tobytes())
        f.write(g.index_bases.tobytes())
    return subprocess.run([exe, str(tmp_path / "batch.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)


def test_compiles_and_fails_loudly_without_gpu(tmp_path):
    from lphash_b200 import api
    try:
        have_gpu = api.device_count() > 0
    except api.LphashError:
        have_gpu = False
    if have_gpu:
        pytest.skip("a GPU is present")
    r = run(tmp_path, load_golden("k31_m20_u64"))
    assert r.returncode == 3 and "CUDA" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_one_contig_per_batch_gives_the_golden_classify(tmp_path, name):
    g = load_golden(name)
    r = run(tmp_path, g)
    assert r.returncode == 0, r.stderr
    raw = open(tmp_path / "out.bin", "rb").read()
    n = int(np.frombuffer(raw, "<u8", 1, 0)[0])
    trip = np.frombuffer(raw, g.triplets.dtype, n, 8)
    pos = 8 + 10 * n
    n_ids = int(np.frombuffer(raw, "<u8", 1, pos)[0])
    ids = np.frombuffer(raw, "<u8", n_ids, pos + 8)
    kmers, mm, batches = np.frombuffer(raw, "<u8", 3, pos + 8 + 8 * n_ids).tolist()
    assert np.array_equal(trip, g.triplets) and np.array_equal(ids, g.coll_ids)
    assert (kmers, mm, batches) == (int(g.n_kmers), int(g.mm_count), len(g.index_offsets) - 1)
