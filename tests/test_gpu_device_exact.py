"""Batches in device buffers with the reference's answers: lphb_query_stream_exact_device (the streaming branch,
non-ACGT quirk included: include/partitioned_mphf.hpp:73-184) and lphb_query_nonstreaming_device (the non-streaming
branch, a non-ACGT byte counts as 'A': :185-195), checked against the reference's golden codes, the bundled config-1
files and the library's host forms."""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_DIR, GOLDEN_NAMES, ROOT, load_golden
from lphash_b200 import api, seqio, synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
ALT_NAMES = ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"]
CFG1 = os.path.join(GOLDEN_DIR, "config1")
SENTINEL = np.uint64(0xA5A5A5A5A5A5A5A5)
GUARD = 256  # codes past the capacity that must stay untouched


def concat(contigs):
    bases = np.frombuffer(b"".join(contigs), dtype=np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in contigs])]).astype(np.uint64)
    return bases, offsets


def capacity(offsets, m):
    return int(np.maximum(np.diff(offsets.astype(np.int64)) - m + 1, 0).sum())


def clean_total(offsets, k):
    return int(np.maximum(np.diff(offsets.astype(np.int64)) - k + 1, 0).sum())


class DeviceBatch:
    """bases and offsets on the device: `lead` junk bytes (N) before the batch, offsets shifted by them; d_bases
    `shift` bytes into its allocation"""

    def __init__(self, bases, offsets, lead=0, shift=0):
        self.raw = np.concatenate([np.full(shift + lead, ord("N"), np.uint8), np.asarray(bases, np.uint8),
                                   np.full(7, ord("N"), np.uint8)])
        self.t = torch.from_numpy(self.raw.copy()).to(DEV)
        self.ptr = self.t.data_ptr() + shift
        self.offsets = offsets.astype(np.uint64) + np.uint64(lead)
        self.d_off = torch.from_numpy(self.offsets.astype(np.int64)).to(DEV)
        self.n = len(offsets) - 1

    def untouched(self):
        return np.array_equal(self.t.cpu().numpy(), self.raw)


def out_buffers(cap, n_contigs):
    d_codes = torch.from_numpy(np.full(cap + GUARD, SENTINEL).view(np.int64)).to(DEV)
    d_code_off = torch.full((n_contigs + 1,), -1, dtype=torch.int64, device=DEV)
    return d_codes, d_code_off


def host(t):
    return t.cpu().numpy().view(np.uint64)


def exact(f, b, cap=None, stream=0):
    """lphb_query_stream_exact_device over a DeviceBatch: (codes, code_offsets); checks the guard region"""
    cap = capacity(b.offsets, f.m) if cap is None else cap
    d_codes, d_code_off = out_buffers(cap, b.n)
    torch.cuda.synchronize()
    n = f.query_device_exact(b.ptr, b.d_off.data_ptr(), b.offsets, d_codes.data_ptr(), cap, d_code_off.data_ptr(), stream)
    codes = host(d_codes)
    assert (codes[cap:] == SENTINEL).all()
    return codes[:n], host(d_code_off)


def nonstreaming(f, b, stream=0):
    """lphb_query_nonstreaming_device over a DeviceBatch: (codes, code_offsets, status)"""
    cap = clean_total(b.offsets, f.k)
    d_codes, d_code_off = out_buffers(cap, b.n)
    d_status = torch.full((4,), -1, dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    f.query_device_nonstreaming(b.ptr, b.d_off.data_ptr(), b.offsets, d_codes.data_ptr(), cap, d_code_off.data_ptr(),
                                d_status.data_ptr(), stream)
    torch.cuda.synchronize()
    codes = host(d_codes)
    assert (codes[cap:] == SENTINEL).all()
    return codes[:cap], host(d_code_off), host(d_status)


@pytest.fixture
def handle():
    opened = []

    def load(name, alt=False):
        g = load_golden(name)
        path = os.path.join(GOLDEN_DIR, ("alt_" if alt else "") + name + ".lph")
        f = api.Mphf.load_alt(path, g.bits) if alt else api.Mphf.load(path, g.bits)
        opened.append(f)
        return g, f

    yield load
    for f in opened:
        f.close()


# ---- the reference's answers ------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", GOLDEN_NAMES)
@pytest.mark.parametrize("wide", [False, True])
def test_exact_form_gives_the_reference_codes(handle, name, wide, monkeypatch):
    if wide:
        monkeypatch.setenv("LPHB_FORCE_WIDE_BUCKETS", "1")
    g, f = handle(name)
    assert not all(g.is_clean())
    codes, code_off = exact(f, DeviceBatch(g.q_bases, g.q_offsets))
    assert np.array_equal(code_off, g.q_code_offsets)
    assert np.array_equal(codes, g.q_codes)
    assert f.stats().dirty_contigs > 0


@pytest.mark.parametrize("name", ALT_NAMES)
def test_unpartitioned_handle_gives_the_reference_codes(handle, name):
    g, f = handle(name, alt=True)
    z = np.load(os.path.join(GOLDEN_DIR, "alt_" + name + ".npz"))
    codes, code_off = exact(f, DeviceBatch(g.q_bases, g.q_offsets))
    assert np.array_equal(code_off, z["q_code_offsets"]) and np.array_equal(codes, z["q_codes"])
    bases, offsets = concat([c for c in g.contigs() if len(c) >= g.k])
    codes, _, _ = nonstreaming(f, DeviceBatch(bases, offsets))
    assert np.array_equal(codes, z["q_codes_ns"])


@pytest.fixture(scope="module")
def cfg1():
    f = api.Mphf.load(os.path.join(CFG1, "se.ust.k31_m16_u128.lph"), 128)
    yield f, json.load(open(os.path.join(CFG1, "expected.json")))["queries"]
    f.close()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<u8").tobytes()).hexdigest()


@pytest.mark.parametrize("name", ["ecoli1", "srr", "self"])
def test_bundled_query_files_match_reference(cfg1, name):
    f, queries = cfg1
    exp = queries[name]
    bases, offsets = seqio.read_batch(os.path.join(CFG1, exp["file"]))
    codes, code_off = exact(f, DeviceBatch(bases, offsets))
    assert len(codes) == exp["n_codes"]
    assert sha(codes) == exp["sha256_codes"]
    assert sha(np.diff(code_off)) == exp["sha256_counts"]
    if name == "self":
        assert np.array_equal(np.sort(codes), np.arange(f.get_kmer_count(), dtype=np.uint64))
    else:
        assert f.stats().dirty_contigs > 0


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_nonstreaming_form_equals_the_host_form_and_leaves_the_bases(handle, name):
    g, f = handle(name)
    want, want_off = f.query_batch(g.q_bases, g.q_offsets, streaming=False)
    b = DeviceBatch(g.q_bases, g.q_offsets)
    codes, code_off, status = nonstreaming(f, b)
    assert np.array_equal(codes, want) and np.array_equal(code_off, want_off)
    assert status[0] == len(want) and status[1] == 0
    assert b.untouched()
    assert not f.dirty_flags().any() and f.stats().dirty_contigs == 0


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
def test_nonstreaming_form_equals_the_stateless_form_on_clean_batches(handle, name):
    g, f = handle(name)
    b = DeviceBatch(g.index_bases, g.index_offsets, lead=5)
    n = clean_total(b.offsets, f.k)
    d_codes, d_code_off = out_buffers(n, b.n)
    d_status = torch.zeros(4, dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    f.query_device(b.ptr, b.d_off.data_ptr(), b.offsets, d_codes.data_ptr(), n, d_code_off.data_ptr(), d_status.data_ptr())
    torch.cuda.synchronize()
    codes, code_off, status = nonstreaming(f, b)
    assert np.array_equal(codes, host(d_codes)[:n]) and np.array_equal(code_off, host(d_code_off))
    assert np.array_equal(np.sort(codes), np.arange(f.get_kmer_count(), dtype=np.uint64))


# ---- layout and edge cases --------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["k31_m20_u64", "k25_m13_u64"])
def test_offsets_not_at_zero_and_unaligned_bases(handle, name):
    g, f = handle(name)
    want_ns, want_ns_off = f.query_batch(g.q_bases, g.q_offsets, streaming=False)
    for lead, shift in [(37, 0), (0, 1), (3, 5), (0, 8), (1, 15), (64, 13)]:
        b = DeviceBatch(g.q_bases, g.q_offsets, lead=lead, shift=shift)
        codes, code_off = exact(f, b)
        assert np.array_equal(codes, g.q_codes) and np.array_equal(code_off, g.q_code_offsets), (lead, shift)
        codes, code_off, _ = nonstreaming(f, b)
        assert np.array_equal(codes, want_ns) and np.array_equal(code_off, want_ns_off), (lead, shift)
        assert b.untouched()


def test_single_records_and_short_spans(handle):
    """one record per batch, dirty ones included, at every alignment; spans shorter than one 16-byte vector"""
    g, f = handle("k31_m20_u64")
    contigs = g.contigs()
    picked = [c for c in contigs if len(c) >= g.k][:6] + [c for c, ok in zip(contigs, g.is_clean()) if not ok][:6]
    picked += [b"ACGTN" * 9, b"NNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNN", b"acgtnACGTxACGT" * 4]
    for i, c in enumerate(picked):
        bases, offsets = concat([c])
        want, want_off = f.query_batch(bases, offsets)
        want_ns, _ = f.query_batch(bases, offsets, streaming=False)
        for shift in (0, i % 16, 15):
            b = DeviceBatch(bases, offsets, lead=shift % 3, shift=shift)
            codes, code_off = exact(f, b)
            assert np.array_equal(codes, want) and np.array_equal(code_off, want_off), (i, shift)
            assert np.array_equal(nonstreaming(f, b)[0], want_ns), (i, shift)
    # spans of 0..40 bytes at every alignment: the copy's head and tail alone
    rng = np.random.default_rng(11)
    for n in range(0, 41):
        seq = bytes(rng.choice(list(b"ACGTNacgt"), size=n).tolist())
        bases, offsets = concat([seq])
        want_ns, _ = f.query_batch(bases, offsets, streaming=False)
        for shift in range(16):
            b = DeviceBatch(bases, offsets, shift=shift)
            assert np.array_equal(nonstreaming(f, b)[0], want_ns), (n, shift)
            assert b.untouched()


def test_empty_batches(handle):
    g, f = handle("k31_m20_u64")
    for offsets in (np.zeros(1, np.uint64), np.zeros(4, np.uint64), np.array([0, 3, 3, 10], np.uint64)):
        bases = np.frombuffer(b"ACGTNNNACG", dtype=np.uint8)[: int(offsets[-1])]
        b = DeviceBatch(bases, offsets, lead=2)
        codes, code_off = exact(f, b)
        assert len(codes) == 0 and not code_off.any()
        codes, code_off, status = nonstreaming(f, b)
        assert len(codes) == 0 and not code_off.any() and status[0] == 0 and status[1] == 0


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k40_m17_u128"])
def test_all_dirty_no_dirty_and_short_contigs_between_dirty_ones(handle, name):
    g, f = handle(name)
    contigs, clean = g.contigs(), g.is_clean()
    dirty = [c for c, ok in zip(contigs, clean) if not ok and len(c) >= g.k]
    spotless = [c for c, ok in zip(contigs, clean) if ok]
    short = [b"ACG", b"N", b"ACGTNACG", b"", b"A" * (g.k - 1), b"NA" * ((g.k - 1) // 2)]
    mixed = []
    for i, c in enumerate(dirty):
        mixed += [c, short[i % len(short)]]
    for contigs_ in (dirty, spotless, mixed, short + dirty[:1] + short):
        bases, offsets = concat(contigs_)
        want, want_off = f.query_batch(bases, offsets)
        host_flags = f.dirty_flags() != 0
        codes, code_off = exact(f, DeviceBatch(bases, offsets, lead=3))
        assert np.array_equal(codes, want) and np.array_equal(code_off, want_off)
        flags = f.dirty_flags() != 0
        assert np.array_equal(flags, host_flags)
        # (a contig shorter than k has no window: a kernel need not look at its bytes)
        long = np.array([len(c) >= g.k for c in contigs_], dtype=bool)
        has_n = np.array([not all(ch in b"ACGTUacgtu" for ch in c) for c in contigs_], dtype=bool)
        assert np.array_equal(flags[long], has_n[long])
        assert f.stats().dirty_contigs == int(flags.sum())


# ---- capacity -----------------------------------------------------------------------------------------------------

def test_capacity_errors_report_the_size_and_write_nothing_past_it(handle):
    g, f = handle("k31_m20_u64")
    b = DeviceBatch(g.q_bases, g.q_offsets, lead=1, shift=3)
    n, clean = len(g.q_codes), clean_total(b.offsets, f.k)
    for cap in sorted({0, 1, n - 1, clean - 1, clean, (n + clean) // 2}):
        if cap >= n:
            continue
        with pytest.raises(api.CapacityError) as e:
            exact(f, b, cap=cap)
        assert e.value.code == api.E_CAPACITY and e.value.n_codes == n, cap
    # a clean batch: its clean total is the final one
    cb = DeviceBatch(g.index_bases, g.index_offsets)
    nc = clean_total(cb.offsets, f.k)
    with pytest.raises(api.CapacityError) as e:
        exact(f, cb, cap=nc - 1)
    assert e.value.n_codes == nc
    assert len(exact(f, cb, cap=nc)[0]) == nc


def test_capacity_at_the_final_total_below_the_clean_total(handle):
    g, f = handle("k31_m20_u64")
    rng = np.random.default_rng(5)
    genome = g.index_bases[: int(g.index_offsets[20])].tobytes()
    contigs = [genome[i:i + 300] + b"N" * 120 + genome[i + 300:i + 700] for i in range(0, 6000, 700)]
    contigs.append(bytes(rng.choice(list(b"ACGT"), size=500).tolist()))
    bases, offsets = concat(contigs)
    want, want_off = f.query_batch(bases, offsets)
    assert len(want) < clean_total(offsets, f.k)
    codes, code_off = exact(f, DeviceBatch(bases, offsets), cap=len(want))
    assert np.array_equal(codes, want) and np.array_equal(code_off, want_off)


# ---- streams and handle state -------------------------------------------------------------------------------------

def test_calls_on_two_streams_interleaved_with_the_other_device_forms(handle):
    """exact and non-streaming calls on two torch streams between lphb_query_stream_device and lphb_lookup_kmers_device
    calls on the same handle, with no host synchronisation but the exact form's own: each result is its own"""
    g, f = handle("k31_m20_u64")
    s1, s2 = torch.cuda.Stream(device=DEV), torch.cuda.Stream(device=DEV)
    rng = np.random.default_rng(9)
    genome = g.index_bases[: int(g.index_offsets[12])]
    jobs = []
    for i in range(6):
        bases, offsets = synth.reads(int(rng.integers(200, 3000)), genome, read_len=int(rng.integers(g.k, 300)),
                                     seed=300 + i)
        bases = bases.copy()
        for r in rng.choice(len(offsets) - 1, size=max(1, (len(offsets) - 1) // 50), replace=False):
            bases[int(offsets[r]) + int(rng.integers(0, int(offsets[r + 1] - offsets[r])))] = ord("N")
        want, want_off = f.query_batch(bases, offsets)
        want_ns, _ = f.query_batch(bases, offsets, streaming=False)
        b = DeviceBatch(bases, offsets, lead=i)
        cap, n_ns = capacity(b.offsets, f.m), clean_total(b.offsets, f.k)
        jobs.append(dict(b=b, want=want, want_off=want_off, want_ns=want_ns, cap=cap, n_ns=n_ns,
                         ex=out_buffers(cap, b.n), ns=out_buffers(n_ns, b.n),
                         ns_status=torch.zeros(4, dtype=torch.int64, device=DEV)))
    kmers = seqio.pack_kmers(g.index_bases, g.index_offsets, g.k, g.bits)
    want_lk = f.lookup(kmers)
    d_kmers = torch.from_numpy(kmers.view(np.int64).copy()).to(DEV)
    d_lk = torch.zeros(len(kmers), dtype=torch.int64, device=DEV)
    ib = DeviceBatch(g.index_bases, g.index_offsets)
    n_idx = clean_total(ib.offsets, f.k)
    d_q, d_q_off = out_buffers(n_idx, ib.n)
    d_q_status = torch.zeros(4, dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    for i, j in enumerate(jobs):
        sa, sb = (s1, s2) if i % 2 == 0 else (s2, s1)
        b = j["b"]
        f.lookup_device(d_kmers.data_ptr(), len(kmers), d_lk.data_ptr(), sa.cuda_stream)
        f.query_device_nonstreaming(b.ptr, b.d_off.data_ptr(), b.offsets, j["ns"][0].data_ptr(), j["n_ns"],
                                    j["ns"][1].data_ptr(), j["ns_status"].data_ptr(), sb.cuda_stream)
        f.query_device(ib.ptr, ib.d_off.data_ptr(), ib.offsets, d_q.data_ptr(), n_idx, d_q_off.data_ptr(),
                       d_q_status.data_ptr(), sa.cuda_stream)
        j["n"] = f.query_device_exact(b.ptr, b.d_off.data_ptr(), b.offsets, j["ex"][0].data_ptr(), j["cap"],
                                      j["ex"][1].data_ptr(), sb.cuda_stream)
    torch.cuda.synchronize()
    for i, j in enumerate(jobs):
        codes = host(j["ex"][0])
        assert j["n"] == len(j["want"]) and np.array_equal(codes[: j["n"]], j["want"]), i
        assert (codes[j["cap"]:] == SENTINEL).all() and np.array_equal(host(j["ex"][1]), j["want_off"]), i
        assert np.array_equal(host(j["ns"][0])[: j["n_ns"]], j["want_ns"]), i
    assert np.array_equal(host(d_lk), want_lk)
    assert np.array_equal(np.sort(host(d_q)[:n_idx]), np.arange(n_idx, dtype=np.uint64))
    assert int(d_q_status[1]) == 0


def test_dirty_flags_and_stats_after_each_call(handle):
    g, f = handle("k63_m24_u128")
    f.query_batch(g.q_bases, g.q_offsets)
    host_flags = f.dirty_flags()
    n_dirty = f.stats().dirty_contigs
    assert n_dirty > 0
    b = DeviceBatch(g.q_bases, g.q_offsets)
    exact(f, b)
    assert np.array_equal(f.dirty_flags() != 0, host_flags != 0)
    st = f.stats()
    assert st.dirty_contigs == n_dirty and st.kernel_launches > 4 and st.kernel_ms > 0
    assert st.h2d_bytes == 0 and st.d2h_bytes > 32
    nonstreaming(f, b)
    assert len(f.dirty_flags()) == b.n and not f.dirty_flags().any()
    st = f.stats()
    assert st.dirty_contigs == 0 and st.kernel_launches == 5 and st.d2h_bytes == 0 and st.kernel_ms > 0
    cb = DeviceBatch(g.index_bases, g.index_offsets)
    exact(f, cb)
    assert len(f.dirty_flags()) == cb.n and not f.dirty_flags().any()
    st = f.stats()
    assert st.dirty_contigs == 0 and st.kernel_launches == 4 and st.d2h_bytes == 32


def test_argument_errors_on_the_device(handle):
    g, f = handle("k31_m20_u64")
    b = DeviceBatch(g.q_bases, g.q_offsets)
    d_codes, d_code_off = out_buffers(capacity(b.offsets, f.m), b.n)
    L = api.lib()
    import ctypes as C
    n = C.c_uint64(0)
    off = b.offsets.ctypes.data
    assert L.lphb_query_stream_exact_device(f._h, None, b.d_off.data_ptr(), off, b.n, d_codes.data_ptr(), 10 ** 6,
                                            d_code_off.data_ptr(), C.byref(n), None) == api.E_ARG
    assert L.lphb_query_stream_exact_device(f._h, b.ptr, b.d_off.data_ptr(), off, b.n, None, 10 ** 6,
                                            d_code_off.data_ptr(), C.byref(n), None) == api.E_ARG
    assert L.lphb_query_nonstreaming_device(f._h, None, b.d_off.data_ptr(), off, b.n, d_codes.data_ptr(), 10 ** 6,
                                            d_code_off.data_ptr(), d_code_off.data_ptr(), None) == api.E_ARG
    # the handle still answers
    codes, _ = exact(f, b)
    assert np.array_equal(codes, g.q_codes)


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_cpp_mirror_device_forms(tmp_path, name):
    g = load_golden(name)
    exe = str(tmp_path / "device_exact_check")
    libdir = os.path.join(ROOT, "lphash_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", f"-DLPHASH_B200_KMER_BITS={g.bits}",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           os.path.join(ROOT, "tests", "cpp", "device_exact_check.cpp"), "-o", exe,
                           "-L", libdir, "-llphash_b200", f"-Wl,-rpath,{libdir}",
                           "-L", os.path.join(cuda, "lib64"), "-lcudart", f"-Wl,-rpath,{os.path.join(cuda, 'lib64')}"])
    offsets = g.q_offsets.astype("<u8")
    (tmp_path / "batch.bin").write_bytes(np.uint64(len(offsets) - 1).tobytes() + offsets.tobytes() +
                                         g.q_bases[: int(offsets[-1])].tobytes())
    r = subprocess.run([exe, g.lph, str(tmp_path / "batch.bin"), str(tmp_path / "out.bin")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = np.fromfile(tmp_path / "out.bin", dtype="<u8")
    n = int(out[0])
    assert np.array_equal(out[1:1 + n], g.q_codes)
    assert np.array_equal(out[1 + n:2 + n + len(offsets) - 1], g.q_code_offsets)
    rest = out[2 + n + len(offsets) - 1:]
    f = api.Mphf.load(g.lph, g.bits)
    try:
        want_ns, _ = f.query_batch(g.q_bases, g.q_offsets, streaming=False)
    finally:
        f.close()
    assert int(rest[0]) == len(want_ns) and np.array_equal(rest[1:], want_ns)
