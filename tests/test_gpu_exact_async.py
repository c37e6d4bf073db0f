"""lphb_query_stream_exact_device_async: the reference's streaming answers (non-ACGT quirk included,
include/partitioned_mphf.hpp:73-184) for a batch in device buffers, enqueued without a host synchronisation.  Checked
against the reference's golden codes, the bundled config-1 files, the CPU oracle on seeded dirty patterns and the
library's other forms; the capacity bound, the guard region past it, asynchrony and ordering on several streams."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, GOLDEN_NAMES, load_golden
from lphash_b200 import api, seqio, synth
from oracle import oracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
CFG1 = os.path.join(GOLDEN_DIR, "config1")
SENTINEL = np.uint64(0xA5A5A5A5A5A5A5A5)
GUARD = 256  # codes past the capacity that must stay untouched
ACGT = np.zeros(256, dtype=bool)
ACGT[np.frombuffer(b"ACGTUacgtu", dtype=np.uint8)] = True


def concat(contigs):
    bases = np.frombuffer(b"".join(contigs), dtype=np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in contigs])]).astype(np.uint64)
    return bases, offsets


def bound(offsets, m):
    return int(np.maximum(np.diff(offsets.astype(np.int64)) - m + 1, 0).sum())


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


class Call:
    """output buffers of one asynchronous call: codes with a guard region past the capacity, code offsets, status"""

    def __init__(self, f, b, cap=None):
        self.f, self.b = f, b
        self.cap = bound(b.offsets, f.m) if cap is None else cap
        self.codes = torch.from_numpy(np.full(self.cap + GUARD, SENTINEL).view(np.int64)).to(DEV)
        self.code_off = torch.full((b.n + 1,), -1, dtype=torch.int64, device=DEV)
        self.status = torch.full((4,), -1, dtype=torch.int64, device=DEV)

    def run(self, stream=0):
        self.f.query_device_exact_async(self.b.ptr, self.b.d_off.data_ptr(), self.b.offsets, self.codes.data_ptr(),
                                        self.cap, self.code_off.data_ptr(), self.status.data_ptr(), stream)
        return self

    def result(self):
        """(codes, code_offsets, status) once the stream is done; checks the guard region"""
        codes = self.codes.cpu().numpy().view(np.uint64)
        assert (codes[self.cap:] == SENTINEL).all()
        status = self.status.cpu().numpy().view(np.uint64)
        return codes[: int(status[0])], self.code_off.cpu().numpy().view(np.uint64), status


def exact_async(f, b, cap=None):
    torch.cuda.synchronize()
    c = Call(f, b, cap).run()
    torch.cuda.synchronize()
    return c.result()


def n_dirty(bases, offsets, shortest=0):
    """contigs of at least `shortest` bytes holding a non-ACGT byte"""
    return sum(1 for c in range(len(offsets) - 1) if offsets[c + 1] - offsets[c] >= shortest and
               not ACGT[bases[int(offsets[c]):int(offsets[c + 1])]].all())


def dirty_count_ok(status, bases, offsets, k):
    """d_status[1] counts the dirty contigs; one shorter than k has no window, and a kernel need not read its bytes"""
    return n_dirty(bases, offsets, k) <= status[1] <= n_dirty(bases, offsets)


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
def test_gives_the_reference_codes(handle, name, wide, monkeypatch):
    if wide:
        monkeypatch.setenv("LPHB_FORCE_WIDE_BUCKETS", "1")
    g, f = handle(name)
    codes, code_off, status = exact_async(f, DeviceBatch(g.q_bases, g.q_offsets))
    assert np.array_equal(code_off, g.q_code_offsets) and np.array_equal(codes, g.q_codes)
    assert dirty_count_ok(status, g.q_bases, g.q_offsets, g.k) and status[1] > 0
    want, want_off = f.query_batch(g.q_bases, g.q_offsets)
    assert np.array_equal(codes, want) and np.array_equal(code_off, want_off)


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
def test_unpartitioned_handle_gives_the_reference_codes(handle, name):
    g, f = handle(name, alt=True)
    z = np.load(os.path.join(GOLDEN_DIR, "alt_" + name + ".npz"))
    codes, code_off, _ = exact_async(f, DeviceBatch(g.q_bases, g.q_offsets))
    assert np.array_equal(code_off, z["q_code_offsets"]) and np.array_equal(codes, z["q_codes"])


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<u8").tobytes()).hexdigest()


@pytest.mark.parametrize("name", ["ecoli1", "srr", "self"])
def test_bundled_query_files_match_reference(name):
    f = api.Mphf.load(os.path.join(CFG1, "se.ust.k31_m16_u128.lph"), 128)
    try:
        exp = json.load(open(os.path.join(CFG1, "expected.json")))["queries"][name]
        bases, offsets = seqio.read_batch(os.path.join(CFG1, exp["file"]))
        codes, code_off, status = exact_async(f, DeviceBatch(bases, offsets))
        assert len(codes) == exp["n_codes"]
        assert sha(codes) == exp["sha256_codes"]
        assert sha(np.diff(code_off)) == exp["sha256_counts"]
        assert (status[1] > 0) == (name != "self")
    finally:
        f.close()


# ---- seeded dirty patterns against the CPU oracle -----------------------------------------------------------------

def patterns(g, rng):
    """contigs of the index's genome with non-ACGT bytes placed at the edges the repair has to get right"""
    k, m = g.k, g.m
    genome = g.index_bases.tobytes()
    at = iter(range(0, 10 ** 9, 97))

    def piece(n):
        i = next(at) % max(1, len(genome) - n)
        return genome[i:i + n]

    out = []
    body = piece(3 * k)
    out += [b"N" + body, body + b"N", b"N" + body + b"N", b"n" + body.lower() + b"n"]
    for run in (m - 1, m, k - 1, k, k + 1):
        out.append(piece(2 * k) + b"N" + piece(run) + b"N" + piece(2 * k))
        out.append(piece(2 * k) + b"NN" + b"".join(piece(run) + b"N" for _ in range(4)) + piece(k + 5))
    out += [b"N" * (3 * k), b"N", b"", piece(k - 1) + b"N", b"N" * k + piece(k)]
    out.append(piece(2 * k).lower() + b"N" + piece(k + 3).lower())
    for junk in (b"X", b"-", b".", b"\x00", b"\xff", b"R", b"*"):
        out.append(piece(2 * k) + junk + piece(m + 2) + junk + piece(2 * k))
    # random sprinkles, short runs and long ones
    for _ in range(30):
        c = bytearray(piece(int(rng.integers(k, 12 * k))))
        for p in rng.choice(len(c), size=int(rng.integers(1, 6)), replace=False):
            c[int(p)] = int(rng.choice(list(b"NNNnX")))
        out.append(bytes(c))
    # a contig longer than one repair chunk (1024 bytes) with runs across chunk boundaries
    long = bytearray(piece(3000))
    for p in (1023, 1024, 1030 + k, 2047, 2048 + m, 2999):
        long[p] = ord("N")
    out.append(bytes(long))
    return out


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
@pytest.mark.parametrize("generic_below", ["0", str(1 << 40)])
def test_seeded_dirty_patterns_match_the_oracle(handle, name, generic_below, monkeypatch):
    monkeypatch.setenv("LPHB_GENERIC_BELOW", generic_below)
    g, f = handle(name)
    o = oracle.OracleMphf(g.lph, g.bits)
    rng = np.random.default_rng(7 + g.k)
    contigs = patterns(g, rng)
    rb, ro = synth.reads(20000, g.index_bases, read_len=150, seed=11)  # a large clean batch
    clean = [rb[int(ro[i]):int(ro[i + 1])].tobytes() for i in range(len(ro) - 1)]
    batches = [contigs, contigs[::-1],
               [contigs[-1]] + clean,               # a dirty contig first: every clean code after it moves
               clean + [contigs[5]],                # ... and last
               clean[:5000] + [contigs[9]] + clean[5000:],
               [c for c in contigs if not ACGT[np.frombuffer(c, np.uint8)].all()]]  # every contig dirty
    for i, cs in enumerate(batches):
        bases, offsets = concat(cs)
        want, want_off = o.query_batch(bases, offsets)
        codes, code_off, status = exact_async(f, DeviceBatch(bases, offsets, lead=i, shift=i % 16))
        assert np.array_equal(code_off, want_off), i
        assert np.array_equal(codes, want), i
        assert dirty_count_ok(status, bases, offsets, g.k), i
        host, host_off = f.query_batch(bases, offsets)
        assert np.array_equal(host, want) and np.array_equal(host_off, want_off), i
        d = DeviceBatch(bases, offsets)
        c = Call(f, d)
        torch.cuda.synchronize()
        n = f.query_device_exact(d.ptr, d.d_off.data_ptr(), d.offsets, c.codes.data_ptr(), c.cap,
                                 c.code_off.data_ptr())
        sync = c.codes.cpu().numpy().view(np.uint64)
        assert n == len(want) and np.array_equal(sync[:n], want), i
    o.close()


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_gaps_of_millions_of_non_acgt_bytes_match_the_oracle(handle, name):
    """a long run, a gap of millions of N (thousands of repair chunks), short runs, a long run: the episode after the
    first run crosses the whole gap, on the asynchronous, the synchronous and the host form"""
    g, f = handle(name)
    o = oracle.OracleMphf(g.lph, g.bits)
    genome, k, m = g.index_bases.tobytes(), g.k, g.m
    short = b"".join(genome[5000 + 60 * i:5000 + 60 * i + m + i % (k - m)] + b"N" * (1 + 700 * i) for i in range(6))
    contigs = [genome[:4000] + b"N" * 3_000_000 + short + genome[6000:9000],
               genome[9000:9000 + 3 * k] + b"n" * 2_500_007 + genome[12000:12000 + k - 1] + b"X" * 70_000 +
               genome[13000:16000],
               b"N" * 1_000_000 + genome[16000:18000] + b"N" * 1_000_003,
               genome[18000:20000]]
    bases, offsets = concat(contigs)
    want, want_off = o.query_batch(bases, offsets)
    o.close()
    codes, code_off, status = exact_async(f, DeviceBatch(bases, offsets, lead=3, shift=5))
    assert np.array_equal(code_off, want_off) and np.array_equal(codes, want)
    assert status[1] == 3
    d = DeviceBatch(bases, offsets)
    c = Call(f, d)
    torch.cuda.synchronize()
    n = f.query_device_exact(d.ptr, d.d_off.data_ptr(), d.offsets, c.codes.data_ptr(), c.cap, c.code_off.data_ptr())
    assert n == len(want) and np.array_equal(c.codes.cpu().numpy().view(np.uint64)[:n], want)
    host, host_off = f.query_batch(bases, offsets)
    assert np.array_equal(host, want) and np.array_equal(host_off, want_off)


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
def test_stateless_form_holds_the_codes_of_windows_in_valid_runs(handle, name):
    """the slots of a dirty contig's windows of k ACGT bytes hold their codes (the repair takes them from there)"""
    g, f = handle(name)
    bases, offsets = concat(patterns(g, np.random.default_rng(3)))
    ns, _ = f.query_batch(bases, offsets, streaming=False)  # equal to the stateless code on an ACGT window
    n = int(np.maximum(np.diff(offsets.astype(np.int64)) - g.k + 1, 0).sum())
    b = DeviceBatch(bases, offsets)
    d_codes = torch.zeros(n + 1, dtype=torch.int64, device=DEV)
    d_off = torch.zeros(b.n + 1, dtype=torch.int64, device=DEV)
    d_status = torch.zeros(4, dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    f.query_device(b.ptr, b.d_off.data_ptr(), b.offsets, d_codes.data_ptr(), n, d_off.data_ptr(), d_status.data_ptr())
    torch.cuda.synchronize()
    got = d_codes.cpu().numpy().view(np.uint64)[:n]
    ok = ACGT[bases]
    mask = []
    for c in range(b.n):
        a, e = int(offsets[c]), int(offsets[c + 1])
        mask += [bool(ok[p:p + g.k].all()) for p in range(a, e - g.k + 1)]
    mask = np.array(mask, dtype=bool)
    assert mask.sum() > 0 and (~mask).sum() > 0
    assert np.array_equal(got[mask], ns[mask])


# ---- edges --------------------------------------------------------------------------------------------------------

def test_single_records_at_every_alignment_and_empty_batches(handle):
    g, f = handle("k31_m20_u64")
    contigs = g.contigs()
    picked = [c for c in contigs if len(c) >= g.k][:4] + [c for c, ok in zip(contigs, g.is_clean()) if not ok][:6]
    picked += [b"ACGTN" * 9, b"N" * 40, b"acgtnACGTxACGT" * 4, b"ACG"]
    for i, c in enumerate(picked):
        bases, offsets = concat([c])
        want, want_off = f.query_batch(bases, offsets)
        for shift in range(16):
            codes, code_off, status = exact_async(f, DeviceBatch(bases, offsets, lead=shift % 3, shift=shift))
            assert np.array_equal(codes, want) and np.array_equal(code_off, want_off), (i, shift)
    for offsets in (np.zeros(1, np.uint64), np.zeros(4, np.uint64), np.array([0, 3, 3, 10], np.uint64)):
        bases = np.frombuffer(b"ACGTNNNACG", dtype=np.uint8)[: int(offsets[-1])]
        codes, code_off, status = exact_async(f, DeviceBatch(bases, offsets, lead=2, shift=5))
        assert len(codes) == 0 and not code_off.any() and status[0] == 0


def test_offsets_not_at_zero_and_unaligned_bases(handle):
    g, f = handle("k63_m24_u128")
    for lead, shift in [(37, 0), (0, 1), (3, 5), (1, 15), (64, 13)]:
        codes, code_off, _ = exact_async(f, DeviceBatch(g.q_bases, g.q_offsets, lead=lead, shift=shift))
        assert np.array_equal(codes, g.q_codes) and np.array_equal(code_off, g.q_code_offsets), (lead, shift)


# ---- capacity -----------------------------------------------------------------------------------------------------

def test_capacity_at_the_bound_passes_and_one_below_enqueues_nothing(handle):
    g, f = handle("k31_m20_u64")
    b = DeviceBatch(g.q_bases, g.q_offsets, lead=1, shift=3)
    cap = bound(b.offsets, f.m)
    codes, code_off, _ = exact_async(f, b, cap=cap)
    assert np.array_equal(codes, g.q_codes)
    c = Call(f, b, cap=cap - 1)
    torch.cuda.synchronize()
    with pytest.raises(api.CapacityError) as e:
        c.run()
    assert e.value.code == api.E_CAPACITY and e.value.n_codes == cap and str(cap) in str(e.value)
    torch.cuda.synchronize()
    assert (c.codes.cpu().numpy().view(np.uint64) == SENTINEL).all()
    assert (c.code_off.cpu().numpy() == -1).all() and (c.status.cpu().numpy() == -1).all()


# ---- asynchrony, streams, workspace -------------------------------------------------------------------------------

def test_returns_before_the_stream_is_done(handle):
    g, f = handle("k31_m20_u64")
    b = DeviceBatch(g.q_bases, g.q_offsets)
    exact_async(f, b)  # the workspace at its size: the call below allocates nothing
    s = torch.cuda.Stream(device=DEV)
    c = Call(f, b)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
    c.run(s.cuda_stream)
    assert not s.query()
    s.synchronize()
    codes, code_off, status = c.result()
    assert np.array_equal(codes, g.q_codes) and np.array_equal(code_off, g.q_code_offsets)
    assert f.stats().kernel_launches > 4 and f.stats().d2h_bytes == 0


def test_calls_on_two_streams_interleaved_with_the_other_device_forms(handle):
    g, f = handle("k31_m20_u64")
    s1, s2 = torch.cuda.Stream(device=DEV), torch.cuda.Stream(device=DEV)
    rng = np.random.default_rng(21)
    genome = g.index_bases[: int(g.index_offsets[12])]
    jobs = []
    for i, reads in enumerate([40000, 30, 5000, 2, 20000, 300]):  # large then small: the workspace is reused
        bases, offsets = synth.reads(reads, genome, read_len=int(rng.integers(g.k, 200)), seed=700 + i)
        bases = bases.copy()
        for r in rng.choice(len(offsets) - 1, size=max(1, (len(offsets) - 1) // 40), replace=False):
            bases[int(offsets[r]) + int(rng.integers(0, int(offsets[r + 1] - offsets[r])))] = ord("N")
        want, want_off = f.query_batch(bases, offsets)
        jobs.append((Call(f, DeviceBatch(bases, offsets, lead=i)), want, want_off))
    kmers = seqio.pack_kmers(g.index_bases, g.index_offsets, g.k, g.bits)
    want_lk = f.lookup(kmers)
    d_kmers = torch.from_numpy(kmers.view(np.int64).copy()).to(DEV)
    d_lk = torch.zeros(len(kmers), dtype=torch.int64, device=DEV)
    ib = DeviceBatch(g.index_bases, g.index_offsets)
    n_idx = int(np.maximum(np.diff(ib.offsets.astype(np.int64)) - g.k + 1, 0).sum())
    d_q = torch.zeros(n_idx, dtype=torch.int64, device=DEV)
    d_q_off = torch.zeros(ib.n + 1, dtype=torch.int64, device=DEV)
    d_q_status = torch.zeros(4, dtype=torch.int64, device=DEV)
    f.check_begin()
    torch.cuda.synchronize()
    for i, (c, _, _) in enumerate(jobs):
        sa, sb = (s1, s2) if i % 2 == 0 else (s2, s1)
        f.lookup_device(d_kmers.data_ptr(), len(kmers), d_lk.data_ptr(), sa.cuda_stream)
        c.run(sb.cuda_stream)
        f.query_device(ib.ptr, ib.d_off.data_ptr(), ib.offsets, d_q.data_ptr(), n_idx, d_q_off.data_ptr(),
                       d_q_status.data_ptr(), sa.cuda_stream)
        if i == 2:  # the index once: a session that sees every k-mer once passes
            f.check_batch_device(ib.ptr, ib.d_off.data_ptr(), ib.offsets, stream=sb.cuda_stream)
    torch.cuda.synchronize()
    report = f.check_end()
    for i, (c, want, want_off) in enumerate(jobs):
        codes, code_off, status = c.result()
        assert np.array_equal(codes, want) and np.array_equal(code_off, want_off), i
        assert status[1] > 0, i
    assert np.array_equal(d_lk.cpu().numpy().view(np.uint64), want_lk)
    assert np.array_equal(np.sort(d_q.cpu().numpy().view(np.uint64)), np.arange(n_idx, dtype=np.uint64))
    assert report.ok and report.kmers == n_idx


def test_dirty_flags_and_stats(handle):
    g, f = handle("k63_m24_u128")
    f.query_batch(g.q_bases, g.q_offsets)
    host_flags = f.dirty_flags() != 0
    _, _, status = exact_async(f, DeviceBatch(g.q_bases, g.q_offsets))
    assert np.array_equal(f.dirty_flags() != 0, host_flags) and status[1] == host_flags.sum()
    st = f.stats()
    assert st.h2d_bytes == 0 and st.d2h_bytes == 0 and st.kernel_launches == 12 and st.kernel_ms > 0
    _, _, status = exact_async(f, DeviceBatch(g.index_bases, g.index_offsets))
    assert status[1] == 0 and not f.dirty_flags().any()


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_cpp_mirror(tmp_path, name):
    import subprocess

    from conftest import ROOT
    g = load_golden(name)
    exe = str(tmp_path / "exact_async_check")
    libdir = os.path.join(ROOT, "lphash_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", f"-DLPHASH_B200_KMER_BITS={g.bits}",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           os.path.join(ROOT, "tests", "cpp", "exact_async_check.cpp"), "-o", exe,
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
    assert n == len(g.q_codes) and dirty_count_ok(out, g.q_bases, g.q_offsets, g.k)
    assert np.array_equal(out[4:4 + n], g.q_codes) and np.array_equal(out[4 + n:], g.q_code_offsets)
