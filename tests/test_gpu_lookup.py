"""Lookup of packed k-mers (lphb_lookup_kmers / lphb_lookup_kmers_device): the code of every k-mer is what the
reference's non-streaming branch returns for the window that encodes it (include/partitioned_mphf.hpp:185-195),
checked against the reference's golden codes, the CPU oracle and the library's own streaming query."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_DIR, GOLDEN_NAMES, ROOT, load_golden
from lphash_b200 import api, seqio

pytestmark = pytest.mark.gpu
ALT_NAMES = ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"]


def batch(contigs):
    bases = np.frombuffer(b"".join(contigs), dtype=np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in contigs])]).astype(np.uint64)
    return bases, offsets


def clean_windows(g):
    """packed windows of the golden's ACGT-only query contigs and the reference's codes for them"""
    contigs, want = [], []
    for c, (seq, ok) in enumerate(zip(g.contigs(), g.is_clean())):
        if ok and len(seq) >= g.k:
            contigs.append(seq)
            want.append(g.q_codes[int(g.q_code_offsets[c]):int(g.q_code_offsets[c + 1])])
    bases, offsets = batch(contigs)
    return seqio.pack_kmers(bases, offsets, g.k, g.bits), np.concatenate(want)


def decode(kmers, k):
    """packed k-mers -> ASCII windows of k bases"""
    words = np.asarray(kmers, dtype=np.uint64).reshape(len(kmers), -1)
    out = []
    for row in words.tolist():
        x = row[0] | (row[1] << 64 if len(row) > 1 else 0)
        out.append(bytes(b"ACGT"[(x >> (2 * (k - 1 - j))) & 3] for j in range(k)))
    return out


def random_kmers(rng, n, k, bits):
    """uniform 2k-bit k-mers in the handle's layout"""
    words = bits // 64
    x = rng.integers(0, 1 << 63, size=(n, words), dtype=np.uint64) * np.uint64(2) + \
        rng.integers(0, 2, size=(n, words), dtype=np.uint64)
    if 2 * k < 64:
        x[:, 0] &= np.uint64((1 << (2 * k)) - 1)
    if words == 2:
        x[:, 1] &= np.uint64((1 << max(2 * k - 64, 0)) - 1)
    return x[:, 0].copy() if words == 1 else x


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


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_windows_of_clean_contigs_give_the_reference_codes(handle, name):
    g, f = handle(name)
    kmers, want = clean_windows(g)
    assert len(want) > 1000
    assert np.array_equal(f.lookup(kmers), want)


@pytest.mark.parametrize("name", ALT_NAMES)
def test_unpartitioned_handle_gives_the_reference_non_streaming_codes(handle, name):
    g, f = handle(name, alt=True)
    z = np.load(os.path.join(GOLDEN_DIR, "alt_" + name + ".npz"))
    bases, offsets = batch([c for c in g.contigs() if len(c) >= g.k])  # non-ACGT bytes count as 'A'
    assert np.array_equal(f.lookup(seqio.pack_kmers(bases, offsets, g.k, g.bits)), z["q_codes_ns"])


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_members_form_a_minimal_perfect_hash_and_fallback_matches_streaming(handle, name):
    g, f = handle(name)
    codes = f.lookup(seqio.pack_kmers(g.index_bases, g.index_offsets, g.k, g.bits))
    n = f.get_kmer_count()
    assert len(codes) == n and np.array_equal(np.sort(codes), np.arange(n, dtype=np.uint64))
    # the k-mers of colliding minimizers (fallback PHF), in the layout lphb_colliding_kmers writes
    coll = g.coll_kmers if g.bits == 128 else g.coll_kmers[:, 0]
    bases, offsets = batch(decode(g.coll_kmers, g.k))
    want, _ = f.query_batch(bases, offsets)
    assert len(coll) > 0 and np.array_equal(f.lookup(coll), want)


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
def test_non_members_match_the_oracle(handle, name):
    from oracle import oracle
    g, f = handle(name)
    kmers = random_kmers(np.random.default_rng(31), 3000, g.k, g.bits)
    o = oracle.OracleMphf(g.lph, g.bits)
    try:
        want = np.concatenate([o.query_stateless(c) for c in decode(kmers, g.k)])
    finally:
        o.close()
    assert np.array_equal(f.lookup(kmers), want)


@pytest.mark.parametrize("name", ["k31_m20_u64", "k31_m16_u128", "k63_m24_u128", "k25_m13_u64"])
def test_bits_above_2k_are_ignored(handle, name):
    g, f = handle(name)
    kmers, want = clean_windows(g)
    rng = np.random.default_rng(7)
    words = g.bits // 64
    used = [min(max(2 * g.k - 64 * w, 0), 64) for w in range(words)]  # bits of each word the k-mer uses
    high = np.array([((1 << 64) - 1) ^ ((1 << u) - 1) for u in used], dtype=np.uint64)
    garbage = rng.integers(0, 1 << 63, size=kmers.shape, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    noisy = kmers | (garbage & (high[0] if words == 1 else high))
    assert not np.array_equal(noisy, kmers)
    assert np.array_equal(f.lookup(noisy), want)


def test_shuffled_input_gives_permuted_codes(handle):
    g, f = handle("k63_m24_u128")
    kmers, want = clean_windows(g)
    perm = np.random.default_rng(3).permutation(len(want))
    assert np.array_equal(f.lookup(kmers[perm]), want[perm])


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_chunked_pipeline_and_small_path_agree(handle, name, monkeypatch):
    g, f = handle(name)
    kmers, want = clean_windows(g)
    assert np.array_equal(f.lookup(kmers), want)  # one small block (input and codes < 1 MB)
    monkeypatch.setenv("LPHB_NO_SMALL_PATH", "1")
    assert np.array_equal(f.lookup(kmers), want)  # one chunk on the handle's stream
    for chunk in ("16", "4000", "65536"):
        monkeypatch.setenv("LPHB_CHUNK_BASES", chunk)
        assert np.array_equal(f.lookup(kmers), want), chunk
        per = max(1, int(chunk) // (g.bits // 8))
        assert f.stats().kernel_launches == -(-len(want) // per)


def test_wide_bucket_table_gives_the_same_codes(handle, monkeypatch):
    monkeypatch.setenv("LPHB_FORCE_WIDE_BUCKETS", "1")
    for name in ("k31_m20_u64", "k63_m24_u128", "k40_m17_u128"):
        g, f = handle(name)
        kmers, want = clean_windows(g)
        assert np.array_equal(f.lookup(kmers), want), name


@pytest.mark.parametrize("no_small", [False, True])
def test_batch_sizes(handle, no_small, monkeypatch):
    if no_small:
        monkeypatch.setenv("LPHB_NO_SMALL_PATH", "1")
    g, f = handle("k63_m24_u128")
    kmers, want = clean_windows(g)
    assert len(f.lookup(kmers[:0])) == 0
    for n in (1, 31, 32, 33, 127, 128, 129, 1025):
        assert np.array_equal(f.lookup(kmers[:n]), want[:n]), n
        assert np.array_equal(f.lookup(kmers[-n:]), want[-n:]), n


def test_shape_must_match_the_handle(handle):
    _, f = handle("k63_m24_u128")
    with pytest.raises(ValueError):
        f.lookup(np.zeros(4, dtype=np.uint64))
    _, f64 = handle("k31_m20_u64")
    with pytest.raises(ValueError):
        f64.lookup(np.zeros((4, 2), dtype=np.uint64))


def test_device_form_on_caller_streams(handle):
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda:0")
    g, f = handle("k31_m16_u128")
    kmers, want = clean_windows(g)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_kmers = torch.from_numpy(kmers.view(np.int64).copy()).to(dev)
    d_codes = torch.full((len(want),), -1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    f.lookup_device(d_kmers.data_ptr(), len(want), d_codes.data_ptr(), s1.cuda_stream)
    # a streaming query of the index contigs on another stream right behind it: the handle orders the two
    bases, offsets = g.index_bases, g.index_offsets
    n_idx = int(f.get_kmer_count())
    d_bases = torch.from_numpy(bases.copy()).to(dev)
    d_off = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    q_codes = torch.zeros(n_idx, dtype=torch.int64, device=dev)
    q_off = torch.empty(len(offsets), dtype=torch.int64, device=dev)
    q_status = torch.zeros(4, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    f.lookup_device(d_kmers.data_ptr(), len(want), d_codes.data_ptr(), s1.cuda_stream)
    f.query_device(d_bases.data_ptr(), d_off.data_ptr(), offsets, q_codes.data_ptr(), n_idx, q_off.data_ptr(),
                   q_status.data_ptr(), s2.cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(d_codes.cpu().numpy().view(np.uint64), want)
    got_q = q_codes.cpu().numpy().view(np.uint64)
    assert int(q_status[1]) == 0 and np.array_equal(np.sort(got_q), np.arange(n_idx, dtype=np.uint64))
    assert np.array_equal(got_q, f.lookup(seqio.pack_kmers(bases, offsets, g.k, g.bits)))
    # n == 0 does nothing; a misaligned 128-bit input is refused
    f.lookup_device(0, 0, 0, s1.cuda_stream)
    with pytest.raises(api.LphashError) as e:
        f.lookup_device(d_kmers.data_ptr() + 8, 1, d_codes.data_ptr(), s1.cuda_stream)
    assert e.value.code == api.E_ARG


def test_dirty_flags_and_stats_after_a_lookup(handle):
    torch = pytest.importorskip("torch")
    g, f = handle("k31_m20_u64")
    f.query_batch(g.q_bases, g.q_offsets)
    assert len(f.dirty_flags()) == len(g.q_offsets) - 1
    kmers, want = clean_windows(g)
    f.stats()
    f.lookup(kmers)
    assert len(f.dirty_flags()) == 0
    st = f.stats()
    assert st.kernel_launches == 1 and st.h2d_bytes == 8 * len(want) and st.d2h_bytes == 8 * len(want)
    assert st.dirty_contigs == 0 and st.kernel_ms > 0
    dev = torch.device("cuda:0")
    d_kmers = torch.from_numpy(kmers.view(np.int64)).to(dev)
    d_codes = torch.empty(len(want), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    f.lookup_device(d_kmers.data_ptr(), len(want), d_codes.data_ptr(), torch.cuda.current_stream().cuda_stream)
    st = f.stats()
    assert st.kernel_launches == 1 and st.h2d_bytes == 0 and st.d2h_bytes == 0 and st.kernel_ms > 0
    assert np.array_equal(d_codes.cpu().numpy().view(np.uint64), want)
    assert len(f.dirty_flags()) == 0


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_cpp_mirror_lookup(tmp_path, name):
    g = load_golden(name)
    exe = str(tmp_path / "lookup_check")
    libdir = os.path.join(ROOT, "lphash_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", f"-DLPHASH_B200_KMER_BITS={g.bits}",
                           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "lookup_check.cpp"),
                           "-o", exe, "-L", libdir, "-llphash_b200", f"-Wl,-rpath,{libdir}"])
    kmers, want = clean_windows(g)
    (tmp_path / "kmers.bin").write_bytes(np.uint64(len(want)).tobytes() + kmers.astype("<u8").tobytes())
    r = subprocess.run([exe, g.lph, str(tmp_path / "kmers.bin"), str(tmp_path / "codes.bin")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(np.fromfile(tmp_path / "codes.bin", dtype="<u8"), want)
