"""Every query and build entry point at every (k, m) of the grid (tests/test_kmgrid_cpu.py: all instantiations of the
tiled kernel, with 64- and 128-bit k-mers, and the edges of the domain the generic kernels serve), on indexes built in
the test with no GPU, bit-exact against the CPU oracle.

Per grid entry the inputs are the index contigs, reads with substitutions, a flood of random non-members, mixed
contigs (members, lower case, N runs, single junk bytes, homopolymers and short-period repeats, records shorter than
m and than k, empty ones) and contig lengths swept across the tile seams of the entry's instantiation and across
16-byte words."""
import numpy as np
import pytest

from lphash_b200 import api, seqio, synth
from oracle import oracle, phf
from test_kmgrid_cpu import (GRID, K_EQ_M, MM_SEED, TILED, cpu_lph, grid_contigs, grid_id, mixed_contigs, sanitize,
                             tile_starts, write_image)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
GENERIC_ALWAYS = str(1 << 62)  # LPHB_GENERIC_BELOW above every batch: the generic (one thread per k-mer) kernel


def concat(contigs):
    bases = np.frombuffer(b"".join(contigs), dtype=np.uint8).copy()
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in contigs])]).astype(np.uint64)
    return bases, offsets


def contigs_of(bases, offsets):
    raw = bases.tobytes()
    return [raw[int(offsets[i]):int(offsets[i + 1])] for i in range(len(offsets) - 1)]


def seam_contigs(bases, k, m, seed):
    """contig lengths around 1, 2 and 3 tiles of the entry's instantiation plus k-1 bases of overlap, lengths
    across a 16-byte word from k-1 up, and one contig of 300 tiles; the sequence is the index's, repeated"""
    tile = tile_starts(k, m)
    rng = np.random.default_rng([k, m, seed, 2])
    src = np.tile(bases, 300 * tile // len(bases) + 2).tobytes()
    lens = [j * tile + k - 1 + d for j in (1, 2, 3) for d in range(-2, 3)] + list(range(k - 1, k + 34))
    lens = [lens[i] for i in rng.permutation(len(lens))] + [300 * tile + k - 1]
    out = []
    for ln in lens:
        a = int(rng.integers(0, len(src) - ln))
        out.append(src[a:a + ln])
    return out


def flood_contigs(k, m, n=300):
    """uniform random contigs (non-members) of 0 to 600 bases"""
    rng = np.random.default_rng([k, m, 3])
    return [synth.random_bases(int(rng.integers(0, 600)), rng).tobytes() for _ in range(n)]


class Entry:
    """one grid entry: the index contigs, its CPU-built image and the query batches"""

    def __init__(self, e, path, bases, offsets):
        self.k, self.m, self.bits = e
        self.path, self.bases, self.offsets = path, bases, offsets
        reads = synth.reads(400, bases, read_len=150, member_frac=0.7, sub_rate=0.01, seed=self.k * 64 + self.m)
        self.batches = {
            "index": (bases, offsets),
            "reads": reads,
            "mixed": concat(mixed_contigs(bases, offsets, self.k, self.m, seed=1)),
            "seams": concat(seam_contigs(bases, self.k, self.m, seed=1)),
            "flood": concat(flood_contigs(self.k, self.m)),
        }

    def clean_batches(self):
        return ["index", "reads", "seams", "flood"]

    def oracle(self):
        return oracle.OracleMphf(self.path, self.bits)

    def load(self):
        return api.Mphf.load(self.path, self.bits)


@pytest.fixture(scope="module")
def grid(tmp_path_factory):
    d = tmp_path_factory.mktemp("kmgrid")
    cache = {}

    def get(e):
        if e not in cache:
            k, m, bits = e
            bases, offsets = grid_contigs(k, m)
            path = write_image(str(d / f"{grid_id(e)}.lph"), cpu_lph(bases, offsets, k, m, bits))
            cache[e] = Entry(e, path, bases, offsets)
        return cache[e]

    return get


@pytest.fixture
def opened():
    """handles (GPU and oracle) closed after the test"""
    hs = []

    def add(h):
        hs.append(h)
        return h

    yield add
    for h in hs:
        h.close()


def check_streaming(f, o, g, names):
    for name in names:
        bases, offsets = g.batches[name]
        want, want_off = o.query_batch(bases, offsets)
        codes, code_off = f.query_batch(bases, offsets)
        assert np.array_equal(code_off, want_off), name
        assert np.array_equal(codes, want), name
        if name == "index":
            assert np.array_equal(np.sort(codes), np.arange(o.info["nkmers"], dtype=np.uint64))


def stateless_oracle(o, bases, offsets):
    """the non-streaming branch: the stateless definition over the contig with every non-ACGT byte as 'A'"""
    want = [o.query_stateless(sanitize(c)) for c in contigs_of(bases, offsets)]
    return np.concatenate(want + [np.zeros(0, np.uint64)]).astype(np.uint64)


def device_batch(bases, offsets, shift):
    """bases on the device `shift` bytes into their allocation (with N padding on both sides) and the offsets"""
    raw = np.concatenate([np.full(shift, ord("N"), np.uint8), bases, np.full(7, ord("N"), np.uint8)])
    t = torch.from_numpy(raw).to(DEV)
    return t, t.data_ptr() + shift, torch.from_numpy(offsets.astype(np.int64)).to(DEV)


def host(t):
    return t.cpu().numpy().view(np.uint64)


# ---- streaming: tiled and generic kernels ---------------------------------------------------------------------

@pytest.mark.parametrize("kernel", ["tiled", "generic"])
@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_streaming_query_matches_the_oracle(grid, opened, monkeypatch, e, kernel):
    """lphb_query_stream: codes and code offsets of every batch; a permutation of [0, n) on the index contigs.
    `tiled` runs the tiled kernel where (k, m) has an instantiation (the generic one elsewhere), `generic` the
    generic kernel for the clean pass (the repair of contigs with non-ACGT bytes keeps the tiled kernel)."""
    if kernel == "generic":
        monkeypatch.setenv("LPHB_GENERIC_BELOW", GENERIC_ALWAYS)
    else:
        monkeypatch.setenv("LPHB_GENERIC_BELOW", "0")
    g = grid(e)
    f, o = opened(g.load()), opened(g.oracle())
    check_streaming(f, o, g, list(g.batches))


@pytest.mark.parametrize("e", [x for x in GRID if x[:2] in TILED], ids=grid_id)
def test_streaming_query_with_wide_bucket_words(grid, opened, monkeypatch, e):
    monkeypatch.setenv("LPHB_FORCE_WIDE_BUCKETS", "1")
    g = grid(e)
    f, o = opened(g.load()), opened(g.oracle())
    check_streaming(f, o, g, ["index", "mixed", "seams"])


# ---- non-streaming, device forms, run-length form -------------------------------------------------------------

@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_nonstreaming_host_and_device_match_the_stateless_oracle(grid, opened, e):
    g = grid(e)
    f, o = opened(g.load()), opened(g.oracle())
    for name in ("mixed", "reads", "seams", "flood"):
        bases, offsets = g.batches[name]
        want = stateless_oracle(o, bases, offsets)
        codes, code_off = f.query_batch(bases, offsets, streaming=False)
        assert np.array_equal(codes, want), name
        assert int(code_off[-1]) == len(want)
        t, ptr, d_off = device_batch(bases, offsets, shift=3)
        d_codes = torch.zeros(max(len(want), 1), dtype=torch.int64, device=DEV)
        d_code_off = torch.zeros(len(offsets), dtype=torch.int64, device=DEV)
        d_status = torch.zeros(4, dtype=torch.int64, device=DEV)
        f.query_device_nonstreaming(ptr, d_off.data_ptr(), offsets, d_codes.data_ptr(), len(want),
                                    d_code_off.data_ptr(), d_status.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(host(d_codes)[:len(want)], want), name
        assert np.array_equal(host(d_code_off), code_off), name


@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_device_forms_match_the_host_form(grid, opened, e):
    """lphb_query_stream_exact_device on every batch, lphb_query_stream_device on the clean ones"""
    g = grid(e)
    f = opened(g.load())
    for name, (bases, offsets) in g.batches.items():
        want, want_off = f.query_batch(bases, offsets)
        t, ptr, d_off = device_batch(bases, offsets, shift=5)
        cap = int(np.maximum(np.diff(offsets.astype(np.int64)) - g.m + 1, 0).sum())
        d_codes = torch.zeros(max(cap, 1), dtype=torch.int64, device=DEV)
        d_code_off = torch.zeros(len(offsets), dtype=torch.int64, device=DEV)
        torch.cuda.synchronize()
        n = f.query_device_exact(ptr, d_off.data_ptr(), offsets, d_codes.data_ptr(), cap, d_code_off.data_ptr())
        assert n == len(want) and np.array_equal(host(d_codes)[:n], want), name
        assert np.array_equal(host(d_code_off), want_off), name
        if name in g.clean_batches():
            d_status = torch.zeros(4, dtype=torch.int64, device=DEV)
            f.query_device(ptr, d_off.data_ptr(), offsets, d_codes.data_ptr(), len(want), d_code_off.data_ptr(),
                           d_status.data_ptr())
            torch.cuda.synchronize()
            assert np.array_equal(host(d_codes)[:len(want)], want), name
            assert np.array_equal(host(d_code_off), want_off), name


@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_run_length_form_expands_to_the_codes(grid, opened, e):
    g = grid(e)
    f = opened(g.load())
    for name in ("mixed", "seams"):
        bases, offsets = g.batches[name]
        want, want_off = f.query_batch(bases, offsets)
        runs, code_off, total = f.query_batch_runs(bases, offsets)
        assert total == len(want) and np.array_equal(code_off, want_off), name
        assert np.array_equal(api.expand_runs(runs), want), name


# ---- lookup of packed k-mers --------------------------------------------------------------------------------

def with_junk_above_2k(kmers, k, bits, rng):
    """random bits at every position >= 2k of the k-mer words"""
    words = bits // 64
    x = np.array(kmers, dtype=np.uint64).reshape(len(kmers), words)
    junk = rng.integers(0, 2**63, size=x.shape, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    for w in range(words):
        used = min(max(2 * k - 64 * w, 0), 64)
        if used < 64:
            x[:, w] |= junk[:, w] & ~np.uint64((1 << used) - 1)
    return x[:, 0].copy() if words == 1 else x


@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_lookup_matches_the_nonstreaming_codes(grid, opened, e):
    g = grid(e)
    f = opened(g.load())
    rng = np.random.default_rng(g.k * 64 + g.m)
    for name in ("index", "mixed", "reads", "flood"):
        bases, offsets = g.batches[name]
        want, _ = f.query_batch(bases, offsets, streaming=False)
        kmers = seqio.pack_kmers(bases, offsets, g.k, g.bits)
        assert len(kmers) == len(want)
        assert np.array_equal(f.lookup(kmers), want), name
        junk = with_junk_above_2k(kmers, g.k, g.bits, rng)
        assert np.array_equal(f.lookup(junk), want), name
        d_kmers = torch.from_numpy(np.ascontiguousarray(junk).view(np.int64)).to(DEV)
        d_codes = torch.zeros(max(len(want), 1), dtype=torch.int64, device=DEV)
        f.lookup_device(d_kmers.data_ptr(), len(want), d_codes.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(host(d_codes)[:len(want)], want), name


# ---- build side -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_build_side_matches_the_oracle_and_rebuilds_the_image(grid, e):
    """scan (the tiled kernel's scan form where (k, m) has one, the generic passes elsewhere), scan + classify,
    the colliding k-mers, and the whole GPU build (oracle/phf.build_lph) equal to the CPU-built image byte for byte"""
    g = grid(e)
    k, m, bits = e
    for name in ("index", "mixed"):
        bases, offsets = g.batches[name]
        want, wk, wmm = oracle.scan(bases, offsets, k, m, seed=MM_SEED, mode=0, mm_count=5)
        got, gk, gmm = api.scan_superkmers(bases, offsets, k, m, seed=MM_SEED, mm_count=5)
        assert (gk, gmm) == (wk, wmm) and np.array_equal(got, want), name
        want0, _, _ = oracle.scan(bases, offsets, k, m, seed=MM_SEED, mode=0)
        trip_w, ids_w = oracle.classify(want0)
        trip, ids, nk, _ = api.scan_classify(bases, offsets, k, m, seed=MM_SEED)
        assert nk == wk and np.array_equal(trip, trip_w) and np.array_equal(ids, ids_w), name
        km_w = oracle.colliding_kmers(bases, offsets, k, m, ids_w, seed=MM_SEED, kmer_bits=bits)
        km = api.colliding_kmers(bases, offsets, k, m, ids, seed=MM_SEED, kmer_bits=bits)
        assert np.array_equal(km, km_w), name
    image = open(g.path, "rb").read()
    assert phf.build_lph(g.bases, g.offsets, k, m, kmer_bits=bits, mm_seed=MM_SEED) == image


@pytest.mark.parametrize("k,m", K_EQ_M)
def test_scan_at_k_equal_m_matches_the_oracle(k, m):
    """W = 1: every k-mer is its own minimizer (no index exists there, the scan is still defined)"""
    bases, offsets = concat(mixed_contigs(*grid_contigs(k, m, 3000), k, m, seed=2))
    want, wk, wmm = oracle.scan(bases, offsets, k, m, seed=MM_SEED, mode=0, mm_count=5)
    got, gk, gmm = api.scan_superkmers(bases, offsets, k, m, seed=MM_SEED, mm_count=5)
    assert (gk, gmm) == (wk, wmm) and np.array_equal(got, want)
    trip_w, ids_w = oracle.classify(oracle.scan(bases, offsets, k, m, seed=MM_SEED, mode=0)[0])
    trip, ids, _, _ = api.scan_classify(bases, offsets, k, m, seed=MM_SEED)
    assert np.array_equal(trip, trip_w) and np.array_equal(ids, ids_w)
