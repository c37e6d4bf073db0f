"""Parity of the CUDA path (through the C ABI, lphash_b200/liblphash_b200.so) with the reference:
against the committed golden vectors generated from the unmodified reference, and against the
CPU oracle on seeded inputs.  Bit-exact (integer work, zero tolerance)."""
import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN_NAMES, load_golden
from lphash_b200 import api, synth
from oracle import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handles():
    cache = {}

    def get(name):
        if name not in cache:
            g = load_golden(name)
            cache[name] = api.Mphf.load(g.lph, g.bits)
        return cache[name]

    yield get
    for h in cache.values():
        h.close()


def test_device_present():
    assert api.device_count() >= 1


def test_info_matches_file(golden, handles):
    f = handles(golden.name)
    o = oracle.OracleMphf(golden.lph, golden.bits)
    assert (f.k, f.m, f.kmer_bits) == (golden.k, golden.m, golden.bits)
    assert f.get_kmer_count() == o.info["nkmers"]
    assert f.get_minimizer_L0() == o.info["distinct_minimizers"]
    for a, b in [("n_maximal", "n_maximal"), ("right_coll_sizes_start", "right_coll_sizes_start"),
                 ("none_sizes_start", "none_sizes_start"), ("none_pos_start", "none_pos_start"),
                 ("fallback_keys", "fb_num_keys"), ("file_bytes", "file_bytes")]:
        assert getattr(f.info, a) == o.info[b]


def test_query_batch_matches_reference_golden(golden, handles):
    """Whole query batch: members, non-members, short/empty contigs, lower case, and contigs with
    non-ACGT bytes (reference streaming quirk reproduced exactly)."""
    f = handles(golden.name)
    codes, code_off = f.query_batch(golden.q_bases, golden.q_offsets)
    assert np.array_equal(code_off, golden.q_code_offsets)
    assert np.array_equal(codes, golden.q_codes)
    assert f.stats().dirty_contigs == sum(1 for c in golden.is_clean() if not c)


def test_single_contig_calls_match(golden, handles):
    """operator()(contig, len) one contig at a time, like the reference driver (query.cpp:52)."""
    f = handles(golden.name)
    off = golden.q_code_offsets
    contigs = golden.contigs()
    for i in list(range(0, 12)) + list(range(len(contigs) - 60, len(contigs))):
        want = golden.q_codes[int(off[i]):int(off[i + 1])]
        got = f(contigs[i])
        assert np.array_equal(got, want), i


@pytest.mark.parametrize("generic_below", [None, "0"])      # library default (generic kernel below 256 K bases) / tiled kernel
@pytest.mark.parametrize("small_path", [True, False])        # one pinned block up, one down / the general path
def test_one_record_per_call_paths(golden, handles, generic_below, small_path, monkeypatch):
    """The reference's own loop hands over one record per call (src/query.cpp:48-56): every contig of the query batch
    alone, streaming and non-streaming, through the small-batch path and the general one, on both kernels - clean
    records, non-members, short and empty records, records with non-ACGT bytes (which leave the small path)."""
    if generic_below is None:
        monkeypatch.delenv("LPHB_GENERIC_BELOW", raising=False)
    else:
        monkeypatch.setenv("LPHB_GENERIC_BELOW", generic_below)
    if not small_path:
        monkeypatch.setenv("LPHB_NO_SMALL_PATH", "1")
    f = handles(golden.name)
    off = golden.q_code_offsets
    contigs = golden.contigs()
    clean = golden.is_clean()
    picks = list(range(0, 16)) + list(range(len(contigs) - 70, len(contigs), 2))
    for i in picks:
        want = golden.q_codes[int(off[i]):int(off[i + 1])]
        got = f(contigs[i])
        assert np.array_equal(got, want), i
        if clean[i] and len(contigs[i]) >= golden.k:  # same codes on ACGT-only input
            assert np.array_equal(f(contigs[i], streaming=False), want), i
    # a few records per call, offsets not starting at zero
    raw = golden.q_bases
    qoff = golden.q_offsets
    sub = qoff[3:9]
    codes, coff = f.query_batch(raw, sub)
    assert np.array_equal(codes, golden.q_codes[int(off[3]):int(off[8])])
    assert np.array_equal(coff, off[3:9] - off[3])


def test_clean_batch_has_no_dirty_contigs_and_is_perfect(golden, handles):
    f = handles(golden.name)
    codes, code_off = f.query_batch(golden.index_bases, golden.index_offsets)
    n = f.get_kmer_count()
    assert f.stats().dirty_contigs == 0
    assert len(codes) == n
    assert np.array_equal(np.sort(codes), np.arange(n, dtype=np.uint64))  # minimal perfect


def test_offsets_not_starting_at_zero(golden, handles):
    f = handles(golden.name)
    skip = 5
    codes, code_off = f.query_batch(golden.q_bases, golden.q_offsets[skip:])
    base = int(golden.q_code_offsets[skip])
    assert np.array_equal(codes, golden.q_codes[base:])
    assert np.array_equal(code_off, golden.q_code_offsets[skip:] - np.uint64(base))


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k15_m7_u64"])
def test_random_reads_match_oracle(name, handles):
    g = load_golden(name)
    f = handles(name)
    o = oracle.OracleMphf(g.lph, g.bits)
    genome = g.index_bases[: int(g.index_offsets[10])]
    bases, offsets = synth.reads(3000, genome, read_len=100 + g.k, seed=0xBEEF + g.k)
    want, want_off = o.query_batch(bases, offsets)
    got, got_off = f.query_batch(bases, offsets)
    assert np.array_equal(got_off, want_off)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("chunk", [1, 700, 5000, 1 << 16])
def test_chunk_pipeline_matches_single_batch(golden, handles, chunk, monkeypatch):
    """lphb_query_stream cuts large batches into chunks that flow through two streams (H2D /
    kernels / D2H overlapped); any chunk size must give the single-batch result, with and
    without contigs that take the non-ACGT quirk path."""
    f = handles(golden.name)
    monkeypatch.setenv("LPHB_CHUNK_BASES", str(chunk))
    codes, code_off = f.query_batch(golden.q_bases, golden.q_offsets)
    assert np.array_equal(code_off, golden.q_code_offsets)
    assert np.array_equal(codes, golden.q_codes)
    codes, code_off = f.query_batch(golden.index_bases, golden.index_offsets)
    assert f.stats().dirty_contigs == 0
    n = f.get_kmer_count()
    assert len(codes) == n and np.array_equal(np.sort(codes), np.arange(n, dtype=np.uint64))
    monkeypatch.setenv("LPHB_CHUNK_BASES", "0")  # pipeline off
    ref_codes, ref_off = f.query_batch(golden.index_bases, golden.index_offsets)
    assert np.array_equal(codes, ref_codes) and np.array_equal(code_off, ref_off)


def test_capacity_error(handles):
    g = load_golden("k31_m20_u64")
    f = handles(g.name)
    out = np.empty(10, dtype=np.uint64)
    with pytest.raises(api.LphashError) as e:
        f.query_batch(g.index_bases, g.index_offsets, out=out)
    assert e.value.code == api.E_CAPACITY


def test_device_resident_variant(handles):
    torch = pytest.importorskip("torch")
    g = load_golden("k31_m20_u64")
    f = handles(g.name)
    dev = torch.device("cuda:0")
    d_bases = torch.from_numpy(g.index_bases.copy()).to(dev)
    offs = g.index_offsets.astype(np.int64)
    d_off = torch.from_numpy(offs).to(dev)
    n = len(offs) - 1
    total = int(np.maximum(np.diff(offs) - g.k + 1, 0).sum())
    d_codes = torch.empty(total, dtype=torch.int64, device=dev)
    d_code_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    d_status = torch.zeros(4, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream()
    f.query_device(d_bases.data_ptr(), d_off.data_ptr(), g.index_offsets, d_codes.data_ptr(), total,
                   d_code_off.data_ptr(), d_status.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    status = d_status.cpu().numpy()
    assert status[0] == total and status[1] == 0
    want, want_off = f.query_batch(g.index_bases, g.index_offsets)
    assert np.array_equal(d_codes.cpu().numpy().view(np.uint64), want)
    assert np.array_equal(d_code_off.cpu().numpy().view(np.uint64), want_off)


# ---- build-side scan ---------------------------------------------------------------------------

def test_scan_matches_reference_golden(golden):
    rec, nk, mm = api.scan_superkmers(golden.index_bases, golden.index_offsets, golden.k, golden.m)
    assert nk == int(golden.n_kmers) and mm == int(golden.mm_count)
    assert rec.dtype == golden.rec.dtype
    assert np.array_equal(rec, golden.rec)


def test_scan_mm_count_carries_over(golden):
    """mm_count is in/out: scanning the set in two batches gives the same stream."""
    off = golden.index_offsets
    half = (len(off) - 1) // 2
    r1, k1, mm1 = api.scan_superkmers(golden.index_bases, off[: half + 1], golden.k, golden.m)
    r2, k2, mm2 = api.scan_superkmers(golden.index_bases, off[half:], golden.k, golden.m, mm_count=mm1)
    assert k1 + k2 == int(golden.n_kmers) and mm2 == int(golden.mm_count)
    assert np.array_equal(np.concatenate([r1, r2]), golden.rec)


def test_scan_short_contigs(golden):
    k, m = golden.k, golden.m
    rng = np.random.Generator(np.random.PCG64(7))
    lens = [0, 1, m - 1, m, k - 1, k, k + 1, 3 * k, 0, 5]
    recs = [synth.random_bases(n, rng).tobytes() for n in lens]
    bases = np.frombuffer(b"".join(recs), dtype=np.uint8)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    want, wk, wmm = oracle.scan(bases, offsets, k, m, mode=0)
    got, gk, gmm = api.scan_superkmers(bases, offsets, k, m)
    assert (gk, gmm) == (wk, wmm)
    assert np.array_equal(got, want)


def test_colliding_kmers_match_reference_golden(golden):
    km = api.colliding_kmers(golden.index_bases, golden.index_offsets, golden.k, golden.m,
                             golden.coll_ids, kmer_bits=golden.bits)
    assert km.shape == golden.coll_kmers.shape
    assert np.array_equal(km, golden.coll_kmers)


def test_scan_then_classify_feeds_the_same_keys(golden):
    """The GPU scan's stream, pushed through classify, yields the key stream PTHash consumes."""
    rec, _, _ = api.scan_superkmers(golden.index_bases, golden.index_offsets, golden.k, golden.m)
    trip, ids = oracle.classify(rec)
    assert np.array_equal(trip, golden.triplets)
    assert np.array_equal(ids, golden.coll_ids)


def test_scan_workspace_is_reused_and_released():
    """The scan keeps its device workspace between calls (lphb_scan_release frees it): calls of
    growing, shrinking and different-(k, m) batches must not see each other's leftovers."""
    rng = np.random.Generator(np.random.PCG64(11))
    for k, m, n in [(31, 20, 4000), (31, 20, 90000), (63, 24, 7000), (31, 20, 500), (25, 13, 20000)]:
        lens = rng.integers(k, 4 * k + 200, size=max(1, n // (2 * k + 100)))
        bases = synth.random_bases(int(lens.sum()), rng)
        offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        want, wk, wmm = oracle.scan(bases, offsets, k, m, mode=0)
        got, gk, gmm = api.scan_superkmers(bases, offsets, k, m)
        assert (gk, gmm) == (wk, wmm)
        assert np.array_equal(got, want), (k, m, n)
    assert api.lib().lphb_scan_release(0) == 0
    assert api.lib().lphb_scan_release(0) == 0  # idempotent
    got, gk, gmm = api.scan_superkmers(bases, offsets, k, m)  # allocates again
    assert np.array_equal(got, want)


@pytest.mark.parametrize("name", ["k63_m24_u128", "k47_m20_u128", "k40_m17_u128"])
def test_wide_windows_long_contigs_match_oracle(name, handles):
    """Windows wider than one thread segment (W = 40, 28 on the tiled kernel; W = 24 generic): long
    contigs, so that most tiles lie inside one contig, plus seams every few tiles."""
    g = load_golden(name)
    f = handles(name)
    o = oracle.OracleMphf(g.lph, g.bits)
    rng = np.random.Generator(np.random.PCG64(0xD1CE + g.k))
    genome = g.index_bases[: int(g.index_offsets[len(g.index_offsets) // 2])]
    lens = [5000, 2999, g.k, 12345, g.k + 1, 931, 929, 1857]
    recs = []
    for ln in lens:
        lo = int(rng.integers(0, max(1, len(genome) - ln)))
        s = genome[lo:lo + ln].copy()
        if len(s) < ln:
            s = np.concatenate([s, synth.random_bases(ln - len(s), rng)])
        recs.append(s)
    bases = np.concatenate(recs)
    offsets = np.concatenate([[0], np.cumsum([len(r) for r in recs])]).astype(np.uint64)
    want, want_off = o.query_batch(bases, offsets)
    got, got_off = f.query_batch(bases, offsets)
    assert np.array_equal(got_off, want_off)
    assert np.array_equal(got, want)


# ---- sort by minimizer + classify ---------------------------------------------------------------

def test_classify_matches_reference_golden(golden):
    """GPU scan -> GPU classify == the reference's classify outputs (the key stream PTHash consumes)."""
    rec, _, _ = api.scan_superkmers(golden.index_bases, golden.index_offsets, golden.k, golden.m)
    trip, ids = api.classify(rec)
    assert trip.dtype == golden.triplets.dtype
    assert np.array_equal(trip, golden.triplets)
    assert np.array_equal(ids, golden.coll_ids)


def test_classify_random_records_match_oracle():
    """Any record order; heavy duplication (groups of 1 .. many), extreme key values, empty input."""
    rng = np.random.Generator(np.random.PCG64(99))
    for n, n_keys in [(0, 1), (1, 1), (2, 1), (1000, 40), (50000, 30000), (200000, 199000)]:
        rec = np.zeros(n, dtype=api.RECORD_DTYPE)
        keys = rng.integers(0, 1 << 62, size=max(n_keys, 1), dtype=np.uint64)
        keys[0] = 0
        keys[-1] = np.uint64(0xFFFFFFFFFFFFFFFF)
        rec["itself"] = keys[rng.integers(0, len(keys), size=n)]
        rec["id"] = rng.permutation(n).astype(np.uint64) * np.uint64(3)
        rec["p1"] = rng.integers(0, 40, size=n)
        rec["size"] = rng.integers(1, 41, size=n)
        want_t, want_i = oracle.classify(rec)
        got_t, got_i = api.classify(rec)
        assert np.array_equal(got_t, want_t), n
        assert np.array_equal(got_i, want_i), n


def test_classify_capacity_error():
    rec = np.zeros(10, dtype=api.RECORD_DTYPE)
    rec["itself"] = np.arange(10)
    rec["size"] = 1
    trip = np.empty(3, dtype=api.TRIPLET_DTYPE)
    ids = np.empty(3, dtype=np.uint64)
    nt, ni = C.c_uint64(0), C.c_uint64(0)
    rc = api.lib().lphb_classify(0, rec.ctypes.data, 10, trip.ctypes.data, 3, C.byref(nt), ids.ctypes.data, 3, C.byref(ni))
    assert rc == api.E_CAPACITY and nt.value == 10 and ni.value == 0


def test_scan_classify_fused_matches_reference_golden(golden):
    trip, ids, nk, mm = api.scan_classify(golden.index_bases, golden.index_offsets, golden.k, golden.m)
    assert nk == int(golden.n_kmers) and mm == int(golden.mm_count)
    assert np.array_equal(trip, golden.triplets)
    assert np.array_equal(ids, golden.coll_ids)


# ---- branches the bundled-size fixtures do not reach on their own -------------------------------

def test_forced_wide_bucket_table_matches_golden(golden, monkeypatch):
    """The 64-bit bucket table (taken on its own only by indexes with a base >= 2^30, i.e. BASELINE
    config 3) forced on every golden through the loader's test hook."""
    monkeypatch.setenv("LPHB_FORCE_WIDE_BUCKETS", "1")
    f = api.Mphf.load(golden.lph, golden.bits)
    monkeypatch.delenv("LPHB_FORCE_WIDE_BUCKETS")
    try:
        narrow = api.Mphf.load(golden.lph, golden.bits)
        assert f.info.device_bytes > narrow.info.device_bytes  # 8 instead of 4 bytes per table slot
        narrow.close()
        codes, code_off = f.query_batch(golden.q_bases, golden.q_offsets)
        assert np.array_equal(code_off, golden.q_code_offsets)
        assert np.array_equal(codes, golden.q_codes)
        codes, _ = f.query_batch(golden.index_bases, golden.index_offsets)
        n = f.get_kmer_count()
        assert len(codes) == n and np.array_equal(np.sort(codes), np.arange(n, dtype=np.uint64))
    finally:
        f.close()


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k21_m11_u64", "k25_m13_u64"])
@pytest.mark.parametrize("wide", [False, True])
def test_non_member_flood_hits_every_table_slot(name, wide, monkeypatch):
    """Random (non-member) sequence probes arbitrary PTHash slots, among them the few whose code
    underflows 64 bits for a non-member offset (hval = base - p with base < p, taken mod 2^64 by
    the reference: SURVEY.md E1 vii) - the entries the 32-bit fast emit must hand to the exact path."""
    g = load_golden(name)
    if wide:
        monkeypatch.setenv("LPHB_FORCE_WIDE_BUCKETS", "1")
    f = api.Mphf.load(g.lph, g.bits)
    try:
        o = oracle.OracleMphf(g.lph, g.bits)
        rng = np.random.Generator(np.random.PCG64(0xF100D + g.k))
        n_bases = int(min(6_000_000, max(1_000_000, 12 * f.get_minimizer_L0() * (g.k - g.m + 2) // 2)))
        bases = synth.random_bases(n_bases, rng)
        cuts = np.sort(rng.choice(np.arange(1, n_bases), size=40, replace=False))
        offsets = np.concatenate([[0], cuts, [n_bases]]).astype(np.uint64)
        want, want_off = o.query_batch(bases, offsets)
        got, got_off = f.query_batch(bases, offsets)
        assert np.array_equal(got_off, want_off)
        assert np.array_equal(got, want)
    finally:
        f.close()


def test_small_probe_chunks_variant():
    """Phase D probes the minimizers of a tile in chunks of 256; the `listcap32` build of the library
    (csrc/Makefile: testvariants) cuts them at 32 so that every tile takes several chunks, and sends
    every bucket with a base below 60000 through the exact 64-bit path that otherwise only codes
    outside 32 bits take."""
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    lib = os.path.join(os.path.dirname(here), "lphash_b200", "liblphash_b200_listcap32.so")
    if not os.path.exists(lib):
        pytest.skip("variant library not built (make -C lphash_b200/csrc testvariants)")
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {os.path.dirname(here)!r}); sys.path.insert(0, {here!r})\n"
        "from conftest import load_golden\n"
        "from lphash_b200 import api\n"
        "for name in ['k31_m20_u64', 'k15_m7_u64', 'k63_m24_u128']:\n"
        "    g = load_golden(name)\n"
        "    f = api.Mphf.load(g.lph, g.bits)\n"
        "    codes, off = f.query_batch(g.q_bases, g.q_offsets)\n"
        "    assert np.array_equal(off, g.q_code_offsets) and np.array_equal(codes, g.q_codes), name\n"
        "    codes, _ = f.query_batch(g.index_bases, g.index_offsets)\n"
        "    assert np.array_equal(np.sort(codes), np.arange(f.get_kmer_count(), dtype=np.uint64)), name\n"
        "    f.close()\n"
        "print('ok')\n")
    env = dict(os.environ, LPHASH_B200_LIB=lib)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


# ---- run-length form of the codes (lphb_query_stream_runs) -----------------------------------------

@pytest.mark.parametrize("chunk", [0, 900, 1 << 16])
def test_run_length_form_expands_to_the_same_codes(golden, handles, chunk, monkeypatch):
    """Members, non-members, colliding minimizers, short contigs and the non-ACGT quirk: the run
    records expand to exactly the vector lphb_query_stream returns, for one-shot and chunk-pipelined
    batches; runs never cross a contig."""
    f = handles(golden.name)
    monkeypatch.setenv("LPHB_CHUNK_BASES", str(chunk))
    for bases, offsets, want, want_off in [(golden.q_bases, golden.q_offsets, golden.q_codes, golden.q_code_offsets),
                                           (golden.index_bases, golden.index_offsets, None, None)]:
        if want is None:
            want, want_off = f.query_batch(bases, offsets)
        runs, code_off, n_codes = f.query_batch_runs(bases, offsets)
        assert n_codes == len(want) and np.array_equal(code_off, want_off)
        assert np.array_equal(api.expand_runs(runs, threads=4), want)
        ends = np.cumsum(np.abs(runs["n"].astype(np.int64)))
        assert np.isin(want_off[1:][np.diff(want_off) > 0], ends).all()  # every contig ends a run
    # compactness on the all-member set: about one run per super-k-mer (2 / (k - m + 2) per k-mer), plus
    # single-code runs for the k-mers of colliding minimizers (frequent in these tiny indexes)
    assert len(runs) < 0.8 * n_codes


def test_run_length_form_capacity_and_count_only(handles):
    g = load_golden("k31_m20_u64")
    f = handles(g.name)
    runs, _, n_codes = f.query_batch_runs(g.index_bases, g.index_offsets)
    small = np.empty(5, dtype=api.RUN_DTYPE)
    with pytest.raises(api.LphashError) as e:
        f.query_batch_runs(g.index_bases, g.index_offsets, out=small)
    assert e.value.code == api.E_CAPACITY
    n_runs, total = C.c_uint64(0), C.c_uint64(0)
    off = np.empty(len(g.index_offsets), dtype=np.uint64)
    bases = np.ascontiguousarray(g.index_bases)
    offsets = np.ascontiguousarray(g.index_offsets, dtype=np.uint64)
    rc = api.lib().lphb_query_stream_runs(f._h, bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1, None, 0,
                                          C.byref(n_runs), off.ctypes.data, C.byref(total))
    assert rc == api.E_CAPACITY or rc == 0
    assert n_runs.value == len(runs) and total.value == n_codes


def test_scan_device_resident_matches_reference_golden(golden):
    """lphb_scan_superkmers_device: bases and offsets already in HBM, records left in HBM."""
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda:0")
    d_bases = torch.from_numpy(golden.index_bases.copy()).to(dev)
    d_off = torch.from_numpy(golden.index_offsets.astype(np.int64)).to(dev)
    torch.cuda.synchronize()
    rec, nrec, nk, mm, ms = api.scan_superkmers_device(d_bases.data_ptr(), d_off.data_ptr(), golden.index_offsets,
                                                       golden.k, golden.m)
    assert nk == int(golden.n_kmers) and mm == int(golden.mm_count) and nrec == len(golden.rec)
    assert np.array_equal(rec, golden.rec)
    assert ms > 0


def test_scan_records_cross_tile_boundaries():
    """Long contigs, so that super-k-mers straddle the 992-start tiles of the fused scan kernel and the
    chained scan over many tiles assigns the record indices; plus seams every few tiles."""
    rng = np.random.Generator(np.random.PCG64(0x5CA9))
    for k, m in [(31, 20), (63, 24), (47, 20), (15, 7), (31, 15)]:
        lens = [40000, k, 5000, 992 + k - 1, 993 + k - 1, 991 + k - 1, 2 * 992 + k, 30000, k + 1, 17]
        bases = synth.random_bases(int(sum(lens)), rng)
        offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        want, wk, wmm = oracle.scan(bases, offsets, k, m, mode=0)
        got, gk, gmm = api.scan_superkmers(bases, offsets, k, m, mm_count=12345)
        assert (gk, gmm) == (wk, wmm + 12345)
        want = want.copy()
        want["id"] += np.uint64(12345)
        assert np.array_equal(got, want), (k, m)


ACGT_BYTES = np.zeros(256, dtype=bool)
ACGT_BYTES[list(b"ACGTUacgtu")] = True


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
def test_non_streaming_branch_matches_the_reference(name, handles):
    """hf(contig, len, streaming=false) (include/partitioned_mphf.hpp:185-195): every window of k bytes,
    a non-ACGT byte counting as 'A' (include/mphf_utils.hpp:108) - contig by contig, on the golden query batch
    (N runs, junk bytes, lower case), against that definition evaluated by the CPU oracle (the stateless query of the
    contig with its non-ACGT bytes made 'A'), which on clean contigs must give the reference's own golden codes (the
    two branches of the reference agree there); and against the unmodified reference (oracle/_ref) where it is built."""
    from oracle import ref
    g = load_golden(name)
    f = handles(name)
    o = oracle.OracleMphf(g.lph, g.bits)
    r = ref.RefMphf(g.lph, g.bits) if ref.available(g.bits) else None
    off = g.q_code_offsets
    wants, contigs = [], []
    n_dirty = 0
    for i, (c, clean) in enumerate(zip(g.contigs(), g.is_clean())):
        if len(c) < g.k:  # the reference is undefined below k (length-k+1 underflows)
            continue
        a = np.frombuffer(c, dtype=np.uint8).copy()
        a[~ACGT_BYTES[a]] = ord("A")
        want = o.query_stateless(a.tobytes())
        assert len(want) == len(c) - g.k + 1
        if clean:
            assert np.array_equal(want, g.q_codes[int(off[i]):int(off[i + 1])])
        if r is not None:
            assert np.array_equal(r.query(c, streaming=False), want)
        assert np.array_equal(f(c, streaming=False), want)
        n_dirty += 0 if clean else 1
        wants.append(want)
        contigs.append(c)
    assert n_dirty >= 5
    # batch form: same codes, clean layout
    bases = np.frombuffer(b"".join(contigs), dtype=np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in contigs])]).astype(np.uint64)
    codes, code_off = f.query_batch(bases, offsets, streaming=False)
    assert np.array_equal(np.diff(code_off).astype(np.int64), np.array([len(c) - g.k + 1 for c in contigs]))
    assert np.array_equal(codes, np.concatenate(wants))
    o.close()
    if r is not None:
        r.close()


@pytest.mark.parametrize("name", ["k31_m20_u64", "k31_m16_u128", "k63_m24_u128", "k47_m20_u128", "k15_m7_u64", "k21_m11_u64",
                                  "k25_m13_u64"])
def test_contig_seams_at_every_tile_alignment(name, handles):
    """Contig lengths swept so that seams fall at every offset of a warp tile (992 / 960 / 928 starts) and of a
    16-byte word: members (substrings of the index contigs), non-members, records shorter than k and than m, empty
    records, lower case, a sprinkle of N - streaming query and build scan against the oracle."""
    g = load_golden(name)
    f = handles(name)
    o = oracle.OracleMphf(g.lph, g.bits)
    rng = np.random.default_rng(g.k * 1000 + g.m)
    idx = g.index_bases
    lens = list(range(0, 70)) + list(range(900, 1040, 3)) + list(range(1880, 2010, 7)) + [5000, 2977, 1, 0, 4093]
    pieces = []
    for i, L in enumerate(lens):
        if i % 3 == 0 and L <= len(idx) - 1:
            s0 = int(rng.integers(0, len(idx) - L))
            p = idx[s0:s0 + L].copy()             # crosses index contig seams: members and non-members mixed
        else:
            p = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), L)
        if i % 11 == 5 and L > 3:
            p[rng.integers(0, L, size=2)] = ord("N")
        if i % 7 == 2:
            p = np.frombuffer(p.tobytes().lower(), dtype=np.uint8)
        pieces.append(p)
    bases = np.concatenate(pieces).astype(np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(p) for p in pieces])]).astype(np.uint64)
    want, want_off = o.query_batch(bases, offsets)
    got, got_off = f.query_batch(bases, offsets)
    assert np.array_equal(got_off, want_off)
    assert np.array_equal(got, want)
    rec_w, nk_w, mm_w = oracle.scan(bases, offsets, g.k, g.m, mode=0)
    rec, nk, mm = api.scan_superkmers(bases, offsets, g.k, g.m)
    assert (nk, mm) == (nk_w, mm_w) and np.array_equal(rec, rec_w)


@pytest.mark.parametrize("small_path", [True, False])
def test_dirty_flags_of_the_last_call(golden, handles, small_path, monkeypatch):
    """lphb_mphf_dirty_flags: one byte per contig of the last query call, nonzero where the contig holds a byte outside
    ACGT/acgt/U/u - after a batch, and after single-record calls on the small-batch path"""
    if not small_path:
        monkeypatch.setenv("LPHB_NO_SMALL_PATH", "1")
    f = handles(golden.name)
    clean = np.array(golden.is_clean())
    lens = np.diff(golden.q_offsets).astype(np.int64)
    f.query_batch(golden.q_bases, golden.q_offsets)
    flags = f.dirty_flags()
    assert len(flags) == len(clean)
    # a contig too short for a k-mer is never looked at by the query kernels: its flag is unspecified
    look = lens >= golden.k
    assert np.array_equal(flags[look] != 0, ~clean[look])
    contigs = golden.contigs()
    for i in [j for j in range(len(contigs)) if look[j]][:6] + [j for j in range(len(contigs)) if look[j] and not clean[j]][:3]:
        f(contigs[i])
        fl = f.dirty_flags()
        assert len(fl) == 1 and bool(fl[0]) == (not clean[i]), i


def test_device_resident_calls_on_several_streams_share_one_handle():
    """lphb_query_stream_device takes the caller's stream, the handle has one device workspace: back-to-back calls on
    DIFFERENT streams (no host synchronisation in between) must not overlap in it - the library orders every call
    behind the previous call's kernels - and each must deliver its own batch's codes."""
    torch = pytest.importorskip("torch")
    g = load_golden("k31_m20_u64")
    f = api.Mphf.load(g.lph, g.bits)
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(3)
    streams = [torch.cuda.Stream(device=dev) for _ in range(4)]
    batches = []
    genome = g.index_bases[: int(g.index_offsets[12])]
    for i in range(12):  # batches of different sizes: different tile counts, different workspace footprints
        bases, offsets = synth.reads(int(rng.integers(200, 6000)), genome, read_len=int(rng.integers(g.k, 400)), seed=100 + i)
        want, want_off = f.query_batch(bases, offsets)
        n = len(offsets) - 1
        batches.append(dict(offsets=offsets, want=want,
                            d_bases=torch.from_numpy(bases.copy()).to(dev),
                            d_off=torch.from_numpy(offsets.astype(np.int64)).to(dev),
                            d_codes=torch.zeros(len(want) + 1, dtype=torch.int64, device=dev),
                            d_code_off=torch.empty(n + 1, dtype=torch.int64, device=dev),
                            d_status=torch.zeros(4, dtype=torch.int64, device=dev)))
    torch.cuda.synchronize()
    for rep in range(3):
        for i, b in enumerate(batches):
            s = streams[(i + rep) % len(streams)]
            f.query_device(b["d_bases"].data_ptr(), b["d_off"].data_ptr(), b["offsets"], b["d_codes"].data_ptr(), len(b["want"]),
                           b["d_code_off"].data_ptr(), b["d_status"].data_ptr(), s.cuda_stream)
        torch.cuda.synchronize()
        for i, b in enumerate(batches):
            st = b["d_status"].cpu().numpy()
            assert st[0] == len(b["want"]) and st[1] == 0, (rep, i, st)
            assert np.array_equal(b["d_codes"].cpu().numpy()[: len(b["want"])].view(np.uint64), b["want"]), (rep, i)
            b["d_codes"].zero_()
    f.close()
