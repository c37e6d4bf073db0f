"""The (k, m) grid: every pair the tiled query kernel is instantiated for and the edges of the (k, m) domain the
generic kernels serve, each on an index built here with no GPU and no reference build-p.

The committed goldens pin eight (k, m) pairs only; the kernels are specialised by k, m and the k-mer width in many
more places (query_tiled.cu pick_cfg, the generic paths at 2k = 64, m-mers across the 64-bit word of a 128-bit
k-mer, windows of 2 to 63 m-mers).  The helpers below make, for any (k, m), a set of contigs with distinct k-mers and
some colliding minimizers (grid_contigs) and the `.lph` image of it (cpu_lph): the CPU oracle's scan, classify and
colliding k-mers, oracle/phf.py's deterministic PHF search, oracle/invindex.py's Part 3 and the host-only
lphb_lph_assemble.  The CPU oracle then answers for any (k, m); tests/test_gpu_kmgrid.py holds every GPU entry point
to it.  Here: the generator and the image are sound, and where the reference build exists (oracle/_ref) the oracle
gives the reference's own answers on the same image."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from lphash_b200 import seqio
from oracle import invindex, oracle, phf, ref

MM_SEED = 42  # the minimizer seed of the reference's build (constants::seed)
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)

# Every (k, m) of pick_cfg in lphash_b200/csrc/query_tiled.cu: 64-bit k-mers where k <= 31, 128-bit always
TILED = [(31, 20), (31, 16), (31, 15), (31, 17), (31, 18), (31, 19), (31, 21), (21, 11), (15, 7), (63, 24), (47, 20)]
# Edges of the domain the generic kernels cover (1 <= m <= 31, m < k <= 31 for 64-bit k-mers, <= 63 for 128-bit):
# m = 31 across the word boundary, m = 1 (W = 63), the first 128-bit k, W = 2 and 3, a window between 50 and 62,
# and a 128-bit k-mer with k <= 31 (fallback hashing with hi = 0)
GENERIC = [(63, 31, 128), (63, 1, 128), (32, 7, 128), (33, 16, 128), (62, 31, 128), (31, 30, 64), (31, 29, 64),
           (25, 13, 128), (11, 5, 64), (63, 10, 128)]
GRID = [(k, m, bits) for k, m in TILED for bits in ((64, 128) if k <= 31 else (128,))] + GENERIC
# k = m: every k-mer is its own minimizer, so no minimizer collides and no index can be built (the fallback PHF
# refuses an empty key set); only the build-side scan is defined
K_EQ_M = [(31, 31), (7, 7)]
N_KMERS = 20_000


def grid_id(e):
    k, m, bits = e
    return f"k{k}_m{m}_u{bits}"


def tile_starts(k, m):
    """k-mer starts per warp tile of the tiled kernel for window W (query_tiled.cu Cfg::Tile): 992 / 960 / 928"""
    w = k - m + 1
    e = max(1, (16 - 1 + w - 1) // 16)
    return 2 * (32 - e) * 16


def _kmer_rows(bases, offsets, k):
    """every window of every contig as one 16-byte value (for uniqueness over any k <= 63)"""
    km = np.ascontiguousarray(seqio.pack_kmers(bases, offsets, k, 128))
    return km.view(np.dtype((np.void, 16))).ravel()


def _concat(pieces):
    bases = np.concatenate(pieces).astype(np.uint8) if pieces else np.zeros(0, np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(p) for p in pieces])]).astype(np.uint64)
    return bases, offsets


def _mmer_value(s):
    v = 0
    for ch in s.tolist():
        v = (v << 2) | int(np.searchsorted(ACGT, ch))
    return v


def grid_contigs(k, m, n_kmers=N_KMERS, seed=0):
    """Contigs for an index at (k, m): about n_kmers distinct k-mers (random pieces of a random genome) and
    min(64, 4^(W-1)) planted copies of one m-base core, W = k - m + 1.

    synth.unitigs cannot serve small windows: its 64 copies of one (m+4)-base core are told apart by 3 tag bases on
    each side, so a k-mer that contains the core and sees fewer than 3 tag bases occurs in several copies.  Here copy
    i carries the same W-1 base tag t_i (i in base 4) on both sides of the core: a k-mer holding the whole core at
    offset j reads t_i[-j:] + core + t_i[:W-1-j], a rotation of t_i around the core, so distinct tags give distinct
    k-mers at every offset.  The core is the m-mer of lowest hash among 512 random ones, so that it is the minimizer
    of most k-mers around it and the copies make it collide.  Windows whose k-mer occurs earlier (random genomes repeat
    k-mers at small k) are dropped by cutting their contig.  Returns (bases, offsets)."""
    rng = np.random.default_rng([k, m, seed])
    w = k - m + 1
    cands = ACGT[rng.integers(0, 4, size=(512, m))]
    hashes = phf.murmur64(np.array([_mmer_value(c) for c in cands], dtype=np.uint64), MM_SEED)
    core = cands[int(np.argmin(hashes))]
    pieces = []
    for i in range(min(64, 4 ** (w - 1))):
        tag = ACGT[[(i >> (2 * d)) & 3 for d in range(w - 1)]]
        left, right = ACGT[rng.integers(0, 4, k + 9)], ACGT[rng.integers(0, 4, k + 9)]
        pieces.append(np.concatenate([left, tag, core, tag, right]))
    total = 0
    while total < n_kmers:  # genome pieces: mostly long, some barely one k-mer long
        ln = k + int(rng.integers(0, 40)) if rng.random() < 0.2 else int(rng.integers(200, 3000))
        pieces.append(ACGT[rng.integers(0, 4, ln)])
        total += ln - k + 1
    order = rng.permutation(len(pieces))
    pieces = [pieces[i] for i in order]
    # keep the first occurrence of every k-mer: cut each piece into runs of windows seen for the first time
    bases, offsets = _concat(pieces)
    rows = _kmer_rows(bases, offsets, k)
    first = np.zeros(len(rows), dtype=bool)
    first[np.unique(rows, return_index=True)[1]] = True
    out, at = [], 0
    for p in pieces:
        good = first[at:at + len(p) - k + 1]
        at += len(p) - k + 1
        edges = np.flatnonzero(np.diff(np.concatenate([[0], good.astype(np.int8), [0]])))
        for a, b in zip(edges[::2], edges[1::2]):  # windows a .. b-1
            out.append(p[a:b + k - 1])
    return _concat(out)


def cpu_lph(bases, offsets, k, m, bits):
    """The `.lph` image of the contigs with no GPU: build-p with c = 3.0, alpha = 0.94 (oracle/phf.build_lph's
    recipe, every part from the CPU restatement).  Raises when no minimizer collides: the reference's build needs a
    non-empty fallback key set."""
    from lphash_b200 import api  # host-only entry points (lphb_lph_assemble)

    rec, nkmers, _ = oracle.scan(bases, offsets, k, m, seed=MM_SEED, mode=0)
    trip, ids = oracle.classify(rec)
    kmers = oracle.colliding_kmers(bases, offsets, k, m, ids, seed=MM_SEED, kmer_bits=bits)
    if len(kmers) == 0:
        raise ValueError(f"k={k} m={m}: no colliding minimizer, the fallback function would have no keys")
    mo = phf.single_phf(phf.murmur64(trip["itself"], phf.PTHASH_SEED))
    orders = oracle.phf_positions(mo, trip["itself"])
    counters, body = invindex.build_inverted_index(trip, orders, k, m)
    values = np.cumsum(invindex.value_lists(trip, orders, k, m))
    universe = int(values[-1]) if len(values) else 0
    ef_bytes = len(invindex.ef_sequence_image(values.tolist(), universe))
    info = api.InvertedIndex(*counters, int((trip["size"] == 0).sum()), universe, len(body) - ef_bytes, ef_bytes, 0.0)
    fh = phf.murmur64(kmers[:, 0], phf.PTHASH_SEED)
    if bits == 128:  # constants.hpp fallback_hasher: murmur(lo, seed) ^ murmur(hi, ~seed)
        fh ^= phf.murmur64(kmers[:, 1], ~phf.PTHASH_SEED & (2**64 - 1))
    fb = phf.single_phf(fh)
    return api.lph_assemble(k, m, MM_SEED, nkmers, len(trip), info, mo, body, fb)


def write_image(path, image):
    with open(path, "wb") as f:
        f.write(image)
    return path


def mixed_contigs(bases, offsets, k, m, seed):
    """a few hundred query contigs: pieces of the index (members, some mutated, some lower case, some with N runs or
    single junk bytes), random non-members, homopolymers and short-period repeats, and records shorter than m, than
    k, and empty"""
    rng = np.random.default_rng([k, m, seed, 1])
    raw = bases.tobytes()
    n = len(offsets) - 1
    out = []
    for _ in range(150):
        c = int(rng.integers(0, n))
        s, e = int(offsets[c]), int(offsets[c + 1])
        a = int(rng.integers(s, e))
        piece = bytearray(raw[a:min(e, a + int(rng.integers(1, 400)))])
        kind = rng.random()
        if kind < 0.2 and piece:
            i = int(rng.integers(0, len(piece)))
            piece[i] = b"ACGT"[(b"ACGT".index(piece[i]) + int(rng.integers(1, 4))) % 4]
        elif kind < 0.35:
            piece = bytearray(piece.lower())
        elif kind < 0.5 and piece:
            i = int(rng.integers(0, len(piece)))
            piece[i:i] = b"N" * int(rng.integers(1, k + 3))
        elif kind < 0.6 and piece:
            piece[int(rng.integers(0, len(piece)))] = bytes([int(rng.choice(list(b"NRn-*.\x00 ")))])[0]
        out.append(bytes(piece))
    for _ in range(60):
        out.append(ACGT[rng.integers(0, 4, int(rng.integers(0, 300)))].tobytes())
    for unit in (b"A", b"C", b"G", b"T", b"AC", b"GT", b"ACG", b"AAT", b"ACGT", b"AACCT", b"ACGTTG", b"AAAAAAAC"):
        for ln in (k - 1, k, k + 1, 3 * k + 5, 400):
            out.append((unit * ln)[:ln])
        out.append((unit * 200)[:200].lower())
    member = raw[int(offsets[0]):int(offsets[0]) + k]
    out += [b"", b"", member[:m - 1], member[:m], member[:k - 1], member[:k - 1].lower(), b"N" * (k - 1)]
    order = rng.permutation(len(out))
    return [out[i] for i in order]


def sanitize(contig):
    """what the non-streaming branch reads: every byte outside ACGTUacgtu counts as 'A'"""
    a = np.frombuffer(contig, dtype=np.uint8).copy()
    ok = np.isin(a, np.frombuffer(b"ACGTUacgtu", dtype=np.uint8))
    a[~ok] = ord("A")
    return a.tobytes()


@pytest.fixture(scope="module")
def built(tmp_path_factory):
    """(bases, offsets, path of the CPU-built image) per grid entry, built once"""
    d = tmp_path_factory.mktemp("kmgrid_cpu")
    cache = {}

    def get(e):
        if e not in cache:
            k, m, bits = e
            bases, offsets = grid_contigs(k, m)
            cache[e] = bases, offsets, write_image(str(d / f"{grid_id(e)}.lph"), cpu_lph(bases, offsets, k, m, bits))
        return cache[e]

    return get


def test_grid_holds_every_tiled_instantiation():
    """an instantiation added to pick_cfg later cannot go untested"""
    src = open(os.path.join(ROOT, "lphash_b200", "csrc", "query_tiled.cu")).read()
    body = src[src.index("bool pick_cfg("):]
    body = body[:body.index("#undef LPHB_CFG")]
    pairs = {(int(a), int(b)) for a, b in re.findall(r"LPHB_CFG\((\d+),\s*(\d+)\)", body)}
    assert len(pairs) >= 11
    for k, m in pairs:
        assert (k, m, 128) in GRID
        assert k > 31 or (k, m, 64) in GRID


@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_index_is_a_minimal_perfect_hash_of_distinct_kmers(built, e):
    k, m, bits = e
    bases, offsets, path = built(e)
    rows = _kmer_rows(bases, offsets, k)
    assert len(np.unique(rows)) == len(rows) >= N_KMERS // 2
    o = oracle.OracleMphf(path, bits)
    try:
        assert (o.k, o.m, o.info["nkmers"]) == (k, m, len(rows))
        assert o.info["fb_num_keys"] > 0
        codes, _ = o.query_batch(bases, offsets)
    finally:
        o.close()
    assert np.array_equal(np.sort(codes), np.arange(len(rows), dtype=np.uint64))


def test_k_equal_m_has_no_index():
    bases, offsets = grid_contigs(31, 31, 2000)
    with pytest.raises(ValueError, match="no colliding minimizer"):
        cpu_lph(bases, offsets, 31, 31, 64)


@pytest.mark.parametrize("k,m", K_EQ_M)
def test_k_equal_m_scan_and_classify_match_the_reference(k, m):
    if not ref.available(64):
        pytest.skip("the reference build (oracle/_ref) is not present")
    bases, offsets = grid_contigs(k, m, 3000)
    rec, nk, mm = oracle.scan(bases, offsets, k, m, seed=MM_SEED, mode=0)
    wrec, wnk, wmm = ref.scan(bases, offsets, k, m, seed=MM_SEED)
    assert (nk, mm) == (wnk, wmm) and np.array_equal(rec, wrec)
    trip, ids = oracle.classify(rec)
    wtrip, wids = ref.classify(bases, offsets, k, m, seed=MM_SEED)
    assert np.array_equal(trip, wtrip) and np.array_equal(ids, wids)


@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_oracle_gives_the_reference_codes_on_the_built_index(built, e):
    """at (k, m) the goldens never pinned: the oracle's streaming and non-streaming codes on mixed contigs are the
    reference's own on the same image"""
    k, m, bits = e
    if not ref.available(bits):
        pytest.skip("the reference build (oracle/_ref) is not present")
    bases, offsets, path = built(e)
    contigs = mixed_contigs(bases, offsets, k, m, seed=3)
    o, r = oracle.OracleMphf(path, bits), ref.RefMphf(path, bits)
    try:
        for c in contigs:
            assert np.array_equal(o.query(c), r.query(c, streaming=True)), c
            clean = c if len(c) >= k else b""
            assert np.array_equal(o.query_stateless(sanitize(clean)), r.query(clean, streaming=False)), c
    finally:
        o.close()
        r.close()

