"""The geometry of the batches tests/test_gpu_repair_geometry.py sends through the device repair of contigs with
non-ACGT bytes (quirk_kernels.cu), checked with no GPU.

The repair's kernels branch on sizes: chunks of kRepairChunk bytes, 32-chunk steps of next_some / prev_some, a
shared table of kTab contigs per kEmitStep output positions in emit_clean, grid-stride loops whose grids are fixed
multiples of the SM count, and a second round per block in the block scans past kRepairScanBlocks * 256 items.
The generators below build batches that cross each of these at its real size; here, for every batch, what each
kernel will see is computed on the host from its bytes, its offsets and the oracle's final code offsets, and the
batch is held to the branch it was made for.  The constants come from the sources, so that a change there fails
here instead of leaving the GPU tests short of their thresholds."""
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT, load_golden
from oracle import oracle

CSRC = os.path.join(ROOT, "lphash_b200", "csrc")


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _const(src, name):
    found = re.findall(r"\b" + name + r"\s*=\s*(\d+)\s*[;,]", src)
    assert len(found) == 1, name
    return int(found[0])


_QK, _QC = _src("query_kernels.cuh"), _src("quirk_kernels.cu")
C = _const(_QK, "kRepairChunk")                  # bytes per chunk of a dirty contig
SCAN_BLOCKS = _const(_QK, "kRepairScanBlocks")   # blocks of the repair's scans (256 threads)
EMIT_STEP = _const(_QC, "kEmitStep")             # output positions per block step of emit_clean
TAB = _const(_QC, "kTab")                        # contigs emit_clean's shared table holds
LOOK = _const(_QC, "kRepLook")                   # bytes before a chunk that its windows reach
THREADS = _const(_QC, "kRepThreads")             # threads of the chunk kernels (k_rep_prep: save_tail)
SMS = 148
G_CHUNKS = SMS * 8    # grid of the chunk kernels (k_rep_prep, k_rep_episodes; save_tail's grid-stride loops)
G_EMIT = SMS * 16     # most blocks emit_clean gets

# where each grid-stride loop or block scan takes its second round
EMIT_WRAP = G_EMIT * EMIT_STEP                # codes after the first dirty contig (in place)
TAIL_CODES_WRAP = G_CHUNKS * THREADS * 4 * 2  # clean codes saved from the first dirty contig on (16-byte vectors)
TAIL_OFF_WRAP = G_CHUNKS * THREADS            # contigs from the first dirty one on (tail_off, i <= fd_rev)
SCAN_WRAP = SCAN_BLOCKS * 256                 # items of a scan (contigs from the first dirty one on, dirty chunks)

ACGT_OK = np.zeros(256, dtype=bool)
ACGT_OK[np.frombuffer(b"ACGTUacgtu", dtype=np.uint8)] = True
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
JUNK = [b"N", b"n", b"X", b"-", b".", b"\x00", b"\xff"]  # the junk bytes the existing dirty patterns use
SCALE_NAMES = ["k31_m20_u64", "k63_m24_u128"]


def test_thresholds_come_from_the_sources():
    assert (C, SCAN_BLOCKS, EMIT_STEP, TAB, LOOK, THREADS) == (1024, 1024, 2048, 128, 64, 256)
    assert "const unsigned g_chunks = 148 * 8;" in _QC
    assert "const unsigned g_dirty = 148 * 8;" in _QC
    assert "grid_for(max_total, kEmitStep, 148 * 16)" in _QC
    # save_tail runs in k_rep_prep at kRepThreads, 4 vectors of 2 codes per thread and tile
    assert "k_rep_prep<<<std::max(g_chunks, grid_for(in_place ? clean_total : 0, 256 * 4, 148 * 8)), kRepThreads" in _QC
    assert "const uint64_t tile = 4 * uint64_t(blockDim.x);" in _QC
    assert "for (; lo + 32 <= hi; lo += 32)" in _QC and "for (; hi >= lo + 32; hi -= 32)" in _QC
    assert (EMIT_WRAP, TAIL_CODES_WRAP, TAIL_OFF_WRAP, SCAN_WRAP) == (4_849_664, 2_424_832, 303_104, 262_144)


# ---- batches ------------------------------------------------------------------------------------------------------

def concat(contigs):
    bases = np.frombuffer(b"".join(contigs), dtype=np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in contigs], dtype=np.int64)]).astype(np.uint64)
    return bases, offsets


class Source:
    """ACGT bytes to cut contigs from: the index's own contigs (members) then seeded random bases (non-members),
    handed out in order and wrapping around"""

    def __init__(self, genome, seed, n=1 << 20):
        g = np.asarray(genome, dtype=np.uint8)
        g = g[ACGT_OK[g]]
        rnd = ACGT[np.random.default_rng([seed, 99]).integers(0, 4, n)]
        self.a = np.concatenate([g, rnd])
        self.at = 0

    def take(self, n):
        if self.at + n > len(self.a):
            self.at = 0
        assert n <= len(self.a)
        out = self.a[self.at:self.at + n].tobytes()
        self.at += n + 7
        return out

    def gather(self, lens, rng):
        """one array of contigs of the given lengths, each from a random place"""
        lens = np.asarray(lens, dtype=np.int64)
        starts = rng.integers(0, len(self.a) - int(lens.max(initial=0)) - 1, len(lens))
        ends = np.cumsum(lens)
        idx = np.repeat(starts - (ends - lens), lens) + np.arange(int(ends[-1]) if len(lens) else 0)
        return self.a[idx].copy(), np.concatenate([[0], ends]).astype(np.uint64)


def sweep_contigs(src, k, m):
    """(name, contig) pairs, every contig dirty, each built to put one edge of the episode walk, the chunk summaries
    or the chunk mask at a chunk seam (contig coordinates, C = kRepairChunk)"""
    w = k - m + 1
    N = b"N"
    P = src.take
    out = []

    def rest():  # short runs, then a long one: spurious codes after a head, then valid codes
        return P(m + 1) + N + P(max(k - 1, 1)) + N + P(2 * k)

    def tail():
        return N + rest()

    for r in (C - 2, C - 1, 0, 1):  # episode heads (last byte of a run of >= k before an N) at p = 2C + r - C
        p = 2 * C + r - (C if r >= C - 2 else 0)
        out.append((f"head p%C={r}", P(p + 1) + tail()))
    out.append(("head p=k-1", P(k) + tail()))
    for L in (k, k + w - 1, k + w, k + w + 1, 2 * w + k):  # the rebuild from a multiple of w bases into the run
        out.append((f"run {L}", P(20) + N + P(L) + tail()))
    for L in (31 * C, 32 * C, 33 * C, 64 * C + 5):  # prev_some over 31 to 64 chunks with no non-ACGT byte
        out.append((f"run {L} from a junk byte", P(100) + N + P(L) + tail()))
        out.append((f"run {L} from the contig start", P(L) + tail()))
    out.append(("run from a chunk start", P(C - 1) + N + P(2 * C) + tail()))
    out.append(("run from one past a chunk start", P(C) + N + P(2 * C) + tail()))
    out.append(("stretch of 1", P(2 * k) + N + P(m) + N + P(2 * k)))
    for d in (-1, 0, 1):  # a stretch whose last byte is the chunk's last one, one short of it, one past it
        out.append((f"stretch to chunk end {d:+d}", P(C + 100) + N * (C - 100 + d) + rest()))
    for j in (31, 32, 33, 63, 64, 65):  # next_some over whole chunks of non-ACGT bytes
        out.append((f"stretch over {j} chunks", P(C - 300) + N * (300 + j * C + 200) + rest()))
        out.append((f"stretch of {j} chunks from a chunk start", P(C) + N * (j * C) + rest()))
    out.append(("stretch to the contig end", P(2 * k) + N * (3 * C + 7)))
    out.append(("short stretch to the contig end", P(k + 3) + N * 5))
    out.append(("stretch from a chunk start to the contig end", P(C) + N * C))
    for j in JUNK:
        out.append((f"junk {j!r}", P(2 * k) + j + P(m + 2) + j * 3 + P(k - 1) + j + P(2 * k)))
    for r in sorted({m - 1, m, k - 1}):  # short runs across a seam after a stretch, then a long run whose k-th byte
        if r < 1:                        # is a chunk's first byte
            continue
        a = 2 * C - r // 2
        head = P(2 * k) + N * (a - 2 * k) + P(r)
        out.append((f"short run {r} across a seam", head + N * (3 * C - k + 1 - len(head)) + P(k + 50)))
    for a in (C, 2 * C):  # the chunk mask's look-back: an N at a - k, a - k + 1, a - 1 before a chunk start a
        for d in (k, k - 1, 1):
            c = bytearray(P(3 * C))
            c[a - d] = ord("N")
            out.append((f"N at {a}-{d}", bytes(c)))
    for j in (1, 2, 33):  # contig lengths at chunk multiples; the last run ends in spurious codes at the contig end
        for d in (-1, 0, 1):
            L = j * C + d
            c = bytearray(P(L))
            c[L // 3] = ord("N")
            c[L - m - 2] = ord("N")
            out.append((f"length {L}", bytes(c)))
    for name, c in out:
        assert not ACGT_OK[np.frombuffer(c, np.uint8)].all() and len(c) >= k, name
    return out


def sweep_groups(contigs):
    """the sweep contigs in groups of at most 31, so that with the filler in front a batch fits one warp of
    k_rep_list (which then lists them in contig order)"""
    return [contigs[i:i + 31] for i in range(0, len(contigs), 31)]


def filler(src, r):
    """a dirty contig of r whole chunks (none for r = 0): the chunks of the contigs after it start r later"""
    if r == 0:
        return []
    c = bytearray(src.take(r * C))
    c[len(c) // 2] = ord("N")
    return [bytes(c)]


def plant_junk(bases, offsets, which, rng, per=1):
    """`per` random bytes of each contig in `which` (of length >= 1) made N"""
    lens = np.diff(offsets.astype(np.int64))
    which = np.asarray(which)[lens[which] > 0]
    for _ in range(per):
        at = offsets[which].astype(np.int64) + (rng.random(len(which)) * lens[which]).astype(np.int64)
        bases[at] = ord("N")
    return which


def many_short(o, src, k, m, n=310_000, seed=0, sixteen=False):
    """contig 0 dirty with a long gap, then n contigs of 0, 1, k-1, k ... k+15 bytes (1 % dirty): emit steps in the
    middle of hundreds of contigs (no shared table).  `sixteen`: n clean contigs of 16 codes each, with a second
    dirty contig halfway; the first dirty contig's count is a multiple of 16 and the second's is not, so the steps
    hold exactly 128 contigs before the second and 129 after it"""
    rng = np.random.default_rng([k, m, seed, 5])
    first = src.take(3000) + b"N" * 100_000 + src.take(m) + b"N" + src.take(k - 1) + b"N" + src.take(2 * k)
    if not sixteen:
        choice = np.array([0, 1, k - 1] + list(range(k, k + 16)))
        bases, offsets = src.gather(choice[rng.integers(0, len(choice), n)], rng)
        plant_junk(bases, offsets, np.flatnonzero(rng.random(n) < 0.01), rng)
        return join([first], (bases, offsets))
    first = fix_count(o, first, src, 0)
    second = fix_count(o, src.take(k + 3) + b"N" + src.take(m + 1), src, 8)
    b1, o1 = src.gather(np.full(n // 2, k + 15), rng)
    b2, o2 = src.gather(np.full(n - n // 2, k + 15), rng)
    return join([first], (b1, o1), [second], (b2, o2))


def fix_count(o, contig, src, want_mod, mod=16):
    """contig with bases added at its end (a run of >= k: one more code per byte) until its code count is want_mod
    modulo mod"""
    contig = contig + src.take(o.k)
    return contig + src.take((want_mod - len(o.query(contig))) % mod)


def read_mix(src, k, m, n_reads, c0_odd, nc_odd, seed=0):
    """150-base reads, 1 % dirty, after a dirty read; a 1-code contig before it makes c0 (the clean codes before the
    first dirty contig) odd, one at the end makes nc (the clean codes from it on) odd"""
    rng = np.random.default_rng([k, m, seed, 6])
    bases, offsets = src.gather(np.full(n_reads, 150), rng)
    plant_junk(bases, offsets, np.flatnonzero(rng.random(n_reads) < 0.01), rng)
    first = bytearray(src.take(150))
    first[70] = ord("N")
    head = [src.take(k)] if c0_odd else []
    per = 150 - k + 1
    nc = per * (n_reads + 1)
    tail = [src.take(k)] if (nc % 2 == 1) != nc_odd else []
    return head + [bytes(first)], bases, offsets, tail


def dirty_reads(src, k, m, n_reads=270_000, seed=0):
    """n_reads reads of 40-150 bases, every one dirty (two N each): more dirty chunks than one round of the
    chunks' block scan"""
    rng = np.random.default_rng([k, m, seed, 7])
    bases, offsets = src.gather(rng.integers(40, 151, n_reads), rng)
    plant_junk(bases, offsets, np.arange(n_reads), rng, per=2)
    return bases, offsets


def join(*parts):
    """one batch of parts in order, each a list of contigs (bytes) or a batch (bases, offsets from 0)"""
    bs, offs, at = [], [np.zeros(1, np.uint64)], np.uint64(0)
    for p in parts:
        b, o = concat(p) if isinstance(p, list) else p
        bs.append(np.asarray(b, np.uint8))
        offs.append(o[1:].astype(np.uint64) + at)
        at += o[-1].astype(np.uint64)
    return np.concatenate(bs), np.concatenate(offs)


# ---- what the kernels see -----------------------------------------------------------------------------------------

def contig_dirty(bases, offsets):
    bad = np.concatenate([[0], np.cumsum(~ACGT_OK[bases], dtype=np.int64)])
    off = offsets.astype(np.int64)
    return bad[off[1:]] > bad[off[:-1]]


class Geometry:
    """what the repair's kernels see for a batch, from its bytes, offsets and final code offsets (the oracle's)"""

    def __init__(self, bases, offsets, final_off, k):
        self.k = k
        off = offsets.astype(np.int64)
        self.lens = np.diff(off)
        self.n = len(self.lens)
        self.dirty = contig_dirty(bases, offsets)
        first = np.flatnonzero(self.dirty)
        assert len(first), "no dirty contig"
        self.fd = int(first[0])
        assert self.lens[self.fd] >= k  # every path flags it: the first dirty contig the kernels see is this one
        self.fd_rev = self.n - self.fd
        clean = np.concatenate([[0], np.cumsum(np.maximum(self.lens - k + 1, 0))])
        self.clean_total = int(clean[-1])
        self.c0 = int(clean[self.fd])
        self.nc = self.clean_total - self.c0
        self.final = final_off.astype(np.int64)
        self.total = int(self.final[-1])
        self.after = self.total - int(self.final[self.fd])
        nch = (self.lens + C - 1) // C
        self.dirty_chunks = int(nch[self.dirty].sum())
        # first chunk ids, where k_rep_list lists the dirty contigs in contig order (one warp: at most 32 contigs)
        self.cb = np.concatenate([[0], np.cumsum(np.where(self.dirty, nch, 0))])[:-1]

    def steps(self, in_place):
        """contigs per block step of emit_clean: from the first dirty contig's final offset in place, else from 0"""
        o0 = int(self.final[self.fd]) if in_place else 0
        if o0 >= self.total:
            return np.zeros(0, np.int64)
        b0 = np.arange(o0, self.total, EMIT_STEP, dtype=np.int64)
        b1 = np.minimum(b0 + EMIT_STEP, self.total)
        lo = np.searchsorted(self.final, b0, "right") - 1
        hi = np.searchsorted(self.final, b1 - 1, "right")
        return hi - lo

    def tail_shift(self, codes_shift=0):
        """tail_shift(codes + c0) for d_codes `codes_shift` codes into a 16-byte aligned allocation"""
        return (codes_shift + self.c0) & 1


# ---- the batches reach their branches -----------------------------------------------------------------------------

@pytest.fixture(scope="module")
def oracles():
    opened = {}

    def get(name):
        if name not in opened:
            g = load_golden(name)
            opened[name] = (g, oracle.OracleMphf(os.path.join(GOLDEN_DIR, name + ".lph"), g.bits))
        return opened[name]

    yield get
    for _, o in opened.values():
        o.close()


def per_contig_matches_batch(o, bases, offsets, sample):
    """the oracle's query_batch over the batch equals its per-contig query, concatenated, on `sample` contigs"""
    want, want_off = o.query_batch(bases, offsets)
    for c in sample:
        a, b = int(offsets[c]), int(offsets[c + 1])
        got = o.query(bases[a:b].tobytes())
        assert np.array_equal(got, want[int(want_off[c]):int(want_off[c + 1])]), c
    return want, want_off


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64", "k15_m7_u64"])
def test_sweep_contigs_reach_their_seams(oracles, name):
    g, o = oracles(name)
    k, m = g.k, g.m
    src = Source(g.index_bases, k)
    named = sweep_contigs(src, k, m)
    contigs = [c for _, c in named]
    total_chunks = 0
    for group in sweep_groups(contigs):
        assert len(group) <= 31
        residues = set()
        for r in range(32):
            bases, offsets = concat(filler(src, r) + group)
            assert len(offsets) - 1 <= 32
            want, want_off = o.query_batch(bases, offsets)
            gm = Geometry(bases, offsets, want_off, k)
            assert gm.dirty.all() and gm.fd == 0
            residues |= {(i, int(gm.cb[i + (r > 0)] % 32)) for i in range(len(group))}
            if r == 0:
                total_chunks += gm.dirty_chunks
        # every contig's first chunk id takes every residue mod 32 (and so mod 8) over the 32 shifts
        assert all(len({s for i2, s in residues if i2 == i}) == 32 for i in range(len(group)))
    assert total_chunks > 600
    # the seams the names promise
    by = dict(named)
    for r in (C - 2, C - 1, 0, 1):
        c = by[f"head p%C={r}"]
        p = c.index(b"N") - 1
        assert p % C == r and p + 1 >= k
    for d in (-1, 0, 1):  # the stretch's last byte at 2C - 1 + d
        ok = ACGT_OK[np.frombuffer(by[f"stretch to chunk end {d:+d}"], np.uint8)]
        assert ok[:C + 100].all() and not ok[C + 100:2 * C + d].any() and ok[2 * C + d]
    for j in (31, 32, 33, 63, 64, 65):
        ok = ACGT_OK[np.frombuffer(by[f"stretch of {j} chunks from a chunk start"], np.uint8)]
        assert ok[:C].all() and not ok[C:(j + 1) * C].any() and ok[(j + 1) * C]
    for a in (C, 2 * C):
        for d in (k, k - 1, 1):
            ok = ACGT_OK[np.frombuffer(by[f"N at {a}-{d}"], np.uint8)]
            assert np.flatnonzero(~ok).tolist() == [a - d] and a - d >= a - LOOK
    for r in sorted({m - 1, m, k - 1}):
        if r < 1:
            continue
        s = np.frombuffer(by[f"short run {r} across a seam"], np.uint8)
        ok = ACGT_OK[s]
        start = 2 * C - r // 2
        assert ok[start:start + r].all() and not ok[start - 1] and not ok[start + r]
        assert start < 2 * C < start + r or r == 1
        long0 = 3 * C - k + 1
        assert not ok[long0 - 1] and ok[long0:].all() and (long0 + k - 1) % C == 0


def test_per_contig_oracle_equals_its_batch_on_sweep_batches(oracles):
    g, o = oracles("k31_m20_u64")
    src = Source(g.index_bases, g.k)
    group = sweep_groups([c for _, c in sweep_contigs(src, g.k, g.m)])[0]
    bases, offsets = concat(filler(src, 5) + group)
    per_contig_matches_batch(o, bases, offsets, range(len(offsets) - 1))


def check_many_short(gm, sixteen):
    """the contigs' scan and tail_off past one round; emit steps past the shared table, and with 16 codes per
    contig, steps of exactly kTab and kTab + 1 contigs"""
    assert gm.fd == 0 and gm.fd_rev > max(TAIL_OFF_WRAP, SCAN_WRAP)
    for in_place in (True, False):
        st = gm.steps(in_place)
        assert (st > TAB).any()
        if sixteen:
            assert (st == TAB).sum() > 100 and (st == TAB + 1).sum() > 100
        else:
            assert (st > TAB).mean() > 0.5
    if sixteen:
        counts = np.diff(gm.final)[gm.dirty]
        assert len(counts) == 2 and counts[0] % 16 == 0 and counts[1] % 16 == 8
        assert (np.diff(gm.final)[~gm.dirty] == 16).all()


def check_read_mix(gm, c0_odd, nc_odd):
    """emit_clean's and save_tail's second grid-stride rounds; c0 and nc of the given parities, so that save_tail's
    head (tail_shift) and trailing code take all four combinations with d_codes 0 and 8 bytes into its allocation"""
    assert gm.c0 % 2 == c0_odd and gm.nc % 2 == nc_odd
    assert gm.after > EMIT_WRAP and gm.nc > TAIL_CODES_WRAP
    assert gm.total < gm.clean_total  # (the not-in-place form runs at the final total)
    for shift in (0, 1):
        assert gm.tail_shift(shift) == (shift + c0_odd) % 2


def check_dirty_reads(gm):
    """the chunks' scan (and the contigs') past one round"""
    assert gm.dirty_chunks > SCAN_WRAP and gm.fd_rev > SCAN_WRAP


def make_read_mix(o, src, c0_odd, nc_odd):
    head, bases, offsets, tail = read_mix(src, o.k, o.m, 70_000, c0_odd, nc_odd)
    return join(head, (bases, offsets), tail)


def make_dirty_reads(o, src):
    bases, offsets = dirty_reads(src, o.k, o.m)
    first = bytearray(src.take(150))  # the first contig at least k long: the first dirty contig on every path
    first[75] = ord("N")
    return join([bytes(first)], (bases, offsets))


# the scale batches: name -> (make(oracle, source) -> (bases, offsets), check(Geometry))
SCALE = {
    "many_short": (lambda o, s: many_short(o, s, o.k, o.m), lambda gm: check_many_short(gm, False)),
    "many_short_16": (lambda o, s: many_short(o, s, o.k, o.m, sixteen=True), lambda gm: check_many_short(gm, True)),
    "read_mix_c0_even_nc_odd": (lambda o, s: make_read_mix(o, s, False, True), lambda gm: check_read_mix(gm, 0, 1)),
    "read_mix_c0_odd_nc_even": (lambda o, s: make_read_mix(o, s, True, False), lambda gm: check_read_mix(gm, 1, 0)),
    "dirty_reads": (make_dirty_reads, check_dirty_reads),
}


def scale_batch(o, genome, kind):
    """(bases, offsets) of a scale batch for the index of oracle o"""
    return SCALE[kind][0](o, Source(genome, o.k))


@pytest.mark.parametrize("name", SCALE_NAMES)
@pytest.mark.parametrize("kind", list(SCALE))
def test_scale_batches_reach_their_thresholds(oracles, name, kind):
    g, o = oracles(name)
    bases, offsets = scale_batch(o, g.index_bases, kind)
    n = len(offsets) - 1
    sample = list(range(0, n, 997)) + [0, 1, n - 1]
    want, want_off = per_contig_matches_batch(o, bases, offsets, sample)
    gm = Geometry(bases, offsets, want_off, g.k)
    assert gm.total <= 10 ** 7
    SCALE[kind][1](gm)
