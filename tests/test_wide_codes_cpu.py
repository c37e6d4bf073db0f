"""Golden indexes rewritten on the host so that their codes, bucket bases and serialized fields reach past 2^32 (and
the other integer edges of the device image), with no GPU and no large build.

Every rewrite keeps a file the reference's reader accepts, and the CPU oracle (all arithmetic mod 2^64) answers on
it.  The transforms:
- header shift: n_maximal += D, nkmers += w*D.  Every non-MAXIMAL code (fallback ones included) adds w*n_maximal in
  mphf::query, so a member's code becomes old + w*D exactly when old >= w*n_maximal;
- targeted shift: the D that puts one chosen bucket's base (LEFT, RIGHT, NONE or the collision base) at a target T;
- sizes_and_positions re-encoded with a larger universe (low widths up to about 50 bits, the codes unchanged), or
  with S added to every value after the encoder's leading 0 (the codes shift like a header shift by S, except those
  of the LEFT bucket of rank 0, which reads that 0);
- the four dictionary vectors of both PHFs at the widest width the loader takes, and their free-slot Elias-Fano
  with a larger universe (the codes unchanged);
- unpartitioned images: S added to num_kmers_in_main_index, nkmers and every value of `sizes` after the leading 0.

tests/test_gpu_wide_codes.py runs every query entry point on these images."""
import struct

import numpy as np
import pytest

from conftest import load_golden
from lphash_b200 import api
from oracle import invindex, oracle, phf

NAMES = ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"]  # tiled 64-bit, tiled 128-bit, generic kernels
S_ADD = (1 << 32) + 12345
EF_UNIVERSES = [1 << 33, 1 << 40, 1 << 50, 1 << 61]
MAX_COMPACT_WIDTH = 57  # the loader's bound (lph_image.cpp Cursor::compact)
PHF_FIXED = 88          # seed, num_keys, table_size, M, dense, sparse, M_dense, M_sparse
LEFT, RIGHT, MAXIMAL, NONE = 0, 1, 2, 3  # OracleMphf.rank_of types


# ---- readers and writers of the serialized structures ---------------------------------------------------------

def header(img):
    k, m, seed, nk, dist, nmax, rs, ns, np_ = struct.unpack_from("<BBQQQQQQQ", img, 0)
    return dict(k=k, m=m, w=k - m + 1, nkmers=nk, distinct=dist, n_maximal=nmax, rs=rs, ns=ns, np=np_)


def read_vec(b, at, dtype):
    n, = struct.unpack_from("<Q", b, at)
    return np.frombuffer(b, dtype=dtype, count=n, offset=at + 8), at + 8 + n * np.dtype(dtype).itemsize


def read_compact(b, at):
    """pthash compact_vector -> (values, width, end)"""
    size, width, _ = struct.unpack_from("<QQQ", b, at)
    words, end = read_vec(b, at + 24, "<u8")
    words = [int(x) for x in words] + [0]
    out = []
    for i in range(size):
        p = i * width
        v = (words[p >> 6] >> (p & 63)) | (words[(p >> 6) + 1] << (64 - (p & 63)) if p & 63 else 0)
        out.append(v & ((1 << width) - 1))
    return out, width, end


def read_ef(b, at):
    """ef_sequence (pthash and lphash share the layout: high bits, darray1, low compact_vector) -> (values, end)"""
    nbits, = struct.unpack_from("<Q", b, at)
    high, at = read_vec(b, at + 8, "<u8")
    at += 8  # darray1: number of positions
    _, at = read_vec(b, at, "<i8")
    _, at = read_vec(b, at, "<u2")
    _, at = read_vec(b, at, "<u8")
    low, width, end = read_compact(b, at)
    ones = np.flatnonzero(np.unpackbits(high.view(np.uint8), bitorder="little")[:nbits])
    return [((int(ones[i]) - i) << width) | low[i] for i in range(len(low))], end


def phf_parts(img, at):
    """offsets of the four dictionary vectors and of the free-slot Elias-Fano of the single_phf at `at`, and its end"""
    starts, p = [], at + PHF_FIXED
    for _ in range(4):
        starts.append(p)
        p = read_compact(img, p)[2]
    free, end = read_ef(img, p)
    return starts, p, free, end


# ---- transforms: bytes -> bytes -------------------------------------------------------------------------------

def header_shift(img, D, nkmers=None):
    """n_maximal += D, nkmers += w*D (or `nkmers`)"""
    h = header(img)
    out = bytearray(img)
    nk = h["nkmers"] + h["w"] * D if nkmers is None else nkmers
    struct.pack_into("<QQQ", out, 10, nk % 2**64, h["distinct"], h["n_maximal"] + D)
    return bytes(out)


def with_nkmers(img, nkmers):
    out = bytearray(img)
    struct.pack_into("<Q", out, 10, nkmers)
    return bytes(out)


def sp_reencode(img, bits, universe=None, add=0):
    """sizes_and_positions with `add` on every value after the encoder's leading 0, at `universe` (default: the
    last value, as the reference encodes it); nkmers grows by `add` too, so that the codes stay below it (the
    loader picks the bucket table's width from nkmers)"""
    sec = api.lph_sections(img, bits)
    vals, end = read_ef(img, sec[2])
    assert end == sec[3] and vals[0] == 0
    vals = [v + add for v in vals[1:]]
    img = with_nkmers(img, header(img)["nkmers"] + add)
    return img[:sec[2]] + invindex.ef_sequence_image(vals, vals[-1] if universe is None else universe) + img[sec[3]:]


def phf_rewrite(img, at, width=None, free_universe=None):
    """the single_phf at `at` with its dictionary vectors at `width` and/or its free slots at `free_universe`"""
    starts, ef_at, free, end = phf_parts(img, at)
    out = img[:starts[0]]
    for s in starts:
        vals, wd, e = read_compact(img, s)
        out += phf._compact(vals, wd if width is None or not vals else width)
    out += phf._ef(free, free_universe) if free_universe is not None and free else img[ef_at:end]
    return out + img[end:]


def both_phfs(img, bits, **kw):
    sec = api.lph_sections(img, bits)
    img = phf_rewrite(img, sec[3], **kw)  # the fallback first: the minimizer PHF's rewrite moves it
    return phf_rewrite(img, sec[0], **kw)


def alt_shift(img, bits, S):
    """mphf_alt: num_kmers_in_main_index += S, nkmers += S, sizes[i] += S for i >= 1"""
    sec = api.lph_sections(img, bits, alt=True)
    vals, end = read_ef(img, sec[2])
    assert end == sec[3] and vals[0] == 0
    out = bytearray(img[:sec[2]])
    nk, dist, main = struct.unpack_from("<QQQ", out, 10)
    struct.pack_into("<QQQ", out, 10, nk + S, dist, main + S)
    new = [v + S for v in vals[1:]]
    return bytes(out) + invindex.ef_sequence_image(new, new[-1]) + img[sec[3]:]


# ---- bucket bases (lph_image.cpp build_buckets) and targeted shifts -------------------------------------------

def bucket_bases(o, img):
    """(kind, base) of every bucket id: kind LEFT / RIGHT / MAXIMAL / NONE, or None for a colliding minimizer;
    and the collision base"""
    h = header(img)
    w, maxblock = h["w"], h["w"] * h["n_maximal"]
    out = []
    for b in range(h["distinct"]):
        t, r = o.rank_of(b)
        if t == LEFT:
            out.append((LEFT, o.sp_access(r) + maxblock))
        elif t == RIGHT:
            v1, v2 = o.sp_pair(h["rs"] + r)
            out.append((None, 0) if v1 == v2 else (RIGHT, v1 + maxblock + h["k"] - h["m"]))
        elif t == MAXIMAL:
            out.append((MAXIMAL, w * r))
        else:
            p1, p2 = o.sp_pair(h["np"] + r)
            out.append((NONE, o.sp_access(h["ns"] + r) + maxblock + p2 - p1))
    return out, o.sp_access(h["np"]) + maxblock


def shift_to(img, bases, kind, T, w):
    """(D, bucket) of the first bucket of `kind` a header shift by D puts at base T"""
    for b, (kd, base) in enumerate(bases):
        if kd == kind and base <= T and (T - base) % w == 0:
            return (T - base) // w, b
    raise AssertionError(f"no bucket of kind {kind} has a base = {T} mod {w}")


def targets(h, fb_keys):
    """name -> (bucket kind or 'collision', target base)"""
    km = h["k"] - h["m"]
    return {"left_last_regular": (LEFT, 2**32 - 1 - km), "left_first_care": (LEFT, 2**32 - km),
            "right_below_2p32": (RIGHT, 2**32 - 1), "right_at_2p32": (RIGHT, 2**32),
            "none_below_2p32": (NONE, 2**32 - 1), "none_at_2p32": (NONE, 2**32),
            "left_at_2p31": (LEFT, 2**31), "right_at_2p31": (RIGHT, 2**31),
            "collision_straddles_2p32": ("collision", 2**32 - fb_keys // 2)}


def fallback_keys(img, bits):
    sec = api.lph_sections(img, bits)
    return struct.unpack_from("<Q", img, sec[3] + 8)[0]


class Source:
    """one golden: its image, the oracle's codes of its index contigs and its bucket bases"""

    def __init__(self, name):
        self.g = g = load_golden(name)
        self.name, self.bits, self.k, self.m = name, g.bits, g.k, g.m
        self.img = open(g.lph, "rb").read()
        self.h = header(self.img)
        o = oracle.OracleMphf(g.lph, g.bits)
        try:
            self.index_codes, _ = o.query_batch(g.index_bases, g.index_offsets)
            self.bases, self.collision_base = bucket_bases(o, self.img)
        finally:
            o.close()
        self.fb_keys = fallback_keys(self.img, g.bits)

    def targeted(self, name):
        kind, T = targets(self.h, self.fb_keys)[name]
        w = self.h["w"]
        if kind == "collision":
            D = (T - self.collision_base) // w
            return header_shift(self.img, D), None, self.collision_base + w * D
        D, b = shift_to(self.img, self.bases, kind, T, w)
        return header_shift(self.img, D), b, T

    def images(self):
        """name -> rewritten image, every transform of this file (the GPU parity set)"""
        h, w, nk = self.h, self.h["w"], self.h["nkmers"]
        out = {"shift_half_above_2p32": header_shift(self.img, ((1 << 32) - nk // 2) // w)}
        for t in targets(h, self.fb_keys):
            out[t] = self.targeted(t)[0]
        for U in EF_UNIVERSES:
            out[f"sp_universe_2p{U.bit_length() - 1}"] = sp_reencode(self.img, self.bits, universe=U)
        out["sp_values_plus_s"] = sp_reencode(self.img, self.bits, add=S_ADD)
        out["sp_values_plus_s_universe_2p61"] = sp_reencode(self.img, self.bits, universe=1 << 61, add=S_ADD)
        out["phf_dicts_width_57"] = both_phfs(self.img, self.bits, width=MAX_COMPACT_WIDTH)
        out["phf_free_slots_universe_2p50"] = both_phfs(self.img, self.bits, free_universe=1 << 50)
        # header nkmers at the top of the range, bases that need the wide table
        out["nkmers_2p64m100_wide"] = header_shift(self.img, (1 << 31) // w, nkmers=2**64 - 100)
        return out


IMAGE_KEYS = ["shift_half_above_2p32", "left_last_regular", "left_first_care", "right_below_2p32", "right_at_2p32",
              "none_below_2p32", "none_at_2p32", "left_at_2p31", "right_at_2p31", "collision_straddles_2p32",
              "sp_universe_2p33", "sp_universe_2p40", "sp_universe_2p50", "sp_universe_2p61", "sp_values_plus_s",
              "sp_values_plus_s_universe_2p61", "phf_dicts_width_57", "phf_free_slots_universe_2p50",
              "nkmers_2p64m100_wide"]
_sources = {}


def source(name):
    if name not in _sources:
        _sources[name] = Source(name)
    return _sources[name]


def shifted(codes, threshold, by):
    return codes + np.where(codes >= np.uint64(threshold), np.uint64(by % 2**64), np.uint64(0))


def oracle_codes(img, bits, bases, offsets, tmp_path, tag="x"):
    p = tmp_path / f"{tag}.lph"
    p.write_bytes(img)
    o = oracle.OracleMphf(str(p), bits)
    try:
        return o.query_batch(bases, offsets)[0]
    finally:
        o.close()


def crossing_probes(o, bases, offsets, base, k, m, want, rng, tries=40):
    """k-mers whose minimizer is that of the slope +1 bucket at `base`, at offset k - m (code base + k - m): members
    of the bucket with their window moved left over random bases, kept where the oracle gives `want`"""
    codes, code_off = o.query_batch(bases, offsets)
    raw = np.asarray(bases, np.uint8).tobytes()
    out = []
    for c in range(len(offsets) - 1):
        for j in range(int(code_off[c]), int(code_off[c + 1])):
            p = int(codes[j]) - base
            if not 0 <= p < k - m:
                continue
            at = int(offsets[c]) + j - int(code_off[c])
            x = raw[at:at + p + m]
            for _ in range(tries):
                y = bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), k - m - p)) + x
                if int(o.query_stateless(y)[0]) == want:
                    out.append(y)
                    break
    return out


# ---- tests ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", NAMES)
def test_reencoding_with_the_original_parameters_gives_the_file(name):
    s = source(name)
    assert sp_reencode(s.img, s.bits) == s.img
    assert both_phfs(s.img, s.bits) == s.img
    for pos in (api.lph_sections(s.img, s.bits)[0], api.lph_sections(s.img, s.bits)[3]):
        starts, ef_at, free, end = phf_parts(s.img, pos)
        assert phf._ef(free) == s.img[ef_at:end]
        for st in starts:
            vals, wd, e = read_compact(s.img, st)
            assert phf._compact(vals, wd) == s.img[st:e]


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
def test_alt_reencoding_gives_the_file_and_shifts_sizes(name):
    g = load_golden(name)
    img = open(g.lph.replace(name, "alt_" + name), "rb").read()
    sec = api.lph_sections(img, g.bits, alt=True)
    sizes, end = read_ef(img, sec[2])
    assert img[:sec[2]] + invindex.ef_sequence_image(sizes[1:], sizes[-1]) + img[sec[3]:] == img
    # the code of bucket b is sizes[b] + positions.diff(b) - p: bucket 0 keeps sizes[0] = 0, so bucket 0 must not be
    # a colliding minimizer (size 0) for the relation new = old + S [old >= sizes[1]] to hold on members
    assert sizes[1] > 0
    new = alt_shift(img, g.bits, S_ADD)
    assert api.lph_sections(new, g.bits, alt=True)[:3] == sec[:3]
    got, _ = read_ef(new, sec[2])
    assert got == [0] + [v + S_ADD for v in sizes[1:]]
    nk, dist, main = struct.unpack_from("<QQQ", new, 10)
    assert (nk, main) == (struct.unpack_from("<Q", img, 10)[0] + S_ADD, struct.unpack_from("<Q", img, 26)[0] + S_ADD)


@pytest.mark.parametrize("name", NAMES)
def test_header_shift_moves_every_non_maximal_code(name, tmp_path):
    s = source(name)
    g, w, nmax = s.g, s.h["w"], s.h["n_maximal"]
    D = ((1 << 32) - s.h["nkmers"] // 2) // w
    got = oracle_codes(s.images()["shift_half_above_2p32"], s.bits, g.index_bases, g.index_offsets, tmp_path)
    assert np.array_equal(got, shifted(s.index_codes, w * nmax, w * D))
    above = int((got >= np.uint64(1 << 32)).sum())
    assert 0.3 * len(got) < above < 0.7 * len(got)  # about half the codes above 2^32


@pytest.mark.parametrize("name", NAMES)
def test_targeted_shift_puts_the_bucket_base_at_the_target(name, tmp_path):
    s = source(name)
    w, nmax = s.h["w"], s.h["n_maximal"]
    for t, (kind, T) in targets(s.h, s.fb_keys).items():
        img, b, base = s.targeted(t)
        D = (header(img)["n_maximal"] - nmax)
        p = tmp_path / f"{t}.lph"
        p.write_bytes(img)
        o = oracle.OracleMphf(str(p), s.bits)
        try:
            bases, cbase = bucket_bases(o, img)
            got, _ = o.query_batch(s.g.index_bases, s.g.index_offsets)
        finally:
            o.close()
        if b is None:
            assert cbase == base and T - w < base <= T, t
        else:
            assert bases[b] == (kind, T), t
        assert np.array_equal(got, shifted(s.index_codes, w * nmax, w * D)), t


@pytest.mark.parametrize("name", NAMES)
def test_sizes_and_positions_reencodings(name, tmp_path):
    """a larger universe leaves the codes; S on every value moves them like a header shift by S"""
    s = source(name)
    g, w, nmax = s.g, s.h["w"], s.h["n_maximal"]
    imgs = s.images()
    q = oracle_codes(s.img, s.bits, g.q_bases, g.q_offsets, tmp_path, "orig")
    for U in EF_UNIVERSES:
        img = imgs[f"sp_universe_2p{U.bit_length() - 1}"]
        assert np.array_equal(oracle_codes(img, s.bits, g.q_bases, g.q_offsets, tmp_path), q), U
    # the encoder's leading 0 stays: LEFT bucket 0 reads EF[0] = 0, so its codes [w*n_maximal, w*n_maximal + EF[1])
    # stay too
    first = read_ef(s.img, api.lph_sections(s.img, s.bits)[2])[0][1]
    for key in ("sp_values_plus_s", "sp_values_plus_s_universe_2p61"):
        got = oracle_codes(imgs[key], s.bits, g.index_bases, g.index_offsets, tmp_path)
        assert np.array_equal(got, shifted(s.index_codes, w * nmax + first, S_ADD)), key
        assert (got >= np.uint64(1 << 32)).any(), key


@pytest.mark.parametrize("name", NAMES)
def test_wide_fields_reach_past_32_bits(name):
    """the rewritten fields really are wide: Elias-Fano low widths above 32 bits, dictionaries at 57 bits"""
    s = source(name)
    imgs = s.images()
    for key, at_least in (("sp_universe_2p50", 33), ("sp_universe_2p61", 44), ("sp_values_plus_s_universe_2p61", 44)):
        img = imgs[key]
        sec = api.lph_sections(img, s.bits)
        p = sec[2] + 8
        _, p = read_vec(img, p, "<u8")
        p += 8
        for dt in ("<i8", "<u2", "<u8"):
            _, p = read_vec(img, p, dt)
        assert struct.unpack_from("<Q", img, p + 8)[0] >= at_least, key
    img = imgs["phf_dicts_width_57"]
    for at in (api.lph_sections(img, s.bits)[0], api.lph_sections(img, s.bits)[3]):
        assert [read_compact(img, st)[1] for st in phf_parts(img, at)[0]] == [MAX_COMPACT_WIDTH] * 4


@pytest.mark.parametrize("name", NAMES)
def test_phf_rewrites_leave_the_codes(name, tmp_path):
    s = source(name)
    g = s.g
    q = oracle_codes(s.img, s.bits, g.q_bases, g.q_offsets, tmp_path, "orig")
    for key in ("phf_dicts_width_57", "phf_free_slots_universe_2p50"):
        assert np.array_equal(oracle_codes(s.images()[key], s.bits, g.q_bases, g.q_offsets, tmp_path), q), key


@pytest.mark.parametrize("name", NAMES)
def test_oracle_loads_every_image_and_nkmers_edges(name, tmp_path):
    s = source(name)
    g = s.g
    assert list(s.images()) == IMAGE_KEYS
    for key, img in s.images().items():
        got = oracle_codes(img, s.bits, g.index_bases, g.index_offsets, tmp_path)
        assert len(got) == len(s.index_codes), key
        # a consistent file: every member's code below the header's nkmers, from which the loader picks the table
        assert int(got.max()) < header(img)["nkmers"], key
    # the header's nkmers alone does not enter a code
    for nk in (2**64 - 1, 2**50):
        got = oracle_codes(with_nkmers(s.img, nk), s.bits, g.index_bases, g.index_offsets, tmp_path)
        assert np.array_equal(got, s.index_codes)


@pytest.mark.parametrize("name", ["k31_m20_u64"])
def test_crossing_probes_cross_2p32(name, tmp_path):
    """slope +1 buckets never give a member the offset k - m (LEFT sizes stay below w): the probes do"""
    s = source(name)
    k, m = s.k, s.m
    for t in ("left_first_care", "left_last_regular"):
        img, b, T = s.targeted(t)
        p = tmp_path / f"{t}.lph"
        p.write_bytes(img)
        o = oracle.OracleMphf(str(p), s.bits)
        try:
            probes = crossing_probes(o, s.g.index_bases, s.g.index_offsets, T, k, m, T + k - m, np.random.default_rng(1))
        finally:
            o.close()
        assert probes, t
