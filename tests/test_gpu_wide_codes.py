"""Codes past 2^32 and the integer edges of the device image, on every query entry point.

The images are goldens rewritten on the host (tests/test_wide_codes_cpu.py): codes straddling 2^32 and 2^31, bucket
bases at the last regular and first exact-path base of both slopes, fallback codes straddling 2^32, Elias-Fano low
fields of up to about 50 bits, 57-bit dictionary fields, unpartitioned images shifted by 2^32 + 12345.  Each entry
point is compared bit for bit with the CPU oracle on the rewritten image (for the unpartitioned ones, with the
relation to the reference's codes).  Also: the loader's bounds on bucket bases (2^30 narrow, 2^62 wide) on both
decoders, the check session on an index of about 2^32 + 2.5x10^4 k-mers (a 512 MB bitmap), and nkmers at the top
of its range."""
import tempfile

import numpy as np
import pytest

from conftest import load_golden
from lphash_b200 import api, seqio
from oracle import oracle
from test_gpu_check import restate
from test_gpu_kmgrid import seam_contigs
from test_kmgrid_cpu import sanitize
from test_wide_codes_cpu import (IMAGE_KEYS, NAMES, S_ADD, alt_shift, crossing_probes, header, header_shift,
                                 read_ef, source, with_nkmers)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
GENERIC_ALWAYS = str(1 << 62)
ALT_NAMES = ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"]


def host(t):
    return t.cpu().numpy().view(np.uint64)


class Case:
    """one rewritten image: its file, the oracle on it and the query batches"""

    def __init__(self, name, key, tmp):
        s = source(name)
        self.s, self.k, self.m, self.bits = s, s.k, s.m, s.bits
        self.img = s.images()[key]
        self.path = str(tmp / f"{name}.{key}.lph")
        open(self.path, "wb").write(self.img)
        g = s.g
        self.batches = {"index": (g.index_bases, g.index_offsets), "query": (g.q_bases, g.q_offsets),
                        "seams": seqio.concat(seam_contigs(g.index_bases, s.k, s.m, seed=1))}
        if key.startswith("left_"):
            o = oracle.OracleMphf(self.path, self.bits)
            try:
                T = s.targeted(key)[2]
                probes = crossing_probes(o, g.index_bases, g.index_offsets, T, s.k, s.m, T + s.k - s.m,
                                         np.random.default_rng(1))
            finally:
                o.close()
            assert probes
            self.batches["probes"] = seqio.concat(probes)
        o = oracle.OracleMphf(self.path, self.bits)
        try:
            self.want = {n: o.query_batch(*b) for n, b in self.batches.items()}
            self.want_ns = {n: np.concatenate([o.query_stateless(sanitize(c)) for c in contigs(*b)] +
                                              [np.zeros(0, np.uint64)]).astype(np.uint64)
                            for n, b in self.batches.items()}
        finally:
            o.close()


def contigs(bases, offsets):
    raw = np.asarray(bases, np.uint8).tobytes()
    return [raw[int(offsets[i]):int(offsets[i + 1])] for i in range(len(offsets) - 1)]


@pytest.fixture(scope="module")
def cases(tmp_path_factory):
    d = tmp_path_factory.mktemp("wide")
    cache = {}

    def get(name, key):
        if (name, key) not in cache:
            cache[name, key] = Case(name, key, d)
        return cache[name, key]

    return get


@pytest.fixture
def opened():
    hs = []

    def add(h):
        hs.append(h)
        return h

    yield add
    for h in hs:
        h.close()


PARAMS = [(n, k) for n in NAMES for k in IMAGE_KEYS]


def pid(p):
    return f"{p[0]}-{p[1]}"


def device_batch(bases, offsets, shift=3):
    raw = np.concatenate([np.full(shift, ord("N"), np.uint8), np.asarray(bases, np.uint8), np.full(7, ord("N"), np.uint8)])
    t = torch.from_numpy(raw).to(DEV)
    return t, t.data_ptr() + shift, torch.from_numpy(np.asarray(offsets).astype(np.int64)).to(DEV)


# ---- streaming: tiled, generic, chunked, run-length -----------------------------------------------------------

@pytest.mark.parametrize("p", PARAMS, ids=pid)
def test_streaming_forms_match_the_oracle(cases, opened, monkeypatch, p):
    c = cases(*p)
    f = opened(api.Mphf.load(c.path, c.bits))
    for mode in ("tiled", "generic", "chunked"):
        monkeypatch.setenv("LPHB_GENERIC_BELOW", GENERIC_ALWAYS if mode == "generic" else "0")
        if mode == "chunked":
            monkeypatch.setenv("LPHB_CHUNK_BASES", "5000")
            monkeypatch.setenv("LPHB_NO_SMALL_PATH", "1")
        for name, (bases, offsets) in c.batches.items():
            want, want_off = c.want[name]
            codes, code_off = f.query_batch(bases, offsets)
            assert np.array_equal(code_off, want_off), (mode, name)
            assert np.array_equal(codes, want), (mode, name)
    for name, (bases, offsets) in c.batches.items():
        want, want_off = c.want[name]
        runs, code_off, total = f.query_batch_runs(bases, offsets)
        assert total == len(want) and np.array_equal(code_off, want_off), name
        assert np.array_equal(api.expand_runs(runs), want), ("runs", name)


@pytest.mark.parametrize("p", PARAMS, ids=pid)
def test_device_forms_match_the_oracle(cases, opened, p):
    """lphb_query_stream_exact_device on every batch, lphb_query_stream_device on the clean ones,
    lphb_query_nonstreaming_device against the stateless oracle"""
    c = cases(*p)
    f = opened(api.Mphf.load(c.path, c.bits))
    for name, (bases, offsets) in c.batches.items():
        want, want_off = c.want[name]
        t, ptr, d_off = device_batch(bases, offsets)
        cap = int(np.maximum(np.diff(np.asarray(offsets).astype(np.int64)) - c.m + 1, 0).sum())
        d_codes = torch.zeros(max(cap, 1), dtype=torch.int64, device=DEV)
        d_code_off = torch.zeros(len(offsets), dtype=torch.int64, device=DEV)
        d_status = torch.zeros(4, dtype=torch.int64, device=DEV)
        n = f.query_device_exact(ptr, d_off.data_ptr(), offsets, d_codes.data_ptr(), cap, d_code_off.data_ptr())
        assert n == len(want) and np.array_equal(host(d_codes)[:n], want), ("exact", name)
        assert np.array_equal(host(d_code_off), want_off), ("exact", name)
        if name != "query":  # clean batches
            d_codes.zero_()
            f.query_device(ptr, d_off.data_ptr(), offsets, d_codes.data_ptr(), len(want), d_code_off.data_ptr(),
                           d_status.data_ptr())
            torch.cuda.synchronize()
            assert np.array_equal(host(d_codes)[:len(want)], want), ("stateless", name)
        ns = c.want_ns[name]
        d_codes.zero_()
        f.query_device_nonstreaming(ptr, d_off.data_ptr(), offsets, d_codes.data_ptr(), cap, d_code_off.data_ptr(),
                                    d_status.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(host(d_codes)[:len(ns)], ns), ("nonstreaming device", name)


@pytest.mark.parametrize("p", PARAMS, ids=pid)
def test_nonstreaming_and_lookup_match_the_oracle(cases, opened, p):
    c = cases(*p)
    f = opened(api.Mphf.load(c.path, c.bits))
    for name, (bases, offsets) in c.batches.items():
        ns = c.want_ns[name]
        codes, _ = f.query_batch(bases, offsets, streaming=False)
        assert np.array_equal(codes, ns), ("nonstreaming", name)
        kmers = seqio.pack_kmers(bases, offsets, c.k, c.bits)
        assert np.array_equal(f.lookup(kmers), ns), ("lookup", name)
        d_kmers = torch.from_numpy(np.ascontiguousarray(kmers).view(np.int64)).to(DEV)
        d_codes = torch.zeros(max(len(ns), 1), dtype=torch.int64, device=DEV)
        f.lookup_device(d_kmers.data_ptr(), len(ns), d_codes.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(host(d_codes)[:len(ns)], ns), ("lookup_device", name)


def decode_both(image, bits, monkeypatch, alt=False):
    """(host-decoded device image, device-decoded one)"""
    out = []
    for hostdec in (True, False):
        if hostdec:
            monkeypatch.setenv("LPHB_HOST_DECODE", "1")
        else:
            monkeypatch.delenv("LPHB_HOST_DECODE", raising=False)
        f = from_bytes(image, bits, alt)
        try:
            out.append(f.device_image())
        finally:
            f.close()
    return out


def from_bytes(image, bits, alt):
    if not alt:
        return api.Mphf.from_bytes(image, bits)
    with tempfile.NamedTemporaryFile(suffix=".lph") as fh:
        fh.write(image)
        fh.flush()
        return api.Mphf.load_alt(fh.name, bits)


@pytest.mark.parametrize("p", PARAMS, ids=pid)
def test_device_decode_equals_host_decode(cases, monkeypatch, p):
    c = cases(*p)
    h, d = decode_both(c.img, c.bits, monkeypatch)
    assert h == d


# ---- loader bounds on bucket bases ----------------------------------------------------------------------------

def load_error(image, bits, monkeypatch, hostdec):
    if hostdec:
        monkeypatch.setenv("LPHB_HOST_DECODE", "1")
    else:
        monkeypatch.delenv("LPHB_HOST_DECODE", raising=False)
    with pytest.raises(api.LphashError) as e:
        api.Mphf.from_bytes(image, bits)
    return e.value.code, str(e.value)


@pytest.mark.parametrize("name", NAMES)
def test_bucket_base_bounds_narrow_and_wide(name, monkeypatch):
    """narrow table: a largest base in [2^30 - w, 2^30 - 1] loads, the next shift is refused; wide table: the same at
    2^62; both decoders agree, on the image and on the error"""
    s = source(name)
    w = s.h["w"]
    top = max(b for kd, b in s.bases if kd not in (None, 2))  # the shifted (non-MAXIMAL) bases
    for limit, nkmers, msg in ((1 << 30, (1 << 30) - 257, "bucket base beyond the number of k-mers"),
                               (1 << 62, None, "bucket base does not fit 62 bits")):
        D = (limit - 1 - top) // w
        ok = header_shift(s.img, D, nkmers)
        assert limit - w <= top + w * D < limit
        h, d = decode_both(ok, s.bits, monkeypatch)
        assert h == d, limit
        f = api.Mphf.from_bytes(ok, s.bits)
        try:
            assert f.info.device_bytes > 0
            codes, _ = f.query_batch(s.g.index_bases, s.g.index_offsets)
            nmax = s.h["n_maximal"]
            want = s.index_codes + np.where(s.index_codes >= np.uint64(w * nmax), np.uint64(w * D), np.uint64(0))
            assert np.array_equal(codes, want), limit
        finally:
            f.close()
        bad = header_shift(s.img, D + 1, nkmers)
        errs = {load_error(bad, s.bits, monkeypatch, hd) for hd in (True, False)}
        assert errs == {(api.E_FORMAT, f"lphash_b200 error {api.E_FORMAT}: {msg}")}, (limit, errs)


# ---- unpartitioned images -------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ALT_NAMES)
def test_unpartitioned_shift_by_s(name, opened, monkeypatch):
    """every main-index code but bucket 0's and every fallback code moves by S: on the members,
    new = old + S [old >= sizes[1]]"""
    g = load_golden(name)
    img = open(g.lph.replace(name, "alt_" + name), "rb").read()
    sizes1 = read_ef(img, api.lph_sections(img, g.bits, alt=True)[2])[0][1]
    new = alt_shift(img, g.bits, S_ADD)
    h, d = decode_both(new, g.bits, monkeypatch, alt=True)
    assert h == d
    f0, f = opened(from_bytes(img, g.bits, True)), opened(from_bytes(new, g.bits, True))
    bases, offsets = g.index_bases, g.index_offsets
    for streaming in (True, False):
        old, _ = f0.query_batch(bases, offsets, streaming=streaming)
        want = old + np.where(old >= np.uint64(sizes1), np.uint64(S_ADD), np.uint64(0))
        codes, _ = f.query_batch(bases, offsets, streaming=streaming)
        assert np.array_equal(codes, want), streaming
        assert (codes >= np.uint64(1 << 32)).any()
    kmers = seqio.pack_kmers(bases, offsets, g.k, g.bits)
    old = f0.lookup(kmers)
    assert np.array_equal(f.lookup(kmers), old + np.where(old >= np.uint64(sizes1), np.uint64(S_ADD), np.uint64(0)))
    runs, _, _ = f.query_batch_runs(bases, offsets)
    assert np.array_equal(api.expand_runs(runs), f.query_batch(bases, offsets)[0])


# ---- the check session past 2^32 ------------------------------------------------------------------------------

def test_check_session_on_codes_past_2p32(cases, opened):
    """nkmers = about 2^32 + 2.5x10^4: the index contigs hit every code but the w*D shifted away"""
    c = cases("k31_m20_u64", "shift_half_above_2p32")
    s = c.s
    h = header(c.img)
    D = h["n_maximal"] - s.h["n_maximal"]
    w = s.h["w"]
    f = opened(api.Mphf.load(c.path, c.bits))
    r = f.check(*c.batches["index"]).as_dict()
    assert r["kmers"] == s.h["nkmers"] and r["missing"] == w * D
    assert r["min_missing_code"] == w * s.h["n_maximal"]
    assert r["duplicates"] == r["out_of_range"] == r["stream_mismatches"] == 0 and r["ok"] == 0
    o = opened(oracle.OracleMphf(c.path, c.bits))
    q = contigs(*c.batches["query"])
    got = f.check(*c.batches["query"]).as_dict()
    want = restate(o, q)
    assert {k: got[k] for k in want} == want
    f.query_batch(*c.batches["index"])  # the handle answers after the sessions


# ---- nkmers at the top of its range ---------------------------------------------------------------------------

@pytest.mark.parametrize("nkmers", [2**64 - 1, 2**50])
def test_check_begin_refuses_a_bitmap_that_cannot_exist(nkmers, opened):
    """the header's nkmers is unbounded: check_begin must refuse before any kernel (never call check_batch here:
    on a build without the bound the session would write past its bitmap)"""
    s = source("k31_m20_u64")
    f = opened(api.Mphf.from_bytes(with_nkmers(s.img, nkmers), s.bits))
    assert f.get_kmer_count() == nkmers
    codes, _ = f.query_batch(s.g.index_bases, s.g.index_offsets)
    assert np.array_equal(codes, s.index_codes)
    with pytest.raises(api.LphashError) as e:
        f.check_begin()
    assert e.value.code == (api.E_ARG if nkmers >= 2**64 - 32 else api.E_NOMEM)
    if nkmers < 2**64 - 32:
        assert str((nkmers + 31) // 32 * 4 + 8) in str(e.value)
    with pytest.raises(api.LphashError):  # no session was left open
        f.check_end()
    codes, _ = f.query_batch(s.g.index_bases, s.g.index_offsets)
    assert np.array_equal(codes, s.index_codes)
    assert np.array_equal(f.lookup(seqio.pack_kmers(s.g.index_bases, s.g.index_offsets, s.k, s.bits)),
                          codes)


def test_nkmers_near_2p64_loads_the_wide_table(cases, opened):
    """nkmers = 2^64 - 100 with bases of 2^31 and more: the wide/narrow choice must not wrap"""
    for name in NAMES:
        c = cases(name, "nkmers_2p64m100_wide")
        f = opened(api.Mphf.load(c.path, c.bits))
        assert f.get_kmer_count() == 2**64 - 100
        codes, code_off = f.query_batch(*c.batches["query"])
        assert np.array_equal(codes, c.want["query"][0]) and np.array_equal(code_off, c.want["query"][1])
        assert (codes >= np.uint64(1 << 31)).any()
