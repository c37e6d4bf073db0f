"""The device repair of contigs with non-ACGT bytes (quirk_kernels.cu) at the sizes and chunk seams its kernels
branch on, bit for bit against the CPU oracle's query_batch (never against the library's host form, which runs the
same two device stages).

The batches come from tests/test_repair_geometry_cpu.py, which checks with no GPU that each one reaches its branch:
  - a seam sweep per index: episode heads, runs, stretches of non-ACGT bytes, short runs after them, the chunk
    mask's look-back and contig lengths, all placed at kRepairChunk seams, in batches of at most 32 contigs behind a
    dirty filler of r = 0..31 chunks, so that every contig's first chunk id takes every residue mod 32;
  - scale batches: 310,000 short contigs after a dirty one (emit_clean without its shared table, steps of exactly
    128 and 129 contigs, the contigs' scan and tail_off past one round), 70,000 reads with millions of codes after
    the first dirty one (the second grid-stride rounds of emit_clean and save_tail, both parities of c0 and nc),
    270,000 dirty reads (the chunks' scan past one round).
Every batch runs through the asynchronous form at the capacity bound, the synchronous device form in place and (where
the final total is below the clean total) not in place, lphb_query_stream with its default and with small pipeline
chunks, and lphb_query_stream_runs."""
import os

import numpy as np
import pytest

import test_repair_geometry_cpu as geo
from conftest import GOLDEN_DIR, load_golden
from lphash_b200 import api
from oracle import oracle
from test_kmgrid_cpu import cpu_lph, grid_contigs

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
SENTINEL = np.uint64(0xA5A5A5A5A5A5A5A5)
GUARD = 256  # codes past the capacity that must stay untouched
GOLDEN = ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64", "k15_m7_u64"]
GRID = [(63, 1), (63, 31)]  # w = 63, the widest window QuirkState's ring takes, and w = 33
SWEEP = GOLDEN + [f"grid_k{k}_m{m}" for k, m in GRID]


class Index:
    def __init__(self, lph, bits, genome):
        self.f = api.Mphf.load(lph, bits)
        self.o = oracle.OracleMphf(lph, bits)
        self.genome = genome
        self.k, self.m = self.o.k, self.o.m

    def close(self):
        self.f.close()
        self.o.close()


@pytest.fixture(scope="module")
def index(tmp_path_factory):
    opened = {}

    def get(name):
        if name not in opened:
            if name.startswith("grid_"):
                k, m = (int(x[1:]) for x in name.split("_")[1:])
                bases, offsets = grid_contigs(k, m)
                path = str(tmp_path_factory.mktemp("repair_grid") / f"{name}.lph")
                with open(path, "wb") as fh:
                    fh.write(cpu_lph(bases, offsets, k, m, 128))
                opened[name] = Index(path, 128, bases)
            else:
                g = load_golden(name)
                opened[name] = Index(os.path.join(GOLDEN_DIR, name + ".lph"), g.bits, g.index_bases)
        return opened[name]

    yield get
    for ix in opened.values():
        ix.close()


def device_batch(bases, offsets):
    """bases (with 7 junk bytes past the end) and offsets on the device"""
    t = torch.from_numpy(np.concatenate([bases, np.full(7, ord("N"), np.uint8)])).to(DEV)
    return t, torch.from_numpy(offsets.astype(np.int64)).to(DEV)


def bound(offsets, m):
    return int(np.maximum(np.diff(offsets.astype(np.int64)) - m + 1, 0).sum())


def run_async(ix, d, offsets, shift=0):
    """the asynchronous form at the capacity bound, d_codes `shift` codes into its allocation; checks the guard
    regions before and past the capacity"""
    cap = bound(offsets, ix.m)
    buf = torch.from_numpy(np.full(shift + cap + GUARD, SENTINEL).view(np.int64)).to(DEV)
    code_off = torch.full((len(offsets),), -1, dtype=torch.int64, device=DEV)
    status = torch.full((4,), -1, dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    ix.f.query_device_exact_async(d[0].data_ptr(), d[1].data_ptr(), offsets, buf.data_ptr() + 8 * shift, cap,
                                  code_off.data_ptr(), status.data_ptr())
    torch.cuda.synchronize()
    out = buf.cpu().numpy().view(np.uint64)
    assert (out[:shift] == SENTINEL).all() and (out[shift + cap:] == SENTINEL).all()
    st = status.cpu().numpy().view(np.uint64)
    return out[shift:shift + int(st[0])], code_off.cpu().numpy().view(np.uint64), st


def run_sync(ix, d, offsets, cap):
    """the synchronous device form with capacity cap (in place when cap holds the clean layout)"""
    buf = torch.from_numpy(np.full(cap + GUARD, SENTINEL).view(np.int64)).to(DEV)
    code_off = torch.full((len(offsets),), -1, dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    n = ix.f.query_device_exact(d[0].data_ptr(), d[1].data_ptr(), offsets, buf.data_ptr(), cap, code_off.data_ptr())
    out = buf.cpu().numpy().view(np.uint64)
    assert (out[cap:] == SENTINEL).all()
    return out[:n], code_off.cpu().numpy().view(np.uint64)


def check_forms(ix, bases, offsets, want, want_off, small_chunk, monkeypatch, shift=0, twice=False, tag=""):
    """every exact form equals the oracle's codes and code offsets"""
    k = ix.k
    lens = np.diff(offsets.astype(np.int64))
    dirty = geo.contig_dirty(bases, offsets)
    fewest, most = int((dirty & (lens >= k)).sum()), int(dirty.sum())  # a contig shorter than k need not be read
    clean_total = int(np.maximum(lens - k + 1, 0).sum())
    d = device_batch(bases, offsets)
    firsts = None
    for i in range(2 if twice else 1):
        codes, code_off, st = run_async(ix, d, offsets, shift)
        assert np.array_equal(code_off, want_off), ("async offsets", tag)
        assert np.array_equal(codes, want), ("async codes", tag)
        assert st[0] == len(want) and fewest <= st[1] <= most, ("async status", tag)
        if firsts is None:
            firsts = codes, code_off
        else:  # the dirty contigs were listed in another order: the same bytes out
            assert codes.tobytes() == firsts[0].tobytes() and code_off.tobytes() == firsts[1].tobytes(), tag
    codes, code_off = run_sync(ix, d, offsets, bound(offsets, ix.m))
    assert np.array_equal(codes, want) and np.array_equal(code_off, want_off), ("sync in place", tag)
    if len(want) < clean_total:
        codes, code_off = run_sync(ix, d, offsets, len(want))
        assert np.array_equal(codes, want) and np.array_equal(code_off, want_off), ("sync not in place", tag)
    for chunk in (None, small_chunk):
        if chunk is None:
            monkeypatch.delenv("LPHB_CHUNK_BASES", raising=False)
        else:
            monkeypatch.setenv("LPHB_CHUNK_BASES", str(chunk))
        codes, code_off = ix.f.query_batch(bases, offsets)
        assert np.array_equal(codes, want) and np.array_equal(code_off, want_off), ("host", chunk, tag)
    monkeypatch.delenv("LPHB_CHUNK_BASES", raising=False)
    runs, code_off, total = ix.f.query_batch_runs(bases, offsets)
    assert total == len(want) and np.array_equal(code_off, want_off), ("runs", tag)
    assert np.array_equal(api.expand_runs(runs), want), ("runs", tag)


@pytest.mark.parametrize("name", SWEEP)
def test_seam_sweep_matches_the_oracle(index, name, monkeypatch):
    ix = index(name)
    src = geo.Source(ix.genome, ix.k)
    named = geo.sweep_contigs(src, ix.k, ix.m)
    fillers = [geo.filler(src, r) for r in range(32)]
    filler_codes = [[ix.o.query(c) for c in fl] for fl in fillers]
    for gi, group in enumerate(geo.sweep_groups([c for _, c in named])):
        group_codes = [ix.o.query(c) for c in group]  # each record starts from a fresh state: cached over the shifts
        for r in range(32):
            contigs = fillers[r] + group
            parts = filler_codes[r] + group_codes
            bases, offsets = geo.concat(contigs)
            want = np.concatenate(parts)
            want_off = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.uint64)
            if r in (0, 17):  # the cache is the batch's answer
                got, got_off = ix.o.query_batch(bases, offsets)
                assert np.array_equal(got, want) and np.array_equal(got_off, want_off)
            assert len(contigs) <= 32  # one warp of k_rep_list: chunk ids in contig order, r chunks later
            check_forms(ix, bases, offsets, want, want_off, 5000, monkeypatch, shift=r % 2, tag=(name, gi, r))


@pytest.mark.parametrize("name", geo.SCALE_NAMES)
@pytest.mark.parametrize("kind", list(geo.SCALE))
def test_scale_batch_matches_the_oracle(index, name, kind, monkeypatch):
    ix = index(name)
    bases, offsets = geo.scale_batch(ix.o, ix.genome, kind)
    want, want_off = ix.o.query_batch(bases, offsets)
    gm = geo.Geometry(bases, offsets, want_off, ix.k)
    assert gm.total <= 10 ** 7
    geo.SCALE[kind][1](gm)
    check_forms(ix, bases, offsets, want, want_off, 200_000, monkeypatch, twice=True, tag=(name, kind))
    if kind.startswith("read_mix"):  # d_codes 8 bytes into its allocation: save_tail's other head and trailing code
        codes, code_off, st = run_async(ix, device_batch(bases, offsets), offsets, shift=1)
        assert np.array_equal(codes, want) and np.array_equal(code_off, want_off)
