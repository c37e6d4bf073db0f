"""The index self-check on the GPU (lphb_check_*: build-p --check, include/mphf_utils.hpp:51-100).

Own contigs: every golden index (partitioned, 64- and 128-bit k-mers; unpartitioned), the config-1 index and every
(k, m) of the grid (tests/test_kmgrid_cpu.py) passes on its own contigs.  Planted failures: the report equals, field
by field, a numpy restatement of the three tests over the CPU oracle's codes (`restate`).  Invariance: the report
does not depend on the batching, the chunking, host versus device form, the alignment of device bases, calls of
other entry points between the batches, or another handle checked at the same time."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_DIR, GOLDEN_NAMES, ROOT, load_golden
from lphash_b200 import api, seqio, synth
from oracle import oracle
from test_check_cpu import build_check_tool
from test_kmgrid_cpu import GRID, cpu_lph, grid_contigs, grid_id, sanitize, write_image

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
NONE = 2**64 - 1
ALT_NAMES = ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"]
CFG1 = os.path.join(GOLDEN_DIR, "config1")
CLEAN = np.zeros(256, dtype=bool)
CLEAN[np.frombuffer(b"ACGTUacgtu", dtype=np.uint8)] = True


def concat(contigs):
    return seqio.concat(list(contigs))


def contigs_of(bases, offsets):
    raw = np.asarray(bases, np.uint8).tobytes()
    return [raw[int(offsets[i]):int(offsets[i + 1])] for i in range(len(offsets) - 1)]


def is_clean(c):
    return bool(CLEAN[np.frombuffer(c, dtype=np.uint8)].all())


def restate(o, contigs, stream=None):
    """the report of one session over `contigs`, from the oracle: non-streaming codes = the stateless codes with every
    non-ACGT byte as 'A'; streaming codes = the oracle's streaming query (or `stream`, a clean-layout array), compared on
    clean contigs only"""
    k, nkmers = o.k, o.info["nkmers"]
    empty = np.zeros(0, np.uint64)
    ns = [o.query_stateless(sanitize(c)) if len(c) >= k else empty for c in contigs]
    codes = np.concatenate(ns + [empty]).astype(np.uint64)
    oor = codes >= np.uint64(nkmers)
    uniq, cnt = np.unique(codes[~oor], return_counts=True)
    # the missing codes without a bitmap of nkmers entries (indexes of 2^32 k-mers and more): uniq is sorted, so the
    # smallest code never hit is the first i with uniq[i] != i, else len(uniq)
    gaps = np.flatnonzero(uniq != np.arange(len(uniq), dtype=np.uint64))
    n_missing = nkmers - len(uniq)
    min_missing = int(gaps[0]) if len(gaps) else len(uniq) if n_missing else NONE
    mism, at = [], 0
    for c, v in zip(contigs, ns):
        if len(v) and is_clean(c):
            st = o.query(c) if stream is None else stream[at:at + len(v)]
            mism.extend((at + np.flatnonzero(st != v)).tolist())
        at += len(v)
    r = dict(kmers=len(codes), contigs=len(contigs), dirty_contigs=sum(not is_clean(c) for c in contigs),
             out_of_range=int(oor.sum()), duplicates=int(cnt.sum() - len(uniq)), missing=n_missing,
             stream_mismatches=len(mism), first_out_of_range=int(np.argmax(oor)) if oor.any() else NONE,
             first_mismatch=min(mism) if mism else NONE,
             min_duplicate_code=int(uniq[cnt > 1][0]) if (cnt > 1).any() else NONE,
             min_missing_code=min_missing)
    r["ok"] = int(r["out_of_range"] == r["duplicates"] == r["missing"] == r["stream_mismatches"] == 0)
    return r


def host_check(f, contigs, parts=1):
    """one session of the host form over `contigs`, cut into `parts` batches"""
    bases, offsets = concat(contigs)
    f.check_begin()
    n = len(contigs)
    for p in range(parts):
        c0, c1 = n * p // parts, n * (p + 1) // parts
        f.check_batch(bases, offsets[c0:c1 + 1])
    return f.check_end().as_dict()


class DeviceBatch:
    """a batch on the device, d_bases `shift` bytes into its allocation"""

    def __init__(self, contigs, shift=0):
        bases, self.offsets = concat(contigs)
        raw = np.concatenate([np.full(shift, ord("N"), np.uint8), bases, np.full(7, ord("N"), np.uint8)])
        self.t = torch.from_numpy(raw).to(DEV)
        self.ptr = self.t.data_ptr() + shift
        self.d_off = torch.from_numpy(self.offsets.astype(np.int64)).to(DEV)
        self.total = int(np.maximum(np.diff(self.offsets.astype(np.int64)), 0).sum())

    def stream_codes(self, f, stream=0):
        """lphb_query_stream_device's codes of the batch (clean layout), on the device"""
        n = int(sum(max(0, int(self.offsets[i + 1] - self.offsets[i]) - f.k + 1) for i in range(len(self.offsets) - 1)))
        d_codes = torch.zeros(max(n, 1), dtype=torch.int64, device=DEV)
        d_code_off = torch.zeros(len(self.offsets), dtype=torch.int64, device=DEV)
        d_status = torch.zeros(4, dtype=torch.int64, device=DEV)
        f.query_device(self.ptr, self.d_off.data_ptr(), self.offsets, d_codes.data_ptr(), n, d_code_off.data_ptr(),
                       d_status.data_ptr(), stream)
        return d_codes


def device_check(f, batches, stream_codes=None, stream=0):
    f.check_begin()
    for i, b in enumerate(batches):
        d = stream_codes[i].data_ptr() if stream_codes is not None else 0
        f.check_batch_device(b.ptr, b.d_off.data_ptr(), b.offsets, d, stream)
    return f.check_end().as_dict()


@pytest.fixture
def opened():
    hs = []

    def add(h):
        hs.append(h)
        return h

    yield add
    for h in hs:
        h.close()


def golden(name, opened, alt=False):
    g = load_golden(name)
    path = os.path.join(GOLDEN_DIR, ("alt_" if alt else "") + name + ".lph")
    f = opened(api.Mphf.load_alt(path, g.bits) if alt else api.Mphf.load(path, g.bits))
    return g, f, path


def assert_passes(r, nkmers):
    assert r["ok"] == 1 and r["kmers"] == nkmers, r
    assert r["out_of_range"] == r["duplicates"] == r["missing"] == r["stream_mismatches"] == 0
    assert r["first_out_of_range"] == r["first_mismatch"] == r["min_duplicate_code"] == r["min_missing_code"] == NONE


# ---- own contigs ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_golden_index_passes_on_its_own_contigs(opened, monkeypatch, name, wide):
    if wide:
        monkeypatch.setenv("LPHB_FORCE_WIDE_BUCKETS", "1")
    g, f, _ = golden(name, opened)
    contigs = contigs_of(g.index_bases, g.index_offsets)
    r = f.check(g.index_bases, g.index_offsets).as_dict()
    assert_passes(r, f.info.nkmers)
    assert r["contigs"] == len(contigs) and r["dirty_contigs"] == 0
    assert device_check(f, [DeviceBatch(contigs)]) == r


@pytest.mark.parametrize("name", ALT_NAMES)
def test_unpartitioned_golden_passes_on_its_own_contigs(opened, name):
    g, f, _ = golden(name, opened, alt=True)
    assert_passes(f.check(g.index_bases, g.index_offsets).as_dict(), f.info.nkmers)


def test_config1_index_passes_on_its_unitigs(opened):
    f = opened(api.Mphf.load(os.path.join(CFG1, "se.ust.k31_m16_u128.lph"), 128))
    bases, offsets = seqio.read_batch(os.path.join(CFG1, "se.ust.k31.fa.gz"))
    r = f.check(bases, offsets).as_dict()
    assert_passes(r, f.info.nkmers)
    assert r["contigs"] == len(offsets) - 1


@pytest.mark.parametrize("e", GRID, ids=grid_id)
def test_grid_index_passes_on_its_own_contigs(opened, tmp_path, e):
    k, m, bits = e
    bases, offsets = grid_contigs(k, m)
    path = write_image(str(tmp_path / f"{grid_id(e)}.lph"), cpu_lph(bases, offsets, k, m, bits))
    f = opened(api.Mphf.load(path, bits))
    r = f.check(bases, offsets).as_dict()
    assert_passes(r, f.info.nkmers)
    assert device_check(f, [DeviceBatch(contigs_of(bases, offsets), shift=3)]) == r


# ---- planted failures -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_one_contig_dropped_reports_the_missing_codes(opened, name):
    g, f, path = golden(name, opened)
    o = opened(oracle.OracleMphf(path, g.bits))
    contigs = contigs_of(g.index_bases, g.index_offsets)
    drop = contigs[:len(contigs) // 2] + contigs[len(contigs) // 2 + 1:]
    r = host_check(f, drop)
    want = restate(o, drop)
    assert r == want and want["missing"] == len(contigs[len(contigs) // 2]) - g.k + 1 and not r["ok"]


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k25_m13_u64"])
def test_key_set_twice_duplicates_every_code(opened, name):
    g, f, _ = golden(name, opened)
    contigs = contigs_of(g.index_bases, g.index_offsets)
    for r in (host_check(f, contigs * 2), host_check(f, contigs * 2, parts=2)):
        assert r["duplicates"] == f.info.nkmers and r["min_duplicate_code"] == 0
        assert r["missing"] == r["out_of_range"] == r["stream_mismatches"] == 0 and not r["ok"]


def flood(k, n=300, seed=7):
    rng = np.random.default_rng(seed)
    return [synth.random_bases(int(rng.integers(k, 4 * k)), rng).tobytes() for _ in range(n)]


def shrunk_copy(name, tmp_path, by):
    """a copy of the golden whose header claims `by` k-mers fewer: the codes of the last `by` keys are out of range"""
    image = bytearray(open(os.path.join(GOLDEN_DIR, name + ".lph"), "rb").read())
    nkmers = int(np.frombuffer(image, "<u8", 1, 10)[0])  # u8 k, u8 m, u64 mm_seed, u64 nkmers
    image[10:18] = np.uint64(nkmers - by).tobytes()
    path = str(tmp_path / f"{name}.shrunk.lph")
    open(path, "wb").write(image)
    return path


@pytest.mark.parametrize("shrink", [0, 5])
@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_query_batches_and_non_members_match_the_restatement(opened, tmp_path, name, shrink):
    g = load_golden(name)
    path = shrunk_copy(name, tmp_path, shrink) if shrink else os.path.join(GOLDEN_DIR, name + ".lph")
    f = opened(api.Mphf.load(path, g.bits))
    o = opened(oracle.OracleMphf(path, g.bits))
    contigs = g.contigs() + [b"", b"ACG", b"N" * (g.k - 1), b"acgtN"] + flood(g.k) + [b""]
    want = restate(o, contigs)
    assert want["dirty_contigs"] > 0 and want["duplicates"] > 0 and not want["ok"]
    assert (want["out_of_range"] > 0) == (shrink > 0)
    assert host_check(f, contigs) == want
    assert host_check(f, contigs, parts=3) == want
    assert device_check(f, [DeviceBatch(contigs, shift=5)]) == want
    assert f.stats().kernel_launches > 0


@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128", "k40_m17_u128"])
def test_changed_pilot_matches_the_restatement(opened, tmp_path, name):
    """a copy of the golden with one value of the pilot dictionary (dense buckets) changed; the oracle loads the same
    bytes"""
    g = load_golden(name)
    image = bytearray(open(os.path.join(GOLDEN_DIR, name + ".lph"), "rb").read())
    sec = api.lph_sections(bytes(image), g.bits)
    at = sec[0] + 88  # single_phf: seed, num_keys, table_size, M (16), dense, sparse, M_dense (16), M_sparse (16)
    ranks_words = int(np.frombuffer(image, "<u8", 1, at + 24)[0])
    at += 32 + 8 * ranks_words  # ranks compact vector {size, width, mask, vector}; then the values
    n_values, width = (int(v) for v in np.frombuffer(image, "<u8", 2, at))
    assert 1 < n_values and 0 < width <= 64
    image[at + 32] ^= 1  # lowest bit of the first pilot value
    path = str(tmp_path / "changed.lph")
    open(path, "wb").write(image)
    f = opened(api.Mphf.load(path, g.bits))
    o = opened(oracle.OracleMphf(path, g.bits))
    contigs = contigs_of(g.index_bases, g.index_offsets)
    want = restate(o, contigs)
    assert not want["ok"] and want["missing"] > 0
    assert host_check(f, contigs) == want
    assert device_check(f, [DeviceBatch(contigs)]) == want


@pytest.mark.parametrize("name", ["k31_m20_u64", "k47_m20_u128", "k25_m13_u64"])
def test_caller_stream_codes_with_a_planted_mismatch(opened, name):
    g, f, path = golden(name, opened)
    o = opened(oracle.OracleMphf(path, g.bits))
    contigs = g.contigs()
    b = DeviceBatch(contigs)
    lens = [max(0, len(c) - g.k + 1) for c in contigs]
    starts = np.concatenate([[0], np.cumsum(lens)])
    clean_c = next(i for i, c in enumerate(contigs) if lens[i] > 3 and is_clean(c))
    dirty_c = next(i for i, c in enumerate(contigs) if lens[i] > 3 and not is_clean(c))
    base = restate(o, contigs)
    codes = b.stream_codes(f)
    torch.cuda.synchronize()
    assert device_check(f, [b], [codes]) == base and base["stream_mismatches"] == 0
    for c, counted in ((clean_c, True), (dirty_c, False)):
        planted = codes.clone()
        j = int(starts[c]) + 2
        planted[j] += 1
        want = restate(o, contigs, stream=planted.cpu().numpy().view(np.uint64))
        r = device_check(f, [b], [planted])
        assert r == want
        assert r["stream_mismatches"] == (1 if counted else 0)
        assert r["first_mismatch"] == (j if counted else NONE)


def test_shrunk_header_reports_out_of_range_codes_on_the_key_set(opened, tmp_path):
    g = load_golden("k31_m20_u64")
    path = shrunk_copy("k31_m20_u64", tmp_path, 3)
    f = opened(api.Mphf.load(path, g.bits))
    o = opened(oracle.OracleMphf(path, g.bits))
    contigs = contigs_of(g.index_bases, g.index_offsets)
    r = host_check(f, contigs)
    assert r == restate(o, contigs)
    assert r["out_of_range"] == 3 and r["missing"] == r["duplicates"] == 0 and not r["ok"]


# ---- invariance -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["k31_m20_u64", "k31_m16_u128", "k63_m24_u128", "k40_m17_u128"])
def test_report_does_not_depend_on_batching_chunking_or_form(opened, monkeypatch, name):
    g, f, path = golden(name, opened)
    o = opened(oracle.OracleMphf(path, g.bits))
    index = contigs_of(g.index_bases, g.index_offsets)
    contigs = index[1:] + g.contigs() + [b""] + index[:3]
    want = restate(o, contigs)
    for parts in (1, 2, 7, len(contigs)):
        assert host_check(f, contigs, parts) == want, parts
    for chunk in ("1", "1000", "20000", "0"):
        monkeypatch.setenv("LPHB_CHUNK_BASES", chunk)
        assert host_check(f, contigs, 2) == want, chunk
    monkeypatch.delenv("LPHB_CHUNK_BASES")
    for shift in range(16):
        parts = [contigs[:40], contigs[40:41], contigs[41:]]
        assert device_check(f, [DeviceBatch(p, shift) for p in parts]) == want, shift
    # dirty flags and stats describe the last batch
    f.check_begin()
    b = DeviceBatch(g.contigs())
    f.check_batch_device(b.ptr, b.d_off.data_ptr(), b.offsets)
    flags = f.dirty_flags()
    assert flags.astype(bool).tolist() == [not c for c in g.is_clean()]
    assert f.stats().kernel_launches >= 4
    f.check_end()


def test_session_interleaved_with_queries_on_two_streams(opened):
    g, f, path = golden("k31_m20_u64", opened)
    _, f2, _ = golden("k63_m24_u128", opened)
    g2 = load_golden("k63_m24_u128")
    o = opened(oracle.OracleMphf(path, g.bits))
    index = contigs_of(g.index_bases, g.index_offsets)
    contigs = g.contigs() + index
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    parts = [DeviceBatch(contigs[i::4]) for i in range(4)]
    want = restate(o, [c for i in range(4) for c in contigs[i::4]])
    kmers = torch.from_numpy(seqio.pack_kmers(g.q_bases, g.q_offsets, g.k, 64).view(np.int64)).to(DEV)
    lookup_out = torch.zeros_like(kmers)
    qb = DeviceBatch(g.contigs())
    other = contigs_of(g2.index_bases, g2.index_offsets)
    f.check_begin()
    f2.check_begin()
    for i, b in enumerate(parts):
        st = s1 if i % 2 else s2
        f.check_batch_device(b.ptr, b.d_off.data_ptr(), b.offsets, 0, st.cuda_stream)
        codes = qb.stream_codes(f, (s2 if i % 2 else s1).cuda_stream)
        f.lookup_device(kmers.data_ptr(), kmers.shape[0], lookup_out.data_ptr(), st.cuda_stream)
        f2.check_batch(*concat(other[i::4]))
    r, r2 = f.check_end().as_dict(), f2.check_end().as_dict()
    torch.cuda.synchronize()
    assert r == want
    assert_passes(r2, f2.info.nkmers)
    assert np.array_equal(lookup_out.cpu().numpy().view(np.uint64), f.lookup(kmers.cpu().numpy().view(np.uint64)))
    assert codes.shape[0] > 0


def test_calls_outside_a_session_are_argument_errors(opened):
    g, f, _ = golden("k31_m20_u64", opened)
    L = api.lib()
    bases, offsets = concat(g.contigs())
    assert L.lphb_check_batch(f._h, bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1) == api.E_ARG
    assert L.lphb_check_end(f._h, None) == api.E_ARG
    assert L.lphb_check_end(f._h, api.CheckReport()) == api.E_ARG
    f.check_begin()
    f.check_end()
    with pytest.raises(api.LphashError):
        f.check_end()
    b = DeviceBatch(g.contigs())
    with pytest.raises(api.LphashError):
        f.check_batch_device(b.ptr, b.d_off.data_ptr(), b.offsets)


# ---- C++ mirror and the example tool ------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_cpp_mirror_gives_the_same_report(opened, tmp_path, name):
    g, f, path = golden(name, opened)
    libdir = os.path.join(ROOT, "lphash_b200")
    exe = str(tmp_path / "check_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O1", f"-DLPHASH_B200_KMER_BITS={g.bits}", "-I",
                           os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "check_mirror.cpp"),
                           "-o", exe, "-L", libdir, "-llphash_b200", f"-Wl,-rpath,{libdir}"])
    contigs = contigs_of(g.index_bases, g.index_offsets)[1:] + g.contigs()
    bases, offsets = concat(contigs)
    batch = tmp_path / "batch.bin"
    batch.write_bytes(np.uint64(len(contigs)).tobytes() + offsets.astype("<u8").tobytes() + bases.tobytes())
    want = host_check(f, contigs)
    for parts in ("1", "3"):
        out = subprocess.run([exe, path, str(batch), parts], capture_output=True, text=True, check=True).stdout
        assert {k: int(v) for k, v in (line.split() for line in out.splitlines())} == want


def test_check_tool_on_config1(tmp_path):
    exe = build_check_tool(tmp_path)
    lph = os.path.join(CFG1, "se.ust.k31_m16_u128.lph")
    fa = os.path.join(CFG1, "se.ust.k31.fa.gz")
    r = subprocess.run([exe, lph, "128", fa, "0", "1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "[Info] Everything is ok" in r.stdout
    row = r.stdout.splitlines()[0].split(",")
    assert row[0] == fa and row[3:7] == ["0", "0", "0", "0"]
    # one record removed: missing codes, exit status 1
    recs = seqio.read_records(fa)
    short = tmp_path / "short.fa"
    short.write_bytes(b"".join(b">r%d\n%s\n" % (i, s) for i, s in enumerate(recs[:5] + recs[6:])))
    r = subprocess.run([exe, lph, "128", str(short)], capture_output=True, text=True)
    assert r.returncode == 1 and "Everything is ok" not in r.stdout
    assert int(r.stdout.splitlines()[0].split(",")[5]) == len(recs[5]) - 31 + 1
