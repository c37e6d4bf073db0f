"""Build sessions (lphb_build_*): Parts 1 + 2 of build-p fed batch by batch must give what one lphb_scan_classify over
the concatenation gives - triplets, ids, k-mer count and m-mer ordinals - whatever the cut, the form of each batch (host
or device) and the number of merge slices; past 2^32 k-mers too, where a single call cannot go."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT
from lphash_b200 import api
from test_gpu_build import dirty_build_batch, parts

pytestmark = pytest.mark.gpu


def contigs_of(bases, offsets):
    raw = np.ascontiguousarray(bases, dtype=np.uint8).tobytes()
    return [raw[int(offsets[i]):int(offsets[i + 1])] for i in range(len(offsets) - 1)]


def concat(contigs):
    bases = np.frombuffer(b"".join(contigs), dtype=np.uint8).copy()
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in contigs])]).astype(np.uint64)
    return bases, offsets


def device_batch(torch, bases, offsets, shift):
    """the batch in device buffers, the first base `shift` bytes into an allocation (offsets unchanged)"""
    t = torch.zeros(len(bases) + shift + 1, dtype=torch.uint8, device="cuda")
    if len(bases):
        t[shift:shift + len(bases)] = torch.from_numpy(bases).cuda()
    o = torch.from_numpy(offsets.astype(np.int64)).cuda()
    torch.cuda.synchronize()
    return t, o, t.data_ptr() + shift


def run_session(k, m, seed, batches, forms=None):
    """batches: lists of contigs (bytes); forms: per batch "host", "host_offset" (offsets not starting at 0) or
    "device" / "device_odd" (device buffers, bases at an even / odd address)"""
    forms = forms or ["host"] * len(batches)
    keep = []
    with api.BuildSession(k, m, seed) as s:
        for contigs, form in zip(batches, forms):
            bases, offsets = concat(contigs)
            if form == "host":
                s.batch(bases, offsets)
            elif form == "host_offset":  # the batch sits 3 bytes into a larger buffer
                s.batch(np.concatenate([np.frombuffer(b"NNN", np.uint8), bases]), offsets + np.uint64(3))
            else:
                import torch
                t, o, ptr = device_batch(torch, bases, offsets, 1 if form == "device_odd" else 0)
                keep.append((t, o))
                s.batch_device(ptr, o.data_ptr(), offsets, torch.cuda.current_stream().cuda_stream)
        return s.end()


def expected(k, m, seed, batches):
    bases, offsets = concat([c for b in batches for c in b])
    return api.scan_classify(bases, offsets, k, m, seed)


def splits(contigs, k, seed):
    """one batch; one contig per batch; random cuts with an empty batch and a batch without a k-mer"""
    rng = np.random.default_rng(seed)
    n = len(contigs)
    cuts = sorted(rng.choice(np.arange(1, n), size=min(4, n - 1), replace=False).tolist())
    rand = [contigs[a:b] for a, b in zip([0] + cuts, cuts + [n])]
    short = contigs[0][: k - 1]  # m-mers but no k-mer: moves the ordinals only
    rand = rand[:1] + [[]] + [[short, short]] + rand[1:]
    return {"one": [contigs], "per_contig": [[c] for c in contigs], "random": rand}


def assert_same(got, want, n_contigs=None):
    trip, ids, rep = got
    wtrip, wids, wnk, wmm = want
    assert np.array_equal(trip, wtrip)
    assert np.array_equal(ids, wids)
    assert (rep.kmers, rep.mm_count, rep.n_triplets, rep.n_ids) == (wnk, wmm, len(wtrip), len(wids))
    assert rep.colliding_minimizers == int((wtrip["size"] == 0).sum())
    if n_contigs is not None:
        assert rep.contigs == n_contigs


@pytest.mark.parametrize("slice_entries", [None, "7"])
def test_every_split_rebuilds_the_golden_index(golden, slice_entries, monkeypatch):
    """every cut of the index contigs gives scan_classify's result on the whole input, and the triplets rebuild the
    reference's `.lph` byte for byte; LPHB_BUILD_SLICE=7 merges in many slices"""
    if slice_entries:
        monkeypatch.setenv("LPHB_BUILD_SLICE", slice_entries)
    image = open(golden.lph, "rb").read()
    p = parts(image, golden.bits)
    k, m, seed = p["k"], p["m"], p["seed"]
    contigs = contigs_of(golden.index_bases, golden.index_offsets)
    for name, batches in splits(contigs, k, seed=len(contigs)).items():
        want = expected(k, m, seed, batches)
        got = run_session(k, m, seed, batches)
        assert got[2].batches == len(batches), name
        assert_same(got, want, sum(len(b) for b in batches))
        if name != "random":  # (the random split adds two short contigs to the input)
            trip = got[0]
            assert got[2].kmers == p["nkmers"] and len(trip) == p["distinct"], name
            info, body = api.build_inverted_index(k, m, p["minimizer_order"], trip)
            out = api.lph_assemble(k, m, seed, got[2].kmers, len(trip), info, p["minimizer_order"], body, p["fallback"])
            assert out == image, name


def test_host_and_device_batches_mix():
    import torch
    z = np.load(os.path.join(GOLDEN_DIR, "k63_m24_u128.npz"))
    k, m = int(z["k"]), int(z["m"])
    contigs = contigs_of(z["index_bases"], z["index_offsets"])
    batches = [contigs[:3], contigs[3:4], [], contigs[4:11], contigs[11:17], contigs[17:]]
    want = expected(k, m, 42, batches)
    for forms in (["host", "device", "device_odd", "host_offset", "device_odd", "host"],
                  ["device_odd", "host_offset", "device", "device", "host", "device_odd"]):
        assert_same(run_session(k, m, 42, batches, forms), want, len(contigs))
    assert torch.cuda.is_available()


@pytest.mark.parametrize("k,m", [(31, 20), (63, 24), (15, 7), (25, 13)])  # tiled scan / generic passes
def test_non_acgt_input_in_batches_matches_the_reference_loop(k, m):
    from oracle import oracle
    bases, offsets = dirty_build_batch(k, m, seed=k)
    rec, wk, wmm = oracle.scan(bases, offsets, k, m, mode=0)
    wtrip, wids = oracle.classify(rec)
    assert len(wids) > 0
    contigs = contigs_of(bases, offsets)
    for cuts in ([1], [2, 5, 8], list(range(1, len(contigs)))):
        batches = [contigs[a:b] for a, b in zip([0] + cuts, cuts + [len(contigs)])]
        forms = ["device_odd" if i % 2 else "host" for i in range(len(batches))]
        assert_same(run_session(k, m, 42, batches, forms), (wtrip, wids, wk, wmm), len(contigs))


def test_part4_in_batches_with_the_session_ids():
    """colliding_kmers batch by batch, with the running mm_count and the session's ids of that batch's m-mer range,
    gives the reference's fallback key set"""
    z = np.load(os.path.join(GOLDEN_DIR, "k31_m20_u64.npz"))
    k, m = int(z["k"]), int(z["m"])
    contigs = contigs_of(z["index_bases"], z["index_offsets"])
    batches = [contigs[:5], contigs[5:6], contigs[6:15], contigs[15:]]
    _, ids, rep = run_session(k, m, 42, batches)
    assert np.array_equal(ids, z["coll_ids"])
    mm, out = 0, []
    for b in batches:
        bases, offsets = concat(b)
        _, _, mm_next = api.scan_superkmers(bases, offsets, k, m, mm_count=mm)
        mine = ids[(ids >= mm) & (ids < mm_next)]
        out.append(api.colliding_kmers(bases, offsets, k, m, mine, kmer_bits=64, mm_count=mm))
        mm = mm_next
    assert mm == rep.mm_count
    assert np.array_equal(np.concatenate(out), z["coll_kmers"])


def test_session_past_2_32_kmers():
    """17 batches of the same 2^28 bases plus one short contig unique to each batch: 4.6e9 k-mers and m-mer ordinals
    past 2^32.  Every minimizer of the repeated part is seen 17 times (it collides, all its ids are in); a minimizer of
    the unique contigs is a singleton exactly when it is seen once in the session."""
    k, m, seed, reps = 63, 24, 42, 17
    rng = np.random.default_rng(2024)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    n_rep, n_pieces, n_u = 1 << 28, 8, 500
    piece = n_rep // n_pieces
    buf = np.empty(n_rep + n_u, dtype=np.uint8)
    buf[:n_rep] = acgt[rng.integers(0, 4, n_rep, dtype=np.uint8)]
    offsets = np.array([i * piece for i in range(n_pieces + 1)] + [n_rep + n_u], dtype=np.uint64)
    rec_r, nk_r, mm_r = api.scan_superkmers(buf[:n_rep], offsets[:-1], k, m, seed)
    mm_u, nk_u = n_u - m + 1, n_u - k + 1
    uniq = [acgt[rng.integers(0, 4, n_u, dtype=np.uint8)] for _ in range(reps)]
    uniq[5] = uniq[3].copy()  # two batches share a contig: its minimizers collide across batches only
    rec_u = []
    with api.BuildSession(k, m, seed) as s:
        for j in range(reps):
            buf[n_rep:] = uniq[j]
            s.batch(buf, offsets)
            start = j * (mm_r + mm_u)
            rec_u.append(api.scan_superkmers(uniq[j], np.array([0, n_u], np.uint64), k, m, seed, mm_count=start + mm_r)[0])
        trip, ids, rep = s.end()
    assert rep.kmers == reps * (nk_r + nk_u) > 1 << 32
    assert rep.mm_count == reps * (mm_r + mm_u) > 1 << 32
    assert rep.records == reps * len(rec_r) + sum(len(r) for r in rec_u)
    # triplets
    keys_r = np.unique(rec_r["itself"])
    all_u = np.concatenate(rec_u)
    ukeys, ucount = np.unique(all_u["itself"], return_counts=True)
    single = ukeys[(ucount == 1) & ~np.isin(ukeys, keys_r)]
    want = np.zeros(len(np.union1d(keys_r, ukeys)), dtype=api.TRIPLET_DTYPE)
    want["itself"] = np.union1d(keys_r, ukeys)
    srec = all_u[np.isin(all_u["itself"], single)]
    at = np.searchsorted(want["itself"], srec["itself"])
    want["p1"][at], want["size"][at] = srec["p1"], srec["size"]
    assert len(single) > 0 and np.array_equal(trip, want)
    # ids, batch by batch
    ids_r = np.sort(rec_r["id"])
    at = 0
    for j in range(reps):
        u = rec_u[j]
        mine = np.sort(np.concatenate([ids_r + np.uint64(j * (mm_r + mm_u)), u["id"][~np.isin(u["itself"], single)]]))
        assert np.array_equal(ids[at:at + len(mine)], mine), j
        at += len(mine)
    assert at == len(ids) == rep.n_ids
    assert ids[-1] > 1 << 32


def test_capacity_and_misuse():
    import ctypes as C
    z = np.load(os.path.join(GOLDEN_DIR, "k21_m11_u64.npz"))
    k, m = int(z["k"]), int(z["m"])
    contigs = contigs_of(z["index_bases"], z["index_offsets"])
    wtrip, wids, wnk, wmm = expected(k, m, 42, [contigs])
    L = api.lib()
    s = api.BuildSession(k, m, 42)
    s.batch(*concat(contigs[:10]))
    bases, offsets = concat(contigs[10:])
    with pytest.raises(api.LphashError) as e:  # decreasing offsets: refused, the session is unchanged
        s.batch(bases, offsets[::-1].copy())
    assert e.value.code == api.E_ARG
    s.batch(bases, offsets)
    r = api.BuildReport()
    assert L.lphb_build_end(s._h, None, 0, None, 0, C.byref(r)) == api.E_CAPACITY
    assert (r.n_triplets, r.n_ids, r.kmers, r.mm_count, r.batches, r.contigs) == \
        (len(wtrip), len(wids), wnk, wmm, 2, len(contigs))
    assert r.device_bytes > 0
    trip = np.empty(r.n_triplets, dtype=api.TRIPLET_DTYPE)
    ids = np.empty(r.n_ids, dtype=np.uint64)
    assert L.lphb_build_end(s._h, trip.ctypes.data, len(trip) - 1, ids.ctypes.data, len(ids), C.byref(r)) == api.E_CAPACITY
    assert L.lphb_build_end(s._h, trip.ctypes.data, len(trip), ids.ctypes.data, len(ids) - 1, C.byref(r)) == api.E_CAPACITY
    assert L.lphb_build_end(s._h, None, len(trip), ids.ctypes.data, len(ids), C.byref(r)) == api.E_ARG
    assert L.lphb_build_end(s._h, trip.ctypes.data, len(trip), ids.ctypes.data, len(ids), C.byref(r)) == api.OK
    assert np.array_equal(trip, wtrip) and np.array_equal(ids, wids)
    # a closed session refuses batches and ends
    with pytest.raises(api.LphashError) as e:
        s.batch(bases, offsets)
    assert e.value.code == api.E_ARG
    assert L.lphb_build_end(s._h, None, 0, None, 0, C.byref(r)) == api.E_ARG
    s.close()
    # an end without batches is an empty result
    with api.BuildSession(k, m, 42) as s:
        trip, ids, r = s.end()
    assert len(trip) == len(ids) == 0 and (r.batches, r.kmers, r.n_triplets) == (0, 0, 0)
    # a batch after an end that asked for the sizes joins the session
    with api.BuildSession(k, m, 42) as s:
        s.batch(*concat(contigs[:10]))
        assert L.lphb_build_end(s._h, None, 0, None, 0, C.byref(r)) == api.E_CAPACITY
        s.batch(bases, offsets)
        trip, ids, r = s.end()
    assert np.array_equal(trip, wtrip) and np.array_equal(ids, wids)


# ---- the literal drop-in with batches forced small -------------------------------------------------------------
CFG1 = os.path.join(GOLDEN_DIR, "config1")


def cli_env(extra):
    env = {k: v for k, v in os.environ.items() if k != "LPHB_GENERIC_BELOW"}
    env.update(extra)
    return env


@pytest.mark.parametrize("cmd", ["build-p", "build-u"])
def test_dropin_builds_in_many_batches(cmd, tmp_path):
    gpu, ref = (os.path.join(ROOT, "oracle", "_ref", n) for n in ("lphash_gpu128", "lphash128"))
    if not (os.path.exists(gpu) and os.path.exists(ref)):
        pytest.skip("drop-in binaries not built (integration/dropin/build_dropin.sh needs the reference tree)")
    src = os.path.join(CFG1, "se.ust.k31.fa.gz")
    outs = {}
    for tag, cli, extra in [("gpu", gpu, ["--check"]), ("ref", ref, [])]:
        out = str(tmp_path / (tag + ".lph"))
        r = subprocess.run([cli, cmd, "-i", src, "-k", "31", "-m", "16", "-o", out, "-d", str(tmp_path), *extra],
                           capture_output=True, text=True, timeout=1800,
                           env=cli_env({"LPHASH_B200_BATCH_BYTES": "100000", "LPHASH_B200_FIRST_CAP": "10"}))
        assert r.returncode == 0, r.stderr
        if extra:
            assert "Everything is ok" in r.stderr, r.stderr[-2000:]
        outs[tag] = (r.stdout, open(out, "rb").read())
    assert outs["gpu"] == outs["ref"]
    if cmd == "build-p":
        assert outs["gpu"][1] == open(os.path.join(CFG1, "se.ust.k31_m16_u128.lph"), "rb").read()
