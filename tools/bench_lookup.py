#!/usr/bin/env python
"""Lookup of packed k-mers (lphb_lookup_kmers) on one GPU, beside the streaming query of the same contigs.

Workloads: config 2 (bench.make_workload: synthetic unitigs, k=31 m=20, 64-bit k-mers) and an index of the same
recipe at k=63 m=24 with 128-bit k-mers (synth.unitigs + oracle.phf.build_lph, cached in bench.CACHE).  Each gives
two rows: `ordered` (every window of every contig in contig order, as seqio.pack_kmers gives them: neighbouring
k-mers share their minimizer) and `shuffled` (the same k-mers in a seeded random order: every probe goes to a random
place of the image).  Before anything is timed, the codes of each row are compared in full with the streaming
query's (lphb_query_stream_device) over the same contigs, and both must be a permutation of 0..n-1.

Per row: the kernel's rate over device-resident k-mers (CUDA events around >= 20 launches after warm-up), its
algorithmic bytes (kmer_bits / 8 in + 8 out per k-mer) over the HBM peak, the end-to-end rate of the host form with
pinned (lphb_host_alloc) and with plain numpy buffers, the streaming query's device rate on the same contigs, a CPU
figure for the reference's non-streaming branch, and the card's name and power limit.  One JSON line per row.

    python tools/bench_lookup.py [--kmers N] [--launches L] [--out rows.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as B  # noqa: E402
from lphash_b200 import api, seqio, synth  # noqa: E402

SEED = 0x100C  # order of the shuffled rows and the CPU sample


def machine():
    """name and power limit of the card, read with a query that changes nothing"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = (x.strip() for x in out[1].split(","))
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the row still stands; the machine is then unknown
        return {"gpu": None, "power_limit": None, "note": f"nvidia-smi: {e}"}


def workload_k63(n_kmers):
    k, m, bits = 63, 24, 128
    bases, offsets = synth.unitigs(n_kmers, k, m)
    lph = os.path.join(B.CACHE, f"lookup_n{n_kmers}_k{k}_m{m}_u{bits}_index{B.INDEX_FORMAT}.lph")
    if not os.path.exists(lph):
        from oracle import phf
        t0 = time.time()
        image = phf.build_lph(bases, offsets, k, m, kmer_bits=bits)
        tmp = f"{lph}.{os.getpid()}.tmp"
        with open(tmp, "wb") as out:
            out.write(image)
        os.replace(tmp, lph)
        B.log(f"[lookup] k=63 index built: {len(image)} bytes ({time.time() - t0:.1f}s)")
    return bases, offsets, lph, k, m, bits


def timed(torch, stream, fn, launches, warmup=3):
    """ms per launch of fn() on stream: CUDA events around `launches` launches after `warmup`"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(launches):
        fn()
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / launches


def cpu_figure(bases, offsets, lph, k, bits, target=10**6):
    """ns per k-mer of the reference's non-streaming branch over a seeded sample of whole contigs (about `target`
    k-mers); the oracle's evaluation of the same definition where the reference library is not built"""
    from oracle import oracle, ref
    rng = np.random.default_rng(SEED)
    order = rng.permutation(len(offsets) - 1)
    contigs, nk = [], 0
    for c in order:
        L = int(offsets[c + 1] - offsets[c])
        if L >= k:
            contigs.append(bases[int(offsets[c]):int(offsets[c + 1])].tobytes())
            nk += L - k + 1
            if nk >= target:
                break
    if ref.available(bits):
        h, kind = ref.RefMphf(lph, bits), "reference (oracle/_ref), RefMphf.query(contig, streaming=False)"
        fn = lambda c: h.query(c, streaming=False)  # noqa: E731
    else:
        h, kind = oracle.OracleMphf(lph, bits), "oracle.OracleMphf.query_stateless (reference library not built)"
        fn = h.query_stateless
    t0 = time.perf_counter()
    got = sum(len(fn(c)) for c in contigs)
    secs = time.perf_counter() - t0
    h.close()
    assert got == nk
    return {"ns_per_kmer": 1e9 * secs / nk, "kmers": nk, "contigs": len(contigs), "threads": 1, "kind": kind}


def host_rates(L, f, kmers, want, reps=3):
    """end-to-end rate of lphb_lookup_kmers with pinned and with plain numpy buffers (median of reps)"""
    n = len(want)
    out = {}
    plain_out = np.empty(n, dtype=np.uint64)
    pin_in, pin_out = C.c_void_p(), C.c_void_p()
    api._check(L.lphb_host_alloc(C.byref(pin_in), kmers.nbytes))
    api._check(L.lphb_host_alloc(C.byref(pin_out), n * 8))
    try:
        h_in = np.frombuffer((C.c_uint8 * kmers.nbytes).from_address(pin_in.value), dtype=np.uint8)
        h_out = np.frombuffer((C.c_uint64 * n).from_address(pin_out.value), dtype=np.uint64)
        h_in[:] = kmers.view(np.uint8).reshape(-1)
        for kind in ("pinned", "numpy"):
            secs = []
            for _ in range(reps + 1):
                t0 = time.perf_counter()
                if kind == "pinned":
                    api._check(L.lphb_lookup_kmers(f._h, pin_in, n, pin_out))
                else:
                    f.lookup(kmers, out=plain_out)
                secs.append(time.perf_counter() - t0)
            got = h_out if kind == "pinned" else plain_out
            assert np.array_equal(got, want), f"{kind}: codes differ"
            st = f.stats()
            out[kind] = {"kmers_per_s": n / float(np.median(secs[1:])), "ms_per_call": 1e3 * float(np.median(secs[1:])),
                         "h2d_bytes": int(st.h2d_bytes), "d2h_bytes": int(st.d2h_bytes),
                         "kernel_launches": int(st.kernel_launches)}
    finally:
        L.lphb_host_free(pin_in)
        L.lphb_host_free(pin_out)
    return out


def run_workload(torch, label, bases, offsets, lph, k, m, bits, launches, gpu, peak, peak_src):
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    f = api.Mphf.load(lph, bits, device=0)
    L = api.lib()
    n = int(np.maximum(np.diff(offsets).astype(np.int64) - k + 1, 0).sum())
    assert n == f.get_kmer_count()
    # the streaming query of the same contigs: the codes every row must reproduce, and the context rate
    d_bases = torch.from_numpy(bases).to(dev)
    d_off = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    d_q = torch.empty(n, dtype=torch.int64, device=dev)
    d_qoff = torch.empty(len(offsets), dtype=torch.int64, device=dev)
    d_status = torch.zeros(4, dtype=torch.int64, device=dev)
    q_ms = timed(torch, stream, lambda: f.query_device(d_bases.data_ptr(), d_off.data_ptr(), offsets, d_q.data_ptr(), n,
                                                       d_qoff.data_ptr(), d_status.data_ptr(), stream.cuda_stream),
                 launches)
    st = d_status.cpu().numpy()
    assert st[0] == n and st[1] == 0, st
    want = d_q.cpu().numpy().view(np.uint64).copy()
    del d_q, d_qoff, d_bases, d_off
    seen = np.zeros(n, dtype=np.uint8)
    seen[want] = 1
    assert int(seen.sum()) == n and int(want.max()) == n - 1, "streaming codes are not a permutation"
    del seen
    t0 = time.time()
    kmers = seqio.pack_kmers(bases, offsets, k, bits)
    B.log(f"[lookup] {label}: {n} k-mers packed ({time.time() - t0:.1f}s)")
    cpu = cpu_figure(bases, offsets, lph, k, bits)
    perm = np.random.default_rng(SEED).permutation(n)
    rows = []
    for order in ("ordered", "shuffled"):
        x = kmers if order == "ordered" else kmers[perm]
        w = want if order == "ordered" else want[perm]
        d_k = torch.from_numpy(x.view(np.int64)).to(dev)
        d_c = torch.full((n,), -1, dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        f.lookup_device(d_k.data_ptr(), n, d_c.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        got = d_c.cpu().numpy().view(np.uint64)
        same = bool(np.array_equal(got, w))
        assert same, f"{label} {order}: lookup codes differ from the streaming query's"
        f.stats()
        ms = timed(torch, stream, lambda: f.lookup_device(d_k.data_ptr(), n, d_c.data_ptr(), stream.cuda_stream),
                   launches)
        st = f.stats()
        del d_k, d_c
        torch.cuda.empty_cache()
        host = host_rates(L, f, x, w)
        algo = n * (bits // 8 + 8)
        achieved = algo / (ms * 1e-3) / 1e9
        row = {"row": f"lookup_{label}_{order}", "metric": "lookup k-mers/sec (device-resident k-mers and codes)",
               "value": n / (ms * 1e-3), "unit": "k-mers/s", "kernel_ms": ms, "launches_timed": launches,
               "kernel_ms_handle_events": float(st.kernel_ms), "kmers": n, "k": k, "m": m, "kmer_bits": bits,
               "order": order, "kernel": f"k_lookup_kmers<{bits // 64}>",
               "roofline": {"bound": "hbm", "algorithmic_bytes": int(algo), "bytes_per_kmer": bits // 8 + 8,
                            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "peak_source": peak_src},
               "e2e": host,
               "streaming_query_device": {"value": n / (q_ms * 1e-3), "unit": "k-mers/s", "kernel_ms": q_ms,
                                          "note": "lphb_query_stream_device over the same contigs, same run"},
               "parity": {"codes_equal_streaming_query": same, "permutation_of_0_to_n_minus_1": True,
                          "note": "full compare of all n codes" + (", permuted like the input" if order == "shuffled" else "")},
               "cpu_baseline": cpu,
               "machine": gpu}
        print(json.dumps(row), flush=True)
        rows.append(row)
    f.close()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--kmers", type=int, default=10**8, help="k-mers of each workload (default 1e8)")
    ap.add_argument("--launches", type=int, default=20, help="timed launches per device figure (>= 20)")
    ap.add_argument("--out", default=None, help="also write the rows to this JSONL file")
    args = ap.parse_args()
    if args.launches < 20:
        ap.error("--launches must be at least 20")
    import torch
    gpu = machine()
    peaks = B.load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (bench.roofline's)"
    rows = []
    bases, offsets, lph = B.make_workload(args.kmers)
    rows += run_workload(torch, "cfg2_k31_m20_u64", bases, offsets, lph, B.K, B.M, B.BITS, args.launches, gpu, peak,
                         peak_src)
    del bases, offsets
    bases, offsets, lph, k, m, bits = workload_k63(args.kmers)
    rows += run_workload(torch, "k63_m24_u128", bases, offsets, lph, k, m, bits, args.launches, gpu, peak, peak_src)
    if args.out:
        with open(args.out, "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
