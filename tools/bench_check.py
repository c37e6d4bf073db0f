#!/usr/bin/env python
"""The index self-check (lphb_check_*: build-p --check) on one GPU, beside the streaming query and the lookup of the
same k-mers.

Workloads: config 2 (bench.make_workload: synthetic unitigs, k=31 m=20, 64-bit k-mers, the index bench.py caches)
and the k=63 m=24 128-bit index of tools/bench_lookup.py.  Before anything is timed, every row checks its index on its
own contigs (ok == 1, kmers == nkmers) and on the same contigs with the first contig dropped (ok == 0, missing ==
that contig's k-mers), both on the device form and on the host form.

Per row: the device-resident session (lphb_check_begin, one lphb_check_batch_device over all contigs, lphb_check_end)
in ms, with the library's streaming pass and with the streaming codes passed in (d_stream_codes); in the same rounds,
alternating with them, lphb_query_stream_device and lphb_lookup_kmers_device over the same k-mers; medians over the
rounds of CUDA events on one stream.  Then the host form's wall time (pinned bases and offsets, median of 3), a CPU
figure for the same three tests on a sample (the oracle's non-streaming and streaming codes of whole contigs and a
bitmap, one thread), and the card's name and power limit.  One JSON line per row.

    python tools/bench_check.py [--kmers N] [--rounds R] [--out rows.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench as B  # noqa: E402
from bench_lookup import machine, workload_k63  # noqa: E402
from lphash_b200 import api, seqio  # noqa: E402

SEED = 0xC4EC


def cpu_figure(bases, offsets, lph, k, bits, nkmers, target=2 * 10**5):
    """ns per k-mer of the three tests on the CPU over a seeded sample of whole contigs: the oracle's non-streaming and
    streaming codes of each contig, the range test, a bitmap of nkmers bits and the comparison, on one thread"""
    from oracle import oracle
    rng = np.random.default_rng(SEED)
    h = oracle.OracleMphf(lph, bits)
    seen = np.zeros(nkmers, dtype=bool)
    nk, bad = 0, 0
    t0 = time.perf_counter()
    for c in rng.permutation(len(offsets) - 1):
        contig = bases[int(offsets[c]):int(offsets[c + 1])].tobytes()
        if len(contig) < k:
            continue
        ns = h.query_stateless(contig)
        st = h.query(contig)
        bad += int((ns >= nkmers).sum()) + int(seen[ns].sum()) + int((st != ns).sum())
        seen[ns] = True
        nk += len(ns)
        if nk >= target:
            break
    secs = time.perf_counter() - t0
    h.close()
    assert bad == 0
    return {"ns_per_kmer": 1e9 * secs / nk, "kmers": nk, "threads": 1,
            "kind": "oracle.OracleMphf query_stateless + query + numpy bitmap, whole contigs"}


def median_ms(torch, stream, fn):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    fn()
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1)


def run_workload(torch, label, bases, offsets, lph, k, m, bits, rounds, gpu):
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(device=dev)
    s = stream.cuda_stream
    f = api.Mphf.load(lph, bits, device=0)
    L = api.lib()
    n = int(np.maximum(np.diff(offsets).astype(np.int64) - k + 1, 0).sum())
    assert n == f.get_kmer_count()
    d_bases = torch.from_numpy(bases).to(dev)
    d_off = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    d_q = torch.empty(n, dtype=torch.int64, device=dev)
    d_qoff = torch.empty(len(offsets), dtype=torch.int64, device=dev)
    d_status = torch.zeros(4, dtype=torch.int64, device=dev)
    d_kmers = torch.from_numpy(seqio.pack_kmers(bases, offsets, k, bits).view(np.int64)).to(dev)
    d_codes = torch.empty(n, dtype=torch.int64, device=dev)

    def query():
        f.query_device(d_bases.data_ptr(), d_off.data_ptr(), offsets, d_q.data_ptr(), n, d_qoff.data_ptr(),
                       d_status.data_ptr(), s)

    def lookup():
        f.lookup_device(d_kmers.data_ptr(), n, d_codes.data_ptr(), s)

    def check(stream_codes=0):
        f.check_begin()
        f.check_batch_device(d_bases.data_ptr(), d_off.data_ptr(), offsets, stream_codes, s)
        return f.check_end()

    # the verdicts every row rests on
    query()
    torch.cuda.synchronize()
    verdicts = {}
    for form, r in (("device", check()), ("device_caller_codes", check(d_q.data_ptr()))):
        assert r.ok == 1 and r.kmers == n and r.missing == 0, (form, r.as_dict())
        verdicts[form] = r.as_dict()
    c0 = int(offsets[1] - offsets[0])
    drop_off = offsets[1:]
    r = f.check(bases, drop_off)
    assert r.ok == 0 and r.missing == c0 - k + 1 and r.duplicates == r.out_of_range == 0, r.as_dict()
    verdicts["host_first_contig_dropped"] = r.as_dict()
    f.check_begin()
    f.check_batch_device(d_bases.data_ptr(), d_off.data_ptr() + 8, drop_off, 0, s)
    r = f.check_end()
    assert r.as_dict() == verdicts["host_first_contig_dropped"], r.as_dict()
    # device-resident legs, alternating within each round
    legs = {"check": check, "check_caller_codes": lambda: check(d_q.data_ptr()), "query_stream_device": query,
            "lookup_kmers_device": lookup}
    for fn in legs.values():  # warm-up
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name in legs}
    for _ in range(rounds):
        for name, fn in legs.items():
            times[name].append(median_ms(torch, stream, fn))
    ms = {name: float(np.median(v)) for name, v in times.items()}
    spread = {name: [float(min(v)), float(max(v))] for name, v in times.items()}
    check()
    st = f.stats()
    del d_kmers, d_codes, d_q, d_qoff
    torch.cuda.empty_cache()
    # host form, pinned buffers
    pin_b, pin_o = C.c_void_p(), C.c_void_p()
    api._check(L.lphb_host_alloc(C.byref(pin_b), len(bases)))
    api._check(L.lphb_host_alloc(C.byref(pin_o), len(offsets) * 8))
    try:
        np.frombuffer((C.c_uint8 * len(bases)).from_address(pin_b.value), dtype=np.uint8)[:] = bases
        np.frombuffer((C.c_uint64 * len(offsets)).from_address(pin_o.value), dtype=np.uint64)[:] = offsets
        secs = []
        for _ in range(4):
            t0 = time.perf_counter()
            api._check(L.lphb_check_begin(f._h))
            api._check(L.lphb_check_batch(f._h, pin_b, pin_o, len(offsets) - 1))
            r = api.CheckReport()
            api._check(L.lphb_check_end(f._h, C.byref(r)))
            secs.append(time.perf_counter() - t0)
            assert r.ok == 1 and r.kmers == n
        host_ms = 1e3 * float(np.median(secs[1:]))
    finally:
        L.lphb_host_free(pin_b)
        L.lphb_host_free(pin_o)
    cpu = cpu_figure(bases, offsets, lph, k, bits, n)
    row = {"row": f"check_{label}", "metric": "check session ms (device-resident contigs: begin, batch, end)",
           "value": ms["check"], "unit": "ms", "kmers": n, "k": k, "m": m, "kmer_bits": bits,
           "contigs": len(offsets) - 1, "bitmap_bytes": (n + 31) // 32 * 4, "rounds": rounds,
           "device_ms_median": ms, "device_ms_min_max": spread,
           "kmers_per_s": {name: n / (v * 1e-3) for name, v in ms.items()},
           "stats_last_check": {"kernel_launches": int(st.kernel_launches)},
           "host_form_pinned_ms": host_ms, "host_form_kmers_per_s": n / (host_ms * 1e-3),
           "verdicts": verdicts, "cpu_baseline": cpu, "machine": gpu}
    print(json.dumps(row), flush=True)
    f.close()
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--kmers", type=int, default=10**8, help="k-mers of each workload (default 1e8)")
    ap.add_argument("--rounds", type=int, default=15, help="timed rounds per device figure")
    ap.add_argument("--out", default=None, help="also write the rows to this JSONL file")
    args = ap.parse_args()
    import torch
    gpu = machine()
    rows = []
    bases, offsets, lph = B.make_workload(args.kmers)
    rows.append(run_workload(torch, "cfg2_k31_m20_u64", bases, offsets, lph, B.K, B.M, B.BITS, args.rounds, gpu))
    del bases, offsets
    bases, offsets, lph, k, m, bits = workload_k63(args.kmers)
    rows.append(run_workload(torch, "k63_m24_u128", bases, offsets, lph, k, m, bits, args.rounds, gpu))
    if args.out:
        with open(args.out, "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
