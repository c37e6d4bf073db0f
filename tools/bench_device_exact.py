#!/usr/bin/env python
"""Queries of batches already in device memory with the reference's answers, on one GPU: the exact streaming form,
synchronous (lphb_query_stream_exact_device) and asynchronous (lphb_query_stream_exact_device_async), beside the
stateless device form (lphb_query_stream_device) and the host form with pinned buffers (lphb_query_stream); the
non-streaming device form (lphb_query_nonstreaming_device) beside the non-streaming host form
(lphb_query_nonstreaming, pinned buffers).

Workloads: the bundled config-1 files ecoli1 (one 4.9 Mbase record with 50 runs of N) and srr (10,000 reads, 105 with
an N) against their k31 m16 index, ecoli1 with a scaffold gap of 10^7 N after its first 2 Mbases (gap_record: the
episode walk across a long gap), and two synthetic read sets of about 10^8 bases (synth.reads over the config-2
genome, bench.make_workload) against the config-2 index: one with an N planted at a seeded position of 1 % of the
reads, and the same reads without any (what a clean batch costs the exact forms).

Before anything is timed, every code of every form is compared with the host form's: the exact and the non-streaming
device forms in full, the stateless form on the contigs without a non-ACGT byte (its other slots are unspecified).

Per form: milliseconds per call and codes per second, and the launches of one call.  Device forms: CUDA events around `--calls` back-to-back calls
on one stream, and the wall time of the same calls ending in a device synchronise.  Host forms: wall time per call.
The figures are the median over `--rounds` rounds, the forms alternating inside each round; min and max give the
run-to-run spread.  One JSON line per workload, with the card's name and power limit.

--no-async leaves the asynchronous form out (a library without it).  --profile instead runs --calls calls of the
asynchronous form per workload under torch.profiler and reports each kernel's mean device time per call (the stages
of the repair), with no timing of the forms.

    python tools/bench_device_exact.py [--reads-bases N] [--calls C] [--rounds R] [--out rows.jsonl] [--no-async]
                                       [--profile]
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

CFG1 = os.path.join(ROOT, "tests", "golden", "config1")
SEED = 0xD1E7  # reads and the planted N


def machine():
    """name and power limit of the card, read with a query that changes nothing"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = (x.strip() for x in out[1].split(","))
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the row still stands; the machine is then unknown
        return {"gpu": None, "power_limit": None, "note": f"nvidia-smi: {e}"}


def planted_reads(genome, n_bases, read_len=150, frac=0.01):
    """synth.reads over `genome`, one N at a seeded position of `frac` of the reads (none for frac = 0)"""
    n_reads = n_bases // read_len
    bases, offsets = synth.reads(n_reads, genome, read_len=read_len, seed=SEED)
    if not frac:
        return bases, offsets
    rng = np.random.default_rng(SEED)
    hit = rng.choice(n_reads, size=max(1, int(n_reads * frac)), replace=False)
    bases[hit.astype(np.int64) * read_len + rng.integers(0, read_len, size=len(hit))] = ord("N")
    return bases, offsets


def gap_record(eco):
    """one record: ecoli1's first 2 Mbases, a scaffold gap of 10^7 N, 20 runs of 20 bases between runs of 5 N, then
    the rest of ecoli1 - the episode after the first 2 Mbases crosses the whole gap"""
    eco = eco.tobytes()
    short = b"".join(eco[2_000_000 + 25 * i:2_000_000 + 25 * i + 20] + b"NNNNN" for i in range(20))
    rec = eco[:2_000_000] + b"N" * 10**7 + short + eco[2_000_500:]
    return np.frombuffer(rec, dtype=np.uint8).copy(), np.array([0, len(rec)], dtype=np.uint64)


class Pinned:
    """a pinned host array (lphb_host_alloc)"""

    def __init__(self, L, n, dtype):
        self.L, self.p = L, C.c_void_p()
        nbytes = max(1, n * np.dtype(dtype).itemsize)
        api._check(L.lphb_host_alloc(C.byref(self.p), nbytes))
        self.a = np.frombuffer((C.c_uint8 * nbytes).from_address(self.p.value), dtype=dtype, count=n)

    def free(self):
        self.L.lphb_host_free(self.p)


def spread(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def run_workload(torch, label, bases, offsets, f, calls, rounds, gpu, with_async=True, profile=False):
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    L = api.lib()
    n_contigs = len(offsets) - 1
    lens = np.diff(offsets).astype(np.int64)
    clean_total = int(np.maximum(lens - f.k + 1, 0).sum())
    cap = int(np.maximum(lens - f.m + 1, 0).sum())
    # host forms with pinned buffers: the reference answers every device form is held to
    h_bases = Pinned(L, len(bases), np.uint8)
    h_bases.a[:] = bases
    h_codes = Pinned(L, max(cap, clean_total), np.uint64)
    h_code_off = np.empty(n_contigs + 1, dtype=np.uint64)
    n_out = C.c_uint64(0)

    def host_call(fn):
        api._check(fn(f._h, h_bases.p, offsets.ctypes.data, n_contigs, h_codes.p, len(h_codes.a),
                      h_code_off.ctypes.data, C.byref(n_out)))
        return n_out.value

    n_exact = host_call(L.lphb_query_stream)
    want, want_off = h_codes.a[:n_exact].copy(), h_code_off.copy()
    host_st = f.stats()
    n_ns = host_call(L.lphb_query_nonstreaming)
    want_ns, want_ns_off = h_codes.a[:n_ns].copy(), h_code_off.copy()
    dirty = np.zeros(n_contigs, dtype=bool)

    d_bases = torch.from_numpy(bases).to(dev)
    d_off = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    d_codes = torch.empty(max(cap, 1), dtype=torch.int64, device=dev)
    d_code_off = torch.empty(n_contigs + 1, dtype=torch.int64, device=dev)
    d_status = torch.zeros(4, dtype=torch.int64, device=dev)
    s = stream.cuda_stream
    args = (d_bases.data_ptr(), d_off.data_ptr(), offsets)

    def exact():
        return f.query_device_exact(*args, d_codes.data_ptr(), cap, d_code_off.data_ptr(), s)

    def exact_async():
        f.query_device_exact_async(*args, d_codes.data_ptr(), cap, d_code_off.data_ptr(), d_status.data_ptr(), s)

    def stateless():
        f.query_device(*args, d_codes.data_ptr(), cap, d_code_off.data_ptr(), d_status.data_ptr(), s)

    def nonstreaming():
        f.query_device_nonstreaming(*args, d_codes.data_ptr(), cap, d_code_off.data_ptr(), d_status.data_ptr(), s)

    def fetch(n):
        torch.cuda.synchronize()
        return d_codes[:n].cpu().numpy().view(np.uint64), d_code_off.cpu().numpy().view(np.uint64)

    # ---- parity, in full, before anything is timed
    torch.cuda.synchronize()
    n = exact()
    dirty[:] = f.dirty_flags() != 0
    exact_st = f.stats()
    got, got_off = fetch(n)
    parity = {"exact_equal_host": bool(n == n_exact and np.array_equal(got, want) and np.array_equal(got_off, want_off))}
    if with_async:
        d_codes.fill_(-1)
        exact_async()
        async_st = f.stats()
        got, got_off = fetch(n_exact)
        parity["exact_async_equal_host"] = bool(int(d_status[0]) == n_exact and int(d_status[1]) == int(dirty.sum())
                                                and np.array_equal(got, want) and np.array_equal(got_off, want_off))
    if profile:
        assert parity.get("exact_async_equal_host"), (label, parity)
        return profile_async(torch, label, exact_async, calls, f, gpu, int(async_st.kernel_launches))
    stateless()
    got, got_off = fetch(clean_total)
    assert int(d_status[0]) == clean_total and int(d_status[1]) == int(dirty.sum())
    # clean contigs have L-k+1 codes in both layouts: compare those slots
    cnt = np.maximum(lens - f.k + 1, 0)
    keep = np.repeat(~dirty, cnt)
    host_keep = np.repeat(~dirty, np.diff(want_off).astype(np.int64))
    parity["stateless_equal_host_on_clean_contigs"] = bool(np.array_equal(got[keep], want[host_keep]))
    parity["stateless_compared_codes"] = int(keep.sum())
    nonstreaming()
    got, got_off = fetch(clean_total)
    parity["nonstreaming_equal_host"] = bool(n_ns == clean_total and np.array_equal(got, want_ns)
                                             and np.array_equal(got_off, want_ns_off))
    assert all(v for k, v in parity.items() if k.endswith("host") or k.endswith("contigs")), (label, parity)

    # ---- timing: the forms alternate inside each round
    def device_ms(fn):
        fn()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(stream)
        for _ in range(calls):
            fn()
        ev1.record(stream)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3 / calls
        return ev0.elapsed_time(ev1) / calls, wall

    def host_ms(fn):
        host_call(fn)
        t0 = time.perf_counter()
        for _ in range(calls):
            host_call(fn)
        return (time.perf_counter() - t0) * 1e3 / calls

    forms = {"exact_device": lambda: device_ms(exact), "stateless_device": lambda: device_ms(stateless),
             "exact_async_device": lambda: device_ms(exact_async),
             "exact_host_pinned": lambda: (None, host_ms(L.lphb_query_stream)),
             "nonstreaming_device": lambda: device_ms(nonstreaming),
             "nonstreaming_host_pinned": lambda: (None, host_ms(L.lphb_query_nonstreaming))}
    if not with_async:
        del forms["exact_async_device"]
    ev = {k: [] for k in forms}
    wall = {k: [] for k in forms}
    launches = {}
    for _ in range(rounds):
        for name, fn in forms.items():
            e, w = fn()
            if e is not None:
                ev[name].append(e)
            wall[name].append(w)
            launches[name] = int(f.stats().kernel_launches)
    codes_of = {"exact_device": n_exact, "exact_async_device": n_exact, "stateless_device": clean_total,
                "exact_host_pinned": n_exact,
                "nonstreaming_device": clean_total, "nonstreaming_host_pinned": clean_total}
    out = {}
    for name in forms:
        r = {"wall_ms_per_call": spread(wall[name]),
             "codes_per_s_wall": codes_of[name] / (float(np.median(wall[name])) * 1e-3),
             "kernel_launches": launches[name]}
        if ev[name]:
            r["event_ms_per_call"] = spread(ev[name])
            r["codes_per_s_events"] = codes_of[name] / (float(np.median(ev[name])) * 1e-3)
        out[name] = r
    h_bases.free()
    h_codes.free()
    row = {"row": f"device_exact_{label}", "contigs": n_contigs, "bases": int(len(bases)), "kmers": clean_total,
           "codes_exact": n_exact, "dirty_contigs": int(dirty.sum()), "k": f.k, "m": f.m, "kmer_bits": f.kmer_bits,
           "calls_per_round": calls, "rounds": rounds, "forms": out, "parity": parity,
           "stats_exact_device": {"d2h_bytes": int(exact_st.d2h_bytes), "h2d_bytes": int(exact_st.h2d_bytes),
                                  "kernel_launches": int(exact_st.kernel_launches)},
           "stats_exact_host": {"d2h_bytes": int(host_st.d2h_bytes), "h2d_bytes": int(host_st.h2d_bytes),
                                "kernel_launches": int(host_st.kernel_launches)},
           "machine": gpu}
    print(json.dumps(row), flush=True)
    return row


def profile_async(torch, label, fn, calls, f, gpu, launches):
    """per kernel of the asynchronous form: mean device time per call under torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t:
            kernels[e.key[:160]] = {"us_per_call": t / calls, "launches_per_call": e.count / calls}
    row = {"row": f"device_exact_async_stages_{label}", "calls": calls, "kernel_launches": launches,
           "us_per_call_sum": sum(v["us_per_call"] for v in kernels.values()), "kernels": kernels, "machine": gpu}
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads-bases", type=int, default=10**8, help="bases of the synthetic read set (default 1e8)")
    ap.add_argument("--kmers", type=int, default=10**8, help="k-mers of the config-2 index the reads are drawn from")
    ap.add_argument("--calls", type=int, default=20, help="calls per form and round (>= 5)")
    ap.add_argument("--rounds", type=int, default=5, help="rounds (>= 3)")
    ap.add_argument("--out", default=None, help="also write the rows to this JSONL file")
    ap.add_argument("--no-async", action="store_true", help="leave out lphb_query_stream_exact_device_async")
    ap.add_argument("--profile", action="store_true", help="per-kernel device time of the asynchronous form only")
    args = ap.parse_args()
    if args.calls < 5 or args.rounds < 3:
        ap.error("--calls must be at least 5 and --rounds at least 3")
    if args.profile and args.no_async:
        ap.error("--profile times the asynchronous form")
    import torch
    gpu = machine()
    opts = (not args.no_async, args.profile)
    rows = []
    exp = json.load(open(os.path.join(CFG1, "expected.json")))["queries"]
    f = api.Mphf.load(os.path.join(CFG1, "se.ust.k31_m16_u128.lph"), 128)
    for name in ("ecoli1", "srr"):
        bases, offsets = seqio.read_batch(os.path.join(CFG1, exp[name]["file"]))
        rows.append(run_workload(torch, "cfg1_" + name, bases, offsets, f, args.calls, args.rounds, gpu, *opts))
    bases, offsets = gap_record(seqio.read_batch(os.path.join(CFG1, exp["ecoli1"]["file"]))[0])
    rows.append(run_workload(torch, "cfg1_ecoli1_gap10M", bases, offsets, f, args.calls, args.rounds, gpu, *opts))
    f.close()
    genome, _, lph = B.make_workload(args.kmers)
    bases, offsets = planted_reads(genome, args.reads_bases)
    f = api.Mphf.load(lph, B.BITS)
    rows.append(run_workload(torch, "reads_1pct_N", bases, offsets, f, args.calls, args.rounds, gpu, *opts))
    bases, offsets = planted_reads(genome, args.reads_bases, frac=0)
    rows.append(run_workload(torch, "reads_clean", bases, offsets, f, args.calls, args.rounds, gpu, *opts))
    f.close()
    if args.out:
        with open(args.out, "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
