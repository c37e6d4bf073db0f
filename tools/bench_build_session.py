#!/usr/bin/env python
"""What a build session (lphb_build_*: Parts 1 + 2 of build-p fed batch by batch) costs against one lphb_scan_classify
call over the same input, and a session past 2^32 k-mers, where one call cannot go.

Workload 1: config 2 (synth.unitigs, 1e8 k-mers, k=31 m=20, the unitigs bench.py indexes).  Rows: one
lphb_scan_classify over all contigs, then sessions of 1, 4, 16 and 64 batches of about equal bases, in host form
(lphb_build_batch from the same numpy arrays) and in device form (lphb_build_batch_device over contigs already in HBM).
Wall-clock medians over the rounds (every call is synchronous); the end phase (merge + copy-out of triplets and ids)
is timed on its own.  Before anything is timed, every session's triplets and ids are compared in full with the single
call's.

Workload 2: 17 batches of 2^28 random bases (one contig each, k=31 m=20), host form: 4.6e9 k-mers and m-mer ordinals
past 2^32.  One run: k-mers/s over the batches, the end phase, the session's device bytes at its end (its peak: every
summary and the merged result are held then).  The card's name and power limit go with every row.

    python tools/bench_build_session.py [--kmers N] [--rounds R] [--out rows.jsonl]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_lookup import machine  # noqa: E402
from lphash_b200 import api, synth  # noqa: E402

K, M, SEED = 31, 20, 42


def cut(offsets, n_batches):
    """contig ranges [a, b) of n_batches batches of about equal bases"""
    n = len(offsets) - 1
    targets = np.linspace(0, int(offsets[-1]), n_batches + 1)[1:-1]
    cuts = np.searchsorted(offsets[1:], targets).tolist()
    edges = [0] + [min(max(c, 0), n) for c in cuts] + [n]
    return list(zip(edges[:-1], edges[1:]))


def session(ranges, add, k=K, m=M):
    """returns (triplets, ids, report, batches_s, end_s)"""
    t0 = time.perf_counter()
    s = api.BuildSession(k, m, SEED)
    for a, b in ranges:
        add(s, a, b)
    t1 = time.perf_counter()
    trip, ids, rep = s.end()
    t2 = time.perf_counter()
    s.close()
    return trip, ids, rep, t1 - t0, t2 - t1


def config2(torch, n_kmers, rounds, gpu):
    bases, offsets = synth.unitigs(n_kmers, K, M)
    n = int(np.maximum(np.diff(offsets).astype(np.int64) - K + 1, 0).sum())
    d_bases = torch.from_numpy(bases).cuda()
    d_off = torch.from_numpy(offsets.astype(np.int64)).cuda()
    torch.cuda.synchronize()

    def single():
        t0 = time.perf_counter()
        r = api.scan_classify(bases, offsets, K, M, SEED)
        return r, time.perf_counter() - t0

    def host_add(s, a, b):
        s.batch(bases, offsets[a:b + 1])

    def device_add(s, a, b):
        s.batch_device(d_bases.data_ptr(), d_off.data_ptr() + 8 * a, offsets[a:b + 1])

    (wtrip, wids, wnk, wmm), _ = single()  # warm-up and the reference result
    legs = {"single_call": None}
    for nb in (1, 4, 16, 64):
        for form, add in (("host", host_add), ("device", device_add)):
            legs[f"session_{nb}_{form}"] = (cut(offsets, nb), add)
    verified = {}
    for name, leg in legs.items():  # every session's result, in full, before any timing
        if leg is None:
            continue
        trip, ids, rep, _, _ = session(*leg)
        ok = np.array_equal(trip, wtrip) and np.array_equal(ids, wids) and (rep.kmers, rep.mm_count) == (wnk, wmm)
        assert ok, name
        verified[name] = {"batches": int(rep.batches), "device_bytes": int(rep.device_bytes)}
    times = {name: [] for name in legs}
    ends = {name: [] for name in legs}
    for _ in range(rounds):
        for name, leg in legs.items():
            if leg is None:
                times[name].append(single()[1])
                continue
            _, _, _, tb, te = session(*leg)
            times[name].append(tb + te)
            ends[name].append(te)
    single_ms = 1e3 * float(np.median(times["single_call"]))
    rows = []
    for name in legs:
        ms = 1e3 * float(np.median(times[name]))
        row = {"row": f"build_session_cfg2_{name}", "metric": "wall ms of Parts 1 + 2 (scan + classify, result in host "
               "memory)", "value": ms, "unit": "ms", "kmers": n, "k": K, "m": M, "contigs": len(offsets) - 1,
               "triplets": len(wtrip), "ids": len(wids), "rounds": rounds,
               "ms_min_max": [1e3 * min(times[name]), 1e3 * max(times[name])],
               "kmers_per_s": n / (ms * 1e-3), "vs_single_call": ms / single_ms, "machine": gpu}
        if name in verified:
            row.update(end_ms=1e3 * float(np.median(ends[name])), **verified[name])
        print(json.dumps(row), flush=True)
        rows.append(row)
    del d_bases, d_off
    torch.cuda.empty_cache()
    return rows


def past_2_32(gpu, reps=17, n_bases=1 << 28):
    rng = np.random.default_rng(7)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    batches = [acgt[rng.integers(0, 4, n_bases, dtype=np.uint8)] for _ in range(reps)]
    offsets = np.array([0, n_bases], dtype=np.uint64)
    trip, ids, rep, tb, te = session([(j, j + 1) for j in range(reps)], lambda s, a, b: s.batch(batches[a], offsets))
    assert rep.kmers == reps * (n_bases - K + 1) > 1 << 32 and rep.mm_count > 1 << 32
    assert len(trip) == rep.n_triplets and np.all(np.diff(trip["itself"].astype(np.uint64)) > 0)
    assert len(ids) == rep.n_ids and np.all(np.diff(ids) > 0)
    row = {"row": "build_session_past_2_32", "metric": "k-mers/s of a host-form session (batches + end)",
           "value": rep.kmers / (tb + te), "unit": "k-mers/s", "kmers": int(rep.kmers), "mm_count": int(rep.mm_count),
           "k": K, "m": M, "batches": reps, "bases_per_batch": n_bases, "records": int(rep.records),
           "triplets": int(rep.n_triplets), "ids": int(rep.n_ids), "batches_s": tb, "end_s": te,
           "peak_device_bytes": int(rep.device_bytes), "machine": gpu}
    print(json.dumps(row), flush=True)
    return [row]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--kmers", type=int, default=10**8, help="k-mers of the config-2 workload (default 1e8)")
    ap.add_argument("--rounds", type=int, default=5, help="timed rounds per config-2 row")
    ap.add_argument("--out", default=None, help="also write the rows to this JSONL file")
    args = ap.parse_args()
    import torch
    gpu = machine()
    rows = config2(torch, args.kmers, args.rounds, gpu)
    rows += past_2_32(gpu)
    if args.out:
        with open(args.out, "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
