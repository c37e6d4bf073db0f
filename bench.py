#!/usr/bin/env python
"""bench.py — streaming query-p throughput of the B200-native LPHash hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg5]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): query-p k-mers/sec (k=31); one "step" = one streaming query pass of the hot path
over the workload's synthetic input.

  one GPU (default)   BASELINE config 2, the configuration the metric is quoted on: synthetic random-genome
                      unitigs, ~1e8 k-mers, k=31 m=20, 64-bit kmer_t, all member k-mers (under torchrun with
                      --workload cfg2: the same-size shard rotated by r contigs per rank, weak scaling).  The
                      line also carries `config5_1gpu`: the reads shape of config 5 on this GPU (8 slabs).
  torchrun, N > 1     BASELINE config 5: 64 slabs x 2^20 reads of 150 bases (1.0066e10 bases; half substrings
                      of the index sequence with 1 % substitutions, half random), generated on the device slab
                      by slab; the slabs are split over the ranks by contiguous range (STRONG scaling: the job
                      is fixed), replicated index, no data-path collective.
The `.lph` index is input preparation outside every timed region: Parts 1-4 of build-p through this library and the
two PTHash functions from a plain pilot search (oracle/phf.py; c=3.0, alpha=0.94), cached in a per-user directory
under the system's temporary directory ($TMPDIR/lphash_b200_bench_<uid>), never in the tree.  Its pilots differ from
those the reference's build-p picks, so the codes are a different (equally valid) minimal perfect hash of the same
k-mers.

Before anything is timed the codes are checked: config 2 - the permutation property, and where the reference library
(oracle/_ref) is built, every one of the 1e8 codes against the reference's answers on the same index; config 5 - every
code of each rank's first slab against the reference's, where it is built.

--dump-outputs DIR (rank 0) writes what the last timed step returned, as float64 .npy files: the codes at a fixed seeded
sample of about 2 M positions (low and high 32 bits in codes_lo / codes_hi, exact; the positions in codes_index), the
code offsets and the status words.  Inputs are a pure function of the arguments, so two builds can be compared file
by file.

--steps K sets the timed steps of every throughput figure (value, config5_1gpu); the host-buffer legs (e2e) are
separate, shorter measurements of min(K, 5) passes (config 5: 2, its one-GPU side line: 1).

Printed JSON (one line, rank 0):
  value      whole-job k-mers/s, inputs resident in HBM, CUDA-event time, max over ranks
  e2e        same metric through lphb_query_stream with pinned HOST buffers (H2D + kernels + D2H of 8 B per
             k-mer); e2e.runs_form: through lphb_query_stream_runs (run records, ~2 B per k-mer back);
             e2e.copy_only_ceiling: the same bytes as plain copies, i.e. what PCIe / host memory allow
  roofline   dominant kernel: algorithmic bytes (L bases in + 8 B per code out) / its launch time
             vs the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the unmodified reference (oracle/_ref) on the host cores, bounded sample (one GPU only)
--impl reference: times the reference's own CPU implementation (all host threads), same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K, M, BITS = 31, 20, 64
INDEX_FORMAT = 1  # part of the cached index's name: bump when oracle/phf.py or the .lph writer changes what it holds


def cache_dir() -> str:
    """This user's directory under the system's temporary directory (the tree may be read-only); a fresh private one
    when that name is taken by someone else or not writable."""
    d = os.path.join(tempfile.gettempdir(), f"lphash_b200_bench_{os.getuid()}")
    try:
        os.makedirs(d, mode=0o700, exist_ok=True)
        if os.stat(d).st_uid == os.getuid() and os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    return tempfile.mkdtemp(prefix="lphash_b200_bench_")


CACHE = cache_dir()


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------
# workload
# ---------------------------------------------------------------------------------------------

def make_workload(n_kmers: int):
    """Config-2 unitigs + their index (cached).  Returns (bases, offsets, lph)."""
    from lphash_b200 import synth
    os.makedirs(CACHE, exist_ok=True)
    lph = index_path(n_kmers)
    t0 = time.time()
    bases, offsets = synth.unitigs(n_kmers, K, M)
    log(f"[bench] synthetic unitigs: {len(offsets) - 1} contigs, {len(bases)} bases ({time.time() - t0:.1f}s)")
    if not os.path.exists(lph):
        from oracle import phf
        t0 = time.time()
        image = phf.build_lph(bases, offsets, K, M, kmer_bits=BITS, device=int(os.environ.get("LOCAL_RANK", "0")))
        tmp = f"{lph}.{os.getpid()}.tmp"
        with open(tmp, "wb") as out:
            out.write(image)
        os.replace(tmp, lph)
        log(f"[bench] index built: {len(image)} bytes ({time.time() - t0:.1f}s)")
    return bases, offsets, lph


def host_threads() -> int:
    """Cores this process may run on (a container's cpuset can be far smaller than os.cpu_count())."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def bind_near_gpu(index: int):
    """Restricts this rank to the cores of the NUMA node its GPU hangs off, before any pinned buffer exists: the
    staging buffers of the end-to-end legs are then node-local (first touch), and the 8 ranks of a box stop
    pulling each other's traffic across the socket link.  Returns a description for the JSON line."""
    try:
        import torch
        p = torch.cuda.get_device_properties(index)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"node": None, "note": "single NUMA node"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return {"node": node, "note": "no allowed core on the GPU's node; affinity left as is"}
        os.sched_setaffinity(0, allowed)
        return {"node": node, "cores": len(allowed)}
    except Exception as e:  # best effort: the bench runs without it
        return {"node": None, "note": f"not bound ({e})"}


def index_path(n_kmers: int) -> str:
    return os.path.join(CACHE, f"cfg2_n{n_kmers}_k{K}_m{M}_u{BITS}_index{INDEX_FORMAT}.lph")


def rotate_contigs(bases, offsets, r: int):
    """Shard r: the same contigs rotated by r positions (same size, different order)."""
    n = len(offsets) - 1
    if r % n == 0:
        return bases, offsets
    r = r % n
    cut = int(offsets[r])
    nb = np.concatenate([bases[cut:], bases[:cut]])
    lens = np.diff(offsets)
    lens = np.concatenate([lens[r:], lens[:r]])
    no = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=no[1:])
    return nb, no


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------

class ClockSampler:
    """SM clock + clock-event reasons of one GPU, polled through NVML from a thread every ~1 ms
    while the timed region runs (the region is tens of ms: `nvidia-smi -lms` is too coarse)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.index = index
        self.sm, self.bits = [], 0
        self.max_sm = None
        self._stop = threading.Event()
        self._thr = None
        self._h = None
        self._nv = None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self._nv = nv
            self._h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = int(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM))
        except Exception as e:  # no NVML: report no samples rather than fail the bench
            log(f"[bench] NVML unavailable: {e}")
            self._h = None
            return
        self._thr = threading.Thread(target=self._poll, daemon=True)
        self._thr.start()

    def _poll(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except AttributeError:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
            except Exception:
                pass
            time.sleep(0.001)

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=2)
        reasons = sorted(name for bit, name in self.REASONS.items() if self.bits & bit)
        return {"sm_mhz": int(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": reasons, "samples": len(self.sm)}


# ---------------------------------------------------------------------------------------------
# config 5: short reads (mixed member / non-member k-mers), generated slab by slab
# ---------------------------------------------------------------------------------------------

READ_LEN = 150
SLAB_READS = 1 << 20            # reads per slab: 157,286,400 bases, 125,829,120 k-mers (k = 31)
CFG5_SLABS = 64                 # 64 slabs = 1.0066e10 bases (BASELINE config 5: >= 10 Gbases)
CFG5_SEED = 0x5EED0005
INDEX_NOTE = ("build-p Parts 1-4 through this library, PTHash functions from oracle/phf.py's pilot search "
              "(c=3.0, alpha=0.94, seeds 42 / 1)")


def reads_slab_device(genome_dev, slab: int, dev):
    """Slab `slab` of the config-5 read set, generated ON THE DEVICE (a pure function of the slab index,
    so every world size sees the same 64 slabs): each read is, with probability 0.5, a 150-base
    substring of the index's sequence with 1 % i.i.d. substitutions (member k-mers cut by mismatches),
    else uniform random (non-members); ACGT only (lphash_b200/synth.py: reads, same distribution)."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(CFG5_SEED + slab)
    R, L = SLAB_READS, READ_LEN
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    out = acgt[torch.randint(0, 4, (R, L), generator=g, device=dev)]
    member = torch.rand(R, generator=g, device=dev) < 0.5
    st = torch.randint(0, genome_dev.numel() - L, (R,), generator=g, device=dev)
    half = R // 4
    for s in range(0, R, half):  # in four parts: the gather index of a whole slab would take 1.3 GB
        idx = st[s:s + half, None] + torch.arange(L, device=dev)[None, :]
        sub = genome_dev[idx].to(torch.int64)
        code = ((sub >> 1) ^ (sub >> 2)) & 3  # A0 C1 G2 T3
        mut = torch.rand((idx.shape[0], L), generator=g, device=dev) < 0.01
        code = torch.where(mut, (code + torch.randint(1, 4, code.shape, generator=g, device=dev)) & 3, code)
        # ACGT by code: A C G T
        by_code = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=dev)
        part = by_code[code]
        m = member[s:s + half, None]
        out[s:s + half] = torch.where(m, part, out[s:s + half])
    return out.reshape(-1)


def cfg5_config(world, slabs_total, n_kmers_total, n_bases_total):
    return {"workload": f"BASELINE config 5: {slabs_total} slabs x {SLAB_READS} synthetic reads of {READ_LEN} bases "
                        f"({n_bases_total} bases, {n_kmers_total} k-mers; half substrings of the index sequence with 1% "
                        f"substitutions, half random), index of config 2 (k={K} m={M}, 1e8 k-mers), streaming query-p, "
                        f"slabs split over {world} GPU(s) by contiguous range",
            "k": K, "m": M, "kmer_bits": BITS, "slabs": slabs_total, "reads_per_slab": SLAB_READS, "read_len": READ_LEN,
            "cache": "per-launch working set (157 MB bases in + 1.0 GB codes out) >> 126 MB L2; no flush needed",
            "index": INDEX_NOTE,
            "sharding": "replicated index, contiguous slab range per rank, no data-path collective"}


# ---------------------------------------------------------------------------------------------
# reference / CPU baseline
# ---------------------------------------------------------------------------------------------

def cpu_reference_run(bases, offsets, lph, steps: int, warmup: int, threads: int):
    """Times the unmodified reference's streaming query (oracle/_ref, `threads` host threads)."""
    from oracle import ref
    f = ref.RefMphf(lph, BITS)
    times, total = [], 0
    for it in range(warmup + steps):
        secs, n, _, _ = f.query_batch(bases, offsets, threads=threads, want_codes=False)
        if it >= warmup:
            times.append(secs)
            total = n
    f.close()
    return total, times


def cpu_reference_codes(bases, offsets, lph, threads: int):
    """Codes of a clean batch from the unmodified reference (the checker of the full-size compare)."""
    from oracle import ref
    f = ref.RefMphf(lph, BITS)
    _, n, codes, code_off = f.query_batch(bases, offsets, threads=threads, want_codes=True, k=K)
    f.close()
    return codes


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    bases, offsets, lph = make_workload(args.kmers)
    threads = host_threads()
    workload = args.workload or ("cfg2" if world == 1 else "cfg5")
    if workload == "cfg2":
        # bounded sample: the full config-2 set is ~4 thread-seconds of CPU work per pass
        n, times = cpu_reference_run(bases, offsets, lph, args.steps, min(args.warmup, 1), threads)
        config = workload_config(args.kmers, n)
        sample = (f"full workload ({n} k-mers) per step, in-memory records, {threads} std::threads over "
                  f"disjoint contig ranges")
        scaling = "weak"
    else:
        from lphash_b200 import synth
        rb, ro = synth.reads(SLAB_READS, bases, read_len=READ_LEN, seed=CFG5_SEED)
        n, times = cpu_reference_run(rb, ro, lph, args.steps, min(args.warmup, 1), threads)
        total_k = CFG5_SLABS * SLAB_READS * (READ_LEN - K + 1)
        config = cfg5_config(world, CFG5_SLABS, total_k, CFG5_SLABS * SLAB_READS * READ_LEN)
        sample = (f"one slab of the read set ({n} k-mers of {total_k}) per step, in-memory records, {threads} "
                  f"std::threads over disjoint read ranges")
        scaling = "strong"
    t = float(np.sum(times))
    value = n * len(times) / t
    line = {"impl": "reference", "metric": "query-p k-mers/sec (k=31)", "value": value,
            "unit": "k-mers/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t / len(times), "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": "k-mers/s", "cores": threads, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_line(line)


def workload_config(n_kmers_requested, n_kmers):
    return {"workload": f"BASELINE config 2: synthetic random-genome unitigs, {n_kmers} k-mers per "
                        f"rank, k={K} m={M}, 64-bit kmer_t, all members, streaming query-p",
            "k": K, "m": M, "kmer_bits": BITS, "kmers_per_rank": int(n_kmers),
            "cache": "per-step working set (bases in + 8 B codes out) ~0.9 GB >> 126 MB L2; no flush needed",
            "index": INDEX_NOTE, "sharding": "replicated index, "
            "same-size contig-rotated shard per rank, no collective"}


# ---------------------------------------------------------------------------------------------
# ours
# ---------------------------------------------------------------------------------------------

def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def roofline(algo_bytes, kern_ms, n_kmers, kernel_name):
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None  # dram bytes read + written by the dominant kernel, from the committed ncu capture
    src = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tr.get("kmers_per_launch") == n_kmers:
            traffic = int(tr["dram_bytes_read"]) + int(tr["dram_bytes_write"])
            src = tr.get("source", "profiles/traffic.json (ncu --set full, one launch)")
    except Exception:
        pass
    achieved = algo_bytes / (kern_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "kernel": kernel_name, "traffic_source": src,
            "algorithmic_bytes_per_launch": int(algo_bytes), "kernel_ms": kern_ms,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
            "input_only_frac": (algo_bytes - 8 * n_kmers) / (kern_ms * 1e-3) / 1e9 / peak}


DUMP_SAMPLE = 2 << 20  # positions drawn per output by --dump-outputs (3 float64 arrays of this size: <= 48 MB)


def snapshot_outputs(torch, args, codes_list, code_off, status):
    """What the last timed step returned, taken on the device right after the timed region: the codes of each output
    buffer at one fixed seeded sample of positions, the code offsets and the status words.  None without
    --dump-outputs."""
    if not args.dump_outputs:
        return None
    n = codes_list[0].numel()
    idx = np.unique(np.random.default_rng(0xD0).integers(0, n, size=min(n, DUMP_SAMPLE // len(codes_list))))
    ti = torch.from_numpy(idx.astype(np.int64)).to(codes_list[0].device)
    codes = torch.stack([c.index_select(0, ti) for c in codes_list]).cpu().numpy().view(np.uint64)
    if len(codes_list) == 1:
        codes = codes[0]
    # codes of non-member k-mers can use all 64 bits: two exact float64 halves
    return {"codes_lo": codes & np.uint64(0xFFFFFFFF), "codes_hi": codes >> np.uint64(32), "codes_index": idx,
            "code_offsets": code_off.cpu().numpy(), "status": status.cpu().numpy()}


def write_outputs(path, outputs):
    if outputs is None:
        return
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a).astype(np.float64))
    log(f"[bench] outputs of the last timed step written to {path}: {', '.join(sorted(outputs))}")


class HostBatch:
    """Pinned host buffers of one batch for the end-to-end calls (inputs copied H2D and results D2H
    inside every timed call)."""

    def __init__(self, torch, bases_np, offsets_np, n_kmers):
        self.bases = torch.from_numpy(np.ascontiguousarray(bases_np)).pin_memory()
        self.offsets = np.ascontiguousarray(offsets_np, dtype=np.uint64)
        self.n_contigs = len(self.offsets) - 1
        self.n_kmers = n_kmers


def e2e_measure(torch, L, f, batches, n_kmers_max, steps, sync_all, check_codes=None):
    """Same metric through the C ABI with HOST buffers, both output forms.  Returns a dict."""
    h_codes = torch.empty(n_kmers_max, dtype=torch.int64).pin_memory()
    run_cap = n_kmers_max // 2 + 1024   # records (12 B each): 6 B per k-mer of pinned capacity
    h_runs = torch.empty(run_cap * 12, dtype=torch.uint8).pin_memory()
    h_code_off = np.empty(max(b.n_contigs for b in batches) + 1, dtype=np.uint64)
    total, n_runs = C.c_uint64(0), C.c_uint64(0)
    out = {}

    def codes_step():
        for b in batches:
            rc = L.lphb_query_stream(f._h, b.bases.data_ptr(), b.offsets.ctypes.data, b.n_contigs,
                                     h_codes.data_ptr(), n_kmers_max, h_code_off.ctypes.data, C.byref(total))
            assert rc == 0 and total.value == b.n_kmers, (rc, L.lphb_last_error())

    def runs_step():
        for b in batches:
            rc = L.lphb_query_stream_runs(f._h, b.bases.data_ptr(), b.offsets.ctypes.data, b.n_contigs,
                                          h_runs.data_ptr(), run_cap, C.byref(n_runs), h_code_off.ctypes.data,
                                          C.byref(total))
            assert rc == 0 and total.value == b.n_kmers, (rc, L.lphb_last_error())

    kmers = sum(b.n_kmers for b in batches)
    for name, step in (("codes", codes_step), ("runs", runs_step)):
        step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        st = f.stats()
        out[name] = {"secs": secs, "kmers": kmers * steps, "h2d": int(st.h2d_bytes), "d2h": int(st.d2h_bytes)}
        if name == "codes" and check_codes is not None:
            assert np.array_equal(h_codes.numpy()[: batches[-1].n_kmers].view(np.uint64), check_codes), \
                "e2e codes differ from the device-resident codes"
        if name == "runs":
            # the run records of the last batch expand to exactly the codes of the 8-byte form
            got = np.empty(batches[-1].n_kmers, dtype=np.uint64)
            n = C.c_uint64(0)
            t0 = time.perf_counter()
            rc = L.lphb_expand_runs(h_runs.data_ptr(), n_runs.value, got.ctypes.data, len(got), C.byref(n), host_threads())
            out["expand_secs"] = time.perf_counter() - t0
            out["expand_kmers"] = int(n.value)
            assert rc == 0 and n.value == batches[-1].n_kmers
            assert np.array_equal(got, h_codes.numpy()[: len(got)].view(np.uint64)), "expanded runs differ from the codes"
            out["runs_bytes_per_kmer"] = 12.0 * n_runs.value / batches[-1].n_kmers
    # copy-only ceiling: the same H2D / D2H bytes with no kernel in between (what PCIe + host memory allow)
    dev_in = torch.empty(max(b.bases.numel() for b in batches), dtype=torch.uint8, device="cuda")
    dev_out = torch.empty(n_kmers_max, dtype=torch.int64, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for form, d2h_elems in (("codes", None), ("runs", out["runs"]["d2h"] // 8)):
        sync_all()
        t0 = time.perf_counter()
        for _ in range(steps):
            for b in batches:
                with torch.cuda.stream(s1):
                    dev_in[: b.bases.numel()].copy_(b.bases, non_blocking=True)
                with torch.cuda.stream(s2):
                    n = b.n_kmers if d2h_elems is None else min(d2h_elems, b.n_kmers)
                    h_codes[:n].copy_(dev_out[:n], non_blocking=True)
        torch.cuda.synchronize()
        out["copy_only_" + form] = {"secs": time.perf_counter() - t0, "kmers": kmers * steps}
    return out


def e2e_object(world, parts, api_note):
    """Aggregates the per-rank e2e measurements (already max-reduced seconds) into the JSON object."""
    o = {"value": parts["codes_kmers"] / parts["codes_secs"], "unit": "k-mers/s",
         "h2d_bytes_per_step": parts["h2d_codes"], "d2h_bytes_per_step": parts["d2h_codes"], "steps": parts["steps"],
         "api": "lphb_query_stream (pinned host buffers, 8 B per k-mer back)" + api_note,
         "runs_form": {"value": parts["runs_kmers"] / parts["runs_secs"], "unit": "k-mers/s",
                       "h2d_bytes_per_step": parts["h2d_runs"], "d2h_bytes_per_step": parts["d2h_runs"],
                       "bytes_per_kmer_back": parts["runs_bpk"],
                       "api": "lphb_query_stream_runs (12-byte run records back; lphb_expand_runs on the host rebuilds the "
                              "identical uint64 vector, checked)",
                       "host_expand_kmers_per_s": parts["expand_rate"]},
         "copy_only_ceiling": {"codes_form": parts["codes_kmers"] / parts["copy_codes_secs"],
                               "runs_form": parts["runs_kmers"] / parts["copy_runs_secs"], "unit": "k-mers/s",
                               "what": "the same H2D and D2H bytes per step as plain cudaMemcpyAsync on two streams, no "
                                       "kernel: the PCIe / host-memory limit of this box for this many ranks"}}
    return o


def run_ours(args):
    import torch
    import torch.distributed as dist

    from lphash_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    workload = args.workload or ("cfg2" if world == 1 else "cfg5")
    # Input preparation comes before any collective: if the index is not cached yet, rank 0 builds it
    # while the other ranks wait on the FILE, not inside an NCCL barrier (whose watchdog would fire
    # during a long build).
    if rank != 0:
        t_wait = time.time()
        while not os.path.exists(index_path(args.kmers)):
            if time.time() - t_wait > 7200:
                raise RuntimeError("rank 0 did not produce the index within 2 h")
            time.sleep(1.0)
    bases, offsets, lph = make_workload(args.kmers)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"),
                                timeout=datetime.timedelta(minutes=30))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    all_cores = os.sched_getaffinity(0)
    threads = len(all_cores)  # the CPU legs use every core the process may run on (affinity restored below)
    numa = bind_near_gpu(local) if not os.environ.get("LPHB_BENCH_NO_NUMA") else {"node": None, "note": "disabled"}
    f = api.Mphf.load(lph, BITS, device=local)
    stream = torch.cuda.Stream(device=dev)  # a real stream: the handle attaches its L2 access-policy window to it
    torch.cuda.set_stream(stream)
    L = api.lib()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    nocheck = bool(os.environ.get("LPHB_BENCH_NOCHECK"))  # kernel-timing experiments with wrong codes only

    if workload == "cfg2":
        line = bench_cfg2(args, torch, dist, api, L, f, dev, stream, rank, world, bases, offsets, lph, sync_all,
                          sampler, nocheck, threads)
        if rank == 0 and world == 1 and not args.no_cfg5:
            # the reads shape of config 5 on this one GPU (8 slabs), beside the headline line
            try:
                line["config5_1gpu"] = bench_cfg5(args, torch, dist, api, L, f, dev, stream, rank, world, bases, lph,
                                                  sync_all, None, nocheck, threads, slabs_total=8, brief=True)
            except Exception as e:
                line["config5_1gpu"] = {"unavailable": str(e)}
    else:
        line = bench_cfg5(args, torch, dist, api, L, f, dev, stream, rank, world, bases, lph, sync_all, sampler,
                          nocheck, threads, slabs_total=args.slabs, brief=False)
    if rank == 0:
        line["config"]["host_numa"] = numa
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cores)
            try:
                if workload == "cfg2":
                    n, times = cpu_reference_run(bases, offsets, lph, steps=3, warmup=1, threads=threads)
                    sample = (f"full workload ({n} k-mers) x3 passes, unmodified reference operator() from {threads} "
                              f"std::threads, records in memory")
                else:
                    from lphash_b200 import synth
                    rb, ro = synth.reads(SLAB_READS, bases, read_len=READ_LEN, seed=CFG5_SEED)
                    n, times = cpu_reference_run(rb, ro, lph, steps=3, warmup=1, threads=threads)
                    sample = (f"one slab ({n} k-mers) x3 passes, unmodified reference operator() from {threads} "
                              f"std::threads, records in memory")
                line["cpu_baseline"] = {"value": n * len(times) / float(np.sum(times)), "unit": "k-mers/s",
                                        "cores": threads, "kind": "reference", "sample": sample}
            except Exception as e:  # the GPU result stands even if the reference .so is absent
                line["cpu_baseline"] = {"unavailable": str(e)}
        emit_line(line)
    f.close()
    if world > 1:
        dist.destroy_process_group()


def bench_cfg2(args, torch, dist, api, L, f, dev, stream, rank, world, bases, offsets, lph, sync_all, sampler,
               nocheck, threads):
    bases, offsets = rotate_contigs(bases, offsets, rank)
    n_contigs = len(offsets) - 1
    n_kmers = int(np.maximum(np.diff(offsets).astype(np.int64) - K + 1, 0).sum())
    d_bases = torch.from_numpy(bases).to(dev)
    d_off = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    d_codes = torch.empty(n_kmers, dtype=torch.int64, device=dev)
    d_code_off = torch.empty(n_contigs + 1, dtype=torch.int64, device=dev)
    d_status = torch.zeros(4, dtype=torch.int64, device=dev)

    def step():
        f.query_device(d_bases.data_ptr(), d_off.data_ptr(), offsets, d_codes.data_ptr(), n_kmers,
                       d_code_off.data_ptr(), d_status.data_ptr(), stream.cuda_stream)

    for _ in range(args.warmup):
        step()
    sync_all()
    st = d_status.cpu().numpy()
    assert st[0] == n_kmers and st[1] == 0, f"unexpected status {st}"
    # correctness gate before timing counts: EVERY code against the unmodified reference's (full compare,
    # SURVEY 8d), and the size-independent property: all members -> a permutation of 0..n-1
    codes_h = d_codes.cpu().numpy().view(np.uint64)
    checked = "none (LPHB_BENCH_NOCHECK)"
    if not nocheck:
        assert int(codes_h.max()) == f.get_kmer_count() - 1 and len(codes_h) == f.get_kmer_count()
        chk = np.zeros(len(codes_h), dtype=np.uint8)
        chk[codes_h] = 1
        assert int(chk.sum()) == len(codes_h), "codes are not a permutation (not a minimal perfect hash)"
        del chk
        checked = "permutation of 0..n-1"
        try:
            want = cpu_reference_codes(bases, offsets, lph, max(1, threads // world))
            assert np.array_equal(codes_h, want), "codes differ from the reference's"
            checked = f"all {len(want)} codes equal the unmodified reference's (oracle/_ref) + permutation of 0..n-1"
            del want
        except (ImportError, OSError, RuntimeError) as e:  # reference library absent on this box
            checked += f" (reference compare unavailable: {e})"

    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f.stats()  # drop the warm-up launches from the handle's per-launch event ring
    sync_all()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    sync_all()
    ms_total = ev0.elapsed_time(ev1)
    st_timed = f.stats()
    outputs = snapshot_outputs(torch, args, [d_codes], d_code_off, d_status) if rank == 0 else None
    if rank == 0:
        # the timed region lasts ~12 ms, a handful of NVML polls: keep the GPU under the identical load
        # (same steps, untimed) until the sampler has seen it for at least 60 ms
        t_end = time.perf_counter() + 0.06
        while time.perf_counter() < t_end:
            for _ in range(args.steps):
                step()
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None  # polled during the timed region and its identical continuation
    if world > 1:
        dist.barrier()
    # dominant-kernel launch time: the handle brackets its main kernel with a CUDA-event pair on
    # the launching stream at EVERY call; stats() returns the mean over the timed region's
    # launches (the most recent 128 of them)
    launches_per_step = int(st_timed.kernel_launches)
    kern_ms_local = float(st_timed.kernel_ms)

    # ---- e2e: HOST (pinned) buffers through the C ABI, both output forms ----------------------
    e2e_steps = max(1, min(args.steps, 5))
    hb = HostBatch(torch, bases, offsets, n_kmers)
    e = e2e_measure(torch, L, f, [hb], n_kmers, e2e_steps, sync_all, None if nocheck else codes_h)

    t = torch.tensor([ms_total, kern_ms_local, e["codes"]["secs"], e["runs"]["secs"], e["copy_only_codes"]["secs"],
                      e["copy_only_runs"]["secs"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, kern_ms, codes_s, runs_s, cc_s, cr_s = (float(x) for x in t.cpu())
    if rank != 0:
        return None
    # the build-side scan of the same resident bases (minimizer::from_string stream; one fused kernel), beside the query
    build_scan = None
    try:
        ms_l, nrec = [], 0
        for _ in range(4):
            _, nrec, nk_s, _, ms = api.scan_superkmers_device(d_bases.data_ptr(), d_off.data_ptr(), offsets, K, M,
                                                              device=dev.index, fetch=False)
            ms_l.append(ms)
        assert nk_s == n_kmers
        api.lib().lphb_scan_release(dev.index)
        s_ms = float(np.mean(ms_l[1:]))
        s_algo = int(offsets[-1] - offsets[0]) + 18 * int(nrec)
        peaks = load_peaks()
        peak = float(peaks.get("hbm_gbs", 6650.0))
        build_scan = {"metric": "build-p scan k-mers/sec (minimizer::from_string stream, bases resident)",
                      "value": n_kmers / (s_ms * 1e-3), "unit": "k-mers/s", "kernel_ms": s_ms, "records": int(nrec),
                      "roofline": {"bound": "hbm", "achieved": s_algo / (s_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                   "frac": s_algo / (s_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": s_algo,
                                   "kernel": "k_query_tiled<31,20,scan> (CUDA events around the kernel, mean of 3 launches)"},
                      "parity": "tools/bench_rows.py scan: all records equal the reference's from_string stream"}
    except Exception as e:  # the headline line stands without it
        build_scan = {"unavailable": str(e)}
    write_outputs(args.dump_outputs, outputs)
    value = world * n_kmers * args.steps / (ms_total * 1e-3)
    algo_bytes = int(offsets[-1] - offsets[0]) + 8 * n_kmers
    parts = {"codes_kmers": world * e["codes"]["kmers"], "codes_secs": codes_s, "runs_kmers": world * e["runs"]["kmers"],
             "runs_secs": runs_s, "h2d_codes": world * e["codes"]["h2d"], "d2h_codes": world * e["codes"]["d2h"],
             "h2d_runs": world * e["runs"]["h2d"], "d2h_runs": world * e["runs"]["d2h"], "runs_bpk": e["runs_bytes_per_kmer"], "steps": e2e_steps,
             "expand_rate": e["expand_kmers"] / e["expand_secs"], "copy_codes_secs": cc_s, "copy_runs_secs": cr_s}
    cfg = workload_config(args.kmers, n_kmers)
    cfg["parity_gate"] = checked
    return {"metric": "query-p k-mers/sec (k=31)", "value": value, "unit": "k-mers/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": cfg, "clocks": clocks,
            "e2e": e2e_object(world, parts, ""),
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline(algo_bytes, kern_ms, n_kmers,
                                 "k_query_tiled<31,20> (mean per launch over the timed region, CUDA events on the launching stream)"),
            "build_scan": build_scan,
            "cpu_baseline": None}


def bench_cfg5(args, torch, dist, api, L, f, dev, stream, rank, world, index_bases, lph, sync_all, sampler, nocheck,
               threads, slabs_total, brief):
    """Config 5: the read set is `slabs_total` slabs; rank r takes the contiguous slab range
    [r * S / world, (r + 1) * S / world) (strong scaling: the job is fixed, the ranks split it)."""
    S = slabs_total
    s0, s1 = rank * S // world, (rank + 1) * S // world
    genome_dev = torch.from_numpy(index_bases).to(dev)
    R, Lr = SLAB_READS, READ_LEN
    offsets = (np.arange(R + 1, dtype=np.uint64) * np.uint64(Lr))
    n_kmers_slab = R * (Lr - K + 1)
    slabs = [reads_slab_device(genome_dev, s, dev) for s in range(s0, s1)]
    del genome_dev
    d_off = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    d_codes = [torch.empty(n_kmers_slab, dtype=torch.int64, device=dev) for _ in slabs]
    d_code_off = torch.empty(R + 1, dtype=torch.int64, device=dev)
    d_status = torch.zeros(4, dtype=torch.int64, device=dev)

    def step():
        for sl, out in zip(slabs, d_codes):
            f.query_device(sl.data_ptr(), d_off.data_ptr(), offsets, out.data_ptr(), n_kmers_slab,
                           d_code_off.data_ptr(), d_status.data_ptr(), stream.cuda_stream)

    for _ in range(max(1, args.warmup if not brief else 1)):
        step()
    sync_all()
    st = d_status.cpu().numpy()
    assert st[0] == n_kmers_slab and st[1] == 0, f"unexpected status {st}"
    # parity gate: this rank's first slab (1.57e8 bases), every code against the unmodified reference
    checked = "none"
    first_codes = None
    if not nocheck and slabs:
        first_codes = d_codes[0].cpu().numpy().view(np.uint64)
        try:
            want = cpu_reference_codes(slabs[0].cpu().numpy(), offsets, lph, max(1, threads // world))
            assert np.array_equal(first_codes, want), "codes differ from the reference's"
            checked = (f"first slab of every rank ({n_kmers_slab} k-mers each, {world * R * Lr} bases in total): all codes "
                       f"equal the unmodified reference's (oracle/_ref)")
            del want
        except (ImportError, OSError, RuntimeError) as e:
            checked = f"reference compare unavailable: {e}"
    steps = args.steps
    if sampler is not None and rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f.stats()
    sync_all()
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    sync_all()
    clocks = sampler.stop() if (sampler is not None and rank == 0) else None
    ms_total = ev0.elapsed_time(ev1)
    outputs = snapshot_outputs(torch, args, d_codes, d_code_off, d_status) if rank == 0 and not brief else None
    st_timed = f.stats()
    launches_per_step = int(st_timed.kernel_launches) * len(slabs)
    kern_ms_local = float(st_timed.kernel_ms)

    # ---- e2e on a bounded number of this rank's slabs ------------------------------------------
    e2e_slabs = min(len(slabs), 4 if not brief else 2)
    e2e_steps = 2 if not brief else 1
    batches = [HostBatch(torch, slabs[i].cpu().numpy(), offsets, n_kmers_slab) for i in range(e2e_slabs)]
    check = None
    if first_codes is not None and e2e_slabs == 1:
        check = first_codes
    e = e2e_measure(torch, L, f, batches, n_kmers_slab, e2e_steps, sync_all, check)

    t = torch.tensor([ms_total, kern_ms_local, e["codes"]["secs"], e["runs"]["secs"], e["copy_only_codes"]["secs"],
                      e["copy_only_runs"]["secs"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, kern_ms, codes_s, runs_s, cc_s, cr_s = (float(x) for x in t.cpu())
    if rank != 0:
        return None
    write_outputs(args.dump_outputs, outputs)
    total_kmers = S * n_kmers_slab
    value = total_kmers * steps / (ms_total * 1e-3)
    algo_bytes = R * Lr + 8 * n_kmers_slab
    e2e_k = world * e["codes"]["kmers"]  # every rank streams the same number of slabs
    parts = {"codes_kmers": e2e_k, "codes_secs": codes_s, "runs_kmers": e2e_k, "runs_secs": runs_s,
             "h2d_codes": e["codes"]["h2d"] * e2e_slabs * world, "d2h_codes": e["codes"]["d2h"] * e2e_slabs * world,
             "h2d_runs": e["runs"]["h2d"] * e2e_slabs * world, "d2h_runs": e["runs"]["d2h"] * e2e_slabs * world,
             "runs_bpk": e["runs_bytes_per_kmer"], "steps": e2e_steps, "expand_rate": e["expand_kmers"] / e["expand_secs"],
             "copy_codes_secs": cc_s, "copy_runs_secs": cr_s}
    cfg = cfg5_config(world, S, total_kmers, S * R * Lr)
    cfg["parity_gate"] = checked
    cfg["e2e_sample"] = f"{e2e_slabs} slab(s) per rank per step through host buffers (bounded sample of the rank's {len(slabs)})"
    line = {"metric": "query-p k-mers/sec (k=31)", "value": value, "unit": "k-mers/s",
            "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms_total / steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": cfg, "clocks": clocks,
            "e2e": e2e_object(world, parts, f"; {e2e_slabs} slab(s) per rank per step"),
            "gpu_launches": launches_per_step * steps,
            "roofline": roofline(algo_bytes, kern_ms, n_kmers_slab,
                                 "k_query_tiled<31,20> on one slab of reads (mean per launch over the timed region, CUDA "
                                 "events on the launching stream)"),
            "cpu_baseline": None}
    if brief:
        return {k: line[k] for k in ("value", "unit", "ms_per_step", "steps", "config", "e2e", "roofline")}
    return line


# stdout carries the one JSON line and nothing else: libraries that print there (NCCL's version banner when the
# environment sets NCCL_DEBUG) are sent to stderr for the whole run, the line goes to the original descriptor
_STDOUT_FD = None


def quiet_stdout():
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _STDOUT_FD is None:
        os.write(1, data)
    else:
        os.write(_STDOUT_FD, data)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kmers", type=int, default=100_000_000)
    ap.add_argument("--workload", default=None, choices=["cfg2", "cfg5"],
                    help="default: cfg2 (BASELINE config 2, the metric's configuration) on one GPU, cfg5 (>= 10 Gbases "
                         "of reads, strong-scaled) under torchrun")
    ap.add_argument("--slabs", type=int, default=CFG5_SLABS, help="slabs of the config-5 read set (64 = 1.0066e10 bases)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg5", action="store_true", help="one GPU: skip the config-5 side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float64, sampled, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
