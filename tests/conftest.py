import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# The library answers batches below 256 K bases with its generic (one thread per k-mer) kernel, which has the
# shorter start-up; the fixtures are that small, so the suite pins the threshold to 0 to keep exercising the tiled
# kernel and lifts it again in the tests of the small-batch path (test_gpu_parity.py).
os.environ.setdefault("LPHB_GENERIC_BELOW", "0")

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
GOLDEN_NAMES = ["k31_m20_u64", "k31_m16_u128", "k63_m24_u128", "k47_m20_u128", "k15_m7_u64",
                "k21_m11_u64",
                "k25_m13_u64", "k40_m17_u128"]  # the last two run on the generic (any k, m) kernels


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


class Golden:
    """One committed fixture generated from the reference by tools/make_golden.py."""

    def __init__(self, name):
        self.name = name
        self.lph = os.path.join(GOLDEN_DIR, name + ".lph")
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        self.z = z
        self.k, self.m, self.bits = int(z["k"]), int(z["m"]), int(z["bits"])

    def __getattr__(self, key):
        return self.z[key]

    def contigs(self):
        raw = self.z["q_bases"].tobytes()
        off = self.z["q_offsets"]
        return [raw[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)]

    def is_clean(self):
        """per query contig: ACGT/acgt/U/u only"""
        ok = np.zeros(256, dtype=bool)
        for ch in b"ACGTUacgtu":
            ok[ch] = True
        return [bool(ok[np.frombuffer(c, dtype=np.uint8)].all()) for c in self.contigs()]


_cache = {}


def load_golden(name):
    if name not in _cache:
        _cache[name] = Golden(name)
    return _cache[name]


@pytest.fixture(params=GOLDEN_NAMES)
def golden(request):
    return load_golden(request.param)


def fnv_fold(codes) -> int:
    """64-bit FNV-1a-style fold over u64 codes (SURVEY.md §8c)."""
    h = 0xCBF29CE484222325
    for v in np.asarray(codes, dtype=np.uint64).tolist():
        h = ((h ^ v) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return h


# ---- synthetic inputs of build-p Part 3 (branches sequence-derived fixtures never reach) ----
def splitmix64(n):
    x = (np.arange(1, n + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15))
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


PART3_FIXTURES = {"sparse": (251100, 200, 20), "maximal": (3000, 31, 20), "mixed": (70000, 63, 24)}
TRIPLET = np.dtype([("itself", "<u8"), ("p1", "u1"), ("size", "u1")])


def part3_triplets(name):
    """the triplet plan of a tests/golden/part3_<name>.npz fixture (tools/make_golden_part3.py): key i = splitmix64(i)"""
    n, k, m = PART3_FIXTURES[name]
    t = np.zeros(n, dtype=TRIPLET)
    t["itself"] = splitmix64(n)
    if name == "sparse":      # 1100 NONE super-k-mers of the largest size among colliding minimizers
        t["p1"][:1100] = 100
        t["size"][:1100] = k - m + 1
    elif name == "maximal":   # nothing but MAXIMAL: sizes_and_positions stays empty
        t["p1"] = k - m
        t["size"] = k - m + 1
    elif name == "mixed":     # every type, sizes spread
        r = np.random.default_rng(5)
        kind = r.integers(0, 5, n)
        w = k - m + 1
        size = r.integers(2, w, n)
        p1 = np.where(kind == 0, size - 1,                      # LEFT (p1 == size-1 < k-m)
             np.where(kind == 1, k - m,                          # RIGHT (size < w)
             np.where(kind == 2, k - m, r.integers(0, 1 << 30, n) % np.maximum(size - 1, 1))))  # MAXIMAL / NONE
        size = np.where(kind == 2, w, size)
        size = np.where(kind == 4, 0, size)                      # colliding
        p1 = np.where(kind == 4, 0, p1)
        t["p1"], t["size"] = p1, size
    return t
