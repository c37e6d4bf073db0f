"""oracle/phf.py: `.lph` indexes made without the reference's build-p (bench.py's input)."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import oracle, phf


@pytest.mark.parametrize("n", [1, 2, 3, 1000, 100_000])
def test_single_phf_is_a_minimal_perfect_hash(n):
    keys = np.unique(np.random.default_rng(n).integers(0, 2**64 - 1, n, dtype=np.uint64))
    image = phf.single_phf(phf.murmur64(keys, phf.PTHASH_SEED))
    assert image == phf.single_phf(phf.murmur64(keys, phf.PTHASH_SEED))  # deterministic
    assert np.array_equal(np.sort(oracle.phf_positions(image, keys)), np.arange(len(keys)))


def test_murmur64_matches_the_oracle():
    v = np.array([0, 1, 42, 2**63 + 7, 2**64 - 1], dtype=np.uint64)
    for seed in (1, 2**64 - 2):
        assert [int(x) for x in phf.murmur64(v, seed)] == [oracle.murmur64(int(x), seed) for x in v]


def test_duplicate_keys_are_refused():
    with pytest.raises(ValueError):
        phf.single_phf(np.array([5, 9, 5], dtype=np.uint64))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_built_index_is_a_minimal_perfect_hash_of_the_kmers(name, tmp_path):
    from lphash_b200 import api

    g = load_golden(name)
    image = phf.build_lph(g.index_bases, g.index_offsets, g.k, g.m, kmer_bits=g.bits)
    path = str(tmp_path / "built.lph")
    with open(path, "wb") as f:
        f.write(image)
    f = api.Mphf.load(path, g.bits)
    codes, _ = f.query_batch(g.index_bases, g.index_offsets)
    f.close()
    assert np.array_equal(np.sort(codes), np.arange(len(codes)))
    want, _ = oracle.OracleMphf(path, g.bits).query_batch(g.index_bases, g.index_offsets)
    assert np.array_equal(codes, want)
