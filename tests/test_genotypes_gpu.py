"""-m gpu: phasing with caller-supplied genotypes (ahs_phase_batch_genotyped) against the CPU oracle with the same dosages,
bit for bit, on every DP kernel (k_thread2 at ploidy 2, k_thread at 3-4, k_thread_canon at 5-6)."""
import copy
import os

import numpy as np
import pytest

from ahsoka_b200 import api, synth
from tests.oracle_genotypes import oracle_phase

pytestmark = pytest.mark.gpu


def with_dosage(batch, dosage):
    b = copy.copy(batch)
    b.allele_dosage = None if dosage is None else np.ascontiguousarray(dosage, dtype=np.uint8)
    return b


def _check(batch, n_threads=0, **kw):
    got = api.phase_batch(batch, **kw)
    bad = got.diff(oracle_phase(batch, n_threads))
    assert not bad, f"GPU differs from oracle in {bad}"
    return got


def _bubbles(batch):
    off = batch.allele_off
    return off[:-1].astype(np.int64), np.diff(off).astype(np.int64)


def _assign(d, a0, k, genotype):
    """the genotype {allele: dosage} for the bubble of k alleles whose first allele is a0"""
    d[a0:a0 + k] = 0
    for a, n in genotype.items():
        d[a0 + a] = n


@pytest.mark.parametrize("ploidy,max_alleles,seed", [(3, 2, 31), (3, 3, 32), (4, 3, 41), (4, 8, 42), (5, 3, 51), (5, 6, 52),
                                                      (6, 2, 61), (6, 12, 62)])
def test_true_dosages_polyploid(ploidy, max_alleles, seed):
    # ploidy 3, 4: ordered tuples (k_thread); 5, 6: canonical tuples (k_thread_canon); 2-bit (<= 3 alleles) and 4-bit codes
    b = synth.generate(synth.params(ploidy, 12, 1, 30, depth=10.0 * ploidy, max_alleles=max_alleles, seed=seed))
    plain = api.phase_batch(b)
    got = _check(with_dosage(b, synth.true_dosage(b)))
    assert got.n_chains_ok == plain.n_chains_ok


def test_cfg4_shape_true_dosages():
    # ploidy 4, 60x: 200-330 final reads per chain, the 4096-state ordered DP
    b = synth.generate(synth.config("cfg4", 0.005))
    got = _check(with_dosage(b, synth.true_dosage(b)), os.cpu_count() or 1)
    assert got.n_chains_ok == b.n_chains and int(np.diff(got.read_off).max()) > 250


def test_cfg5_shape_true_dosages():
    # ploidy 6, 80x, Zipf-skewed chain sizes with one forced 600-bubble chain: the canonical-tuple DP over long chains
    b = synth.generate(synth.params(6, 24, 2, 500, 2, 600, 1.2, 1, depth=80.0, seed=0xA450CA05))
    got = _check(with_dosage(b, synth.true_dosage(b)), os.cpu_count() or 1)
    assert got.n_chains_ok >= 20


def diploid_non_default(b, seed):
    """Ploidy 2: homozygous {a:2} at a random 20 % of the bubbles, {1:1, 2:1} at the other bubbles of 3+ alleles, the truth
    ({0:1, 1:1}) elsewhere.  Where the consensus alleles cannot meet the genotype, every state is allowed."""
    rng = np.random.default_rng(seed)
    d = synth.true_dosage(b)
    a0s, ks = _bubbles(b)
    for a0, k in zip(a0s, ks):
        if rng.random() < 0.2:
            _assign(d, a0, k, {int(rng.integers(0, k)): 2})
        elif k >= 3:
            _assign(d, a0, k, {1: 1, 2: 1})
    return d


@pytest.mark.parametrize("max_alleles,seed", [(2, 1), (3, 2), (6, 3)])
def test_diploid_non_default_genotypes(max_alleles, seed):
    b = synth.generate(synth.params(2, 40, 1, 24, depth=30.0, max_alleles=max_alleles, seed=seed))
    gb = with_dosage(b, diploid_non_default(b, seed))
    got = _check(gb)
    assert got.diff(api.phase_batch(b))                             # the genotypes did change the threading


def test_mixed_known_unknown_and_wrong_genotypes():
    # ploidy 4: a random 30 % of the bubbles unknown, 20 % a wrong but valid dosage vector, the rest the truth
    b = synth.generate(synth.params(4, 16, 1, 40, depth=40.0, max_alleles=4, seed=44))
    rng = np.random.default_rng(44)
    d = synth.true_dosage(b)
    a0s, ks = _bubbles(b)
    for a0, k in zip(a0s, ks):
        u = rng.random()
        if u < 0.3:
            d[a0:a0 + k] = 0
        elif u < 0.5:
            d[a0:a0 + k] = np.bincount(rng.integers(0, k, 4), minlength=k)
    _check(with_dosage(b, d))


@pytest.mark.parametrize("ploidy,seed", [(2, 12), (4, 43), (6, 63)])
def test_null_and_all_zero_dosage_equal_the_plain_call(ploidy, seed):
    b = synth.generate(synth.params(ploidy, 20, 1, 30, depth=10.0 * ploidy, seed=seed))
    plain = api.phase_batch(b)
    assert not api.phase_batch(with_dosage(b, np.zeros(int(b.allele_off[-1]), np.uint8))).diff(plain)
    lib = api.load_library()
    import ctypes as C
    s, o, dev = b.c_struct(), api.BatchOut(), (C.c_int * 1)(0)
    assert lib.ahs_phase_batch_genotyped(C.byref(s), None, C.byref(o), dev, 1) == 0          # NULL dosage pointer
    try:
        assert not api.result_from_struct(o).diff(plain)
    finally:
        lib.ahs_free_out(C.byref(o))
    if ploidy == 2:                                                 # the diploid truth is the built-in genotype
        assert not api.phase_batch(with_dosage(b, synth.true_dosage(b))).diff(plain)


@pytest.mark.parametrize("chunks", ["1", "2", "4"])
def test_chunked_and_devices_list_are_result_identical(chunks, monkeypatch):
    # every chunk of chains (AHS_CHUNKS) indexes its own slice of the dosages
    b = synth.generate(synth.config("cfg2", 0.25))
    gb = with_dosage(b, diploid_non_default(b, 5))
    want = oracle_phase(gb, os.cpu_count() or 1)
    monkeypatch.setenv("AHS_CHUNKS", chunks)
    assert not api.phase_batch(gb).diff(want)
    assert not api.phase_batch(gb, devices=[0]).diff(want)


def test_multi_device_genotyped():
    if api.load_library().ahs_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    b = synth.generate(synth.config("cfg2", 0.02))
    gb = with_dosage(b, diploid_non_default(b, 6))
    assert not api.phase_batch(gb, devices=[0, 1]).diff(oracle_phase(gb))


def test_malformed_dosages_are_rejected():
    b = synth.generate(synth.params(3, 60, 1, 3, min_len=1, depth=20.0, max_alleles=3, seed=93))
    good = synth.true_dosage(b)
    a0s, ks = _bubbles(b)
    nb = np.diff(b.bubble_off)
    short = int(np.flatnonzero(nb == 1)[0])                         # a chain of one bubble: never phased (status 1)
    cases = []
    d = good.copy(); d[a0s[5]] += 1; cases.append(d)                # a bubble summing to p + 1
    d = good.copy(); d[a0s[7]:a0s[7] + ks[7]] = 0; d[a0s[7]] = 4; cases.append(d)      # one allele with p + 1
    d = good.copy(); g = int(b.bubble_off[short]); d[a0s[g]:a0s[g] + ks[g]] = 0; d[a0s[g]] = 1; cases.append(d)   # sum 1
    for d in cases:
        with pytest.raises(RuntimeError, match="allele_dosage"):
            api.phase_batch(with_dosage(b, d))
        with pytest.raises(RuntimeError, match="allele_dosage"):
            api.phase_batch(with_dosage(b, d), devices=[0])
    # the library is still usable afterwards
    _check(with_dosage(b, good))
    assert not api.phase_batch(b).diff(oracle_phase(b))
