"""Caller-supplied genotypes (allele dosages per bubble) in the threading DP: the CPU oracle's rule, the Batch plumbing and
the C entry point without a device.  The GPU against the oracle: tests/test_genotypes_gpu.py."""
import copy
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

from ahsoka_b200 import api, synth
from tests.oracle_genotypes import oracle_phase


def with_dosage(batch, dosage):
    b = copy.copy(batch)
    b.allele_dosage = None if dosage is None else np.ascontiguousarray(dosage, dtype=np.uint8)
    return b


@pytest.mark.parametrize("ploidy,seed", [(2, 1), (4, 41), (6, 61)])
def test_oracle_all_zero_dosage_is_the_plain_rule(ploidy, seed):
    b = synth.generate(synth.params(ploidy, 12, 1, 30, depth=10.0 * ploidy, seed=seed))
    plain = oracle_phase(b)
    assert not oracle_phase(with_dosage(b, np.zeros(int(b.allele_off[-1]), np.uint8))).diff(plain)


def test_oracle_diploid_builtin_genotype_stated_explicitly():
    # ploidy 2 threads against {0:1, 1:1} at every position: the same genotype supplied as dosages changes nothing
    b = synth.generate(synth.params(2, 30, 1, 24, depth=30.0, max_alleles=4, seed=7))
    d = np.zeros(int(b.allele_off[-1]), np.uint8)
    d[b.allele_off[:-1]] = 1
    d[b.allele_off[:-1] + 1] = 1
    assert not oracle_phase(with_dosage(b, d)).diff(oracle_phase(b))
    # the generator's diploid truth is that genotype too
    assert np.array_equal(synth.true_dosage(b), d)


def test_oracle_true_tetraploid_dosages_reach_the_dp():
    b = synth.generate(synth.params(4, 12, 1, 30, depth=40.0, max_alleles=3, seed=41))
    d = synth.true_dosage(b)
    assert set(np.unique(d).tolist()) >= {1, 2, 3}                  # {0:3,1:1}, {0:2,1:2}, ... occur
    plain, gt = oracle_phase(b), oracle_phase(with_dosage(b, d))
    assert {"path", "hap_allele"} & set(gt.diff(plain))
    # the read x bubble matrix and the clusters do not depend on the genotypes
    for k in ("status", "read_off", "read_id", "read_cluster", "cell_off", "cell_pos", "cell_allele", "pos_off", "pos"):
        assert np.array_equal(getattr(gt, k), getattr(plain, k)), k


_A = [1, 2, 4, 5, 7, 8, 10]           # haplotype A: allele 0 at bubbles 0, 1, 2
_B = [1, 3, 4, 6, 7, 9, 10]           # haplotype B: allele 1 at bubbles 0, 1, 2


def two_haplotype_chain(dosage=None):
    """One diploid chain of three bubbles (alleles [src, inner, sink]) and eight reads over all of it, four from each haplotype."""
    reads = [_A, _B] * 4
    n = len(reads)
    return api.Batch(2, [0], [0, 3], [0, 2, 4, 6], [0, 3, 6, 9, 12, 15, 18], [1, 2, 4, 1, 3, 4, 4, 5, 7, 4, 6, 7, 7, 8, 10, 7, 9, 10],
                     [2, 1, 0], [0, n], [0, n], np.cumsum([0] + [len(r) for r in reads]), sum(reads, []), list(range(n)), [0.99] * n,
                     allele_dosage=dosage)


def test_hand_derived_homozygous_genotype_forces_a_switch():
    # Two clusters, every column covMap = [0, 1] (equal coverage 1/2: ascending id), consensus of cluster 0 = allele 0 (the reads
    # of haplotype A), of cluster 1 = allele 1.  Ordered states (t0, t1), code t0 * 2 + t1.
    # Plain: {0:1,1:1} admits (0,1) and (1,0) at every column, coverage cost 0 (cov 1/2 in [1/4, 3/4]); no switch: cost 0, the
    # lowest final code (0,1) everywhere.
    # Bubble 1 given {0:2}: only (0,0) conforms (consensus {0,0}); its coverage cost is 2 (cov 1/2 outside [3/4, 5/4], twice).
    # From column 0, (0,1) -> (0,0) and (1,0) -> (0,0) each switch one haplotype: 32 + 8 = 40, tie -> lower code (0,1):
    # D1(0,0) = 0 + 40 + 2 = 42.  Column 2 ({0:1,1:1}): (0,1) and (1,0) each cost 42 + 40 = 82, lowest code (0,1).
    # Path (0,1), (0,0), (0,1); hap_allele the same; dp_cost 82.  Given {1:2} instead: (1,1) in the middle, by the same steps.
    plain = oracle_phase(two_haplotype_chain())
    assert list(plain.read_cluster) == [0, 0, 0, 0, 1, 1, 1, 1]      # stage B creates the reads allele by allele: A's first
    assert list(plain.path) == [0, 1] * 3 and list(plain.hap_allele) == [0, 1] * 3 and plain.dp_cost[0] == 0
    hom0 = oracle_phase(two_haplotype_chain(np.array([0, 0, 2, 0, 0, 0], np.uint8)))
    assert list(hom0.path) == [0, 1, 0, 0, 0, 1] and list(hom0.hap_allele) == [0, 1, 0, 0, 0, 1] and hom0.dp_cost[0] == 82
    hom1 = oracle_phase(two_haplotype_chain(np.array([0, 0, 0, 2, 0, 0], np.uint8)))
    assert list(hom1.path) == [0, 1, 1, 1, 0, 1] and list(hom1.hap_allele) == [0, 1, 1, 1, 0, 1] and hom1.dp_cost[0] == 82
    # the built-in genotype stated at every bubble changes nothing
    assert not oracle_phase(two_haplotype_chain(np.array([1, 1, 1, 1, 1, 1], np.uint8))).diff(plain)


def test_oracle_rejects_malformed_dosages():
    with pytest.raises(RuntimeError, match=r"failed \(1\)"):          # AHS_ERR_ARG
        oracle_phase(two_haplotype_chain(np.array([0, 0, 2, 1, 0, 0], np.uint8)))


def test_batch_select_save_load_keep_allele_dosage():
    b = synth.generate(synth.params(4, 10, 1, 12, depth=20.0, max_alleles=3, seed=5))
    b.allele_dosage = synth.true_dosage(b)
    perm = np.array([7, 2, 5])
    s = b.select(perm)
    want = np.concatenate([b.allele_dosage[b.allele_off[b.bubble_off[c]]:b.allele_off[b.bubble_off[c + 1]]] for c in perm])
    assert s.allele_dosage.dtype == np.uint8 and np.array_equal(s.allele_dosage, want)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "b.npz")
        b.save(path)
        back = api.Batch.load(path)
        assert back.allele_dosage is not None and np.array_equal(back.allele_dosage, b.allele_dosage)
        plain = copy.copy(b); plain.allele_dosage = None
        plain.save(path)
        assert api.Batch.load(path).allele_dosage is None
    assert with_dosage(b, None).select(perm).allele_dosage is None


def test_genotyped_call_without_a_device():
    lib = api.load_library()
    if lib.ahs_device_count() > 0:
        pytest.skip("a CUDA device is present")
    b = synth.generate(synth.params(4, 4, 1, 8, depth=20.0, seed=3))
    b.allele_dosage = synth.true_dosage(b)
    with pytest.raises(RuntimeError, match=r"failed \(2\)"):          # AHS_ERR_CUDA
        api.phase_batch(b)
    s, o, dev = b.c_struct(), api.BatchOut(), (C.c_int * 1)(0)
    assert lib.ahs_phase_batch_genotyped(C.byref(s), b.dosage_ptr(), C.byref(o), dev, 1) == 2


def test_python_side_checks_of_allele_dosage():
    b = synth.generate(synth.params(2, 4, 1, 8, depth=10.0, seed=3))
    with pytest.raises(ValueError, match="allele_dosage"):            # the resident timing mode has no genotyped variant
        api.phase_batch(with_dosage(b, synth.true_dosage(b)), resident_iters=1)
    with pytest.raises(ValueError, match="allele_dosage"):            # one entry per allele
        api.phase_batch(with_dosage(b, np.zeros(3, np.uint8)))
