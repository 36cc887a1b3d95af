"""Synthetic bubble-chain workloads (binding of ahsoka_b200/csrc/synth.cpp) and the named
configurations of BASELINE.json (SURVEY.md §8d)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .api import ROOT, Batch, BatchIn

SYNTH_LIB = os.path.join(ROOT, "ahsoka_b200", "lib", "libahsoka_synth.so")


class SynthParams(C.Structure):
    _fields_ = [("ploidy", C.c_int32), ("n_chains", C.c_int32), ("len_mode", C.c_int32), ("mean_len", C.c_int32),
                ("min_len", C.c_int32), ("max_len", C.c_int32), ("zipf_alpha", C.c_double), ("n_forced_max", C.c_int32),
                ("depth", C.c_double), ("mean_span", C.c_double), ("span_sigma", C.c_double), ("err", C.c_double),
                ("miss", C.c_double), ("max_alleles", C.c_int32), ("dup_lines", C.c_int32), ("seed", C.c_uint64)]


_lib = None


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(SYNTH_LIB):
            raise RuntimeError(f"{SYNTH_LIB} missing: run __graft_entry__.build()")
        lib = C.CDLL(SYNTH_LIB)
        lib.ahs_synth_generate.argtypes = [C.POINTER(SynthParams), C.POINTER(C.c_void_p)]
        lib.ahs_synth_batch_in.argtypes = [C.c_void_p]
        lib.ahs_synth_batch_in.restype = C.POINTER(BatchIn)
        lib.ahs_synth_counts.argtypes = [C.c_void_p, C.c_int]
        lib.ahs_synth_counts.restype = C.c_int64
        lib.ahs_synth_truth_read_hap.argtypes = [C.c_void_p]
        lib.ahs_synth_truth_read_hap.restype = C.POINTER(C.c_int32)
        lib.ahs_synth_truth_hap_allele.argtypes = [C.c_void_p]
        lib.ahs_synth_truth_hap_allele.restype = C.POINTER(C.c_uint8)
        lib.ahs_synth_write_gfa_gaf.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        lib.ahs_synth_free.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def params(ploidy=2, n_chains=1, len_mode=0, mean_len=40, min_len=2, max_len=0, zipf_alpha=1.2, n_forced_max=0,
           depth=30.0, mean_span=16.0, span_sigma=0.5, err=0.05, miss=0.02, max_alleles=None, dup_lines=0, seed=0xA450CA00):
    if max_alleles is None:
        max_alleles = max(2, ploidy)
    return SynthParams(ploidy, n_chains, len_mode, mean_len, min_len, max_len, zipf_alpha, n_forced_max, depth, mean_span,
                       span_sigma, err, miss, max_alleles, dup_lines, seed)


# BASELINE.json configs -> generator parameters (SURVEY.md §8d).  `scale` shrinks the chain count.
def config(name: str, scale: float = 1.0) -> SynthParams:
    n = lambda x: max(1, int(round(x * scale)))
    if name == "cfg1":      # 1 chain of 1k bubbles, 2k ONT-like reads
        return params(2, 1, 0, 1000, depth=32.0, seed=0xA450CA01)
    if name == "cfg2":      # diploid human-scale: 50k chains, 2M bubbles, 30x
        return params(2, n(50000), 1, 40, depth=30.0, seed=0xA450CA02)
    if name == "cfg3":      # triploid: 20k chains, 1M bubbles, 40x
        return params(3, n(20000), 1, 50, depth=40.0, seed=0xA450CA03)
    if name == "cfg4":      # tetraploid: 10k chains, 800k bubbles, 60x
        return params(4, n(10000), 1, 80, depth=60.0, seed=0xA450CA04)
    if name == "cfg5":      # hexaploid, Zipf-skewed chain sizes up to 10k bubbles, 80x
        return params(6, n(2000), 2, 500, 2, 10000, 1.2, max(1, n(4)), depth=80.0, seed=0xA450CA05)
    if name == "cfg5cap":   # cfg5 with the chain length capped at 1000 bubbles (<= ~3,600 final reads per chain: inside the cluster-editing limit)
        return params(6, n(2000), 2, 500, 2, 1000, 1.2, max(1, n(4)), depth=80.0, seed=0xA450CA05)
    if name == "zipf2":     # diploid, Zipf-skewed chain sizes up to 10k bubbles, 30x: the load-balancing stress of SURVEY 8e
        return params(2, n(4000), 2, 500, 2, 10000, 1.2, max(1, n(4)), depth=30.0, seed=0xA450CA06)
    raise KeyError(name)


def generate(p: SynthParams, gfa_gaf_prefix: str | None = None) -> Batch:
    lib = _load()
    h = C.c_void_p()
    rc = lib.ahs_synth_generate(C.byref(p), C.byref(h))
    if rc != 0:
        raise RuntimeError(f"ahs_synth_generate failed ({rc})")
    try:
        s = lib.ahs_synth_batch_in(h).contents
        cnt = [int(lib.ahs_synth_counts(h, i)) for i in range(8)]
        Cn, NB, NA, NAN, NR, NE, NEN, NN = cnt

        def arr(ptr, n, dt):
            return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dt, copy=True) if n else np.zeros(0, dtype=dt)
        b = Batch(s.ploidy, arr(s.chain_id, Cn, np.int32), arr(s.bubble_off, Cn + 1, np.int64), arr(s.allele_off, NB + 1, np.int64),
                  arr(s.anode_off, NA + 1, np.int64), arr(s.anode, NAN, np.int32), arr(s.stage_a_order, NB, np.int32),
                  arr(s.read_off, Cn + 1, np.int64), arr(s.entry_off, Cn + 1, np.int64), arr(s.enode_off, NE + 1, np.int64),
                  arr(s.enode, NEN, np.int32), arr(s.entry_read, NE, np.int32), arr(s.entry_identity, NE, np.float32))
        b.truth = {"read_hap": arr(lib.ahs_synth_truth_read_hap(h), NE, np.int32),
                   "hap_allele": arr(lib.ahs_synth_truth_hap_allele(h), NB * s.ploidy, np.uint8), "n_nodes": NN}
        if gfa_gaf_prefix is not None:
            rc = lib.ahs_synth_write_gfa_gaf(h, (gfa_gaf_prefix + ".gfa").encode(), (gfa_gaf_prefix + ".gaf").encode())
            if rc != 0:
                raise RuntimeError("ahs_synth_write_gfa_gaf failed")
        return b
    finally:
        lib.ahs_synth_free(h)


def true_dosage(batch: Batch) -> np.ndarray:
    """Per-allele dosages of the generator's haplotypes (batch.truth["hap_allele"]), indexed like allele_off: the number of
    haplotypes that carry each allele of each bubble.  Every haplotype gets a distinct allele while the bubble has at least
    ploidy alleles (diploid truth is always {0:1, 1:1}); the remaining haplotypes draw one at random."""
    p = int(batch.ploidy)
    hap = batch.truth["hap_allele"].reshape(-1, p).astype(np.int64)
    idx = batch.allele_off[:-1, None] + hap
    return np.bincount(idx.ravel(), minlength=int(batch.allele_off[-1])).astype(np.uint8)
