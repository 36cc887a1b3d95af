"""ctypes binding of oracle/_ref/liboracle_gt.so (tests/native/oracle_genotypes.cpp): the CPU oracle with caller-supplied
genotypes.  TEST INFRASTRUCTURE, imported only by tests/.

oracle_phase(batch) is tests.oracle_binding.oracle_phase when batch.allele_dosage is None, and the same oracle with the
batch's allele dosages (the rule of ahs_phase_batch_genotyped) otherwise."""
import ctypes as C
import os

from ahsoka_b200.api import ROOT, Batch, BatchIn, BatchOut, PhaseResult, result_from_struct
from tests import oracle_binding

ORACLE_GT_LIB = os.path.join(ROOT, "oracle", "_ref", "liboracle_gt.so")
_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_GT_LIB):
            import __graft_entry__
            __graft_entry__.build()
        lib = C.CDLL(ORACLE_GT_LIB)
        lib.ahs_oracle_phase_batch_gt.argtypes = [C.POINTER(BatchIn), C.POINTER(C.c_uint8), C.POINTER(BatchOut), C.c_int]
        lib.ahs_oracle_phase_batch_gt.restype = C.c_int
        lib.ahs_oracle_free_out.argtypes = [C.POINTER(BatchOut)]
        _lib = lib
    return _lib


def oracle_phase(batch: Batch, n_threads: int = 0) -> PhaseResult:
    if batch.allele_dosage is None:
        return oracle_binding.oracle_phase(batch, n_threads)
    lib = load()
    s, o = batch.c_struct(), BatchOut()
    rc = lib.ahs_oracle_phase_batch_gt(C.byref(s), batch.dosage_ptr(), C.byref(o), n_threads)
    if rc != 0:
        raise RuntimeError(f"oracle failed ({rc})")
    try:
        return result_from_struct(o)
    finally:
        lib.ahs_oracle_free_out(C.byref(o))
