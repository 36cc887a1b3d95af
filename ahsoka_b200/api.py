"""ctypes binding of include/ahsoka_b200.h.

``phase_batch`` is the call a user makes: host buffers in, host buffers out, everything in
between on the GPU.  There is no CPU fallback: if the CUDA library is missing or no device is
usable the call raises (reference seam: src/polyassembly.cpp:171).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(ROOT, "ahsoka_b200", "lib", "libahsoka_b200.so")

i32p, i64p, u8p, f32p, f64p = (C.POINTER(t) for t in (C.c_int32, C.c_int64, C.c_uint8, C.c_float, C.c_double))


class BatchIn(C.Structure):
    _fields_ = [("n_chains", C.c_int32), ("ploidy", C.c_int32), ("chain_id", i32p),
                ("bubble_off", i64p), ("allele_off", i64p), ("anode_off", i64p), ("anode", i32p),
                ("stage_a_order", i32p), ("read_off", i64p), ("entry_off", i64p), ("enode_off", i64p),
                ("enode", i32p), ("entry_read", i32p), ("entry_identity", f32p)]


class BatchOut(C.Structure):
    _fields_ = [("n_chains", C.c_int32), ("ploidy", C.c_int32), ("status", i32p),
                ("read_off", i64p), ("read_id", i32p), ("read_mapq", i32p), ("read_cluster", i32p),
                ("cell_off", i64p), ("cell_pos", i32p), ("cell_allele", u8p),
                ("n_clusters", i32p), ("pos_off", i64p), ("pos", i32p), ("path", i32p), ("hap_allele", u8p),
                ("dp_cost", f64p), ("maxpos", i32p),
                ("n_cells", C.c_int64), ("n_pairs", C.c_int64), ("n_chains_ok", C.c_int64),
                ("ms_h2d", C.c_float), ("ms_project", C.c_float), ("ms_rows", C.c_float), ("ms_score", C.c_float),
                ("ms_cluster", C.c_float), ("ms_consensus", C.c_float), ("ms_thread", C.c_float), ("ms_d2h", C.c_float),
                ("ms_total_device", C.c_float), ("n_launches", C.c_int32), ("reserved", C.c_int32),
                ("bytes_project", C.c_int64), ("bytes_score", C.c_int64), ("bytes_consensus", C.c_int64)]


class Limits(C.Structure):
    _fields_ = [("max_ploidy", C.c_int32), ("max_alleles", C.c_int32), ("max_reads_cluster", C.c_int32),
                ("max_positions", C.c_int32), ("max_clusters_position", C.c_int32), ("reserved", C.c_int32 * 3)]


_I32 = ("chain_id", "anode", "stage_a_order", "enode", "entry_read")
_I64 = ("bubble_off", "allele_off", "anode_off", "read_off", "entry_off", "enode_off")


@dataclass
class Batch:
    """Host-side CSR batch (numpy arrays own the memory the C struct points to)."""
    ploidy: int
    chain_id: np.ndarray
    bubble_off: np.ndarray
    allele_off: np.ndarray
    anode_off: np.ndarray
    anode: np.ndarray
    stage_a_order: np.ndarray
    read_off: np.ndarray
    entry_off: np.ndarray
    enode_off: np.ndarray
    enode: np.ndarray
    entry_read: np.ndarray
    entry_identity: np.ndarray
    truth: dict = field(default_factory=dict)
    # optional caller genotypes, one uint8 per allele (indexed like allele_off): how many haplotypes carry the allele.
    # Per bubble all 0 (unknown) or summing to the ploidy; see ahs_phase_batch_genotyped in include/ahsoka_b200.h.
    allele_dosage: np.ndarray | None = None

    def __post_init__(self):
        for k in _I32:
            setattr(self, k, np.ascontiguousarray(getattr(self, k), dtype=np.int32))
        for k in _I64:
            setattr(self, k, np.ascontiguousarray(getattr(self, k), dtype=np.int64))
        self.entry_identity = np.ascontiguousarray(self.entry_identity, dtype=np.float32)
        if self.allele_dosage is not None:
            self.allele_dosage = np.ascontiguousarray(self.allele_dosage, dtype=np.uint8)

    def dosage_ptr(self):
        """ctypes pointer to allele_dosage, after checking that it has one entry per allele."""
        n_alleles = int(self.allele_off[-1]) if len(self.allele_off) else 0
        if self.allele_dosage.shape != (n_alleles,):
            raise ValueError(f"allele_dosage has shape {self.allele_dosage.shape}, the batch has {n_alleles} alleles")
        return self.allele_dosage.ctypes.data_as(u8p)

    @property
    def n_chains(self):
        return int(self.chain_id.shape[0])

    def c_struct(self) -> BatchIn:
        s = BatchIn()
        s.n_chains, s.ploidy = self.n_chains, int(self.ploidy)
        for k in _I32:
            setattr(s, k, getattr(self, k).ctypes.data_as(i32p))
        for k in _I64:
            setattr(s, k, getattr(self, k).ctypes.data_as(i64p))
        s.entry_identity = self.entry_identity.ctypes.data_as(f32p)
        return s

    def nbytes(self) -> int:
        return int(sum(getattr(self, k).nbytes for k in _I32 + _I64) + self.entry_identity.nbytes)

    def select(self, chains) -> "Batch":
        """Sub-batch with the given chain indices (in the given order).  Used for sharding."""
        chains = np.asarray(chains, dtype=np.int64)

        def span(off, idx):
            lo, hi = off[idx], off[idx + 1]
            n = hi - lo
            new_off = np.zeros(len(idx) + 1, dtype=np.int64)
            np.cumsum(n, out=new_off[1:])
            tot = int(new_off[-1])
            # gather indices lo[i] .. hi[i]-1
            if tot == 0:
                return new_off, np.zeros(0, dtype=np.int64)
            rep = np.repeat(lo - new_off[:-1], n)
            return new_off, rep + np.arange(tot, dtype=np.int64)

        b_off, b_idx = span(self.bubble_off, chains)
        a_off_rel, a_idx = span(self.allele_off, b_idx)
        an_off, an_idx = span(self.anode_off, a_idx)
        e_off, e_idx = span(self.entry_off, chains)
        en_off, en_idx = span(self.enode_off, e_idx)
        r_n = self.read_off[chains + 1] - self.read_off[chains]
        r_off = np.zeros(len(chains) + 1, dtype=np.int64)
        np.cumsum(r_n, out=r_off[1:])
        return Batch(self.ploidy, self.chain_id[chains], b_off, a_off_rel, an_off, self.anode[an_idx],
                     self.stage_a_order[b_idx], r_off, e_off, en_off, self.enode[en_idx],
                     self.entry_read[e_idx], self.entry_identity[e_idx],
                     allele_dosage=None if self.allele_dosage is None else self.allele_dosage[a_idx])

    def save(self, path):
        extra = {} if self.allele_dosage is None else {"allele_dosage": self.allele_dosage}
        np.savez_compressed(path, ploidy=self.ploidy, **{k: getattr(self, k) for k in _I32 + _I64},
                            entry_identity=self.entry_identity, **extra)

    @staticmethod
    def load(path) -> "Batch":
        z = np.load(path)
        return Batch(int(z["ploidy"]), *[z[k] for k in ("chain_id", "bubble_off", "allele_off", "anode_off", "anode",
                                                        "stage_a_order", "read_off", "entry_off", "enode_off", "enode",
                                                        "entry_read", "entry_identity")],
                     allele_dosage=z["allele_dosage"] if "allele_dosage" in z.files else None)

    @staticmethod
    def from_dump(path) -> "Batch":
        """Read the raw dump written by the host drop-in (AHSOKA_DUMP_BATCH)."""
        raw = open(path, "rb").read()
        hdr = np.frombuffer(raw, dtype=np.int64, count=7)
        C_, p, NB, NA, NAN, NE, NEN = (int(x) for x in hdr)
        o = 56

        def take(dt, n):
            nonlocal o
            a = np.frombuffer(raw, dtype=dt, count=n, offset=o).copy()
            o += a.nbytes
            return a
        chain_id = take(np.int32, C_); bubble_off = take(np.int64, C_ + 1); allele_off = take(np.int64, NB + 1)
        anode_off = take(np.int64, NA + 1); anode = take(np.int32, NAN); sao = take(np.int32, NB)
        read_off = take(np.int64, C_ + 1); entry_off = take(np.int64, C_ + 1); enode_off = take(np.int64, NE + 1)
        enode = take(np.int32, NEN); entry_read = take(np.int32, NE); ident = take(np.float32, NE)
        return Batch(p, chain_id, bubble_off, allele_off, anode_off, anode, sao, read_off, entry_off, enode_off, enode,
                     entry_read, ident)


@dataclass
class PhaseResult:
    ploidy: int
    status: np.ndarray
    read_off: np.ndarray
    read_id: np.ndarray
    read_mapq: np.ndarray
    read_cluster: np.ndarray
    cell_off: np.ndarray
    cell_pos: np.ndarray
    cell_allele: np.ndarray
    n_clusters: np.ndarray
    pos_off: np.ndarray
    pos: np.ndarray
    path: np.ndarray
    hap_allele: np.ndarray
    dp_cost: np.ndarray
    maxpos: np.ndarray
    n_cells: int
    n_pairs: int
    n_chains_ok: int
    timings: dict
    _owner: object = None          # (lib, BatchOut) while the arrays are views of the library's pinned buffers

    ARRAYS = ("status", "read_off", "read_id", "read_mapq", "read_cluster", "cell_off", "cell_pos", "cell_allele",
              "n_clusters", "pos_off", "pos", "path", "hap_allele", "dp_cost", "maxpos")

    def release(self):
        """Give the library's output buffers back (only needed for results obtained with copy=False)."""
        if self._owner is not None:
            lib, o = self._owner
            self._owner = None
            for k in self.ARRAYS:
                setattr(self, k, None)
            lib.ahs_free_out(C.byref(o))

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def diff(self, other: "PhaseResult"):
        """Names of the arrays that differ (bit-exact comparison)."""
        bad = [k for k in self.ARRAYS if not np.array_equal(getattr(self, k), getattr(other, k))]
        for k in ("n_cells", "n_pairs", "n_chains_ok"):
            if getattr(self, k) != getattr(other, k):
                bad.append(k)
        return bad


def _np(ptr, n, dtype, copy=True):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    a = np.ctypeslib.as_array(ptr, shape=(n,))
    return a.astype(dtype, copy=True) if copy else a


def result_from_struct(o: BatchOut, copy: bool = True) -> PhaseResult:
    """numpy view of an ahs_batch_out.  copy=False: zero-copy views of the library's (pinned) output
    buffers, valid until PhaseResult.release()."""
    def g(ptr, n, dtype):
        return _np(ptr, n, dtype, copy)
    Cn, p = o.n_chains, o.ploidy
    read_off = g(o.read_off, Cn + 1, np.int64)
    nr = int(read_off[-1])
    cell_off = g(o.cell_off, nr + 1, np.int64)
    nc = int(cell_off[-1])
    pos_off = g(o.pos_off, Cn + 1, np.int64)
    npos = int(pos_off[-1])
    t = {k: float(getattr(o, k)) for k in ("ms_h2d", "ms_project", "ms_rows", "ms_score", "ms_cluster", "ms_consensus",
                                           "ms_thread", "ms_d2h", "ms_total_device")}
    t.update({k: int(getattr(o, k)) for k in ("n_launches", "bytes_project", "bytes_score", "bytes_consensus")})
    return PhaseResult(p, g(o.status, Cn, np.int32), read_off, g(o.read_id, nr, np.int32), g(o.read_mapq, nr, np.int32),
                       g(o.read_cluster, nr, np.int32), cell_off, g(o.cell_pos, nc, np.int32), g(o.cell_allele, nc, np.uint8),
                       g(o.n_clusters, Cn, np.int32), pos_off, g(o.pos, npos, np.int32), g(o.path, npos * p, np.int32),
                       g(o.hap_allele, npos * p, np.uint8), g(o.dp_cost, Cn, np.float64), g(o.maxpos, Cn, np.int32),
                       int(o.n_cells), int(o.n_pairs), int(o.n_chains_ok), t)


_lib = None


def load_library(path: str = LIB_PATH):
    """Load the CUDA library.  Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the phasing path has no CPU fallback)")
    lib = C.CDLL(path)
    lib.ahs_abi_version.restype = C.c_int
    lib.ahs_device_count.restype = C.c_int
    lib.ahs_get_limits.argtypes = [C.POINTER(Limits)]
    lib.ahs_phase_batch.argtypes = [C.POINTER(BatchIn), C.POINTER(BatchOut), C.c_int]
    lib.ahs_phase_batch.restype = C.c_int
    lib.ahs_phase_batch_multi.argtypes = [C.POINTER(BatchIn), C.POINTER(BatchOut), C.POINTER(C.c_int), C.c_int]
    lib.ahs_phase_batch_multi.restype = C.c_int
    lib.ahs_phase_batch_resident.argtypes = [C.POINTER(BatchIn), C.POINTER(BatchOut), C.c_int, C.c_int, C.c_int]
    lib.ahs_phase_batch_resident.restype = C.c_int
    lib.ahs_phase_batch_genotyped.argtypes = [C.POINTER(BatchIn), u8p, C.POINTER(BatchOut), C.POINTER(C.c_int), C.c_int]
    lib.ahs_phase_batch_genotyped.restype = C.c_int
    lib.ahs_free_out.argtypes = [C.POINTER(BatchOut)]
    lib.ahs_last_error.restype = C.c_char_p
    lib.ahs_chain_cost.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int]
    lib.ahs_chain_cost.restype = C.c_double
    lib.ahs_plan_shares.argtypes = [C.POINTER(C.c_double), C.c_int64, C.c_int, C.POINTER(C.c_int64)]
    lib.ahs_plan_shares.restype = C.c_int
    lib.ahs_warmup.argtypes = [C.c_int, C.c_uint64, C.c_uint64]
    lib.ahs_warmup.restype = C.c_int
    lib.ahs_pin_host.argtypes = [C.c_void_p, C.c_uint64]
    lib.ahs_pin_host.restype = C.c_int
    lib.ahs_unpin_host.argtypes = [C.c_void_p]
    lib.ahs_unpin_host.restype = C.c_int
    lib.ahs_debug_std_sort.argtypes = [i32p, i32p, C.c_int32, C.c_int, C.c_int]
    lib.ahs_debug_std_sort.restype = C.c_int
    _lib = lib
    return lib


def pin_batch(batch: Batch) -> None:
    """Page-lock the batch's host arrays (bench: H2D from pinned memory)."""
    lib = load_library()
    for k in _I32 + _I64 + ("entry_identity",):
        a = getattr(batch, k)
        if a.nbytes:
            rc = lib.ahs_pin_host(a.ctypes.data, a.nbytes)
            if rc != 0:
                raise RuntimeError("ahs_pin_host failed: " + lib.ahs_last_error().decode())


def unpin_batch(batch: Batch) -> None:
    lib = load_library()
    for k in _I32 + _I64 + ("entry_identity",):
        a = getattr(batch, k)
        if a.nbytes:
            lib.ahs_unpin_host(a.ctypes.data)


def debug_std_sort(keys, values, descending=False, device=0):
    """Device replay of libstdc++'s std::sort (comparator on the key only); returns sorted copies."""
    lib = load_library()
    k = np.ascontiguousarray(keys, dtype=np.int32).copy(); v = np.ascontiguousarray(values, dtype=np.int32).copy()
    rc = lib.ahs_debug_std_sort(k.ctypes.data_as(i32p), v.ctypes.data_as(i32p), len(k), int(descending), device)
    if rc != 0:
        raise RuntimeError(f"ahs_debug_std_sort failed ({rc}): {lib.ahs_last_error().decode()}")
    return k, v


def limits() -> Limits:
    lim = Limits()
    load_library().ahs_get_limits(C.byref(lim))
    return lim


def phase_batch(batch: Batch, device: int = 0, devices=None, resident_iters: int = 0, warmup: int = 0,
                copy: bool = True) -> PhaseResult:
    """Phase a batch on the GPU (host buffers in / out).

    copy=False returns zero-copy numpy views of the library-owned output buffers (the C ABI's own contract:
    valid until ahs_free_out); call .release() on the result before the next call on the same device.
    devices: list of CUDA ordinals -> ahs_phase_batch_multi (one contiguous, cost-balanced share of the chains per device).
    resident_iters > 0 -> ahs_phase_batch_resident (device-only timing over resident inputs).
    batch.allele_dosage set -> ahs_phase_batch_genotyped on `device` or `devices` (not with resident_iters).
    """
    lib = load_library()
    s, o = batch.c_struct(), BatchOut()
    if batch.allele_dosage is not None:
        if resident_iters > 0:
            raise ValueError("allele_dosage: the resident-input timing mode has no genotyped variant; "
                             "phase without resident_iters, or set allele_dosage to None")
        devs = list(devices) if devices is not None else [device]
        arr = (C.c_int * len(devs))(*devs)
        rc = lib.ahs_phase_batch_genotyped(C.byref(s), batch.dosage_ptr(), C.byref(o), arr, len(devs))
    elif devices is not None:
        arr = (C.c_int * len(devices))(*devices)
        rc = lib.ahs_phase_batch_multi(C.byref(s), C.byref(o), arr, len(devices))
    elif resident_iters > 0:
        rc = lib.ahs_phase_batch_resident(C.byref(s), C.byref(o), device, warmup, resident_iters)
    else:
        rc = lib.ahs_phase_batch(C.byref(s), C.byref(o), device)
    if rc != 0:
        raise RuntimeError(f"ahs_phase_batch failed ({rc}): {lib.ahs_last_error().decode()}")
    if not copy:
        r = result_from_struct(o, copy=False)
        r._owner = (lib, o)
        return r
    try:
        return result_from_struct(o)
    finally:
        lib.ahs_free_out(C.byref(o))
