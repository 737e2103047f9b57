"""ctypes bindings of the CPU oracle (oracle/liboracle.so) and of oracle/_ref.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  Nothing under coast_b200/
imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

K_CRC16, K_SHA256, K_AES128, K_MM_U32, K_GEMM_TF32, K_QSORT, K_CHSTONE_SHA, K_CHSTONE_AES = range(8)
F_COUNT_ERRORS, F_COUNT_SYNCS, F_NO_MEM_REPLICATION, F_MAJORITY = 1, 2, 4, 0x100
F_STORE_DATA_SYNC, F_NO_STORE_DATA_SYNC, F_NO_LOAD_SYNC, F_NO_STORE_ADDR_SYNC = 0x200, 0x400, 0x800, 0x1000
PLAN_NONE, PLAN_BERNOULLI, PLAN_TABLE = 0, 1, 2
AES_DECRYPT, AES_KEY_PER_UNIT = 1, 2
NO_FAULT_UNIT = 0xFFFFFFFFFFFFFFFF


class OrcPlan(C.Structure):
    _fields_ = [("mode", C.c_uint32), ("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32),
                ("threshold", C.c_uint32), ("table", C.c_void_p)]


class OrcFault(C.Structure):
    _fields_ = [("active", C.c_int), ("replica", C.c_uint32), ("site", C.c_uint32), ("bit", C.c_uint32)]


class OrcStats(C.Structure):
    _fields_ = [("errors_corrected", C.c_uint64), ("dwc_detected", C.c_uint64), ("syncs", C.c_uint64),
                ("injected", C.c_uint64), ("first_fault_unit", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class OrcDesc(C.Structure):
    _fields_ = [("kernel", C.c_uint32), ("num_clones", C.c_uint32), ("flags", C.c_uint32), ("mode", C.c_uint32),
                ("n_units", C.c_uint64), ("unit_base", C.c_uint64),
                ("unit_bytes", C.c_uint32), ("M", C.c_uint32), ("N", C.c_uint32), ("K", C.c_uint32),
                ("inp", C.c_void_p), ("out", C.c_void_p), ("aux", C.c_void_p),
                ("key", C.c_uint8 * 16), ("plan", C.POINTER(OrcPlan))]


def build(force: bool = False) -> None:
    """Compile liboracle.so (always) and oracle/_ref (only where /root/reference exists)."""
    if force or not os.path.exists(os.path.join(HERE, "liboracle.so")) or \
            os.path.getmtime(os.path.join(HERE, "liboracle.so")) < os.path.getmtime(os.path.join(HERE, "coast_oracle.c")):
        subprocess.run(["make", "-s", "-C", HERE, "liboracle.so"], check=True)
    if os.path.exists("/root/reference/tests/crc16/crc16.c"):
        subprocess.run(["make", "-s", "-C", HERE, "ref"], check=True)


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(os.path.join(HERE, "liboracle.so"))
        L.orc_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.orc_fill_philox.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32]
        L.orc_fault_sites.argtypes = [C.c_uint32] * 3
        L.orc_fault_sites.restype = C.c_uint32
        L.orc_fault_site_bits.argtypes = [C.c_uint32] * 4
        L.orc_fault_site_bits.restype = C.c_uint32
        L.orc_out_bytes_per_unit.argtypes = [C.c_uint32]
        L.orc_out_bytes_per_unit.restype = C.c_uint32
        L.orc_votes_per_unit.argtypes = [C.c_uint32]
        L.orc_votes_per_unit.restype = C.c_uint32
        L.orc_fault_for_unit.argtypes = [C.POINTER(OrcPlan), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                         C.c_uint64, C.c_uint64, C.POINTER(OrcFault)]
        L.orc_crc16.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(OrcFault)]
        L.orc_crc16.restype = C.c_uint16
        L.orc_sha256.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(OrcFault)]
        L.orc_aes128.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(OrcFault)]
        L.orc_chstone_sha.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(OrcFault)]
        L.orc_run.argtypes = [C.POINTER(OrcDesc), C.POINTER(OrcStats)]
        L.orc_run_mt.argtypes = [C.POINTER(OrcDesc), C.c_int, C.POINTER(OrcStats)]
        _lib = L
    return _lib


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(c, k, o)
    return list(o)


def fill_philox(n_words: int, word_base: int, seed: int) -> np.ndarray:
    out = np.empty(n_words, dtype=np.uint32)
    lib().orc_fill_philox(out.ctypes.data, n_words, word_base, seed)
    return out


def fault_sites(kernel, unit_bytes=0, K=0):
    return int(lib().orc_fault_sites(kernel, unit_bytes, K))


def fault_site_bits(kernel, unit_bytes, K, site):
    return int(lib().orc_fault_site_bits(kernel, unit_bytes, K, site))


def out_bytes_per_unit(kernel):
    return int(lib().orc_out_bytes_per_unit(kernel))


def votes_per_unit(kernel):
    return int(lib().orc_votes_per_unit(kernel))


def fault_entry(replica, site, bit):
    return 0x80000000 | ((replica & 3) << 29) | ((site & 0xFFFFFF) << 5) | (bit & 31)


def fault_for_unit(plan, kernel, num_clones, unit_bytes, K, unit, local=None):
    f = OrcFault()
    lib().orc_fault_for_unit(C.byref(plan) if plan is not None else None, kernel, num_clones, unit_bytes, K,
                             unit, unit if local is None else local, C.byref(f))
    return (f.replica, f.site, f.bit) if f.active else None


def make_plan(mode=PLAN_NONE, seed=0, p=0.0, table: np.ndarray | None = None, threshold=None):
    pl = OrcPlan()
    pl.mode = mode
    pl.seed_lo = seed & 0xFFFFFFFF
    pl.seed_hi = (seed >> 32) & 0xFFFFFFFF
    pl.threshold = int(threshold if threshold is not None else min(int(p * 2 ** 32), 0xFFFFFFFF))
    pl.table = table.ctypes.data if table is not None else None
    pl._keep = table
    return pl


def run(kernel, num_clones, inp: np.ndarray, n_units, *, flags=0, mode=0, unit_bytes=0, M=0, N=0, K=0,
        aux: np.ndarray | None = None, key: bytes | None = None, plan: OrcPlan | None = None, unit_base=0,
        threads=1):
    """Run the protected region on the CPU oracle.  Returns (out: np.ndarray[uint8], stats: dict)."""
    L = lib()
    ob = unit_bytes if kernel == K_QSORT else out_bytes_per_unit(kernel)
    out = np.zeros(n_units * ob, dtype=np.uint8)
    d = OrcDesc()
    d.kernel, d.num_clones, d.flags, d.mode = kernel, num_clones, flags, mode
    d.n_units, d.unit_base, d.unit_bytes = n_units, unit_base, unit_bytes
    d.M, d.N, d.K = M, N, K
    inp = np.ascontiguousarray(inp)
    d.inp = inp.ctypes.data
    d.out = out.ctypes.data
    if aux is not None:
        aux = np.ascontiguousarray(aux)
        d.aux = aux.ctypes.data
    if key is not None:
        d.key = (C.c_uint8 * 16)(*key)
    if plan is not None:
        d.plan = C.pointer(plan)
    st = OrcStats()
    st.first_fault_unit = NO_FAULT_UNIT
    rc = L.orc_run_mt(C.byref(d), threads, C.byref(st)) if threads > 1 else L.orc_run(C.byref(d), C.byref(st))
    if rc != 0:
        raise ValueError("orc_run: bad descriptor")
    return out, st.as_dict()


def crc16(data: bytes) -> int:
    buf = np.frombuffer(data, dtype=np.uint8)
    return int(lib().orc_crc16(buf.ctypes.data, len(data), None))


def sha256(data: bytes) -> bytes:
    buf = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, dtype=np.uint8)
    out = np.zeros(32, dtype=np.uint8)
    lib().orc_sha256(buf.ctypes.data, len(data), out.ctypes.data, None)
    return out.tobytes()


def chstone_sha(data: bytes) -> list:
    """sha_info_digest[5] of tests/chstone/sha for one stream (len(data) % 64 == 0)."""
    buf = np.frombuffer(data, dtype=np.uint8)
    out = np.zeros(5, dtype=np.uint32)
    lib().orc_chstone_sha(buf.ctypes.data, len(data), out.ctypes.data, None)
    return [int(x) for x in out]


def chstone_site_of_input_bit(byte: int, bit: int):
    """(site, bit) of the fault plan that flips `bit` of input byte `byte` as the replica loads it (little-endian W[])."""
    return 421 * (byte // 64) + (byte % 64) // 4, 8 * (byte % 4) + bit


def aes128(state: bytes, key: bytes, direction: int):
    s = np.frombuffer(state, dtype=np.uint8).copy()
    k = np.frombuffer(key, dtype=np.uint8).copy()
    lib().orc_aes128(s.ctypes.data, k.ctypes.data, direction, None)
    return s.tobytes(), k.tobytes()


# ---------------------------------------------------------------------------
# oracle/_ref: the reference's own sources, compiled from /root/reference.
# ---------------------------------------------------------------------------
class RefStats(C.Structure):
    _fields_ = OrcStats._fields_

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class RefFault(C.Structure):
    _fields_ = [("replica", C.c_int), ("byte", C.c_int), ("bit", C.c_int)]


def ref_available() -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", "libref_sha256.so"))


_refs = {}


def ref(name: str):
    """Load oracle/_ref/libref_<name>.so (RTLD_LOCAL: the reference reuses global names across tests)."""
    if name not in _refs:
        path = os.path.join(HERE, "_ref", f"libref_{name}.so")
        if not os.path.exists(path):
            build()
        _refs[name] = C.CDLL(path, mode=os.RTLD_LOCAL if hasattr(os, "RTLD_LOCAL") else 0)
    return _refs[name]
