"""ctypes access to the CPU oracle (oracle/libcdoracle.so).  TEST INFRASTRUCTURE ONLY.

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs; the product package never imports this module.
PARITY UNPINNED — see oracle/cdoracle.h for why and for the reference citations.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcdoracle.so")
FAKE_NVML = os.path.join(HERE, "..", "tests", "fake_nvml", "libnvidia-ml.so.1")
MAX_GPUS = 16
MAX_LINKS = 18
_N2 = MAX_GPUS * MAX_GPUS

FLAG_LEGACY_CLIQUE = 0x1
FLAG_NO_ENUMERATE = 0x2
FLAG_NO_IMEX_CTL = 0x4
FLAG_THREADS = 0x8


class NvmlT(C.Structure):
    _fields_ = [
        ("n", C.c_uint32),
        ("reach", C.c_uint8 * _N2),
        ("link_active", (C.c_uint8 * MAX_LINKS) * MAX_GPUS),
        ("n_links", C.c_uint8 * MAX_GPUS),
        ("mig_enabled", C.c_uint8 * MAX_GPUS),
        ("fabric_state", C.c_uint8 * MAX_GPUS),
        ("fabric_ret", C.c_int32 * MAX_GPUS),
        ("fabric_status", C.c_int32 * MAX_GPUS),
        ("fabric_clique", C.c_uint32 * MAX_GPUS),
        ("cluster_uuid", (C.c_uint8 * 16) * MAX_GPUS),
        ("p2p_read", C.c_int32 * _N2),
        ("p2p_write", C.c_int32 * _N2),
        ("p2p_nvlink", C.c_int32 * _N2),
        ("uuid", (C.c_char * 96) * MAX_GPUS),
        ("name", (C.c_char * 96) * MAX_GPUS),
        ("pci_bus_id", (C.c_char * 32) * MAX_GPUS),
        ("memory_total", C.c_uint64 * MAX_GPUS),
        ("minor", C.c_int32 * MAX_GPUS),
        ("cc_major", C.c_int32 * MAX_GPUS),
        ("cc_minor", C.c_int32 * MAX_GPUS),
        ("driver_version", C.c_char * 96),
        ("cuda_driver_version", C.c_int32),
        ("clique_id", C.c_char * 96),
        ("clique_err", C.c_int32),
        ("clique_err_text", C.c_char * 160),
        ("imex_gate", C.c_int32),
        ("nvml_calls", C.c_uint32),
        ("init_ms", C.c_double),
        ("enumerate_ms", C.c_double),
        ("fabric_ms", C.c_double),
        ("link_poll_ms", C.c_double),
        ("p2p_poll_ms", C.c_double),
        ("imex_ms", C.c_double),
        ("shutdown_ms", C.c_double),
        ("total_ms", C.c_double),
    ]

    def reach_matrix(self):
        return [[self.reach[i * MAX_GPUS + j] for j in range(self.n)] for i in range(self.n)]

    def uuids(self):
        return [self.uuid[i].value.decode() for i in range(self.n)]


class PlanT(C.Structure):
    _fields_ = [
        ("n", C.c_uint32),
        ("rounds", C.c_uint32),
        ("n_slots", C.c_uint32),
        ("n_slices", C.c_uint32),
        ("bytes_per_pair", C.c_uint64),
        ("src_bytes", C.c_uint64),
        ("land_bytes", C.c_uint64),
        ("partner", (C.c_int8 * MAX_GPUS) * MAX_GPUS),
    ]


_lib = None


def build() -> None:
    subprocess.run(["make", "-C", HERE, "-s"], check=True, capture_output=True)


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build()
    L = C.CDLL(LIB_PATH)
    u64, u32 = C.c_uint64, C.c_uint32
    L.cdoracle_nvml_poll.restype = C.c_int
    L.cdoracle_nvml_poll.argtypes = [u32, u32, C.POINTER(NvmlT)]
    L.cdoracle_splitmix64.restype = u64
    L.cdoracle_splitmix64.argtypes = [u64]
    L.cdoracle_src_word.restype = u64
    L.cdoracle_src_word.argtypes = [u64, u32, u64]
    L.cdoracle_write_salt.restype = u64
    L.cdoracle_write_salt.argtypes = [u64, u32, u32, u64]
    L.cdoracle_write_word.restype = u64
    L.cdoracle_write_word.argtypes = [u64, u64]
    L.cdoracle_checksum.restype = None
    L.cdoracle_checksum.argtypes = [C.POINTER(u64), u64, C.POINTER(u64), C.POINTER(u64)]
    L.cdoracle_src_checksum.restype = None
    L.cdoracle_src_checksum.argtypes = [u64, u32, u64, u64, C.POINTER(u64), C.POINTER(u64)]
    L.cdoracle_write_checksum.restype = None
    L.cdoracle_write_checksum.argtypes = [u64, u32, u32, u64, u64, C.POINTER(u64), C.POINTER(u64)]
    L.cdoracle_plan.restype = C.c_int
    L.cdoracle_plan.argtypes = [u32, u64, u32, u32, C.POINTER(PlanT)]
    L.cdoracle_slot.restype = u32
    L.cdoracle_slot.argtypes = [u32, u32]
    _lib = L
    return L


DEFAULT_SEED = 0xCD5EED0000000001


def nvml_poll(n_max: int = 0, flags: int = 0) -> NvmlT:
    out = NvmlT()
    rc = lib().cdoracle_nvml_poll(n_max, flags, C.byref(out))
    if rc != 0:
        raise RuntimeError(f"cdoracle_nvml_poll failed: rc={rc} (-1: libnvidia-ml.so.1 not loadable)")
    return out


def nvml_poll_rc(n_max: int = 0, flags: int = 0):
    out = NvmlT()
    rc = lib().cdoracle_nvml_poll(n_max, flags, C.byref(out))
    return rc, out


def src_checksum(seed: int, rank: int, first_word: int, n_words: int):
    s, x = C.c_uint64(), C.c_uint64()
    lib().cdoracle_src_checksum(seed, rank, first_word, n_words, C.byref(s), C.byref(x))
    return s.value, x.value


def write_checksum(seed: int, src: int, dst: int, run_seq: int, n_words: int):
    s, x = C.c_uint64(), C.c_uint64()
    lib().cdoracle_write_checksum(seed, src, dst, run_seq, n_words, C.byref(s), C.byref(x))
    return s.value, x.value


def checksum(words):
    """(S, X) of a numpy.uint64 array of words, by cdoracle_checksum (granules counted from words[0])."""
    import numpy as np

    w = np.ascontiguousarray(words, dtype=np.uint64)
    s, x = C.c_uint64(), C.c_uint64()
    lib().cdoracle_checksum(w.ctypes.data_as(C.POINTER(C.c_uint64)), w.size, C.byref(s), C.byref(x))
    return s.value, x.value


_GOLDEN = 0x9E3779B97F4A7C15
_WRITE_TAG = 0x5752495445  # "WRITE"
_M64 = (1 << 64) - 1


def _splitmix64_np(x):
    """pattern.c's cdoracle_splitmix64 over a numpy.uint64 array (wrapping arithmetic)."""
    import numpy as np

    u = np.uint64
    z = x + u(_GOLDEN)
    z ^= z >> u(30)
    z *= u(0xBF58476D1CE4E5B9)
    z ^= z >> u(27)
    z *= u(0x94D049BB133111EB)
    z ^= z >> u(31)
    return z


def src_words(seed: int, rank: int, first_word: int, n: int):
    """Words first_word .. first_word + n - 1 of rank `rank`'s source buffer, as a numpy.uint64 array
    (vectorised restatement of cdoracle_src_word: splitmix64(seed ^ rank << 56 ^ k))."""
    import numpy as np

    k = np.arange(n, dtype=np.uint64) + np.uint64(first_word)
    return _splitmix64_np(k ^ np.uint64((seed ^ (rank << 56)) & _M64))


def write_words(seed: int, src: int, dst: int, run_seq: int, first_word: int, n: int):
    """Words first_word .. first_word + n - 1 of what rank `src` stores into rank `dst`'s landing slot in run
    `run_seq`, as a numpy.uint64 array (cdoracle_write_salt + cdoracle_write_word: z = (salt + k) * golden,
    w = z ^ z >> 32)."""
    import numpy as np

    x = (seed ^ _WRITE_TAG ^ (src << 56) ^ (dst << 48) ^ run_seq) & _M64
    salt = _splitmix64_np(np.array([x], dtype=np.uint64))[0]
    z = (np.arange(n, dtype=np.uint64) + np.uint64(first_word) + salt) * np.uint64(_GOLDEN)
    return z ^ (z >> np.uint64(32))


def plan(n: int, nbytes: int, mode: int, diag: bool = False) -> PlanT:
    p = PlanT()
    rc = lib().cdoracle_plan(n, nbytes, mode, 1 if diag else 0, C.byref(p))
    if rc != 0:
        raise ValueError("cdoracle_plan: bad argument")
    return p


def expected_read(seed: int, n: int, nbytes: int, mode: int, issuer: int, owner: int, diag: bool = False):
    """(S, X) the read probe of `issuer` must compute on `owner`'s source buffer."""
    p = plan(n, nbytes, mode, diag)
    words = p.bytes_per_pair // 8
    if mode == 2:
        first = 0
    elif issuer == owner:
        first = (n - 1) * words
    else:
        first = lib().cdoracle_slot(issuer, owner) * words
    return src_checksum(seed, owner, first, words)
