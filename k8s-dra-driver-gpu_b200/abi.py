"""ctypes mirror of include/cdprobe.h (the structs a cgo shim would see as C.cdprobe_*_t)."""
from __future__ import annotations

import ctypes as C
import os

MAX_GPUS = 16
MAX_PHASES = 64
ABI_VERSION = 2

OK = 0
ERR_ABI, ERR_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_TIMEOUT = -1, -2, -3, -4, -5
ERR_RENDEZVOUS, ERR_NOMEM, ERR_UNSUPPORTED, ERR_STATE, ERR_INTEGRITY = -6, -7, -8, -9, -10

MODE_REACH_ONLY, MODE_SLICED, MODE_FULL = 0, 1, 2
OP_READ, OP_WRITE = 1, 2
FLAG_FABRIC_HANDLES = 0x01
FLAG_MIG_AWARE = 0x02
FLAG_LOCAL_DIAG = 0x04
FLAG_PATH_LDST = 0x08
FLAG_NO_COOPERATIVE = 0x10
FLAG_OVERLAP_VERIFY = 0x20
FLAG_ALLOW_SAME_DEVICE = 0x40
FLAG_UNIDIRECTIONAL = 0x80
FLAG_SERIAL_VERIFY = 0x100
FLAG_SIMULATE_MIG = 0x200
FLAG_ALL_RANK_BARRIERS = 0x400
FLAG_PAIR_BARRIERS = 0x800

OPT_EVENT_TIMING, OPT_CTAS, OPT_PATH, OPT_TIMEOUT_MS, OPT_OVERLAP_VERIFY, OPT_VERIFY_CTAS = 1, 2, 3, 4, 5, 6
OPT_UNIDIRECTIONAL = 7
OPT_WARMUP, OPT_WARMUP_BYTES, OPT_DEBUG_SKIP_RANK = 8, 9, 10
OPT_CTAS_RANK, OPT_MIN_FRACTION_PPM, OPT_LINK_PEAK_MBPS, OPT_SOLO_RANK, OPT_ALL_RANK_BARRIERS = 11, 12, 13, 14, 15
OPT_PAIR_BARRIERS = 16
OPT_DEBUG_DAMAGE_WRITE = 17

_N2 = MAX_GPUS * MAX_GPUS


class ConfigT(C.Structure):
    _fields_ = [
        ("abi", C.c_uint32),
        ("n_gpus", C.c_uint32),
        ("ordinals", C.c_int32 * MAX_GPUS),
        ("bytes", C.c_uint64),
        ("mode", C.c_uint32),
        ("ops", C.c_uint32),
        ("timeout_ms", C.c_uint32),
        ("flags", C.c_uint32),
        ("seed", C.c_uint64),
        ("min_fraction", C.c_float),
        ("link_peak_gbps", C.c_float),
        ("ctas", C.c_uint32),
        ("world_size", C.c_uint32),
        ("rank", C.c_uint32),
        ("reserved0", C.c_uint32),
        ("session", C.c_char * 64),
    ]


class ResultT(C.Structure):
    _fields_ = [
        ("abi", C.c_uint32),
        ("n", C.c_uint32),
        ("row_mask", C.c_uint32),
        ("verdict", C.c_uint32),
        ("reach_read", C.c_uint8 * _N2),
        ("reach_write", C.c_uint8 * _N2),
        ("gbps_read", C.c_float * _N2),
        ("gbps_write", C.c_float * _N2),
        ("status", C.c_int32 * _N2),
        ("sum_read", C.c_uint64 * _N2),
        ("xor_read", C.c_uint64 * _N2),
        ("sum_write", C.c_uint64 * _N2),
        ("xor_write", C.c_uint64 * _N2),
        ("bytes_per_pair", C.c_uint64),
        ("run_seq", C.c_uint64),
        ("rounds", C.c_uint32),
        ("phases", C.c_uint32),
        ("launches", C.c_uint32),
        ("aborted", C.c_uint32),
        ("warmed", C.c_uint32),
        ("reserved1", C.c_uint32),
        ("probe_ms", C.c_double),
        ("device_ms", C.c_double * MAX_GPUS),
        ("barrier_us", C.c_double * MAX_GPUS),
        ("event_ms", C.c_double * MAX_GPUS),
        ("min_gbps_read", C.c_float),
        ("min_gbps_write", C.c_float),
        ("gate_gbps_read", C.c_float),
        ("gate_gbps_write", C.c_float),
        ("kernel_ms", C.c_double * MAX_GPUS),
        ("unreachable_pairs", C.c_uint32),
        ("slow_pairs", C.c_uint32),
    ]


class InfoT(C.Structure):
    _fields_ = [
        ("abi", C.c_uint32),
        ("n", C.c_uint32),
        ("n_local", C.c_uint32),
        ("first_local_rank", C.c_uint32),
        ("ordinal", C.c_int32 * MAX_GPUS),
        ("sm_count", C.c_uint32 * MAX_GPUS),
        ("ctas", C.c_uint32 * MAX_GPUS),
        ("mig", C.c_uint32 * MAX_GPUS),
        ("uuid", (C.c_char * 48) * MAX_GPUS),
        ("handle_type", C.c_uint32),
        ("path", C.c_uint32),
        ("bytes_per_pair", C.c_uint64),
        ("alloc_bytes", C.c_uint64),
        ("src_sum", (C.c_uint64 * MAX_GPUS) * MAX_GPUS),
        ("src_xor", (C.c_uint64 * MAX_GPUS) * MAX_GPUS),
        ("n_slices", C.c_uint32),
        ("smem_bytes", C.c_uint32),
        ("open_ms", C.c_double),
        ("fill_ms", C.c_double),
    ]


class PlanT(C.Structure):
    _fields_ = [
        ("abi", C.c_uint32),
        ("n", C.c_uint32),
        ("rounds", C.c_uint32),
        ("n_slots", C.c_uint32),
        ("n_slices", C.c_uint32),
        ("reserved", C.c_uint32),
        ("bytes_per_pair", C.c_uint64),
        ("src_bytes", C.c_uint64),
        ("land_bytes", C.c_uint64),
        ("partner", (C.c_int8 * MAX_GPUS) * MAX_GPUS),
    ]


class TraceT(C.Structure):
    _fields_ = [
        ("abi", C.c_uint32),
        ("n_phases", C.c_uint32),
        ("kind0", C.c_uint8 * MAX_PHASES),
        ("kind1", C.c_uint8 * MAX_PHASES),
        ("peer0", C.c_int8 * MAX_PHASES),
        ("peer1", C.c_int8 * MAX_PHASES),
        ("sync_all", C.c_uint8 * MAX_PHASES),
        ("sync_mask", C.c_uint16 * MAX_PHASES),
        ("post_mask", C.c_uint16 * MAX_PHASES),
        ("t_start", C.c_uint64 * MAX_PHASES),
        ("t_end0", C.c_uint64 * MAX_PHASES),
        ("t_end1", C.c_uint64 * MAX_PHASES),
        ("t_arrive", C.c_uint64 * MAX_PHASES),
    ]


class TopologyT(C.Structure):
    _fields_ = [
        ("abi", C.c_uint32),
        ("n", C.c_uint32),
        ("uuid", (C.c_char * 96) * MAX_GPUS),
        ("pci_bus_id", (C.c_char * 32) * MAX_GPUS),
        ("mig", C.c_uint8 * MAX_GPUS),
        ("links_active", C.c_uint8 * MAX_GPUS),
        ("link_mask", C.c_uint32 * MAX_GPUS),
        ("fabric_state", C.c_uint8 * MAX_GPUS),
        ("clique_id", C.c_char * 96),
        ("clique_error", C.c_char * 160),
    ]


class ScheduleT(C.Structure):
    _fields_ = [
        ("abi", C.c_uint32),
        ("n_phases", C.c_uint32),
        ("peer_mask", C.c_uint32),
        ("reserved", C.c_uint32),
        ("kind", (C.c_uint8 * MAX_PHASES) * 2),
        ("peer", (C.c_int8 * MAX_PHASES) * 2),
        ("slot", (C.c_uint8 * MAX_PHASES) * 2),
        ("writer", (C.c_uint8 * MAX_PHASES) * 2),
        ("cta0", (C.c_uint16 * MAX_PHASES) * 2),
        ("nctas", (C.c_uint16 * MAX_PHASES) * 2),
        ("sync_all", C.c_uint8 * MAX_PHASES),
        ("sync_mask", C.c_uint16 * MAX_PHASES),
        ("post_mask", C.c_uint16 * MAX_PHASES),
        ("wait_barrier", (C.c_uint8 * MAX_PHASES) * 2),
    ]


# Every symbol include/cdprobe.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "cdprobe_abi_version": (C.c_uint32, []),
    "cdprobe_strerror": (C.c_char_p, [C.c_int]),
    "cdprobe_last_error": (C.c_char_p, []),
    "cdprobe_open": (C.c_int, [C.POINTER(ConfigT), C.POINTER(C.c_void_p)]),
    "cdprobe_run": (C.c_int, [C.c_void_p, C.POINTER(ResultT)]),
    "cdprobe_gather": (C.c_int, [C.c_void_p, C.POINTER(ResultT)]),
    "cdprobe_info": (C.c_int, [C.c_void_p, C.POINTER(InfoT)]),
    "cdprobe_trace": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(TraceT)]),
    "cdprobe_set_option": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64]),
    "cdprobe_remap_peer": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "cdprobe_unmap_peer": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "cdprobe_corrupt": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64]),
    "cdprobe_peek": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]),
    "cdprobe_ce_copy": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_uint32,
                                  C.c_uint64, C.c_uint32, C.POINTER(C.c_double)]),
    "cdprobe_close": (None, [C.c_void_p]),
    "cdprobe_plan": (C.c_int, [C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(PlanT)]),
    "cdprobe_topology": (C.c_int, [C.c_uint32, C.POINTER(TopologyT)]),
    "cdprobe_schedule": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                   C.c_uint32, C.POINTER(ScheduleT)]),
    "cdprobe_rendezvous_selftest": (C.c_int, [C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "cdprobe_gate": (C.c_int, [C.POINTER(ConfigT), C.c_uint32, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
}

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libcdprobe.so")
_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen libcdprobe.so (lazily, like go-nvml does for NVML) and type every entry point.

    There is no fallback: a missing library is an error, never a silent CPU path.
    """
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise OSError(f"{p} not found: build it with `python k8s-dra-driver-gpu_b200/build.py` (needs nvcc)")
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib
