"""Host-side mirror of the Go shim ``pkg/fabricprobe`` (SURVEY.md §8b).

Go signature being mirrored (see INTEGRATION.md for the cgo file)::

    type Config struct{ Ordinals []int; Bytes uint64; Mode, Ops, TimeoutMs, Flags uint32; ... }
    type Result struct{ N int; ReachRead, ReachWrite []bool /* N x N row-major */
                        GBpsRead, GBpsWrite []float32; ProbeMs float64; ... }
    func Open(Config) (*Probe, error)
    func (*Probe) Run(ctx) (Result, error)
    func (*Probe) Close()

Caller in the reference tree: ``run()`` in cmd/compute-domain-daemon/main.go:212-347
owns the probe; ``check()`` (main.go:435-459) reads its cached verdict.  Errors
follow the daemon's convention: a Python exception here is a Go ``error`` there;
``ErrUnsupported`` is what the ``!cgo`` stub returns.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import List, Optional, Sequence

from . import abi


class ProbeError(RuntimeError):
    def __init__(self, code: int, what: str, detail: str = ""):
        self.code = code
        self.detail = detail
        super().__init__(f"{what}: {detail}" if detail else what)


class ErrUnsupported(ProbeError):
    """No CUDA driver / no sm_100 GPU: the probe cannot run and nothing stands in for it."""


@dataclasses.dataclass
class Config:
    ordinals: Optional[Sequence[int]] = None  # None = all visible GPUs
    bytes: int = 1 << 30
    mode: int = abi.MODE_SLICED
    ops: int = abi.OP_READ | abi.OP_WRITE
    timeout_ms: int = 5000
    flags: int = 0
    seed: int = 0
    min_fraction: float = 0.0  # 0 = library default (0.90 of the calibrated reference; 0.65 of an explicit peak)
    link_peak_gbps: float = 0.0  # 0 = calibrated reference (include/cdprobe.h); > 0 = absolute GB/s
    ctas: int = 0
    world_size: int = 1
    rank: int = 0
    session: str = ""

    def to_c(self) -> abi.ConfigT:
        c = abi.ConfigT()
        c.abi = abi.ABI_VERSION
        if self.ordinals is None:
            c.n_gpus = 0
        else:
            c.n_gpus = len(self.ordinals)
            for i, o in enumerate(self.ordinals):
                c.ordinals[i] = int(o)
        c.bytes = int(self.bytes)
        c.mode = self.mode
        c.ops = self.ops
        c.timeout_ms = self.timeout_ms
        c.flags = self.flags
        c.seed = self.seed
        c.min_fraction = self.min_fraction
        c.link_peak_gbps = self.link_peak_gbps
        c.ctas = self.ctas
        c.world_size = self.world_size
        c.rank = self.rank
        c.session = self.session.encode()[:63]
        return c


@dataclasses.dataclass
class Result:
    n: int
    row_mask: int
    verdict: bool
    reach_read: List[List[int]]
    reach_write: List[List[int]]
    gbps_read: List[List[float]]
    gbps_write: List[List[float]]
    status: List[List[int]]
    sum_read: List[List[int]]
    xor_read: List[List[int]]
    sum_write: List[List[int]]
    xor_write: List[List[int]]
    bytes_per_pair: int
    run_seq: int
    rounds: int
    phases: int
    launches: int
    aborted: bool
    warmed: bool
    probe_ms: float
    device_ms: List[float]
    barrier_us: List[float]
    event_ms: List[float]
    min_gbps_read: float
    min_gbps_write: float
    gate_gbps_read: float = 0.0
    gate_gbps_write: float = 0.0
    unreachable_pairs: int = 0
    slow_pairs: int = 0
    kernel_ms: List[float] = dataclasses.field(default_factory=list)
    raw: abi.ResultT = dataclasses.field(repr=False, default=None)

    @property
    def reach(self) -> List[List[int]]:
        """reach_read AND reach_write — what is compared with the NVML oracle (SURVEY §8c)."""
        return [[a & b for a, b in zip(ra, rb)] for ra, rb in zip(self.reach_read, self.reach_write)]

    @staticmethod
    def from_c(r: abi.ResultT) -> "Result":
        n = r.n

        def mat(a):
            return [[a[i * abi.MAX_GPUS + j] for j in range(n)] for i in range(n)]

        return Result(
            n=n,
            row_mask=r.row_mask,
            verdict=bool(r.verdict),
            reach_read=mat(r.reach_read),
            reach_write=mat(r.reach_write),
            gbps_read=mat(r.gbps_read),
            gbps_write=mat(r.gbps_write),
            status=mat(r.status),
            sum_read=mat(r.sum_read),
            xor_read=mat(r.xor_read),
            sum_write=mat(r.sum_write),
            xor_write=mat(r.xor_write),
            bytes_per_pair=r.bytes_per_pair,
            run_seq=r.run_seq,
            rounds=r.rounds,
            phases=r.phases,
            launches=r.launches,
            aborted=bool(r.aborted),
            warmed=bool(r.warmed),
            probe_ms=r.probe_ms,
            device_ms=list(r.device_ms)[:n],
            barrier_us=list(r.barrier_us)[:n],
            event_ms=list(r.event_ms)[:n],
            min_gbps_read=r.min_gbps_read,
            min_gbps_write=r.min_gbps_write,
            gate_gbps_read=r.gate_gbps_read,
            gate_gbps_write=r.gate_gbps_write,
            unreachable_pairs=r.unreachable_pairs,
            slow_pairs=r.slow_pairs,
            kernel_ms=list(r.kernel_ms)[:n],
            raw=r,
        )


def _raise(lib, rc: int, what: str):
    msg = lib.cdprobe_strerror(rc).decode()
    detail = lib.cdprobe_last_error().decode()
    cls = ErrUnsupported if rc in (abi.ERR_NO_DEVICE, abi.ERR_UNSUPPORTED) else ProbeError
    raise cls(rc, f"{what}: {msg}", detail)


class Probe:
    """One probe domain handle (not thread-safe, like the C handle)."""

    def __init__(self, cfg: Config):
        self._lib = abi.load_library()
        self._h = C.c_void_p()
        self.cfg = cfg
        c = cfg.to_c()
        rc = self._lib.cdprobe_open(C.byref(c), C.byref(self._h))
        if rc != abi.OK:
            self._h = C.c_void_p()
            _raise(self._lib, rc, "cdprobe_open")

    # -- Go: (*Probe).Run -------------------------------------------------------------
    def Run(self, gather: bool = False, allow_timeout: bool = False) -> Result:
        r = abi.ResultT()
        rc = self._lib.cdprobe_run(self._h, C.byref(r))
        if rc != abi.OK and not (allow_timeout and rc == abi.ERR_TIMEOUT):
            _raise(self._lib, rc, "cdprobe_run")
        if gather:
            rc2 = self._lib.cdprobe_gather(self._h, C.byref(r))
            if rc2 != abi.OK:
                _raise(self._lib, rc2, "cdprobe_gather")
        return Result.from_c(r)

    def run_raw(self, out: abi.ResultT) -> int:
        """The bare ABI call (bench.py times this)."""
        return self._lib.cdprobe_run(self._h, C.byref(out))

    def Info(self) -> abi.InfoT:
        i = abi.InfoT()
        rc = self._lib.cdprobe_info(self._h, C.byref(i))
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_info")
        return i

    def Trace(self, local: int = 0):
        """Per-phase timeline of the last run: list of dicts (ns relative to the first barrier release)."""
        t = abi.TraceT()
        rc = self._lib.cdprobe_trace(self._h, local, C.byref(t))
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_trace")
        names = {0: "-", 1: "read", 2: "write", 3: "verify", 4: "warm"}
        return [{"job0": names[t.kind0[p]], "peer0": t.peer0[p], "job1": names[t.kind1[p]], "peer1": t.peer1[p],
                 "sync_all": int(t.sync_all[p]), "sync_mask": int(t.sync_mask[p]), "post_mask": int(t.post_mask[p]), "t_start": t.t_start[p], "t_end0": t.t_end0[p], "t_end1": t.t_end1[p],
                 "t_arrive": t.t_arrive[p]} for p in range(t.n_phases)]

    def SetOption(self, option: int, value: int) -> None:
        rc = self._lib.cdprobe_set_option(self._h, option, value)
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_set_option")

    def UnmapPeer(self, local: int, peer: int) -> None:
        rc = self._lib.cdprobe_unmap_peer(self._h, local, peer)
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_unmap_peer")

    def RemapPeer(self, local: int, peer: int) -> None:
        rc = self._lib.cdprobe_remap_peer(self._h, local, peer)
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_remap_peer")

    def CeCopy(self, copies, push: bool = True, nbytes: int = 0, reps: int = 4):
        """Copy-engine reference on the probe's buffers: `copies` = [(local rank, peer rank), ...] run concurrently;
        returns [(ms for `reps` copies, GB/s), ...].  Not part of a probe: the same-box ceiling quoted beside it."""
        k = len(copies)
        loc = (C.c_uint32 * k)(*[c[0] for c in copies])
        peer = (C.c_uint32 * k)(*[c[1] for c in copies])
        ms = (C.c_double * k)()
        rc = self._lib.cdprobe_ce_copy(self._h, k, loc, peer, 1 if push else 0, nbytes, reps, ms)
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_ce_copy")
        info = self.Info()
        pl = plan(info.n, self.cfg.bytes, self.cfg.mode, self.cfg.flags)
        nb = min(x for x in (nbytes or pl.src_bytes, pl.src_bytes, pl.land_bytes))
        return [(ms[i], nb * reps / (ms[i] * 1e-3) / 1e9 if ms[i] > 0 else 0.0) for i in range(k)]

    def Corrupt(self, local: int, byte_offset: int, xor_mask: int) -> None:
        rc = self._lib.cdprobe_corrupt(self._h, local, byte_offset, xor_mask)
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_corrupt")

    def Peek(self, local: int, byte_offset: int, nbytes: int) -> bytes:
        """`nbytes` of local rank `local`'s own allocation from `byte_offset` (Ctrl, source, landing slots; DESIGN §4)."""
        buf = C.create_string_buffer(nbytes) if nbytes > 0 else None
        rc = self._lib.cdprobe_peek(self._h, local, byte_offset, nbytes, buf)
        if rc != abi.OK:
            _raise(self._lib, rc, "cdprobe_peek")
        return buf.raw

    def Close(self) -> None:
        if self._h:
            self._lib.cdprobe_close(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.Close()

    def __del__(self):
        try:
            self.Close()
        except Exception:
            pass


def Open(cfg: Config) -> Probe:
    return Probe(cfg)


def topology(strict: bool = True) -> abi.TopologyT:
    """internal/common topology enumeration (NVML only, no CUDA)."""
    lib = abi.load_library()
    t = abi.TopologyT()
    rc = lib.cdprobe_topology(1 if strict else 0, C.byref(t))
    if rc != abi.OK:
        _raise(lib, rc, "cdprobe_topology")
    return t


def gate(cfg: Config, n_total: int):
    """(read, write) GB/s threshold the verdict of an n_total-rank domain with this config applies (host-only)."""
    lib = abi.load_library()
    r, w = C.c_float(), C.c_float()
    c = cfg.to_c()
    rc = lib.cdprobe_gate(C.byref(c), n_total, C.byref(r), C.byref(w))
    if rc != abi.OK:
        _raise(lib, rc, "cdprobe_gate")
    return r.value, w.value


def plan(n: int, nbytes: int, mode: int, flags: int = 0) -> abi.PlanT:
    lib = abi.load_library()
    p = abi.PlanT()
    rc = lib.cdprobe_plan(n, nbytes, mode, flags, C.byref(p))
    if rc != abi.OK:
        _raise(lib, rc, "cdprobe_plan")
    return p
