"""Read-back checker: the bytes a rank's probe allocation holds, word for word against the pattern oracle.

Shared by tests/test_gpu_readback.py and the one-process-per-rank children it starts.  The layout is computed
from the oracle's plan (oracle/pattern.c), not from the library, and checked against the allocation size the
library reports.  Regions of at most 64 MiB are compared whole; larger ones on windows: the first and the last
MiB (the tail unit) and +-1 MiB around byte offsets 2^31 and 2^32 of the region.
"""
from __future__ import annotations

import dataclasses

import numpy as np

from oracle import oracle

SEED = oracle.DEFAULT_SEED
MiB = 1 << 20
VMM_GRANULE = 2 * MiB       # every region of the allocation starts on a 2 MiB boundary (DESIGN §4)
FULL_COMPARE_MAX = 64 * MiB
FLAG_LOCAL_DIAG = 0x04
OP_READ, OP_WRITE = 1, 2


def _roundup(v: int, a: int) -> int:
    return (v + a - 1) // a * a


@dataclasses.dataclass
class Mismatch:
    where: str
    first_byte: int          # allocation offset of the first byte that differs
    bad_words: int           # words that differ (within the compared windows)
    word_offsets: list       # allocation offsets of the first bad words (at most 8)
    got: int                 # first bad word as read back
    expected: int

    def __str__(self):
        return (f"{self.where}: first bad byte at allocation offset {self.first_byte:#x}, {self.bad_words} bad "
                f"word(s) (read {self.got:#018x}, expected {self.expected:#018x})")


def report(mismatches) -> str:
    return "\n".join(str(m) for m in mismatches)


class Layout:
    """Where things are in one rank's allocation: Ctrl at 0, source at 2 MiB, landing slots after the source
    rounded up to 2 MiB, the allocation ending at the landing slots rounded up to 2 MiB."""

    def __init__(self, probe):
        info = probe.Info()
        cfg = probe.cfg
        self.n, self.n_local, self.first = info.n, info.n_local, info.first_local_rank
        self.diag = self.n == 1 or bool(cfg.flags & FLAG_LOCAL_DIAG)
        self.ops = cfg.ops or (OP_READ | OP_WRITE)
        pl = oracle.plan(self.n, cfg.bytes, cfg.mode, self.diag)
        self.bpp, self.n_slots, self.n_slices = pl.bytes_per_pair, pl.n_slots, pl.n_slices
        self.src_bytes, self.land_bytes = pl.src_bytes, pl.land_bytes
        self.src_off = VMM_GRANULE
        self.land_off = self.src_off + _roundup(self.src_bytes, VMM_GRANULE)
        self.alloc = info.alloc_bytes
        assert info.bytes_per_pair == self.bpp
        assert self.alloc == self.land_off + _roundup(self.land_bytes, VMM_GRANULE), \
            f"allocation layout changed: {self.alloc:#x} bytes, expected landing slots at {self.land_off:#x} + " \
            f"{self.land_bytes:#x} rounded up to 2 MiB (DESIGN §4)"

    def slot(self, writer: int, owner: int) -> int:
        """Landing slot of `owner` that `writer` fills: its index among owner's peers; the diagonal slot last."""
        if writer == owner:
            return self.n - 1
        return writer if writer < owner else writer - 1

    def slice_of(self, reader: int, owner: int) -> int:
        """Source slice of `owner` that `reader` loads."""
        return 0 if self.n_slices == 1 else self.slot(reader, owner)

    def padding(self):
        """The bytes between the regions' ends and the next 2 MiB boundary: nobody may write them."""
        return [(a, b) for a, b in ((self.src_off + self.src_bytes, self.land_off),
                                    (self.land_off + self.land_bytes, self.alloc)) if b > a]


def windows(nbytes: int):
    """Byte ranges [a, b) of a region of `nbytes` that are compared word for word."""
    if nbytes <= FULL_COMPARE_MAX:
        return [(0, nbytes)]
    w = [(0, MiB), (nbytes - MiB, nbytes)]
    for c in (1 << 31, 1 << 32):
        if c < nbytes:
            w.append((max(0, c - MiB), min(nbytes, c + MiB)))
    merged = []
    for a, b in sorted(w):
        if merged and a <= merged[-1][1]:
            merged[-1] = (merged[-1][0], max(merged[-1][1], b))
        else:
            merged.append((a, b))
    return merged


def compare(got: bytes, expected, where: str, base: int):
    """None when `got` equals the numpy.uint64 array `expected`, else a Mismatch; `base` is the allocation
    offset of got[0]."""
    g = np.frombuffer(got, dtype=np.uint64)
    assert g.shape == expected.shape
    bad = np.flatnonzero(g != expected)
    if bad.size == 0:
        return None
    k = int(bad[0])
    diff = int(g[k]) ^ int(expected[k])
    low_byte = ((diff & -diff).bit_length() - 1) // 8  # little-endian: the lowest differing bit's byte comes first
    return Mismatch(where, base + 8 * k + low_byte, int(bad.size), [base + 8 * int(i) for i in bad[:8]],
                    int(g[k]), int(expected[k]))


def check_region(probe, local: int, off: int, nbytes: int, expect, where: str):
    """Peek [off, off + nbytes) of local rank `local` and compare it with expect(first_word, n_words)."""
    out = []
    for a, b in windows(nbytes):
        m = compare(probe.Peek(local, off + a, b - a), expect(a // 8, (b - a) // 8), where, off + a)
        if m is not None:
            out.append(m)
    return out


def source_mismatches(probe, lay: Layout):
    """Every source slice of every local rank equals src_words (reads never write)."""
    out = []
    for li in range(lay.n_local):
        g = lay.first + li
        for s in range(lay.n_slices):
            k0 = s * lay.bpp // 8
            out += check_region(probe, li, lay.src_off + s * lay.bpp, lay.bpp,
                                lambda k, n: oracle.src_words(SEED, g, k0 + k, n), f"rank {g} source slice {s}")
    return out


def landing_mismatches(probe, lay: Layout, res):
    """Landing slots of every local rank after run `res`:
      - a cell res marks write-reachable: exactly this run's pattern from that writer;
      - an unreachable cell: exactly this run's or exactly the previous run's pattern, never a mix;
      - without OP_WRITE: all zero, as open left them."""
    out = []
    zeros = lambda k, n: np.zeros(n, dtype=np.uint64)
    for li in range(lay.n_local):
        j = lay.first + li
        for i in range(lay.n):
            if i == j and not lay.diag:
                continue
            slot = lay.slot(i, j)
            off = lay.land_off + slot * lay.bpp
            where = f"rank {j} landing slot {slot} (writer {i}, run_seq {res.run_seq})"
            if not lay.ops & OP_WRITE:
                out += check_region(probe, li, off, lay.bpp, zeros, where + ", ops = READ")
                continue
            now = check_region(probe, li, off, lay.bpp,
                               lambda k, n: oracle.write_words(SEED, i, j, res.run_seq, k, n), where)
            if now and not res.reach_write[i][j]:
                before = check_region(probe, li, off, lay.bpp,
                                      lambda k, n: oracle.write_words(SEED, i, j, res.run_seq - 1, k, n), where)
                if before:
                    for m in now:
                        m.where += ", unreachable cell: neither this run's nor the previous run's pattern"
                else:
                    now = []
            out += now
    return out


def snapshot_padding(probe, lay: Layout):
    return {(li, a, b): probe.Peek(li, a, b - a) for li in range(lay.n_local) for a, b in lay.padding()}


def padding_mismatches(probe, lay: Layout, snap):
    out = []
    for (li, a, b), before in snap.items():
        m = compare(probe.Peek(li, a, b - a), np.frombuffer(before, dtype=np.uint64).copy(),
                    f"rank {lay.first + li} padding [{a:#x}, {b:#x})", a)
        if m is not None:
            out.append(m)
    return out


def all_mismatches(probe, lay: Layout, res, snap):
    return source_mismatches(probe, lay) + landing_mismatches(probe, lay, res) + padding_mismatches(probe, lay, snap)
