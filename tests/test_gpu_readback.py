"""Read-back tests: the bytes the probe kernels leave in HBM, word for word against the pattern oracle.

test_gpu_parity.py compares (S, X) checksums, and the checksum cannot see every placement error (DESIGN §5:
words reordered inside a 16 KiB granule, granules swapped whose fold6 is equal, stores outside the slot a
verifier reads).  Here cdprobe_peek copies a rank's own allocation back, and tests/readback_check.py holds it
against oracle.src_words / oracle.write_words:
  - the source is exact right after open and after every run (reads never write);
  - after run r every landing slot of a write-reachable cell holds exactly r's pattern from its writer; an
    unreachable cell's slot holds r's or r - 1's pattern, never a mix; with ops = READ the slots stay zero;
  - the padding up to the next 2 MiB boundary after the source and after the landing slots is never written.
Every configuration runs twice, so the re-salted pattern of the second run is checked too.  A failure names
the first bad byte's allocation offset and the number of bad words.
"""
import ctypes as C
import functools
import json
import subprocess
import sys
import textwrap
import uuid

import pytest

import readback_check as rb
from conftest import ROOT, gpu_count

NGPU = gpu_count()
SEED = rb.SEED
SAME = 0x40 | 0x10  # ALLOW_SAME_DEVICE | NO_COOPERATIVE: several ranks on one device
UNIT, GRANULE = 8192, 16384
PATHS, PATH_IDS = [0, 1, 2], ["tma", "ldst128", "ldst256"]
N1_SIZES = [128, 8064, 8192, 8192 + 128, 16384 * 3 + 640, (1 << 23) + 128 * 77, (64 << 20) + 384]
SAME_DEV_BYTES = (2 << 20) + 128 * 9
BIG_BYTES = (4 << 30) + 3 * 8192 + 640  # bytes_per_pair > 2^32
gpu = pytest.mark.gpu


def assert_clean(mismatches):
    assert not mismatches, "\n" + rb.report(mismatches)


def ones(n):
    return [[1] * n for _ in range(n)]


def open_checked(pkg, cfg, path):
    """Open, select the data path, check the source as the fill kernel left it; returns (probe, layout, padding)."""
    p = pkg.Open(cfg)
    try:
        p.SetOption(pkg.abi.OPT_PATH, path)
        assert p.Info().path == path
        lay = rb.Layout(p)
        assert_clean(rb.source_mismatches(p, lay))
        return p, lay, rb.snapshot_padding(p, lay)
    except BaseException:
        p.Close()
        raise


def run_checked(p, lay, pad, runs=2, reach=True):
    """`runs` probe runs, every invariant after each; with `reach`, every cell of the ops in use is reachable."""
    for _ in range(runs):
        r = p.Run()
        assert not r.aborted
        if reach:
            if lay.ops & rb.OP_READ:
                assert r.reach_read == ones(lay.n)
            if lay.ops & rb.OP_WRITE:
                assert r.reach_write == ones(lay.n)
        assert_clean(rb.all_mismatches(p, lay, r, pad))
    return r


def same_device(pkg, n, nbytes=SAME_DEV_BYTES, mode=1, flags=0, ops=3, ctas=8):
    return pkg.Config(ordinals=[0] * n, bytes=nbytes, mode=mode, ops=ops, flags=SAME | flags, ctas=ctas,
                      timeout_ms=20000)


# ---------------------------------------------------------------------------------------------- CPU ----
def test_peek_rejects_a_null_handle(pkg):
    lib = pkg.abi.load_library()
    buf = C.create_string_buffer(16)
    assert lib.cdprobe_peek(None, 0, 0, 8, buf) == pkg.abi.ERR_ARG


def test_layout_windows_cover_the_edges():
    """The windows a large region is compared on: first and last MiB, +-1 MiB around 2^31 and 2^32."""
    MiB = rb.MiB
    assert rb.windows(64 * MiB) == [(0, 64 * MiB)]
    n = BIG_BYTES
    # the last MiB of a 4 GiB + 24.6 KiB slice overlaps the window around 2^32: one window to the end
    assert rb.windows(n) == [(0, MiB), ((1 << 31) - MiB, (1 << 31) + MiB), ((1 << 32) - MiB, n)]
    assert rb.windows(3 << 32) == [(0, MiB), ((1 << 31) - MiB, (1 << 31) + MiB), ((1 << 32) - MiB, (1 << 32) + MiB),
                                   ((3 << 32) - MiB, 3 << 32)]
    assert rb.windows((64 << 20) + 384) == [(0, MiB), ((63 << 20) + 384, (64 << 20) + 384)]


def test_comparator_names_the_first_bad_byte(oracle):
    exp = oracle.src_words(SEED, 0, 0, 4096)
    got = exp.copy()
    got[1000] ^= rb.np.uint64(1 << 43)  # byte 5 of word 1000
    got[3000] ^= rb.np.uint64(1)
    m = rb.compare(got.tobytes(), exp, "x", 0x200000)
    assert m.first_byte == 0x200000 + 8 * 1000 + 5 and m.bad_words == 2
    assert m.word_offsets == [0x200000 + 8000, 0x200000 + 24000]
    assert rb.compare(exp.tobytes(), exp, "x", 0) is None


# ------------------------------------------------------------------------------------ N = 1 loop-back ----
@gpu
@pytest.mark.parametrize("ctas", [0, 5], ids=["default-grid", "5-ctas"])
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("nbytes", N1_SIZES)
def test_single_gpu_bytes_are_exact(pkg, nbytes, path, ctas):
    """5 CTAs give each warp many units, so the 3-stage TMA ring wraps several times at the larger sizes."""
    p, lay, pad = open_checked(pkg, pkg.Config(ordinals=[0], bytes=nbytes, ctas=ctas), path)
    with p:
        run_checked(p, lay, pad)


# ----------------------------------------------------------------- several ranks on one device ----
@gpu
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("n", [2, 3, 4, 5, 8])
def test_same_device_ranks_bytes_are_exact(pkg, n, path):
    p, lay, pad = open_checked(pkg, same_device(pkg, n), path)
    with p:
        run_checked(p, lay, pad)


@gpu
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("n,mode,flags", [(2, 2, 0), (3, 2, 0), (4, 0, 0), (4, 1, 0x04)],
                         ids=["n2-full", "n3-full", "n4-reach-only", "n4-local-diag"])
def test_same_device_modes_bytes_are_exact(pkg, n, mode, flags, path):
    p, lay, pad = open_checked(pkg, same_device(pkg, n, mode=mode, flags=flags), path)
    with p:
        run_checked(p, lay, pad)


@gpu
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("flags", [0x80, 0x100, 0x800, 0x400],
                         ids=["unidirectional", "serial-verify", "pair-barriers", "all-rank-barriers"])
def test_slot_contents_do_not_depend_on_the_schedule(pkg, flags, path):
    p, lay, pad = open_checked(pkg, same_device(pkg, 4, flags=flags), path)
    with p:
        run_checked(p, lay, pad)


@gpu
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("ops", [1, 2], ids=["read-only", "write-only"])
def test_single_op_bytes_are_exact(pkg, ops, path):
    """READ only: the landing slots stay as open zeroed them.  WRITE only: the source is still untouched."""
    p, lay, pad = open_checked(pkg, same_device(pkg, 4, ops=ops), path)
    with p:
        run_checked(p, lay, pad)


@gpu
def test_unmapped_pair_leaves_whole_patterns_and_remap_restores(pkg):
    n = 4
    p, lay, pad = open_checked(pkg, same_device(pkg, n), 0)
    with p:
        run_checked(p, lay, pad, runs=1)
        p.UnmapPeer(1, 2)
        r = p.Run()  # one run only: the rule for an unreachable cell is "this run's or the previous run's"
        exp = ones(n)
        exp[1][2] = exp[2][1] = 0
        assert r.reach == exp and not r.aborted
        assert_clean(rb.all_mismatches(p, lay, r, pad))
        p.RemapPeer(1, 2)
        run_checked(p, lay, pad)


@gpu
def test_copy_engine_scribbles_are_overwritten(pkg):
    p, lay, pad = open_checked(pkg, same_device(pkg, 2), 0)
    with p:
        r = run_checked(p, lay, pad, runs=1)
        p.CeCopy([(0, 1)], push=True, reps=1)
        p.CeCopy([(0, 1), (1, 0)], push=False, reps=1)
        # the copies put source bytes into the landing slots (visibly), and nowhere else
        assert rb.landing_mismatches(p, lay, r)
        assert_clean(rb.source_mismatches(p, lay) + rb.padding_mismatches(p, lay, pad))
        run_checked(p, lay, pad)


# ---------------------------------------------------------------------------- slices of 4 GiB and more ----
@functools.lru_cache(maxsize=None)
def _src_checksum(oracle, rank, n_words):
    return oracle.src_checksum(SEED, rank, 0, n_words)


@functools.lru_cache(maxsize=None)
def _write_checksum(oracle, i, j, run_seq, n_words):
    return oracle.write_checksum(SEED, i, j, run_seq, n_words)


def _big_slice_checks(oracle, p, lay, pad):
    words = lay.bpp // 8
    info = p.Info()
    for li in range(lay.n_local):
        assert (info.src_sum[li][0], info.src_xor[li][0]) == _src_checksum(oracle, li, words)
    for _ in range(2):
        r = p.Run()
        assert not r.aborted and r.reach == ones(lay.n)
        for i in range(lay.n):
            for j in range(lay.n):
                if i != j or lay.diag:
                    assert (r.sum_read[i][j], r.xor_read[i][j]) == _src_checksum(oracle, j, words), (i, j)
                    assert (r.sum_write[i][j], r.xor_write[i][j]) == _write_checksum(oracle, i, j, r.run_seq, words)
        assert_clean(rb.all_mismatches(p, lay, r, pad))


@gpu
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
def test_slice_over_4_gib_single_gpu(pkg, oracle, path):
    """bytes_per_pair > 2^32 (an ~8 GiB allocation): byte offsets past 2^31 and 2^32 in the source and the
    landing slot; checksums against the oracle over the whole slice, bytes on windows around those offsets."""
    cfg = pkg.Config(ordinals=[0], bytes=BIG_BYTES, mode=pkg.abi.MODE_FULL, timeout_ms=60000)
    p, lay, pad = open_checked(pkg, cfg, path)
    with p:
        assert lay.bpp == BIG_BYTES > 1 << 32
        _big_slice_checks(oracle, p, lay, pad)


@gpu
def test_slice_over_4_gib_same_device_pair(pkg, oracle):
    cfg = same_device(pkg, 2, nbytes=BIG_BYTES, mode=pkg.abi.MODE_FULL)
    cfg.timeout_ms = 60000
    p, lay, pad = open_checked(pkg, cfg, 0)
    with p:
        _big_slice_checks(oracle, p, lay, pad)


# ------------------------------------------------------------------------------------- real NVLink ----
@gpu
@pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("mode,nbytes", [(1, 64 << 20), (2, 16 << 20)], ids=["sliced-64MiB", "full-16MiB"])
def test_real_nvlink_bytes_are_exact(pkg, mode, nbytes, path):
    n = min(NGPU, 8)
    cfg = pkg.Config(ordinals=list(range(n)), bytes=nbytes, mode=mode, timeout_ms=20000)
    p, lay, pad = open_checked(pkg, cfg, path)
    with p:
        run_checked(p, lay, pad)


# --------------------------------------------------------------------------- one process per rank ----
CHILD = textwrap.dedent(
    """
    import json, os, sys
    sys.path.insert(0, %r)
    sys.path.insert(0, os.path.join(%r, "tests"))
    import cdprobe_pkg
    import readback_check as rb
    m = cdprobe_pkg.load()
    session, rank, world, ordinal, nbytes, flags, ctas = sys.argv[1:8]
    cfg = m.Config(ordinals=[int(ordinal)], bytes=int(nbytes), world_size=int(world), rank=int(rank), session=session,
                   flags=int(flags), ctas=int(ctas), timeout_ms=30000)
    out = []
    with m.Open(cfg) as p:
        lay = rb.Layout(p)
        bad = rb.source_mismatches(p, lay)
        pad = rb.snapshot_padding(p, lay)
        for _ in range(2):
            r = p.Run(gather=True)
            bad += rb.all_mismatches(p, lay, r, pad)
            out.append({"n": r.n, "row_mask": r.row_mask, "reach_read": r.reach_read, "reach_write": r.reach_write,
                        "aborted": r.aborted})
    print("RESULT " + json.dumps({"runs": out, "mismatches": [str(b) for b in bad]}))
    """
) % (ROOT, ROOT)


def run_world(world, ordinals, nbytes, flags, ctas):
    session = f"rb-{uuid.uuid4().hex[:12]}"
    procs = [subprocess.Popen([sys.executable, "-c", CHILD, session, str(r), str(world), str(ordinals[r]), str(nbytes),
                               str(flags), str(ctas)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for r in range(world)]
    outs = []
    for p in procs:
        so, se = p.communicate(timeout=300)
        assert p.returncode == 0, se[-2000:]
        outs.append(json.loads([l for l in so.splitlines() if l.startswith("RESULT ")][-1][7:]))
    return outs


def check_world(outs, world):
    for rank, o in enumerate(outs):
        assert not o["mismatches"], f"rank {rank}:\n" + "\n".join(o["mismatches"])
        for r in o["runs"]:
            assert r["n"] == world and r["row_mask"] == (1 << world) - 1 and not r["aborted"]
            assert r["reach_read"] == ones(world) and r["reach_write"] == ones(world)


@gpu
def test_two_processes_on_one_gpu_bytes_are_exact(pkg):
    check_world(run_world(2, [0, 0], SAME_DEV_BYTES, 0x40, 8), 2)


@gpu
@pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs")
def test_one_process_per_gpu_bytes_are_exact(pkg):
    n = min(NGPU, 8)
    check_world(run_world(n, list(range(n)), 32 << 20, 0, 0), n)


# ---------------------------------------------------------------------- edges of the detection contract ----
EDGE_BPP = 16384 * 3 + 640  # six full 8 KiB units, three granules, a 640-byte tail unit
EDGES = {"word-0": 0, "last-word": EDGE_BPP - 8, "last-word-of-unit-0": UNIT - 8, "first-word-of-unit-1": UNIT,
         "first-word-of-granule-1": GRANULE, "first-word-of-tail-unit": EDGE_BPP // UNIT * UNIT}


@gpu
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("n", [1, 3])
def test_one_flipped_word_fails_exactly_its_reader(pkg, oracle, n, path):
    """A flipped source word at a unit, granule or tail edge fails exactly the reader of that slice; the
    read-back names its offset; flipping it back restores parity."""
    nbytes = EDGE_BPP * max(n - 1, 1)
    cfg = pkg.Config(ordinals=[0], bytes=nbytes) if n == 1 else same_device(pkg, n, nbytes=nbytes)
    reader, owner = (0, 0) if n == 1 else (2, 0)
    p, lay, pad = open_checked(pkg, cfg, path)
    with p:
        assert lay.bpp == EDGE_BPP
        run_checked(p, lay, pad, runs=1)
        base = lay.slice_of(reader, owner) * lay.bpp
        for e, (name, pos) in enumerate(EDGES.items()):
            bit = (13 * e + 5) % 64
            word = int(oracle.src_words(SEED, owner, (base + pos) // 8, 1)[0])
            p.Corrupt(owner, base + pos, 1 << bit)
            off = lay.src_off + base + pos
            assert int.from_bytes(p.Peek(owner, off, 8), "little") == word ^ (1 << bit), name
            (m,) = rb.source_mismatches(p, lay)
            assert m.first_byte == off + bit // 8 and m.bad_words == 1, (name, str(m))
            r = p.Run()
            exp = ones(n)
            exp[reader][owner] = 0
            assert r.reach_read == exp, name
            assert r.reach_write == ones(n), name
            p.Corrupt(owner, base + pos, 1 << bit)
            r = p.Run()
            assert r.reach == ones(n), name
            for i in range(n):
                for j in range(n):
                    if i != j or n == 1:
                        assert (r.sum_read[i][j], r.xor_read[i][j]) == oracle.expected_read(SEED, n, nbytes, 1, i, j)
            assert_clean(rb.all_mismatches(p, lay, r, pad))


# ------------------------------------------------------------------------- the comparator is not vacuous ----
@gpu
def test_peek_rejects_out_of_range_arguments(pkg):
    p, lay, _ = open_checked(pkg, pkg.Config(ordinals=[0], bytes=1 << 20), 0)
    with p:
        lib, h = p._lib, p._h
        buf = C.create_string_buffer(16)
        assert lib.cdprobe_peek(h, 0, lay.alloc - 8, 8, buf) == pkg.abi.OK  # the last word is readable
        assert lib.cdprobe_peek(h, 0, lay.alloc - 8, 16, buf) == pkg.abi.ERR_ARG
        assert lib.cdprobe_peek(h, 0, (1 << 64) - 8, 16, buf) == pkg.abi.ERR_ARG  # offset + bytes wraps
        assert lib.cdprobe_peek(h, 0, 0, 0, buf) == pkg.abi.ERR_ARG
        assert lib.cdprobe_peek(h, 1, 0, 8, buf) == pkg.abi.ERR_ARG
        assert lib.cdprobe_peek(h, 0, 0, 8, None) == pkg.abi.ERR_ARG
        with pytest.raises(pkg.ProbeError):
            p.Peek(0, lay.alloc, 8)


@gpu
def test_swapped_words_inside_a_granule_pass_the_checksum_but_not_the_readback(pkg):
    """The checksum's known blind spot, pinned (DESIGN §5): two source words of one 16 KiB granule swapped leave
    S and X unchanged, so the reader still reports the slice reachable; only the read-back sees it.  A stronger
    checksum would turn reach_read to 0 here: update this test together with it."""
    p, lay, pad = open_checked(pkg, pkg.Config(ordinals=[0], bytes=1 << 20), 0)
    with p:
        a, b = GRANULE + 8 * 3, GRANULE + 8 * 500
        wa = int.from_bytes(p.Peek(0, lay.src_off + a, 8), "little")
        wb = int.from_bytes(p.Peek(0, lay.src_off + b, 8), "little")
        p.Corrupt(0, a, wa ^ wb)
        p.Corrupt(0, b, wa ^ wb)
        (m,) = rb.source_mismatches(p, lay)
        assert m.bad_words == 2 and m.word_offsets == [lay.src_off + a, lay.src_off + b], str(m)
        r = p.Run()
        assert r.reach_read[0][0] == 1 and r.reach_write[0][0] == 1
