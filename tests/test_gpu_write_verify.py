"""The write half of reachability, seen to fail: a landing slot damaged after its writer is done.

reach_write[i][j] is 1 when rank j's verify job reads the landing slot that rank i filled and gets the (S, X) that
i published (`publish_verdicts` in probe_kernels.cu), and i's host then decodes run_seq * 4 + Ok (`assemble` in
handle.cc).  Unmapping a pair, aborting or running a rank alone make the cell 0 without any verify job running, and
cdprobe_corrupt only touches the source, which only the read path checks.  CDPROBE_OPT_DEBUG_DAMAGE_WRITE makes the
barrier that closes a write phase damage the slot before the verifier may read it:
  1  flip bit 0 of the first word          (S and X change)
  2  flip bit 63 of the last word          (the tail of a partial unit when bytes_per_pair % 8192 != 0)
  3  first word + D, last word - D         (S unchanged: only X can see it)
  4  swap words 0 and 1                    (S and X unchanged: the checksum's blind spot, the verify passes)
For every case the expected outcome comes from the oracle: the verify passes exactly when
cdoracle_checksum(damaged pattern) == cdoracle_checksum(pattern).  Then:
  - reach_write[i][j] is that prediction, every other cell is reachable, and every checksum the writers report is
    still the clean oracle value (a writer sums what it generated);
  - status stays 0; a failed verify counts one unreachable pair (off the diagonal) and turns the verdict to 0;
  - Ctrl read back pins the branch: the writer's verdict word is run_seq * 4 + 2 (mismatch) or + 1 (ok), the
    verifier's published entry is the clean checksum with seq == run_seq;
  - the read-back finds exactly the damaged words in that slot, and nothing anywhere else;
  - with the option cleared the next run is clean.
"""
import json
import os
import subprocess
import sys
import textwrap
import uuid

import numpy as np
import pytest

import readback_check as rb
from conftest import ROOT, gpu_count

NGPU = gpu_count()
SEED = rb.SEED
SAME = 0x40 | 0x10  # ALLOW_SAME_DEVICE | NO_COOPERATIVE: several ranks on one device
PATHS, PATH_IDS = [0, 1, 2], ["tma", "ldst128", "ldst256"]
CODES = [1, 2, 3, 4]
N1_SIZES = [128, 8192 + 128, 16384 * 3 + 640, 1 << 20, (8 << 20) + 128 * 77]
SAME_DEV_BYTES = (2 << 20) + 128 * 9
BIG_BYTES = (4 << 30) + 3 * 8192 + 640  # the slot's last word lies past byte 2^32
M64 = (1 << 64) - 1
DELTA = 0x9E3779B97F4A7C15  # code 3's constant (kGolden in probe_types.h)
GRANULE_WORDS = 2048

# Ctrl (probe_types.h), pinned by test_ctrl_offsets_match_probe_types
CTRL_WR, WRPUB_BYTES, CTRL_VERDICT = 2048, 32, 2560
VERDICT_OK, VERDICT_MISMATCH = 1, 2
gpu = pytest.mark.gpu


def damage_value(local, target, code):
    return ((local + 1) << 16) | (target << 8) | code


def damage_changes(n_words, code, word):
    """{word index: damaged value} of a slot of `n_words` whose clean word k is word(k)."""
    last = n_words - 1
    if code == 1:
        return {0: word(0) ^ 1}
    if code == 2:
        return {last: word(last) ^ (1 << 63)}
    if code == 3:
        return {0: (word(0) + DELTA) & M64, last: (word(last) - DELTA) & M64}
    if code == 4:
        return {0: word(1), 1: word(0)}
    raise ValueError(code)


def fold6(g):
    return (g ^ (g >> 6) ^ (g >> 12) ^ (g >> 18) ^ (g >> 24) ^ (g >> 30)) & 63


def rotl64(x, r):
    r &= 63
    return ((x << r) | (x >> (64 - r))) & M64 if r else x


def checksum_after(clean, changes, word):
    """(S, X) of a slot whose checksum is `clean` once `changes` are applied, without touching the other words:
    S moves by the differences, X by each changed word's xor rotated like its granule."""
    s, x = clean
    for k, new in changes.items():
        old = word(k)
        s = (s + new - old) & M64
        x ^= rotl64(old ^ new, fold6(k // GRANULE_WORDS))
    return s, x


def writer_word(i, j, run_seq):
    return lambda k: int(rb.oracle.write_words(SEED, i, j, run_seq, k, 1)[0])


def predict(oracle, lay, i, j, run_seq, code):
    """(clean (S, X), damaged (S, X), changes) of cell i -> j: cdoracle_checksum over the whole slot up to 64 MiB,
    the exact update rule above past that (checked against cdoracle_checksum in the CPU tests)."""
    words = lay.bpp // 8
    word = writer_word(i, j, run_seq)
    ch = damage_changes(words, code, word)
    if lay.bpp <= rb.FULL_COMPARE_MAX:
        w = oracle.write_words(SEED, i, j, run_seq, 0, words)
        clean = oracle.checksum(w)
        for k, v in ch.items():
            w[k] = np.uint64(v)
        return clean, oracle.checksum(w), ch
    clean = oracle.write_checksum(SEED, i, j, run_seq, words)
    return clean, checksum_after(clean, ch, word), ch


def peek_u64(p, local, off, n=1):
    return [int(v) for v in np.frombuffer(p.Peek(local, off, 8 * n), dtype=np.uint64)]


def landing_mismatches(p, lay, run_seq, cell, changes):
    """Every landing slot of every local rank against run_seq's pattern, with `changes` applied to `cell`'s slot."""
    out = []
    for li in range(lay.n_local):
        j = lay.first + li
        for i in range(lay.n):
            if i == j and not lay.diag:
                continue
            ch = changes if (i, j) == cell else {}

            def expect(k, n, i=i, j=j, ch=ch):
                w = rb.oracle.write_words(SEED, i, j, run_seq, k, n)
                for idx, v in ch.items():
                    if k <= idx < k + n:
                        w[idx - k] = np.uint64(v)
                return w

            out += rb.check_region(p, li, lay.land_off + lay.slot(i, j) * lay.bpp, lay.bpp, expect,
                                   f"rank {j} landing slot {lay.slot(i, j)} (writer {i}, run_seq {run_seq})")
    return out


def open_probe(pkg, cfg, path):
    p = pkg.Open(cfg)
    try:
        p.SetOption(pkg.abi.OPT_PATH, path)
        lay = rb.Layout(p)
        return p, lay, rb.snapshot_padding(p, lay)
    except BaseException:
        p.Close()
        raise


def check_damaged_run(oracle, p, lay, pad, r, writer, target, code):
    """One run with `writer`'s slot in `target` damaged by `code`; every invariant of the module docstring."""
    n, seq = lay.n, r.run_seq
    clean, damaged, ch = predict(oracle, lay, writer, target, seq, code)
    passes = damaged == clean
    if code in (1, 2, 3):
        assert not passes, f"code {code} must be visible to the checksum at {lay.bpp} bytes per pair"
    what = f"code {code}, cell {writer} -> {target}, {lay.bpp} bytes per pair"
    assert not r.aborted, what
    assert r.status == [[0] * n for _ in range(n)], what
    exp = [[1] * n for _ in range(n)]
    exp[writer][target] = 1 if passes else 0
    assert r.reach_write == exp, what
    assert r.reach_read == [[1] * n for _ in range(n)], what
    for i in range(n):
        for j in range(n):
            if i != j or lay.diag:
                w = oracle.write_checksum(SEED, i, j, seq, lay.bpp // 8) if (i, j) != (writer, target) else clean
                assert (r.sum_write[i][j], r.xor_write[i][j]) == w, (what, i, j)
    assert r.unreachable_pairs == (0 if passes or writer == target else 1), what
    if not passes:
        assert not r.verdict, what
    # the branch publish_verdicts took, and what the verifier compared with
    if lay.first <= writer < lay.first + lay.n_local:
        (v,) = peek_u64(p, writer - lay.first, CTRL_VERDICT + 8 * target)
        assert v == seq * 4 + (VERDICT_OK if passes else VERDICT_MISMATCH), (what, v, seq)
    if lay.first <= target < lay.first + lay.n_local:
        s, x, q = peek_u64(p, target - lay.first, CTRL_WR + WRPUB_BYTES * lay.slot(writer, target), 3)
        assert (s, x) == clean and q == seq, what
    # bytes: exactly the damaged words differ from the pattern, in that slot only
    if lay.first <= target < lay.first + lay.n_local:
        off = lay.land_off + lay.slot(writer, target) * lay.bpp
        (m,) = rb.check_region(p, target - lay.first, off, lay.bpp,
                               lambda k, nw: oracle.write_words(SEED, writer, target, seq, k, nw), what)
        assert sorted(m.word_offsets) == [off + 8 * k for k in sorted(ch)], (what, str(m))
    bad = (rb.source_mismatches(p, lay) + landing_mismatches(p, lay, seq, (writer, target), ch)
           + rb.padding_mismatches(p, lay, pad))
    assert not bad, what + "\n" + rb.report(bad)
    return passes


def check_clean_run(p, lay, pad, r):
    n = lay.n
    assert not r.aborted and r.reach == [[1] * n for _ in range(n)] and r.unreachable_pairs == 0
    bad = rb.all_mismatches(p, lay, r, pad)
    assert not bad, "\n" + rb.report(bad)


def damage_each_code(pkg, oracle, p, lay, pad, writer, target, codes=CODES):
    for code in codes:
        p.SetOption(pkg.abi.OPT_DEBUG_DAMAGE_WRITE, damage_value(writer - lay.first, target, code))
        check_damaged_run(oracle, p, lay, pad, p.Run(), writer, target, code)
    p.SetOption(pkg.abi.OPT_DEBUG_DAMAGE_WRITE, 0)
    check_clean_run(p, lay, pad, p.Run())


# ---------------------------------------------------------------------------------------------- CPU ----
def test_ctrl_offsets_match_probe_types(tmp_path):
    """The Ctrl offsets this module peeks at, taken from probe_types.h by the host compiler."""
    hdr = os.path.join(ROOT, "k8s-dra-driver-gpu_b200", "csrc", "probe_types.h")
    src = tmp_path / "ctrl.cc"
    src.write_text(f'#include <stdio.h>\n#include "{hdr}"\nint main() {{ printf("%zu %zu %zu\\n", '
                   "offsetof(cdp::Ctrl, wr), offsetof(cdp::Ctrl, verdict), sizeof(cdp::WrPub)); return 0; }\n")
    exe = tmp_path / "ctrl"
    subprocess.run(["g++", "-std=c++17", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out] == [CTRL_WR, CTRL_VERDICT, WRPUB_BYTES]


def test_damage_option_constant(pkg):
    text = open(os.path.join(ROOT, "include", "cdprobe.h")).read()
    assert "#define CDPROBE_OPT_DEBUG_DAMAGE_WRITE 17u" in text
    assert pkg.abi.OPT_DEBUG_DAMAGE_WRITE == 17
    assert pkg.abi.load_library().cdprobe_set_option(None, 17, damage_value(0, 0, 1)) == pkg.abi.ERR_ARG


@pytest.mark.parametrize("nbytes", N1_SIZES + [(64 << 20) + 384])
def test_damage_prediction_matches_the_oracle(oracle, nbytes):
    """The update rule used past 64 MiB equals cdoracle_checksum over the damaged slot; codes 1-3 are visible to
    the checksum at every size the GPU tests use, code 4 is not."""
    words = nbytes // 8
    w = oracle.write_words(SEED, 0, 0, 2, 0, words)
    word = lambda k: int(w[k])
    clean = oracle.checksum(w)
    assert clean == oracle.write_checksum(SEED, 0, 0, 2, words)
    for code in CODES:
        ch = damage_changes(words, code, word)
        d = w.copy()
        for k, v in ch.items():
            d[k] = np.uint64(v)
        got = oracle.checksum(d)
        assert got == checksum_after(clean, ch, word), code
        assert (got == clean) == (code == 4), code
        if code == 3:
            assert got[0] == clean[0] and got[1] != clean[1]  # only X sees it


def test_damage_prediction_past_4_gib(oracle):
    """Codes 1-3 move the checksum of the slot over 4 GiB too (its last word lies past byte 2^32)."""
    words = BIG_BYTES // 8
    word = writer_word(0, 0, 2)
    clean = (0, 0)
    for code in (1, 2, 3):
        assert checksum_after(clean, damage_changes(words, code, word), word) != clean


# ------------------------------------------------------------------------------------ N = 1 loop-back ----
@gpu
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("nbytes", N1_SIZES)
def test_loopback_verify_catches_a_damaged_slot(pkg, oracle, nbytes, path):
    """The diagonal verify starts when the barrier releases the grid, without waiting for a signal: the damage
    must already be in HBM then."""
    p, lay, pad = open_probe(pkg, pkg.Config(ordinals=[0], bytes=nbytes), path)
    with p:
        assert lay.bpp == nbytes
        damage_each_code(pkg, oracle, p, lay, pad, 0, 0)


@gpu
def test_loopback_slot_over_4_gib(pkg, oracle):
    cfg = pkg.Config(ordinals=[0], bytes=BIG_BYTES, mode=pkg.abi.MODE_FULL, timeout_ms=60000)
    p, lay, pad = open_probe(pkg, cfg, 0)
    with p:
        assert lay.bpp == BIG_BYTES > 1 << 32
        damage_each_code(pkg, oracle, p, lay, pad, 0, 0, codes=[2])


# ----------------------------------------------------------------- several ranks on one device ----
SCHEDULES = {"default": 0, "pair-barriers": 0x800, "unidirectional": 0x80, "serial-verify": 0x100}
CELLS = {2: (1, 0), 3: (0, 2), 4: (3, 1), 8: (5, 2)}


@gpu
@pytest.mark.parametrize("sched", list(SCHEDULES))
@pytest.mark.parametrize("n", [2, 3, 4, 8])
def test_same_device_verify_catches_one_damaged_cell(pkg, oracle, n, sched):
    """Default: the writer only signals after its write (post barrier), the verify polls for it; pair-barriers:
    a sync barrier; unidirectional: one writer at a time; serial-verify: the verify runs after every round."""
    path = [0, 1, 2][(n + len(sched)) % 3]
    cfg = pkg.Config(ordinals=[0] * n, bytes=SAME_DEV_BYTES, flags=SAME | SCHEDULES[sched], ctas=8, timeout_ms=20000)
    p, lay, pad = open_probe(pkg, cfg, path)
    with p:
        writer, target = CELLS[n]
        damage_each_code(pkg, oracle, p, lay, pad, writer, target)


@gpu
def test_damage_option_rejects_bad_values(pkg):
    cfg = pkg.Config(ordinals=[0] * 3, bytes=SAME_DEV_BYTES, flags=SAME, ctas=8, timeout_ms=20000)
    with pkg.Open(cfg) as p:
        set_opt = lambda v: p._lib.cdprobe_set_option(p._h, pkg.abi.OPT_DEBUG_DAMAGE_WRITE, v)
        for v in (damage_value(-1, 1, 1), damage_value(3, 1, 1), damage_value(0, 3, 1), damage_value(0, 0, 1),
                  damage_value(0, 1, 0), damage_value(0, 1, 5), damage_value(0, 1, 255), 1 << 40):
            assert set_opt(v) == pkg.abi.ERR_ARG, hex(v)
        assert set_opt(damage_value(2, 0, 4)) == pkg.abi.OK
        assert set_opt(0) == pkg.abi.OK
        r = p.Run()
        assert r.reach == [[1] * 3 for _ in range(3)] and r.unreachable_pairs == 0
    with pkg.Open(pkg.Config(ordinals=[0], bytes=1 << 20)) as p:
        assert p._lib.cdprobe_set_option(p._h, pkg.abi.OPT_DEBUG_DAMAGE_WRITE, damage_value(0, 0, 3)) == pkg.abi.OK


# ------------------------------------------------------------------------------------- real NVLink ----
@gpu
@pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("path", PATHS, ids=PATH_IDS)
def test_real_nvlink_verify_catches_a_damaged_slot(pkg, oracle, path):
    n = min(NGPU, 8)
    cfg = pkg.Config(ordinals=list(range(n)), bytes=16 << 20, mode=pkg.abi.MODE_FULL, timeout_ms=20000)
    p, lay, pad = open_probe(pkg, cfg, path)
    with p:
        damage_each_code(pkg, oracle, p, lay, pad, n - 1, 0)


# --------------------------------------------------------------------------- one process per rank ----
CHILD = textwrap.dedent(
    """
    import json, os, sys
    sys.path.insert(0, %r)
    sys.path.insert(0, os.path.join(%r, "tests"))
    import numpy as np
    import cdprobe_pkg
    import readback_check as rb
    m = cdprobe_pkg.load()
    session, rank, world, ordinal, nbytes, flags, writer, target, code = sys.argv[1:10]
    rank, writer, target = int(rank), int(writer), int(target)
    cfg = m.Config(ordinals=[int(ordinal)], bytes=int(nbytes), world_size=int(world), rank=rank, session=session,
                   flags=int(flags), ctas=8, timeout_ms=30000)
    out = []
    with m.Open(cfg) as p:
        lay = rb.Layout(p)
        if rank == writer:
            p.SetOption(m.abi.OPT_DEBUG_DAMAGE_WRITE, (1 << 16) | (target << 8) | int(code))
        for k in range(2):
            r = p.Run(gather=True)
            ctrl = np.frombuffer(p.Peek(0, 0, 4096), dtype=np.uint64)
            out.append({"run_seq": r.run_seq, "reach_read": r.reach_read, "reach_write": r.reach_write,
                        "sum_write": r.sum_write, "xor_write": r.xor_write, "status": r.status,
                        "unreachable_pairs": r.unreachable_pairs, "verdict": r.verdict, "aborted": r.aborted,
                        "ctrl": [int(v) for v in ctrl[:%d]], "slot": [lay.slot(i, rank) for i in range(lay.n)],
                        "bpp": lay.bpp})
            if rank == writer:
                p.SetOption(m.abi.OPT_DEBUG_DAMAGE_WRITE, 0)
    print("RESULT " + json.dumps(out))
    """
) % (ROOT, ROOT, (CTRL_VERDICT // 8) + 16)


def run_world(ordinals, nbytes, flags, writer, target, code):
    world = len(ordinals)
    session = f"wv-{uuid.uuid4().hex[:12]}"
    procs = [subprocess.Popen([sys.executable, "-c", CHILD, session, str(r), str(world), str(ordinals[r]), str(nbytes),
                               str(flags), str(writer), str(target), str(code)],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(world)]
    outs = []
    for p in procs:
        so, se = p.communicate(timeout=300)
        assert p.returncode == 0, se[-2000:]
        outs.append(json.loads([l for l in so.splitlines() if l.startswith("RESULT ")][-1][7:]))
    return outs


def check_world(oracle, outs, writer, target, code):
    n = len(outs)
    for rank, runs in enumerate(outs):
        for k, r in enumerate(runs):
            seq, bpp = r["run_seq"], r["bpp"]
            clean = oracle.write_checksum(SEED, writer, target, seq, bpp // 8)
            word = writer_word(writer, target, seq)
            passes = k == 1 or checksum_after(clean, damage_changes(bpp // 8, code, word), word) == clean
            exp = [[1] * n for _ in range(n)]
            exp[writer][target] = 1 if passes else 0
            what = f"rank {rank}, run {k}"
            assert not r["aborted"] and r["reach_read"] == [[1] * n for _ in range(n)], what
            assert r["reach_write"] == exp and r["unreachable_pairs"] == (0 if passes else 1), what
            assert r["status"] == [[0] * n for _ in range(n)], what
            if not passes:
                assert not r["verdict"], what
            for i in range(n):
                for j in range(n):
                    if i != j:
                        assert (r["sum_write"][i][j], r["xor_write"][i][j]) == \
                            oracle.write_checksum(SEED, i, j, seq, bpp // 8), (what, i, j)
            ctrl = r["ctrl"]
            if rank == writer:
                assert ctrl[CTRL_VERDICT // 8 + target] == seq * 4 + (VERDICT_OK if passes else VERDICT_MISMATCH)
            if rank == target:
                e = (CTRL_WR + WRPUB_BYTES * r["slot"][writer]) // 8
                assert tuple(ctrl[e:e + 2]) == clean and ctrl[e + 2] == seq, what


@gpu
@pytest.mark.parametrize("code", [1, 3])
def test_two_processes_on_one_gpu_verify_catches_a_damaged_slot(pkg, oracle, code):
    """The writer's process damages the slot; the verify and its verdict cross the process boundary."""
    check_world(oracle, run_world([0, 0], SAME_DEV_BYTES, 0x40, 1, 0, code), 1, 0, code)


@gpu
@pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs")
def test_one_process_per_gpu_verify_catches_a_damaged_slot(pkg, oracle):
    n = min(NGPU, 8)
    check_world(oracle, run_world(list(range(n)), 32 << 20, 0, 0, n - 1, 3), 0, n - 1, 3)
