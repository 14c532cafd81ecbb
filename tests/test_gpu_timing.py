"""GB/s and the timeline, held against references the kernel does not control.

  - Host arithmetic: every field the host derives from the kernels' timestamps (per-pair GB/s, the minima, slow and
    unreachable pairs, verdict, device_ms, barrier_us) equals tests/result_model.py's prediction bit for bit, from
    the trace of the same run, over modes, ops, schedules, data paths, faults and a two-process gather.
  - Timeline invariants: t_start[0] == 0, t_start <= t_end <= t_arrive <= next t_start for every job present, and
    device_ms <= kernel_ms <= event_ms (+ eps) <= probe_ms (+ eps).
  - An independent clock: a one-phase loop-back read's time against CUDA events around the kernel, at 148, 32 and 8
    CTAs, and its growth with the byte count.
  - Physical ceilings: loop-back jobs under the HBM3e data-sheet figure, NVLink cells under 900 GB/s and near the
    copy engine on the same pair.
  - The %globaltimer tick, printed (DESIGN §5).
Absolute bounds quote the B200 data sheet; the measured ratios are printed with -s.
"""
import functools
import json
import math
import subprocess
import sys
import textwrap
import uuid

import pytest

import result_model as rm
from conftest import ROOT, gpu_count

NGPU = gpu_count()
SAME = 0x40 | 0x10  # ALLOW_SAME_DEVICE | NO_COOPERATIVE
HBM_GBPS = 7700.0   # HGX B200 data sheet, HBM3e per GPU: 7.7 TB/s
NVLINK_GBPS = 900.0  # NVLink 5, per direction per GPU
EPS_MS = 0.05       # two clocks (globaltimer, CUDA events) and a host clock: slack between them
GiB = 1 << 30
OPT_EVENT_TIMING = 1  # CDPROBE_OPT_EVENT_TIMING
gpu = pytest.mark.gpu


def traces(p, n_local):
    return [p.Trace(li) for li in range(n_local)]


def check_model(p, r, ops, diag):
    """The result equals the model's prediction from the same run's trace, bit for bit."""
    info = p.Info()
    d = rm.as_dict(r)
    tr = traces(p, info.n_local)
    pred = rm.predict(d, tr, info.first_local_rank, ops, diag)
    for k in rm.DERIVED:
        assert d[k] == pred[k], (k, d[k], pred[k])
    assert d["device_ms"][:info.n_local] == pred["device_ms"]
    assert d["barrier_us"][:info.n_local] == pred["barrier_us"]
    return tr


def check_timeline(r, tr, n_local, events=True):
    for li, t in enumerate(tr):
        assert t and t[0]["t_start"] == 0, li
        for p, ph in enumerate(t):
            for job, end in (("job0", "t_end0"), ("job1", "t_end1")):
                if ph[job] != "-":
                    assert ph["t_start"] <= ph[end] <= ph["t_arrive"], (li, p, job, ph)
            assert ph["t_start"] <= ph["t_arrive"], (li, p, ph)
            if p + 1 < len(t):
                assert ph["t_arrive"] <= t[p + 1]["t_start"], (li, p)
        if events:
            dev, ker, ev = r.device_ms[li], r.kernel_ms[li], r.event_ms[li]
            assert 0 < dev <= ker <= ev + EPS_MS, (li, dev, ker, ev)
            assert ev <= r.probe_ms + EPS_MS, (li, ev, r.probe_ms)


def run_and_check(p, ops, diag, runs=2):
    n_local = p.Info().n_local
    p.SetOption(OPT_EVENT_TIMING, 1)
    out = []
    for _ in range(runs):
        r = p.Run()
        tr = check_model(p, r, ops, diag)
        check_timeline(r, tr, n_local)
        out.append((r, tr))
    return out


# ------------------------------------------------------------------------------------ host arithmetic ----
@gpu
@pytest.mark.parametrize("ops", [1, 2, 3], ids=["read", "write", "read-write"])
@pytest.mark.parametrize("mode", [0, 1, 2], ids=["reach-only", "sliced", "full"])
def test_single_gpu_result_is_the_model(pkg, mode, ops):
    with pkg.Open(pkg.Config(ordinals=[0], bytes=(1 << 20) + 640, mode=mode, ops=ops)) as p:
        run_and_check(p, ops, True)


SCHED = {"default": 0, "uni": 0x80, "serial": 0x100, "pair-barriers": 0x800, "all-rank": 0x400}


@gpu
@pytest.mark.parametrize("sched", list(SCHED))
@pytest.mark.parametrize("n", [2, 3, 5, 8])
def test_same_device_result_is_the_model(pkg, n, sched):
    cfg = pkg.Config(ordinals=[0] * n, bytes=(2 << 20) + 128 * 9, flags=SAME | SCHED[sched], ctas=8, timeout_ms=20000)
    with pkg.Open(cfg) as p:
        run_and_check(p, 3, False)


@gpu
@pytest.mark.parametrize("path", [0, 1, 2], ids=["tma", "ldst128", "ldst256"])
def test_result_is_the_model_on_every_path(pkg, path):
    for cfg in (pkg.Config(ordinals=[0], bytes=8 << 20),
                pkg.Config(ordinals=[0] * 3, bytes=4 << 20, flags=SAME, ctas=8, timeout_ms=20000)):
        with pkg.Open(cfg) as p:
            p.SetOption(pkg.abi.OPT_PATH, path)
            run_and_check(p, 3, cfg.ordinals == [0])


@gpu
def test_result_is_the_model_under_faults(pkg):
    a = pkg.abi
    base = dict(bytes=(2 << 20) + 128 * 9, ctas=8, timeout_ms=20000)
    # simulated MIG: every peer pair is excluded, nothing is unreachable
    with pkg.Open(pkg.Config(ordinals=[0] * 3, flags=SAME | a.FLAG_SIMULATE_MIG, **base)) as p:
        ((r, _), _) = run_and_check(p, 3, False)
        assert r.unreachable_pairs == 0
    with pkg.Open(pkg.Config(ordinals=[0] * 4, flags=SAME, **base)) as p:
        p.UnmapPeer(1, 2)
        ((r, _), _) = run_and_check(p, 3, False)
        assert r.unreachable_pairs >= 1 and not r.verdict
        p.RemapPeer(1, 2)
        p.SetOption(a.OPT_CTAS_RANK, (1 << 16) | 1)  # local rank 0 throttled to one CTA
        run_and_check(p, 3, False)
        p.SetOption(a.OPT_LINK_PEAK_MBPS, 100_000_000)  # a gate of 65 TB/s: nobody meets it
        ((r, _), _) = run_and_check(p, 3, False)
        assert not r.verdict and r.slow_pairs == 4 * 3 and r.unreachable_pairs == 0


# ------------------------------------------------------------------------ two processes, one gather ----
CHILD = textwrap.dedent(
    """
    import ctypes as C, json, os, sys
    sys.path.insert(0, %r)
    sys.path.insert(0, os.path.join(%r, "tests"))
    import cdprobe_pkg
    import result_model as rm
    m = cdprobe_pkg.load()
    session, rank, world = sys.argv[1:4]
    cfg = m.Config(ordinals=[0], bytes=(2 << 20) + 128 * 9, world_size=int(world), rank=int(rank), session=session,
                   flags=0x40, ctas=8, timeout_ms=30000)
    out = []
    with m.Open(cfg) as p:
        for _ in range(2):
            raw = m.abi.ResultT()
            assert p._lib.cdprobe_run(p._h, C.byref(raw)) == 0
            pre = rm.as_dict(m.Result.from_c(raw))
            tr = p.Trace(0)
            assert p._lib.cdprobe_gather(p._h, C.byref(raw)) == 0
            out.append({"pre": pre, "trace": tr, "gathered": rm.as_dict(m.Result.from_c(raw))})
    print("RESULT " + json.dumps(out))
    """
) % (ROOT, ROOT)


@gpu
def test_two_process_gather_is_the_model_merge(pkg):
    world = 2
    session = f"tm-{uuid.uuid4().hex[:12]}"
    procs = [subprocess.Popen([sys.executable, "-c", CHILD, session, str(r), str(world)], stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(world)]
    outs = []
    for p in procs:
        so, se = p.communicate(timeout=300)
        assert p.returncode == 0, se[-2000:]
        outs.append(json.loads([l for l in so.splitlines() if l.startswith("RESULT ")][-1][7:]))
    for k in range(2):
        pres = [o[k]["pre"] for o in outs]
        for rank, o in enumerate(outs):
            pre, tr = o[k]["pre"], o[k]["trace"]
            pred = rm.predict(pre, [tr], rank, 3, False)
            for f in rm.DERIVED:
                assert pre[f] == pred[f], (rank, f)
            assert pre["device_ms"][:1] == pred["device_ms"] and pre["barrier_us"][:1] == pred["barrier_us"]
            check_timeline(None, [tr], 1, events=False)
            merged = rm.merge(pre, [pres[q] for q in range(world) if q != rank])
            for f in rm.MERGED:
                assert o[k]["gathered"][f] == merged[f], (rank, f)
            assert merged["row_mask"] == 3


# ------------------------------------------------------------------------------- an independent clock ----
def loopback_read(pkg, nbytes, ctas=0, runs=3):
    """[(phase ns from the reported GB/s, event ms, trace)] of `runs` N = 1 read-only runs."""
    out = []
    with pkg.Open(pkg.Config(ordinals=[0], bytes=nbytes, mode=pkg.abi.MODE_FULL, ops=1, timeout_ms=60000)) as p:
        p.SetOption(pkg.abi.OPT_EVENT_TIMING, 1)
        if ctas:
            p.SetOption(pkg.abi.OPT_CTAS, ctas)
        p.Run()
        for _ in range(runs):
            r = p.Run()
            assert r.reach_read == [[1]] and not r.aborted
            tr = check_model(p, r, 1, True)
            check_timeline(r, tr, 1)
            out.append((nbytes / r.gbps_read[0][0], r.event_ms[0], tr))
    return out


@gpu
@pytest.mark.parametrize("ctas", [148, 32, 8])
def test_phase_time_follows_cuda_events(pkg, ctas):
    """4 GiB read once: the kernel is one phase, so the phase time is most of the event time, whatever the speed."""
    rs = loopback_read(pkg, 4 * GiB, ctas)
    for t_ns, ev_ms, tr in rs:
        assert len(tr) == 1, tr
        ratio = t_ns / 1e6 / ev_ms
        print(f"\n[timing] ctas {ctas}: phase {t_ns / 1e6:.4f} ms, event {ev_ms:.4f} ms, ratio {ratio:.4f}")
        assert 0.85 <= ratio <= 1.0, (ctas, t_ns, ev_ms)


@gpu
def test_phase_time_scales_with_bytes(pkg):
    t = {g: min(x[0] for x in loopback_read(pkg, g * GiB)) for g in (1, 2, 4)}
    print(f"\n[timing] phase ns: {t}; 2/1 {t[2] / t[1]:.4f}, 4/2 {t[4] / t[2]:.4f}")
    assert 1.85 <= t[2] / t[1] <= 2.1 and 1.85 <= t[4] / t[2] <= 2.1, t


# ------------------------------------------------------------------------------- physical ceilings ----
@gpu
@pytest.mark.parametrize("path", [0, 1, 2], ids=["tma", "ldst128", "ldst256"])
def test_loopback_jobs_stay_under_hbm_bandwidth(pkg, path):
    """4 GiB per job: the 126 MB L2 can hide at most 3 % of the bytes."""
    with pkg.Open(pkg.Config(ordinals=[0], bytes=4 * GiB, mode=pkg.abi.MODE_FULL, timeout_ms=60000)) as p:
        p.SetOption(pkg.abi.OPT_PATH, path)
        for r, tr in run_and_check(p, 3, True, runs=3):
            bpp = r.bytes_per_pair
            rates = [bpp / (ph[e] - ph["t_start"]) for ph in tr[0] for j, e in (("job0", "t_end0"), ("job1", "t_end1"))
                     if ph[j] in ("read", "write", "verify")]
            print(f"\n[timing] path {path}: loop-back job GB/s {[round(x) for x in rates]}")
            assert rates and max(rates) < HBM_GBPS, rates
            assert r.gbps_read[0][0] < HBM_GBPS and r.gbps_write[0][0] < HBM_GBPS


@gpu
@pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("mode,nbytes", [(0, 0), (1, GiB), (2, 256 << 20)], ids=["reach-only", "sliced-1GiB", "full"])
def test_nvlink_cells_stay_under_the_link_rate(pkg, mode, nbytes):
    n = min(NGPU, 8)
    with pkg.Open(pkg.Config(ordinals=list(range(n)), bytes=nbytes or GiB, mode=mode, timeout_ms=20000)) as p:
        for r, _ in run_and_check(p, 3, False):
            for i in range(n):
                for j in range(n):
                    if i != j:
                        assert 0 < r.gbps_read[i][j] < NVLINK_GBPS and 0 < r.gbps_write[i][j] < NVLINK_GBPS, (i, j)


@gpu
@pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("uni", [False, True], ids=["both-ways", "one-way"])
def test_nvlink_cells_are_near_the_copy_engine(pkg, uni):
    """The SM probe of pair (0, 1) against the copy engine on the same pair, direction and schedule."""
    flags = pkg.abi.FLAG_UNIDIRECTIONAL if uni else 0
    with pkg.Open(pkg.Config(ordinals=[0, 1], bytes=GiB, mode=pkg.abi.MODE_FULL, flags=flags)) as p:
        rs = [x[0] for x in run_and_check(p, 3, False, runs=3)]
        for push, key in ((True, "gbps_write"), (False, "gbps_read")):
            copies = [(0, 1)] if uni else [(0, 1), (1, 0)]
            ce = [g for _, g in p.CeCopy(copies, push=push, reps=4)]
            for (i, j), c in zip(copies, ce):
                sm = max(getattr(r, key)[i][j] for r in rs)
                print(f"\n[timing] {key} {i}->{j} {'one-way' if uni else 'both-ways'}: SM {sm:.0f}, CE {c:.0f}, "
                      f"ratio {sm / c:.3f}")
                assert 0.6 <= sm / c <= 1.15, (key, i, j, sm, c)


# ------------------------------------------------------------------------------------- timer tick ----
@gpu
def test_timer_tick_is_reported_and_reach_does_not_depend_on_it(pkg):
    """50 loop-back runs of 128 B, the shortest phases the suite has: every cell is reachable in every run, and
    the smallest nonzero phase time and the gcd of all stamps are printed."""
    stamps, phases = [], []
    with pkg.Open(pkg.Config(ordinals=[0], bytes=128)) as p:
        for _ in range(50):
            r = p.Run()
            assert r.reach == [[1]] and r.verdict and not r.aborted
            tr = check_model(p, r, 3, True)
            check_timeline(r, tr, 1, events=False)
            for ph in tr[0]:
                stamps += [ph[k] for k in ("t_start", "t_end0", "t_end1", "t_arrive") if ph[k]]
                if ph["job0"] in ("read", "write"):
                    phases.append(ph["t_end0"] - ph["t_start"])
    g = functools.reduce(math.gcd, stamps)
    nz = [x for x in phases if x > 0]
    print(f"\n[timing] globaltimer: gcd of {len(stamps)} stamps {g} ns, smallest phase {min(nz) if nz else None} ns, "
          f"zero-length phases {len(phases) - len(nz)} of {len(phases)}")
    assert all(x > 0 for x in phases)
