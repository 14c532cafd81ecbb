#!/usr/bin/env python3
"""bench.py — the ComputeDomain fabric probe benchmark (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA probe
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU/NVML poll
    python bench.py --config c2|c3-full|c5 ...                # BASELINE configs 2 / 3 (full mode) / 5 (storm)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's results as DIR/*.npy

A "step" is one pass of the hot path: one `cdprobe_run` over the N-GPU domain (sliced mode,
1 GiB per GPU, read + write + verify) — BASELINE.json configs[2] at N GPUs; at N = 1 the same
kernel runs its loop-back phases against local HBM.  One process per GPU (torchrun for N > 1);
the data path is NVLink P2P between cuMem-mapped buffers with a hand-rolled device barrier —
torch.distributed (NCCL) is used only to bracket the timed region and take max-over-ranks.

metric  = nvlink_probe_ms (lower is better): time to produce the N x N reachability + GB/s
          matrix.  `value` is the probe kernel's duration by CUDA events on its launch stream
          (median of the K timed steps, max over ranks; buffers resident in HBM; the mean and the worst
          step are in `value_mean_ms` / `value_max_ms`); `e2e.value` is the same probe through the
          public C ABI call from the host: launch, kernel, result rows written to pinned host
          memory and read back.  Per-pair GB/s vs the 900 GB/s/dir NVLink-5 peak is in
          `per_link_gbps`; `roofline` is the dominant kernel against its bound (HBM at N = 1,
          NVLink at N > 1).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the benchmark leaves the tree as the build left it (it may be read-only): no bytecode caches next to the sources
sys.dont_write_bytecode = True

GIB = 1 << 30
NVLINK_PEAK_GBPS = 900.0        # nominal per direction per GPU (BASELINE.md §2)
# (the profiling guide quotes a 770 GB/s peer copy; it is not used: every N > 1 line carries the SAME-BOX copy-engine
#  figures measured next to the probe on the probe's own buffers, roofline.peak_measured_ce_{uni,bidi})
HBM_FALLBACK_GBPS = 6650.0
# Bytes on the NVLink wire per payload byte of SM-issued traffic, from ncu's nvltx/nvlrx counters on the solo probe
# kernel (profiles/r02_ncu_nvlink_{read,write}.csv; 1 GiB of payload each): a read costs 1.125 B of response in the
# payload direction (32 B per 256-B response) and 0.1875 B of request in the opposite one (48 B per 256 B); a write
# costs 1.1875 B in the payload direction and ~0.003 B of acknowledgement back.
WIRE = {"read_rx": 1207959648 / 1073741888, "read_tx_req": 201326656 / 1073741888,
        "write_tx": 1275068544 / 1073741888, "write_rx_ack": 3453312 / 1073741888}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": HBM_FALLBACK_GBPS}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.025):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml

            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        return {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "samples": len(self.samples),
            "reasons": sorted(self.reasons),
        }


def nvlink_counters(index: int):
    """NVLink data TX/RX KiB of one GPU through NVML field values 138/139: the aggregate over its links
    (scopeId 0xFFFFFFFF) and each of the 18 physical links (scopeId = link) — or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        out = {}
        for name, fid in (("tx_kib", 138), ("rx_kib", 139)):
            vals = pynvml.nvmlDeviceGetFieldValues(h, [(fid, 0xFFFFFFFF)] + [(fid, l) for l in range(18)])
            if vals[0].nvmlReturn != 0:
                return None
            out[name] = int(vals[0].value.ullVal)
            out[name + "_per_link"] = [int(v.value.ullVal) if v.nvmlReturn == 0 else None for v in vals[1:]]
        return out
    except Exception:
        return None


def per_link_delta(a, b, key):
    """Per physical link KiB moved between two samples, and how evenly the GPU spread them over its links."""
    x, y = a.get(key + "_per_link"), b.get(key + "_per_link")
    if not x or not y or any(v is None for v in x + y):
        return None
    d = [q - p for p, q in zip(x, y)]
    active = [v for v in d if v > 0]
    if not active:
        return None
    mean = sum(active) / len(active)
    return {"kib": d, "links_carrying_traffic": len(active), "min_share_of_mean": min(active) / mean,
            "max_share_of_mean": max(active) / mean}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def workload_name(n: int, mode: str, nbytes: int) -> str:
    """The workload both arms answer: validate the N-GPU domain's fabric (N x N reachability matrix)."""
    if n > 1:
        return (f"{n}-GPU all-pairs NVLink probe, {mode} mode, {nbytes >> 20} MiB per GPU, "
                f"read+write+verify (BASELINE configs[2] at {n} GPU)")
    return f"1-GPU loop-back probe, {nbytes >> 20} MiB buffer, read+write+verify"


# --------------------------------------------------------------------- reference arm ----
def cpu_poll_timing(n_gpus: int, steps: int, warmup: int, budget_s: float, flags: int = 0):
    """Times the reference's CPU path (oracle/nvml_poll.c: the NVML enumerate + NvLinkState + P2PStatus
    poll the north_star names) on this box's host cores; flags = 8 runs the link/P2P polls on one thread
    per GPU."""
    from oracle import oracle as o

    o.lib()
    times, last = [], None
    t_stop = time.perf_counter() + budget_s
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        last = o.nvml_poll(n_gpus, flags)
        dt = (time.perf_counter() - t0) * 1e3
        if i >= warmup:
            times.append(dt)
        if time.perf_counter() > t_stop and len(times) >= 3:
            break
    return times, last


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return 0
    line = {"impl": "reference", "metric": "nvlink_probe_ms", "unit": "ms", "n_gpus": args.gpus,
            "higher_is_better": False, "data": "synthetic", "dtype": "u64", "vs_baseline": None, "scaling": "weak",
            "gpu_launches": 0}
    try:
        # both variants the survey asks for: one thread (NVML serialises in the RM) and one thread per GPU;
        # the line reports the faster one
        t1, last = cpu_poll_timing(args.gpus, args.steps, args.warmup, budget_s=60.0)
        tn, last_n = cpu_poll_timing(args.gpus, args.steps, args.warmup, budget_s=60.0, flags=8)
    except Exception as e:  # NVML missing etc.: say so, do not fake a number
        line["unavailable"] = f"NVML poll could not run: {e}"
        print(json.dumps(line))
        return 0
    threaded = last.n > 1 and statistics.median(tn) < statistics.median(t1)
    times = tn if threaded else t1
    cores = last.n if threaded else 1
    # the distribution has a 10-50x tail (first nvmlInit of a process, RM lock contention): the median is the
    # typical poll, mean and max ride beside it
    v = statistics.median(times)
    sample = (f"{len(times)} polls of the {last.n}-GPU node: nvmlInitWithFlags + enumerate + fabric info + "
              f"{18 * last.n} NvLinkState + {3 * last.n * (last.n - 1)} P2PStatus + nvmlShutdown "
              f"({last.nvml_calls} NVML calls per poll)")
    line.update({
        "value": v, "ms_per_step": statistics.mean(times), "steps": len(times), "warmup": args.warmup,
        "config": {"workload": workload_name(args.gpus, args.mode, args.bytes),
                   "reference_path": (f"the reference's CPU answer to the same question: NVML enumerate + NvLinkState + "
                                      f"P2PStatus poll of {last.n} GPU(s) -> N x N reachability matrix (it moves no bytes "
                                      f"and measures no bandwidth: SURVEY.md F1)"),
                   "n_gpus_polled": last.n, "threads": cores},
        "cpu_baseline": {"value": v, "unit": "ms", "cores": cores, "kind": "port", "sample": sample,
                         "single_thread_ms": statistics.median(t1), "thread_per_gpu_ms": statistics.median(tn),
                         "host_cores": os.cpu_count(), "statistic": "median", "mean_ms": statistics.mean(times),
                         "median_ms": statistics.median(times), "max_ms": max(times),
                         "phases_ms": {"init": last.init_ms, "enumerate": last.enumerate_ms, "fabric": last.fabric_ms,
                                       "link_poll": last.link_poll_ms, "p2p_poll": last.p2p_poll_ms,
                                       "shutdown": last.shutdown_ms}},
        "e2e": {"value": v, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reach_all_ones": all(last.reach[i * 16 + j] for i in range(last.n) for j in range(last.n)),
    })
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- our arm ----
CONFIGS = {
    # BASELINE.json configs[1]: 2-GPU P2P read/write reachability matrix, 64 MiB buffers, IMEX channel 0
    "c2": {"gpus": 2, "bytes": 64 << 20, "mode": "full", "fabric": True,
           "name": "BASELINE configs[1]: 2-GPU P2P read/write reachability matrix, 64 MiB buffers, full mode, "
                   "fabric handles iff IMEX channel 0 exists"},
    # configs[2] in full mode: every ordered pair moves the whole 1 GiB buffer (56 GiB over the fabric at N = 8)
    "c3-full": {"gpus": None, "bytes": GIB, "mode": "full", "fabric": False,
                "name": "BASELINE configs[2] in FULL mode: {n}-GPU all-pairs NVLink probe, 1 GiB per ordered pair"},
    # configs[4]: reconcile storm — one probe per NodePrepare/Unprepare cycle, a peer mapping torn down and rebuilt each cycle
    "c5": {"gpus": None, "bytes": GIB, "mode": "sliced", "fabric": False,
           "name": "BASELINE configs[4]: reconcile storm, {cycles} prepare/unprepare cycles (unmap + remap of one peer, "
                   "then a full probe) on {n} GPU(s)"},
}


def parity_block(pkg, oracle, res, n, nbytes, mode_id, uuids, seed):
    """Driver-visible parity (VERDICT r01 next #1), outside every timed region: every cell's checksums against
    the CPU oracle's restatement of the patterns, and reach_read AND reach_write against the reachability
    matrix the oracle derives from the NVML poll (nvlib.go:208-363; go-nvml device.go:281-285,1652-1661),
    matched by GPU UUID."""
    diag = n == 1
    cells = [(i, j) for i in range(n) for j in range(n) if i != j or diag]
    bad = []
    words = res.bytes_per_pair // 8
    for i, j in cells:
        exp_r = oracle.expected_read(seed, n, nbytes, mode_id, i, j, diag)
        exp_w = oracle.write_checksum(seed, i, j, res.run_seq, words)
        if (res.sum_read[i][j], res.xor_read[i][j]) != exp_r:
            bad.append(["read", i, j])
        if (res.sum_write[i][j], res.xor_write[i][j]) != exp_w:
            bad.append(["write", i, j])
    block = {"cells": len(cells), "checksum_ok": not bad, "checksum_mismatches": bad[:8],
             "words_per_cell": words, "oracle": "oracle/pattern.c (scalar C restatement), oracle/nvml_poll.c"}
    try:
        o = oracle.nvml_poll()
        by_uuid = {u: k for k, u in enumerate(o.uuids())}
        idx = [by_uuid[u] for u in uuids]
        om = o.reach_matrix()
        exp = [[om[idx[i]][idx[j]] for j in range(n)] for i in range(n)]
        block["reach_vs_nvml_ok"] = res.reach == exp
        block["reach_cells_one"] = sum(sum(row) for row in res.reach)
        block["nvml_gpus_polled"] = o.n
        if res.reach != exp:
            block["reach_mismatches"] = [[i, j, res.reach[i][j], exp[i][j]] for i in range(n) for j in range(n)
                                         if res.reach[i][j] != exp[i][j]][:8]
    except Exception as e:  # no NVML on the box: say so; never assume
        block["reach_vs_nvml_ok"] = None
        block["reach_vs_nvml_error"] = str(e)
    return block


def dump_outputs(res, out_dir):
    """Writes the N x N matrices the last timed cdprobe_run handed its caller (completed across ranks) as
    out_dir/<name>.npy, so that two builds run with the same arguments can be compared file for file.
    Every value written is computed, not measured: the source patterns are seeded and the write pattern is
    salted by the run count, which the arguments fix.  The per-pair GB/s and the timings differ from run to
    run and stay in the JSON line.  A 64-bit checksum does not fit a float64 mantissa, so each one is stored
    as its (high, low) 32-bit halves along a last axis of length 2."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"reach_read": np.array(res.reach_read, np.float32), "reach_write": np.array(res.reach_write, np.float32),
              "status": np.array(res.status, np.float32)}
    for name in ("sum_read", "xor_read", "sum_write", "xor_write"):
        a = np.array(getattr(res, name), np.uint64)
        arrays[name] = np.stack([a >> np.uint64(32), a & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_probe(args):
    import torch

    import cdprobe_pkg

    pkg = cdprobe_pkg.load()
    abi = pkg.abi
    rank, world, local = dist_env()
    conf = CONFIGS.get(args.config) if args.config else None
    if conf:
        args.bytes, args.mode = conf["bytes"], conf["mode"]
        if conf["gpus"] and args.gpus != conf["gpus"]:
            raise SystemExit(f"--config {args.config} is defined on {conf['gpus']} GPUs (launch with --gpus {conf['gpus']})")
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch N > 1 with torchrun: one process per GPU")
    n = args.gpus
    # one visible GPU per rank (a launcher that sets CUDA_VISIBLE_DEVICES per process): the ordinal is 0
    if torch.cuda.device_count() <= local:
        local = 0
    torch.cuda.set_device(local)
    grp = pkg.distutil.RankGroup(backend="gloo")  # host-side only: barrier + max; the data path uses no collective library

    def barrier():
        grp.barrier()
        torch.cuda.synchronize()

    max_over_ranks = grp.max

    session = grp.session()
    flags = abi.FLAG_PATH_LDST if args.path == "ldst" else 0
    if conf and conf["fabric"]:
        flags |= abi.FLAG_FABRIC_HANDLES
    if args.all_rank_barriers:
        flags |= abi.FLAG_ALL_RANK_BARRIERS
    mode_id = {"sliced": 1, "full": 2, "reach": 0}[args.mode]
    cfg = pkg.Config(ordinals=[local], bytes=args.bytes, mode=mode_id, ops=3, flags=flags, ctas=args.ctas,
                     world_size=world, rank=rank, session=session, timeout_ms=args.timeout_ms)
    # what a daemon pod pays before its first verdict: contexts + VMM + mapping + fill + source checksums (open),
    # then one cold probe.  Wall clock around the public calls, max over ranks.
    barrier()
    t_open0 = time.perf_counter()
    probe = pkg.Open(cfg)
    t_open1 = time.perf_counter()
    out = abi.ResultT()

    def step():
        rc = probe.run_raw(out)
        if rc != abi.OK:
            raise RuntimeError(f"cdprobe_run rc={rc}: {abi.load_library().cdprobe_last_error().decode()}")

    step()
    t_first = time.perf_counter()
    info = probe.Info()
    daemon_cost = {
        "open_call_ms": max_over_ranks((t_open1 - t_open0) * 1e3),
        "open_ms": max_over_ranks(info.open_ms), "fill_and_checksum_ms": max_over_ranks(info.fill_ms),
        "first_run_ms": max_over_ranks((t_first - t_open1) * 1e3),
        "cold_first_verdict_ms": max_over_ranks((t_first - t_open0) * 1e3),
        "note": "cdprobe_open (CUDA contexts, cuMemCreate/Map of every rank's buffer, pattern fill, source "
                "checksums, rendezvous) + the first cdprobe_run; the steady-state `value`/`e2e` exclude it",
    }

    if args.config == "c5":
        return run_storm(args, pkg, probe, grp, info, n, rank, local, daemon_cost, conf)

    # ---- warm-up (untimed) --------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step()

    sampler = ClockSampler(local)
    sampler.start()
    nvl0 = nvlink_counters(local) if n > 1 else None

    # ---- loop A: kernel durations by CUDA events on the launch stream -> `value`, roofline
    probe.SetOption(abi.OPT_EVENT_TIMING, 1)
    step()
    ev, dev_ms, rd, wr, bar_us, ker_ms = [], [], [], [], [], []
    barrier()
    for _ in range(args.steps):
        step()
        ev.append(out.event_ms[0])
        dev_ms.append(out.device_ms[0])
        rd.append(out.min_gbps_read)
        wr.append(out.min_gbps_write)
        bar_us.append(out.barrier_us[0])
        ker_ms.append(out.kernel_ms[0])
    barrier()
    probe.SetOption(abi.OPT_EVENT_TIMING, 0)

    # ---- loop B: EXACTLY K steps through the public ABI, barrier + sync on both sides -> e2e
    step()
    host_ms = []
    warmed = 0
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
        host_ms.append(out.probe_ms)
        warmed += int(out.warmed)
    torch.cuda.synchronize()
    t_local = (time.perf_counter() - t0) * 1e3
    barrier()
    nvl1 = nvlink_counters(local) if n > 1 else None
    clocks = sampler.stop()

    wall_ms = max_over_ranks(t_local)
    ms_per_step = wall_ms / args.steps
    # `value` is the typical probe: the MEDIAN of the K event-timed kernels (max over ranks), like the reference arm's
    # median poll.  One host hiccup in K steps (a rank launching a few ms late parks every other rank's kernel in the
    # opening barrier) moves the mean by tens of us; the mean and the worst step ride beside it.
    value = max_over_ranks(statistics.median(ev))
    value_mean = max_over_ranks(statistics.mean(ev))
    value_max = max_over_ranks(max(ev))
    device_ms = max_over_ranks(statistics.median(dev_ms))
    e2e_ms = max_over_ranks(statistics.median(host_ms))
    e2e_mean = max_over_ranks(statistics.mean(host_ms))
    barrier_us = max_over_ranks(statistics.median(bar_us))
    kernel_ms = max_over_ranks(statistics.median(ker_ms))

    # per-pair GB/s over the whole domain: the last timed step's rows, completed across ranks
    rc = abi.load_library().cdprobe_gather(probe._h, ctypes.byref(out))
    if rc != abi.OK:
        raise RuntimeError(f"cdprobe_gather rc={rc}")
    res = pkg.Result.from_c(out)
    warmed_steps = max_over_ranks(float(warmed))

    # ---- parity self-check (untimed, every N): rank 0 holds the gathered matrices ----------------
    uuids = grp.gather_objects(info.uuid[0].value.decode())
    parity = None
    if rank == 0:
        from oracle import oracle as o  # the checker: never on the measured path

        o.lib()
        parity = parity_block(pkg, o, res, n, args.bytes, mode_id, uuids, o.DEFAULT_SEED)
        if args.dump_outputs:
            dump_outputs(res, args.dump_outputs)
    parity_ok = grp.gather_objects(None if parity is None else
                                   bool(parity["checksum_ok"] and parity["reach_vs_nvml_ok"] is not False))[0]

    # the daemon's situation: ONE probe after the GPUs sat idle (NVLink leaves its active state);
    # the library's automatic wake-up phase is part of this number
    time.sleep(1.0)
    barrier()
    cold = probe.Run(gather=True)
    cold_pairs = [(i, j) for i in range(n) for j in range(n) if i != j or n == 1]
    cold_start = {"idle_s": 1.0, "probe_ms": max_over_ranks(cold.probe_ms), "warmed": bool(cold.warmed),
                  "read_min": min(cold.gbps_read[i][j] for i, j in cold_pairs),
                  "write_min": min(cold.gbps_write[i][j] for i, j in cold_pairs), "verdict": bool(cold.verdict)}
    bpp = res.bytes_per_pair
    pairs_r = [res.gbps_read[i][j] for i in range(n) for j in range(n) if i != j or n == 1]
    pairs_w = [res.gbps_write[i][j] for i in range(n) for j in range(n) if i != j or n == 1]
    reach_ok = all(res.reach[i][j] == 1 for i in range(n) for j in range(n))

    def pct(v, f):
        v = sorted(v)
        return v[min(len(v) - 1, max(0, int(round(f * (len(v) - 1)))))]

    # run-to-run repeatability of this rank's slowest pair: central 90 % spread (p95 - p5) / median, and
    # the worst single step; max over ranks
    spread_r = max_over_ranks((pct(rd, 0.95) - pct(rd, 0.05)) / statistics.median(rd))
    spread_w = max_over_ranks((pct(wr, 0.95) - pct(wr, 0.05)) / statistics.median(wr))
    worst_r = max_over_ranks((statistics.median(rd) - min(rd)) / statistics.median(rd))
    worst_w = max_over_ranks((statistics.median(wr) - min(wr)) / statistics.median(wr))
    ev_spread = max_over_ranks((max(ev) - min(ev)) / statistics.median(ev))

    # per-link figure with one-way payload (each ordered pair alone on its two ports): a few extra,
    # untimed-for-the-headline runs with the unidirectional schedule
    uni = None
    ce = None
    if n > 1:
        probe.SetOption(abi.OPT_UNIDIRECTIONAL, 1)
        for _ in range(2):
            probe.Run()
        ur = [probe.Run(gather=True) for _ in range(3)]
        probe.SetOption(abi.OPT_UNIDIRECTIONAL, 0)
        u_r = [statistics.median(u.gbps_read[i][j] for u in ur) for i in range(n) for j in range(n) if i != j]
        u_w = [statistics.median(u.gbps_write[i][j] for u in ur) for i in range(n) for j in range(n) if i != j]
        uni = {"read_min": min(u_r), "read_median": statistics.median(u_r), "write_min": min(u_w),
               "write_median": statistics.median(u_w), "probe_ms": statistics.median(u.probe_ms for u in ur),
               "frac_min_of_900": min(min(u_r), min(u_w)) / NVLINK_PEAK_GBPS,
               "reach_all_ones": all(all(all(c == 1 for c in row) for row in u.reach) for u in ur)}
        # ---- the same-box ceiling: the copy engine on the very same buffers, ranks 0 <-> 1 (untimed for the
        # headline).  One way: rank 0 pushes alone.  Both ways: ranks 0 and 1 push to each other at once (each
        # process enqueues `reps` back-to-back copies after a host barrier; ~10 ms of copy hides the skew).
        reps = 8
        barrier()
        uni_push = probe.CeCopy([(0, 1)], push=True, reps=reps)[0][1] if rank == 0 else 0.0
        barrier()
        uni_pull = probe.CeCopy([(0, 1)], push=False, reps=reps)[0][1] if rank == 0 else 0.0
        barrier()
        bidi = probe.CeCopy([(0, 1 - rank)], push=True, reps=reps)[0][1] if rank < 2 else 1e30
        barrier()
        ce = {"uni_push": max_over_ranks(uni_push), "uni_pull": max_over_ranks(uni_pull), "bidi_push_min": grp.min(bidi),
              "bytes_per_copy": min(bpp * (n - 1), args.bytes if args.mode != "full" else bpp), "copies": reps,
              "how": "cudaMemcpyAsync (copy engine) between rank 0's and rank 1's probe buffers, CUDA events on the "
                     "issuing rank's stream; bidi = both ranks pushing at once"}
        uni["frac_min_of_ce_uni"] = min(min(u_r), min(u_w)) / max(ce["uni_push"], ce["uni_pull"])

    peaks, peak_kind = measured_peaks()
    passes = 3  # read B, write B, verify B per GPU per probe
    a_gpu = (n - 1 if n > 1 else 1) * bpp
    algo_bytes = passes * a_gpu  # per launch (= per GPU per probe)
    achieved = algo_bytes / (value * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f).get(f"n{n}_{args.path}")
        if t and args.bytes == GIB and args.mode == "sliced":
            traffic = t["dram_bytes_read"] + t["dram_bytes_write"]
    except Exception:
        traffic = None
    if n == 1:
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                    "traffic_source": "profiles/ncu_traffic.json (ncu --set full capture of this kernel)" if traffic else None, "peak_kind": f"{peak_kind} copy bandwidth",
                    "kernel": "cdprobe_kernel", "algorithmic_bytes_per_launch": algo_bytes,
                    "note": "N=1 loop-back: read 1 GiB + write 1 GiB + verify 1 GiB of local HBM per launch"}
    else:
        # NVLink-bound phases: read (ingress) and write (egress) each move a_gpu bytes per GPU; verify is local
        link_bytes = 2 * a_gpu
        link_achieved = min(min(pairs_r), min(pairs_w))
        roofline = {"bound": "nvlink", "achieved": link_achieved, "peak": NVLINK_PEAK_GBPS, "unit": "GB/s",
                    "frac": link_achieved / NVLINK_PEAK_GBPS, "traffic": None,
                    "peak_kind": "nominal NVLink 5 per direction per GPU; the same-box copy-engine ceilings are beside it",
                    "peak_measured_ce_uni": max(ce["uni_push"], ce["uni_pull"]), "peak_measured_ce_bidi": ce["bidi_push_min"],
                    "frac_of_ce_bidi": link_achieved / ce["bidi_push_min"],
                    "frac_read_of_ce_bidi": min(pairs_r) / ce["bidi_push_min"],
                    "frac_write_of_ce_bidi": min(pairs_w) / ce["bidi_push_min"],
                    "ce": ce,
                    # wire-level view: with both directions loaded a port's direction carries, per payload byte of its own
                    # op, the payload + protocol of that op plus the requests/acks of the opposite direction's op
                    "wire_bytes_per_payload_byte": WIRE,
                    "wire_gbps_read_phase": min(pairs_r) * (WIRE["read_rx"] + WIRE["read_tx_req"]),
                    "wire_gbps_write_phase": min(pairs_w) * (WIRE["write_tx"] + WIRE["write_rx_ack"]),
                    "frac_wire_read_phase_of_900": min(pairs_r) * (WIRE["read_rx"] + WIRE["read_tx_req"]) / NVLINK_PEAK_GBPS,
                    "frac_wire_write_phase_of_900": min(pairs_w) * (WIRE["write_tx"] + WIRE["write_rx_ack"]) / NVLINK_PEAK_GBPS,
                    "payload_ceiling_read_bidi": NVLINK_PEAK_GBPS / (WIRE["read_rx"] + WIRE["read_tx_req"]),
                    "payload_ceiling_write_bidi": NVLINK_PEAK_GBPS / (WIRE["write_tx"] + WIRE["write_rx_ack"]),
                    "wire_source": "profiles/r02_ncu_nvlink_read.csv, profiles/r02_ncu_nvlink_write.csv (ncu nvltx__/nvlrx__ "
                                   "bytes of the solo probe kernel)",
                    "kernel": "cdprobe_kernel", "algorithmic_bytes_per_launch": algo_bytes,
                    "nvlink_bytes_per_launch_per_direction": a_gpu,
                    "aggregate_link_gbps_per_gpu": link_bytes / (value * 1e-3) / 1e9,
                    "note": "achieved = slowest ordered pair with exclusive endpoints (tournament round), both "
                            "directions of every port loaded; SM-issued peer stores cap at ~715 GB/s one way on "
                            "every store shape (profiles/r02_linkbench_n2.jsonl)"}

    if rank == 0:
        wl = conf["name"].format(n=n, cycles=0) if conf else workload_name(n, args.mode, args.bytes)
        line = {
            "metric": "nvlink_probe_ms", "value": value, "unit": "ms", "n_gpus": n, "steps": args.steps,
            "value_statistic": "median of the timed steps (max over ranks)", "value_mean_ms": value_mean, "value_max_ms": value_max,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": False, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {
                "workload": wl, "config": args.config or "c3-sliced",
                "bytes_per_gpu": args.bytes, "bytes_per_pair": bpp, "mode": args.mode, "path": args.path,
                "ctas": int(info.ctas[0]), "rounds": res.rounds, "phases": res.phases,
                "barriers": "all-rank" if args.all_rank_barriers else "neighbourhood",
                "parallelism": f"{n} ranks, one process per GPU, no data-path collective",
                "l2": "inputs (1 GiB per pass) exceed the 126 MB L2; no explicit flush",
                "handle_type": int(info.handle_type),
            },
            "device_ms_globaltimer": device_ms, "kernel_ms_globaltimer": kernel_ms, "barrier_us": barrier_us,
            "time_breakdown_note": "value (CUDA events around the launch) >= kernel_ms (CTA 0 entry -> result row published) "
                                   ">= device_ms (first barrier release -> last phase done); the differences are launch/"
                                   "completion latency and the residency barrier + row output",
            "e2e": {"value": e2e_ms, "unit": "ms", "h2d_bytes_per_step": 2768,
                    "d2h_bytes_per_step": 48 + 120 * int(res.phases), "mean_ms": e2e_mean,
                    "note": "cdprobe_run from a host thread: kernel parameters (2768 B) in, result row "
                            "(pinned host memory written by the kernel) out; the probe's inputs are "
                            "generated on the device by design"},
            "gpu_launches": args.steps * n,
            "per_link_gbps": {
                "read_min": min(pairs_r), "read_median": statistics.median(pairs_r), "read_max": max(pairs_r),
                "write_min": min(pairs_w), "write_median": statistics.median(pairs_w), "write_max": max(pairs_w),
                "peak": NVLINK_PEAK_GBPS if n > 1 else peaks["hbm_gbs"],
                "frac_min": min(min(pairs_r), min(pairs_w)) / (NVLINK_PEAK_GBPS if n > 1 else peaks["hbm_gbs"]),
                "run_to_run_spread_read": spread_r, "run_to_run_spread_write": spread_w,
                "worst_step_drop_read": worst_r, "worst_step_drop_write": worst_w, "probe_ms_spread": ev_spread,
                "gate_gbps_read": res.gate_gbps_read, "gate_gbps_write": res.gate_gbps_write,
            },
            "job_throughput_gbps": (n * passes * a_gpu / (value * 1e-3) / 1e9) if n == 1 else
                                   (n * 2 * a_gpu / (value * 1e-3) / 1e9),
            "job_throughput_note": "whole-job bytes per probe / probe time: N x (read + write) payload over NVLink "
                                   "(N = 1: read + write + verify through HBM)",
            "reachability_all_ones": reach_ok, "verdict": bool(res.verdict),
            "parity": parity, "daemon_cost": daemon_cost,
            "cold_start": cold_start, "timed_steps_with_wakeup_phase_traffic": warmed_steps,
            "roofline": roofline, "clocks": clocks,
        }
        if uni is not None:
            line["per_link_gbps_unidirectional"] = uni
        if nvl0 and nvl1:
            line["nvlink_counters"] = {
                "tx_kib_delta": nvl1["tx_kib"] - nvl0["tx_kib"], "rx_kib_delta": nvl1["rx_kib"] - nvl0["rx_kib"],
                "algorithmic_kib_per_direction": (2 * args.steps + 2) * 2 * a_gpu // 1024,
                "per_physical_link_tx": per_link_delta(nvl0, nvl1, "tx_kib"),
                "per_physical_link_rx": per_link_delta(nvl0, nvl1, "rx_kib"),
                "note": "NVML fields 138/139 (NVLink data TX/RX KiB) on rank 0's GPU across both timed loops "
                        "(2 x steps + 2 probes); per probe each direction carries the write payload and the "
                        "read responses: 2 x (N-1) x bytes_per_pair.  per_physical_link_*: the same counters per link "
                        "(scopeId = link 0..17): a port spreads a pair's traffic over all its links, so a weak link "
                        "shows up here as an outlier share before it shows in the pair's GB/s"}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_subprocess(n)
    # every rank lets go of its buffers before the daemon twin takes the box (rank 0 only; the others wait in close())
    probe.Close()
    grp.barrier()
    if rank == 0:
        if not args.no_daemon:
            line["daemon_cost"]["daemon_process"] = daemon_once(n)
        print(json.dumps(line))
    grp.close()
    if parity_ok is False:
        if rank == 0:
            sys.stderr.write("PARITY FAILURE: " + json.dumps(parity) + "\n")
        return 3
    return 0


def daemon_once(n: int):
    """What a daemon pod really pays: a FRESH process (`cdprobe-daemon run --once`, the C++ twin of the Go daemon's
    probe slice) that creates the CUDA contexts of every visible GPU, opens the probe in one process, runs one cold
    pass with the daemon's defaults (1 GiB per GPU, sliced, library gate) and writes its verdict.  Wall clock of the
    process; not part of any timed region."""
    import subprocess
    import tempfile

    exe = os.path.join(ROOT, "k8s-dra-driver-gpu_b200", "cdprobe-daemon")
    lib = os.path.join(ROOT, "k8s-dra-driver-gpu_b200", "libcdprobe.so")
    with tempfile.TemporaryDirectory() as td:
        vp = os.path.join(td, "fabricprobe.json")
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "CUDA_VISIBLE_DEVICES")}
        vis = [x for x in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if x] or [str(i) for i in range(n)]
        env.update({"COMPUTE_DOMAIN_UUID": "bench", "CDPROBE_LIBRARY": lib, "FABRIC_PROBE_VERDICT_PATH": vp, "POD_UID": "bench",
                    "CUDA_VISIBLE_DEVICES": ",".join(vis[:n])})  # the same N GPUs this bench line is about
        try:
            t0 = time.perf_counter()
            cp = subprocess.run([exe, "run", "--once"], env=env, capture_output=True, text=True, timeout=300)
            wall = (time.perf_counter() - t0) * 1e3
            v = json.load(open(vp))
            tp = [l for l in cp.stderr.splitlines() if l.startswith("t_fabric_probe")]
            return {"wall_ms": wall, "exit": cp.returncode, "n_gpus": v["n"], "ok": v["ok"], "probe_ms": v["probe_ms"],
                    "t_fabric_probe_s": float(tp[-1].split()[1]) if tp else None,
                    "unreachable_pairs": v["unreachable_pairs"], "slow_pairs": v["slow_pairs"],
                    "note": "fresh `cdprobe-daemon run --once` over every visible GPU in one process: CUDA context creation + "
                            "cdprobe_open + one cold probe + verdict file"}
        except Exception as e:
            return {"wall_ms": None, "error": str(e)}


def cpu_baseline_subprocess(n: int):
    """The reference's CPU path in a fresh process (its `check` is exec'ed per kubelet probe: NVML init is never
    amortised), bounded to ~10-20 polls: the reference arm of this same script."""
    try:
        import subprocess

        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
        steps = 20 if n == 1 else 8
        cp = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--gpus", str(n),
                             "--steps", str(steps), "--warmup", "2"], capture_output=True, text=True, timeout=180, env=env)
        ref = json.loads([l for l in cp.stdout.splitlines() if l.startswith("{")][-1])
        return ref.get("cpu_baseline") or {"value": None, "unit": "ms", "cores": 1, "kind": "port",
                                           "sample": ref.get("unavailable")}
    except Exception as e:
        return {"value": None, "unit": "ms", "cores": 1, "kind": "port", "sample": f"unavailable: {e}"}


def run_storm(args, pkg, probe, grp, info, n, rank, local, daemon_cost, conf):
    """BASELINE configs[4] (SURVEY §8d C5): `--steps` prepare/unprepare cycles on one open handle; every cycle
    tears down and rebuilds this rank's mapping of one peer (the NodeUnprepare/NodePrepare churn a live domain
    sees, cmd/compute-domain-kubelet-plugin/driver.go:165-232) and then runs a full probe.  Reports p50/p99 per
    cycle, device memory and fd deltas (leak check), and the parity block of the LAST cycle."""
    import torch

    abi = pkg.abi
    cycles = args.steps
    out = abi.ResultT()

    def fd_count():
        try:
            return len(os.listdir("/proc/self/fd"))
        except OSError:
            return -1

    def cycle(k):
        t0 = time.perf_counter()
        if n > 1:
            peer = (rank + 1 + k % (n - 1)) % n
            probe.RemapPeer(0, peer)
        t1 = time.perf_counter()
        rc = probe.run_raw(out)
        if rc != abi.OK:
            raise RuntimeError(f"cycle {k}: cdprobe_run rc={rc}: {abi.load_library().cdprobe_last_error().decode()}")
        t2 = time.perf_counter()
        return (t1 - t0) * 1e3, (t2 - t1) * 1e3, bool(out.verdict), out.min_gbps_read, out.min_gbps_write

    for k in range(max(args.warmup, 3)):
        cycle(k)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    fds0 = fd_count()
    sampler = ClockSampler(local)
    sampler.start()
    grp.barrier()
    t0 = time.perf_counter()
    rows = [cycle(k) for k in range(cycles)]
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    grp.barrier()
    clocks = sampler.stop()
    free1, _ = torch.cuda.mem_get_info()
    fds1 = fd_count()

    def pct(v, f):
        v = sorted(v)
        return v[min(len(v) - 1, max(0, int(round(f * (len(v) - 1)))))]

    cyc = [a + b for a, b, *_ in rows]
    probe_ms = [b for _, b, *_ in rows]
    remap_ms = [a for a, *_ in rows]
    stats = {"cycles": cycles, "wall_ms": grp.max(wall),
             "cycle_ms_p50": grp.max(pct(cyc, 0.5)), "cycle_ms_p99": grp.max(pct(cyc, 0.99)), "cycle_ms_max": grp.max(max(cyc)),
             "probe_ms_p50": grp.max(pct(probe_ms, 0.5)), "probe_ms_p99": grp.max(pct(probe_ms, 0.99)),
             "remap_ms_p50": grp.max(pct(remap_ms, 0.5)), "remap_ms_p99": grp.max(pct(remap_ms, 0.99)),
             "verdict_failures": int(grp.max(float(sum(1 for r in rows if not r[2])))),
             "read_min_gbps": grp.min(min(r[3] for r in rows)), "write_min_gbps": grp.min(min(r[4] for r in rows)),
             "device_free_delta_bytes": int(grp.max(float(abs(free0 - free1)))), "fd_delta": int(grp.max(float(abs(fds1 - fds0))))}
    rc = abi.load_library().cdprobe_gather(probe._h, ctypes.byref(out))
    if rc != abi.OK:
        raise RuntimeError(f"cdprobe_gather rc={rc}")
    res = pkg.Result.from_c(out)
    uuids = grp.gather_objects(info.uuid[0].value.decode())
    parity = None
    if rank == 0:
        from oracle import oracle as o

        o.lib()
        parity = parity_block(pkg, o, res, n, args.bytes, 1, uuids, o.DEFAULT_SEED)
        if args.dump_outputs:
            dump_outputs(res, args.dump_outputs)
        line = {"metric": "nvlink_probe_ms", "value": stats["probe_ms_p50"], "unit": "ms", "n_gpus": n, "steps": cycles,
                "warmup": max(args.warmup, 3), "ms_per_step": stats["wall_ms"] / cycles, "higher_is_better": False,
                "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": conf["name"].format(n=n, cycles=cycles), "config": "c5", "bytes_per_gpu": args.bytes,
                           "bytes_per_pair": res.bytes_per_pair, "mode": "sliced",
                           "parallelism": f"{n} ranks, one process per GPU, no data-path collective"},
                "e2e": {"value": stats["cycle_ms_p50"], "unit": "ms", "h2d_bytes_per_step": 2768,
                        "d2h_bytes_per_step": 48 + 120 * int(res.phases),
                        "note": "one reconcile cycle through the public ABI: cdprobe_remap_peer + cdprobe_run (p50)"},
                "gpu_launches": cycles * n, "storm": stats, "parity": parity, "daemon_cost": daemon_cost,
                "reachability_all_ones": all(all(c == 1 for c in row) for row in res.reach), "verdict": bool(res.verdict),
                "clocks": clocks}
        print(json.dumps(line))
    ok = grp.gather_objects(None if parity is None else bool(parity["checksum_ok"] and parity["reach_vs_nvml_ok"] is not False))[0]
    probe.Close()
    grp.close()
    return 3 if ok is False else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cdprobe", choices=["cdprobe", "reference"])
    ap.add_argument("--bytes", type=int, default=GIB)
    ap.add_argument("--mode", default="sliced", choices=["sliced", "full", "reach"])
    ap.add_argument("--path", default="tma", choices=["tma", "ldst"])
    ap.add_argument("--ctas", type=int, default=0)
    ap.add_argument("--timeout-ms", type=int, default=10000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-daemon", action="store_true", help="skip the fresh-process daemon timing (daemon_cost.daemon_process)")
    ap.add_argument("--config", default="", choices=["", "c2", "c3-full", "c5"],
                    help="BASELINE.json configs beyond the headline: c2 (2 GPUs, 64 MiB, full), c3-full (1 GiB per ordered "
                         "pair), c5 (reconcile storm: --steps cycles)")
    ap.add_argument("--all-rank-barriers", action="store_true", help="round-1 barrier schedule (comparison)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the reachability, status and checksum matrices of the last "
                         "timed step as DIR/<name>.npy (rank 0; the same arguments give the same files)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the probe's results; the reference arm has none")
    if args.impl == "reference":
        return run_reference(args)
    return run_probe(args)


if __name__ == "__main__":
    sys.exit(main())
