"""What the host must make of the kernels' timestamps: a pure-Python restatement of `assemble()` and of the merge
in `cdprobe_gather` (handle.cc).

From each local rank's trace (Probe.Trace(): ns relative to the first barrier release) and the result's reach
bits, mapping status, gates and bytes_per_pair, `predict` gives the fields the host derives, exactly:
  - gbps_read / gbps_write of every probed cell: float32 of bytes_per_pair / (t_end0 - t_start) in double, 0 for
    a job that did not finish after it started;
  - min_gbps_read / min_gbps_write over the off-diagonal cells (the diagonal when n == 1);
  - slow_pairs (reachable but under the gate), unreachable_pairs (MIG-excluded cells skipped) and verdict,
    including the n == 1 loop-back rule (reachability only);
  - device_ms (= t_arrive of the last phase / 1e6) and barrier_us (sum of next t_start - t_arrive, / 1e3).
`merge` is the gather: rows another process filled are copied, counts add up, the verdict is the AND.
Results and predictions are plain dicts keyed like fabricprobe.Result's fields, matrices as n x n lists.
"""
from __future__ import annotations

import numpy as np

OP_READ, OP_WRITE = 1, 2
ERR_UNSUPPORTED = -8  # CDPROBE_ERR_UNSUPPORTED: the mapping status of a MIG-excluded pair

DERIVED = ("gbps_read", "gbps_write", "min_gbps_read", "min_gbps_write", "slow_pairs", "unreachable_pairs", "verdict")
MERGED = ("reach_read", "reach_write", "gbps_read", "gbps_write", "status", "sum_read", "xor_read", "sum_write",
          "xor_write", "row_mask", "verdict", "aborted", "unreachable_pairs", "slow_pairs", "min_gbps_read",
          "min_gbps_write")


def f32(x: float) -> float:
    return float(np.float32(x))


def as_dict(r) -> dict:
    """The fields of a fabricprobe.Result the model reads or predicts."""
    keys = set(MERGED) | {"n", "bytes_per_pair", "gate_gbps_read", "gate_gbps_write", "device_ms", "barrier_us",
                          "event_ms", "kernel_ms", "probe_ms", "run_seq"}
    return {k: getattr(r, k) for k in keys}


def predict(res: dict, traces, first: int, ops: int, diag: bool) -> dict:
    """Fields assemble() derives for local ranks first .. first + len(traces) - 1 of result `res`."""
    n, bpp = res["n"], res["bytes_per_pair"]
    ops = ops or (OP_READ | OP_WRITE)
    gate = {"read": res["gate_gbps_read"], "write": res["gate_gbps_write"]}
    reach = {"read": res["reach_read"], "write": res["reach_write"]}
    out = {"gbps_read": [[0.0] * n for _ in range(n)], "gbps_write": [[0.0] * n for _ in range(n)],
           "slow_pairs": 0, "unreachable_pairs": 0, "device_ms": [], "barrier_us": []}
    mins = {"read": None, "write": None}
    verdict = True
    for li, tr in enumerate(traces):
        g = first + li
        slow = [False] * n
        bar_ns = 0.0
        for p, ph in enumerate(tr):
            if p + 1 < len(tr) and tr[p + 1]["t_start"] > ph["t_arrive"]:
                bar_ns += float(tr[p + 1]["t_start"] - ph["t_arrive"])
            op = ph["job0"]
            if op not in ("read", "write"):
                continue
            j = ph["peer0"]
            done = not res["aborted"] and ph["t_end0"] > ph["t_start"]
            gbps = f32(bpp / float(ph["t_end0"] - ph["t_start"])) if done else 0.0
            out["gbps_" + op][g][j] = gbps
            if j != g or n == 1:
                if mins[op] is None or gbps < mins[op]:
                    mins[op] = gbps
                if reach[op][g][j] and j != g and gbps < gate[op]:
                    slow[j] = True
        last = tr[-1]["t_arrive"] if tr else 0
        out["device_ms"].append(float(last) / 1e6 if last > 0 else 0.0)
        out["barrier_us"].append(bar_ns / 1e3)
        for j in range(n):
            if j == g or res["status"][g][j] == ERR_UNSUPPORTED or res["status"][j][g] == ERR_UNSUPPORTED:
                continue
            unreachable = bool((ops & OP_READ and not res["reach_read"][g][j]) or
                               (ops & OP_WRITE and not res["reach_write"][g][j]))
            if unreachable:
                out["unreachable_pairs"] += 1
            elif slow[j]:
                out["slow_pairs"] += 1
            if unreachable or slow[j]:
                verdict = False
        if n == 1 and diag:
            if (ops & OP_READ and not res["reach_read"][g][g]) or (ops & OP_WRITE and not res["reach_write"][g][g]):
                verdict = False
    out["min_gbps_read"] = mins["read"] or 0.0
    out["min_gbps_write"] = mins["write"] or 0.0
    out["verdict"] = verdict and not res["aborted"]
    return out


def merge(mine: dict, others) -> dict:
    """cdprobe_gather: `mine` completed with the results of the other processes, in rank order."""
    m = {k: (v if not isinstance(v, list) else [list(row) if isinstance(row, list) else row for row in v])
         for k, v in mine.items()}
    n = m["n"]
    for o in others:
        for g in range(n):
            if not (o["row_mask"] >> g) & 1 or (m["row_mask"] >> g) & 1:
                continue
            for k in ("reach_read", "reach_write", "gbps_read", "gbps_write", "status", "sum_read", "xor_read",
                      "sum_write", "xor_write"):
                m[k][g] = list(o[k][g])
            m["row_mask"] |= 1 << g
        m["verdict"] = bool(m["verdict"]) and bool(o["verdict"])
        m["aborted"] = bool(m["aborted"]) or bool(o["aborted"])
        m["unreachable_pairs"] += o["unreachable_pairs"]
        m["slow_pairs"] += o["slow_pairs"]
        for k in ("min_gbps_read", "min_gbps_write"):
            if o[k] > 0.0 and (m[k] == 0.0 or o[k] < m[k]):
                m[k] = o[k]
    return m
