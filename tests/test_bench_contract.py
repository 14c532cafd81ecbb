"""The bench.py JSON contract, checked on the lines recorded on the B200 boxes (profiles/r01_final_*, profiles/r02_*):
every key the driver reads is present with the right type and the numbers are internally consistent.
(The lines themselves were produced by `bench.py` on GPU; this guards the schema on CPU.)"""
import json
import os

import pytest

from conftest import ROOT

PROFILES = os.path.join(ROOT, "profiles")
REQUIRED = {"metric": str, "value": float, "unit": str, "n_gpus": int, "steps": int, "warmup": int,
            "ms_per_step": float, "higher_is_better": bool, "scaling": str, "dtype": str, "data": str, "config": dict,
            "e2e": dict, "gpu_launches": int, "roofline": dict, "clocks": dict}


def load(name):
    p = os.path.join(PROFILES, name)
    if not os.path.exists(p):
        pytest.skip(f"{name} not recorded")
    return json.loads([l for l in open(p) if l.startswith("{")][-1])


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_our_arm_line(n):
    j = load(f"r01_final_bench_n{n}.json")
    for k, t in REQUIRED.items():
        assert k in j, k
        assert isinstance(j[k], t) or (t is float and isinstance(j[k], int)), (k, type(j[k]))
    assert j["metric"] == "nvlink_probe_ms" and j["unit"] == "ms" and j["higher_is_better"] is False
    assert j["n_gpus"] == n and j["vs_baseline"] is None and j["data"] == "synthetic" and j["scaling"] == "weak"
    assert j["warmup"] >= 3 and j["gpu_launches"] == j["steps"] * n
    assert "workload" in j["config"] and "model" not in j["config"]
    e = j["e2e"]
    assert e["unit"] == "ms" and e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    r = j["roofline"]
    assert set(["bound", "achieved", "peak", "unit", "frac", "traffic"]) <= set(r)
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["unit"] == "GB/s"
    c = j["clocks"]
    assert c["sm_mhz"] and c["sm_max_mhz"] and isinstance(c["reasons"], list)
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert j["reachability_all_ones"] is True and j["verdict"] is True
    # the wall clock of the timed loop agrees with the per-call figure (no work hidden outside the loop)
    assert abs(j["ms_per_step"] - e["value"]) / e["value"] < 0.05
    if n == 1:
        assert r["bound"] == "hbm" and 0.5 < r["frac"] < 1.1 and r["traffic"] >= r["algorithmic_bytes_per_launch"]
        cb = j["cpu_baseline"]
        assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
    else:
        assert r["bound"] == "nvlink" and 0.5 < r["frac"] < 1.0
        nv = j["nvlink_counters"]
        assert abs(nv["tx_kib_delta"] / nv["algorithmic_kib_per_direction"] - 1) < 1e-3  # counters == algorithmic bytes
        assert j["per_link_gbps"]["run_to_run_spread_read"] < 0.02 and j["per_link_gbps"]["run_to_run_spread_write"] < 0.02
        assert j["value"] < 5.0  # north_star: < 5 ms


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_reference_arm_line(n):
    j = load(f"r01_final_ref_n{n}.json")
    assert j["impl"] == "reference" and j["metric"] == "nvlink_probe_ms" and j["unit"] == "ms"
    assert j["higher_is_better"] is False and j["n_gpus"] == n and j["gpu_launches"] == 0 and j["value"] > 0
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    ours = load(f"r01_final_bench_n{n}.json")
    if "workload" in j["config"] and "reference_path" in j["config"]:
        assert j["config"]["workload"] == ours["config"]["workload"]  # both arms answer the same question


# ---- round 2 lines: parity block, same-box CE ceilings, daemon cost, configs c2 / c3-full / c5 ----------------
def _common_r02(j, n):
    for k, t in REQUIRED.items():
        if k == "roofline" and j["config"].get("config") == "c5":
            continue
        assert k in j, k
        assert isinstance(j[k], t) or (t is float and isinstance(j[k], int)), (k, type(j[k]))
    assert j["metric"] == "nvlink_probe_ms" and j["unit"] == "ms" and j["higher_is_better"] is False
    assert j["n_gpus"] == n and j["vs_baseline"] is None and j["scaling"] == "weak" and j["warmup"] >= 3
    p = j["parity"]
    assert p["cells"] == (n * (n - 1) if n > 1 else 1) and p["checksum_ok"] is True and p["reach_vs_nvml_ok"] is True
    assert p["checksum_mismatches"] == [] and p["nvml_gpus_polled"] >= n
    d = j["daemon_cost"]
    assert d["cold_first_verdict_ms"] >= d["open_ms"] > 0 and d["first_run_ms"] > 0
    assert j["reachability_all_ones"] is True and j["verdict"] is True
    c = j["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_r02_headline_line(n):
    j = load(f"r02_bench_n{n}.json")
    _common_r02(j, n)
    assert j["gpu_launches"] == j["steps"] * n
    assert j["value"] >= j["kernel_ms_globaltimer"] >= j["device_ms_globaltimer"] > 0
    e = j["e2e"]
    assert abs(j["ms_per_step"] - e["value"]) / e["value"] < 0.05 and e["d2h_bytes_per_step"] == 48 + 120 * j["config"]["phases"]
    dp = j["daemon_cost"]["daemon_process"]  # a fresh `cdprobe-daemon run --once` over the same N GPUs
    assert dp["exit"] == 0 and dp["ok"] is True and dp["n_gpus"] == n and dp["unreachable_pairs"] == dp["slow_pairs"] == 0
    assert dp["wall_ms"] > dp["probe_ms"] > 0
    r = j["roofline"]
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["statistic"] == "median" and cb["value"] == cb["median_ms"] <= cb["mean_ms"] * 1.5
    if n == 1:
        assert r["bound"] == "hbm" and 0.9 < r["frac"] < 1.05
    else:
        assert r["bound"] == "nvlink" and j["value"] < 5.0
        assert 700 < r["peak_measured_ce_bidi"] < 900 and 700 < r["peak_measured_ce_uni"] < 900
        assert 0.8 < r["frac_read_of_ce_bidi"] < 1.0 and 0.8 < r["frac_write_of_ce_bidi"] < 1.0
        # wire view: payload + protocol bytes of both directions' ops fill the 900 GB/s a direction has
        assert 0.9 < r["frac_wire_read_phase_of_900"] < 1.0 and 0.85 < r["frac_wire_write_phase_of_900"] < 1.0
        nv = j["nvlink_counters"]
        assert abs(nv["tx_kib_delta"] / nv["algorithmic_kib_per_direction"] - 1) < 1e-3
        if nv.get("per_physical_link_tx"):  # the 18 links of the port carry equal shares (a weak link would stand out)
            pl = nv["per_physical_link_tx"]
            assert pl["links_carrying_traffic"] == 18 and sum(pl["kib"]) == nv["tx_kib_delta"]
            assert 0.98 < pl["min_share_of_mean"] <= 1.0 <= pl["max_share_of_mean"] < 1.02
        g = j["per_link_gbps"]
        assert g["read_min"] > g["gate_gbps_read"] > 500 and g["write_min"] > g["gate_gbps_write"] > 500
        assert j["config"]["barriers"] == "neighbourhood"
        if n == 8:
            assert j["barrier_us"] < 60  # round 1: ~93-110 us with 15 all-rank exchanges (VERDICT r01 next #3)
            assert j["value"] < 3.30    # round 1: 3.328-3.330 ms


@pytest.mark.parametrize("name,n,cfg", [("r02_bench_c2_n2.json", 2, "c2"), ("r02_bench_c3full_n8.json", 8, "c3-full")])
def test_r02_config_lines(name, n, cfg):
    j = load(name)
    _common_r02(j, n)
    assert j["config"]["config"] == cfg and j["config"]["mode"] == "full"
    assert j["config"]["bytes_per_pair"] == j["config"]["bytes_per_gpu"] == ((64 << 20) if cfg == "c2" else (1 << 30))


@pytest.mark.parametrize("n", [2, 8])
def test_r02_storm_line(n):
    j = load(f"r02_bench_c5_n{n}.json")
    _common_r02(j, n)
    st = j["storm"]
    assert j["config"]["config"] == "c5" and st["cycles"] == j["steps"] and (n != 8 or st["cycles"] == 1000)
    assert st["verdict_failures"] == 0 and st["device_free_delta_bytes"] == 0 and st["fd_delta"] == 0
    assert st["cycle_ms_p99"] >= st["cycle_ms_p50"] >= st["probe_ms_p50"] > 0 and j["gpu_launches"] == st["cycles"] * n


# ---- the parity self-check of bench.py is not vacuous: a wrong checksum or a wrong reach bit is caught -------------
def test_parity_block_catches_mismatches(pkg, oracle, monkeypatch):
    import types

    import bench

    n, nbytes, mode = 3, 3 << 12, 1
    bpp = oracle.plan(n, nbytes, mode).bytes_per_pair
    words = bpp // 8
    seed, run_seq = oracle.DEFAULT_SEED, 7

    def result():
        r = types.SimpleNamespace(bytes_per_pair=bpp, run_seq=run_seq)
        z = [[0] * n for _ in range(n)]
        r.sum_read, r.xor_read, r.sum_write, r.xor_write = ([row[:] for row in z] for _ in range(4))
        r.reach = [[1] * n for _ in range(n)]
        for i in range(n):
            for j in range(n):
                if i != j:
                    r.sum_read[i][j], r.xor_read[i][j] = oracle.expected_read(seed, n, nbytes, mode, i, j)
                    r.sum_write[i][j], r.xor_write[i][j] = oracle.write_checksum(seed, i, j, run_seq, words)
        return r

    # no NVML in this container: the reach half must say so (None), never assume
    good = bench.parity_block(pkg, oracle, result(), n, nbytes, mode, [f"GPU-{i}" for i in range(n)], seed)
    assert good["cells"] == 6 and good["checksum_ok"] is True and good["reach_vs_nvml_ok"] is None and good["reach_vs_nvml_error"]
    bad = result()
    bad.xor_write[2][0] ^= 1 << 40
    blk = bench.parity_block(pkg, oracle, bad, n, nbytes, mode, [f"GPU-{i}" for i in range(n)], seed)
    assert blk["checksum_ok"] is False and blk["checksum_mismatches"] == [["write", 2, 0]]
    # with an NVML that answers (the fake one): an unreachable cell the NVML poll calls reachable is a parity failure
    fake = types.SimpleNamespace(uuids=lambda: [f"GPU-{i}" for i in range(n)], reach_matrix=lambda: [[1] * n for _ in range(n)], n=n)
    monkeypatch.setattr(oracle, "nvml_poll", lambda *a, **k: fake)
    r = result()
    assert bench.parity_block(pkg, oracle, r, n, nbytes, mode, [f"GPU-{i}" for i in (2, 0, 1)], seed)["reach_vs_nvml_ok"] is True
    r.reach[1][2] = 0
    blk = bench.parity_block(pkg, oracle, r, n, nbytes, mode, [f"GPU-{i}" for i in range(n)], seed)
    assert blk["reach_vs_nvml_ok"] is False and blk["reach_mismatches"] == [[1, 2, 0, 1]]


@pytest.mark.gpu
def test_bench_runs_end_to_end_with_parity(tmp_path):
    """bench.py itself on the GPU box (N = 1, a few steps): exit 0, one JSON line, parity block green, roofline
    against the measured peak — what the driver runs, exercised by `pytest -m gpu` too."""
    import subprocess
    import sys

    cp = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "10", "--warmup", "3",
                         "--no-cpu-baseline", "--no-daemon"], capture_output=True, text=True, timeout=300)
    assert cp.returncode == 0, cp.stderr[-2000:]
    lines = [l for l in cp.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["n_gpus"] == 1 and j["gpu_launches"] == 10 and j["parity"]["checksum_ok"] is True
    assert j["parity"]["reach_vs_nvml_ok"] is True and j["verdict"] is True and 0.5 < j["roofline"]["frac"] < 1.1


def _load_dump(d):
    import numpy as np

    out = {}
    for f in sorted(os.listdir(d)):
        a = np.load(os.path.join(d, f))
        assert a.dtype in (np.float32, np.float64), (f, a.dtype)
        out[f[:-len(".npy")]] = a
    return out


def test_dump_outputs_keeps_every_checksum_bit(tmp_path):
    """--dump-outputs stores float arrays only: a u64 checksum goes out as its exact (high, low) 32-bit halves."""
    import types

    import numpy as np

    import bench

    n = 2
    big = [[0xFFFFFFFFFFFFFFFF, 0x8000000000000001], [(1 << 53) + 1, 12345]]
    r = types.SimpleNamespace(reach_read=[[1, 0], [1, 1]], reach_write=[[1, 1], [0, 1]], status=[[0, -4], [0, 0]],
                              sum_read=big, xor_read=big, sum_write=big, xor_write=big)
    bench.dump_outputs(r, str(tmp_path / "out"))
    d = _load_dump(tmp_path / "out")
    assert set(d) == {"reach_read", "reach_write", "status", "sum_read", "xor_read", "sum_write", "xor_write"}
    assert d["reach_read"].tolist() == r.reach_read and d["status"].tolist() == r.status
    for name in ("sum_read", "xor_read", "sum_write", "xor_write"):
        a = d[name]
        assert a.shape == (n, n, 2)
        assert [[(int(a[i, j, 0]) << 32) | int(a[i, j, 1]) for j in range(n)] for i in range(n)] == big


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_and_match_the_oracle(tmp_path, oracle):
    """Two runs with the same arguments dump the same files; the dumped read checksum is the oracle's, and the
    dumped matrices are the ones the line's parity block checked."""
    import subprocess
    import sys

    nbytes = 16 << 20
    dumps = []
    for k in range(2):
        d = tmp_path / f"out{k}"
        cp = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "5", "--warmup", "3",
                             "--bytes", str(nbytes), "--no-cpu-baseline", "--no-daemon", "--dump-outputs", str(d)],
                            capture_output=True, text=True, timeout=300)
        assert cp.returncode == 0, cp.stderr[-2000:]
        j = json.loads([l for l in cp.stdout.splitlines() if l.startswith("{")][-1])
        assert j["steps"] == 5 and j["parity"]["checksum_ok"] is True
        dumps.append(_load_dump(d))
    a, b = dumps
    assert set(a) == set(b) and all((a[k] == b[k]).all() for k in a)
    assert a["reach_read"].tolist() == a["reach_write"].tolist() == [[1.0]] and a["status"].tolist() == [[0.0]]
    s, x = (int(a[k][0, 0, 0]) << 32 | int(a[k][0, 0, 1]) for k in ("sum_read", "xor_read"))
    assert (s, x) == oracle.expected_read(oracle.DEFAULT_SEED, 1, nbytes, 1, 0, 0, True)
