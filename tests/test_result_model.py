"""CPU checks of tests/result_model.py on hand-built traces: the arithmetic the GPU timing tests hold the library to."""
import numpy as np

import result_model as rm


def ph(job0, peer0, t_start, t_end0, t_arrive, job1="-", t_end1=0):
    return {"job0": job0, "peer0": peer0, "job1": job1, "peer1": peer0, "t_start": t_start, "t_end0": t_end0,
            "t_end1": t_end1, "t_arrive": t_arrive}


def res(n, bpp, reach_read=None, reach_write=None, status=None, gate=(0.0, 0.0), aborted=False, row_mask=1):
    ones = [[1] * n for _ in range(n)]
    z = [[0] * n for _ in range(n)]
    return {"n": n, "bytes_per_pair": bpp, "reach_read": reach_read or ones, "reach_write": reach_write or ones,
            "status": status or z, "gate_gbps_read": gate[0], "gate_gbps_write": gate[1], "aborted": aborted,
            "row_mask": row_mask, "gbps_read": [[0.0] * n for _ in range(n)], "gbps_write": [[0.0] * n for _ in range(n)],
            "sum_read": z, "xor_read": z, "sum_write": z, "xor_write": z, "verdict": True, "unreachable_pairs": 0,
            "slow_pairs": 0, "min_gbps_read": 0.0, "min_gbps_write": 0.0}


def test_loopback_gbps_device_ms_and_barrier_time():
    bpp = 3 << 20
    tr = [ph("write", 0, 0, 1000, 1200), ph("read", 0, 1500, 4500, 4700, "verify", 4600)]
    out = rm.predict(res(1, bpp), [tr], 0, 3, True)
    assert out["gbps_write"] == [[float(np.float32(bpp / 1000.0))]]
    assert out["gbps_read"] == [[float(np.float32(bpp / 3000.0))]]
    assert out["min_gbps_read"] == out["gbps_read"][0][0] and out["min_gbps_write"] == out["gbps_write"][0][0]
    assert out["device_ms"] == [4700 / 1e6] and out["barrier_us"] == [300 / 1e3]
    assert out["verdict"] and out["unreachable_pairs"] == 0 and out["slow_pairs"] == 0


def test_loopback_rule_fails_the_verdict_without_counting_a_pair():
    r = res(1, 128, reach_write=[[0]])
    out = rm.predict(r, [[ph("write", 0, 0, 10, 20), ph("read", 0, 20, 30, 40)]], 0, 3, True)
    assert not out["verdict"] and out["unreachable_pairs"] == 0
    assert rm.predict(r, [[ph("read", 0, 0, 30, 40)]], 0, 1, True)["verdict"]  # reads only: the write bit is not judged


def test_a_phase_that_did_not_advance_the_clock_reports_zero():
    out = rm.predict(res(1, 128), [[ph("read", 0, 500, 500, 600)]], 0, 1, True)
    assert out["gbps_read"] == [[0.0]] and out["min_gbps_read"] == 0.0


def test_slow_unreachable_and_mig_excluded_cells():
    n, bpp = 4, 1 << 30
    reach_w = [[1] * n for _ in range(n)]
    reach_w[1][2] = 0
    status = [[0] * n for _ in range(n)]
    status[3][1] = rm.ERR_UNSUPPORTED
    r = res(n, bpp, reach_write=reach_w, status=status, gate=(500.0, 500.0))
    # rank 1: reads 0 at 1000 GB/s, writes 0 at 250 GB/s (slow), write to 2 unverified, nothing probed with 3
    tr = [ph("write", 0, 0, bpp // 250, bpp // 250 + 10), ph("read", 0, bpp // 250 + 20, bpp // 250 + 20 + bpp // 1000,
                                                             bpp // 250 + 30 + bpp // 1000),
          ph("write", 2, bpp // 100, bpp // 100 + bpp // 700, bpp // 100 + bpp // 700 + 5)]
    out = rm.predict(r, [tr], 1, 3, False)
    assert out["gbps_write"][1][0] == float(np.float32(bpp / float(bpp // 250)))
    assert out["slow_pairs"] == 1            # 1 -> 0
    assert out["unreachable_pairs"] == 1     # 1 -> 2 unverified; 1 -> 3 is excluded by status[3][1]
    assert not out["verdict"]
    assert out["min_gbps_write"] == out["gbps_write"][1][0]
    assert out["device_ms"] == [tr[-1]["t_arrive"] / 1e6]


def test_aborted_rows_report_no_bandwidth():
    out = rm.predict(res(2, 1 << 20, aborted=True), [[ph("read", 1, 0, 100, 200)]], 0, 1, False)
    assert out["gbps_read"][0][1] == 0.0 and not out["verdict"]


def test_merge_completes_rows_and_combines_counts():
    n = 2
    a, b = res(n, 128, row_mask=1), res(n, 128, row_mask=2)
    a["gbps_read"][0][1], b["gbps_read"][1][0] = 5.0, 3.0
    a["min_gbps_read"], b["min_gbps_read"] = 5.0, 3.0
    a["min_gbps_write"], b["min_gbps_write"] = 2.0, 0.0
    b["verdict"], b["slow_pairs"], b["unreachable_pairs"] = False, 1, 2
    m = rm.merge(a, [b])
    assert m["row_mask"] == 3 and m["gbps_read"] == [[0.0, 5.0], [3.0, 0.0]]
    assert m["min_gbps_read"] == 3.0 and m["min_gbps_write"] == 2.0  # a zero minimum from another process is ignored
    assert not m["verdict"] and m["slow_pairs"] == 1 and m["unreachable_pairs"] == 2
    assert a["row_mask"] == 1 and a["gbps_read"][1][0] == 0.0  # the input is not modified
