"""CPU: the oracle's node-local scorers (NodeResourcesFit LeastAllocated, BalancedAllocation) against a plain Python
restatement of the reference's arithmetic, on a table of rows at the edges where the kernels' fp32 shortcuts could slip
(tests/score_edges.py). The GPU side of the same comparison is in tests/test_gpu_engine_matrix.py."""
import numpy as np
import pytest

import score_edges as se
from oracle import binding as oracle


def test_least_and_balanced_known_answers():
    assert se.least_requested(0, 0) == 0 and se.least_requested(5, 4) == 0 and se.least_requested(4, 4) == 0
    assert se.least_requested(0, 7) == 100 and se.least_requested(1, 7) == 85      # 600 // 7
    for r, c in se.FP32_REPAIR_CASES:
        assert se.least_requested(r, c) == ((c - r) * 100) // c
    assert se.least_requested(*se.FP32_REPAIR_CASES[0]) == 31
    assert se.least_requested(*se.FP32_REPAIR_CASES[1]) == 75
    # Go's float64: (1 - 0.68/2) * 100 = 65.99999999999999 -> 65 (exact arithmetic would say 66)
    assert se.balanced_score(1000, 1000, 680, 0) == 65
    assert se.balanced_score(1000, 0, 680, 0) == 100 and se.balanced_score(0, 0, 1, 1) == 100
    assert se.balanced_score(10, 10, 20, 0) == 50                                        # clipped fraction
    assert se.least_score(1000, 0, 500, 7, 1, 1) == 50 and se.least_score(1000, 1000, 500, 0, 3, 7) == (50 * 3 + 100 * 7) // 10


def test_edge_table_covers_the_edges():
    rows = se.edge_rows()
    assert len(rows) >= 100_000
    for r in rows:
        for a, q in ((r[0], r[2]), (r[1], r[3])):
            assert 0 <= a <= se.CAP_MAX and q >= 0
            q7 = q + 7 * max(se.CLONE_CPU, se.CLONE_MEM)
            assert q7 < se.INT64_MAX
            if q7 <= a:
                assert (a - q) * 100 <= se.INT64_MAX          # (c - r) * 100 never overflows int64
    cpu = {(r[0], r[2]) for r in rows}
    for c in se.CAPACITIES:
        for q in range(101):
            r0 = c - (-(-q * c // 100))
            assert all((c, r0 + d) in cpu for d in (-2, -1, 0, 1, 2) if 0 <= r0 + d <= c + 1), (c, q)
        assert (c, c) in cpu and (c, c + 1) in cpu
    assert any(r[1] == 0 for r in rows) and any(r[0] == 0 for r in rows)
    assert any(r[2] > r[0] > 0 for r in rows) and any(r[2] > (1 << 53) and r[0] > (1 << 53) for r in rows)
    # balanced values within 1e-12 of an integer, on both sides of it
    below = above = 0
    for a0, a1, q0, q1 in rows:
        if a0 and a1:
            f0, f1 = min(float(q0) / float(a0), 1.0), min(float(q1) / float(a1), 1.0)
            v = (1 - abs((f0 - f1) / 2)) * 100.0
            d = v - round(v)
            below += -1e-12 < d < 0
            above += 0 < d < 1e-12
    assert below >= 20 and above >= 20, (below, above)


def _f32_least(x100, c):
    return int(np.float32(np.float32(x100) / np.float32(c)))


def test_edge_table_reaches_the_fp32_shortcuts():
    """Emulated fp32 (correctly rounded; the device's approximate divide is within 2 ulp of it): the table holds rows where the
    least quotient estimate is off by one in both directions, and near-integer balanced rows whose fp32 screen value lands
    on the other side of the integer than the float64 value, within the 1/64 margin where the kernel must not trust it."""
    lo = hi = 0
    screen_flips = 0
    for a0, a1, q0, q1 in se.edge_rows():
        for a, q in ((a0, q0), (a1, q1)):
            if 0 < a and q <= a:
                x100 = (a - q) * 100
                e, t = _f32_least(x100, a), x100 // a
                lo += e < t
                hi += e > t
        if a0 > 0 and a1 > 0:
            g0 = min(np.float32(np.float32(q0) / np.float32(a0)), np.float32(1))
            g1 = min(np.float32(np.float32(q1) / np.float32(a1)), np.float32(1))
            v = (np.float32(1) - abs(g0 - g1) * np.float32(0.5)) * np.float32(100)
            fl = np.floor(v)
            if int(fl) != se.balanced_score(a0, a1, q0, q1):
                fr = float(v - fl)
                assert not (0.015625 < fr < 0.984375), (a0, a1, q0, q1)   # the screen's margin covers every emulated slip
                screen_flips += 1
    assert lo >= 10 and hi >= 10, (lo, hi)
    assert screen_flips >= 10, screen_flips


@pytest.mark.parametrize("weights", se.WEIGHTS)
def test_oracle_scorers_match_python_reference(built, weights):
    snap = se.edge_snapshot()
    t = se.probe_template(weights)
    for clones in (se.CLONES if weights == se.WEIGHTS[0] else (0,)):
        want = se.reference_scores(weights, clones)
        got = oracle.node_scores(snap, t, clones)
        for name, g, w in zip(("total", "least", "balanced"), got, want):
            bad = np.nonzero(g != w)[0]
            assert len(bad) == 0, "%s differs on %d rows, first %s: oracle %d, reference %d" % (
                name, len(bad), se.edge_rows()[bad[0]], g[bad[0]], w[bad[0]])
