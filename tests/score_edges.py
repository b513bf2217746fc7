"""The node-local scorers restated in plain Python, and a table of (allocatable, requested) rows at their arithmetic edges.

leastRequestedScore / leastResourceScorer (noderesources/least_allocated.go:30-61) in Python ints, balancedResourceScorer
(noderesources/balanced_allocation.go:146-180) in Python floats: IEEE double, one rounding per operation, int() truncation like
Go's int64(). Neither depends on the oracle or the kernels, so both can be checked against them.

The kernels take shortcuts exactly here: the least score is an fp32 quotient estimate repaired with an int64 remainder, the
balanced score trusts an fp32 screen unless it lies within 1/64 of an integer (ccsim_device.cuh). The table puts requests on
every quotient boundary of a range of capacities, near-integer balanced values, clipped fractions, zero allocatable and
operands above 2^53, so that a wrong shortcut changes some row's score.
"""
import functools
import importlib

import numpy as np

abi = importlib.import_module("cluster-capacity_b200._abi")

INT64_MAX = (1 << 63) - 1
CAP_MAX = INT64_MAX // 100            # the largest capacity whose (capacity - requested) * 100 cannot overflow int64
CAPACITIES = [1, 2, 7, 100, 1000, (1 << 24) - 1, (1 << 24) + 1, 10**9 + 7, 64000, 512 << 30, 1 << 40, (1 << 53) - 1, (1 << 53) + 1, CAP_MAX]
# (requested, capacity) pairs where an fp32 estimate of the least quotient is off by one in either direction
FP32_REPAIR_CASES = [(52903383750351562, 76671570652683425), (11329731028648695, 47207212619369554)]
# (w_fit, w_balanced, least_w_cpu, least_w_mem): the default, uneven resource weights (no `>> 1` shortcut), score-weight sums
# up to 40 (scores up to 4000: every bit of the 12-bit packed score field), a resource weight of 0
WEIGHTS = [(1, 1, 1, 1), (1, 1, 3, 7), (3, 7, 1, 1), (20, 20, 1, 1), (40, 0, 2, 5), (0, 40, 1, 1), (13, 27, 1, 0)]
CLONES = (0, 1, 7)
# per clone, the probe templates add this much to Requested and NonZeroRequested (least / balanced pod requests are 0, so that
# clone 0 sees the table's values exactly and clones 1 and 7 step over the neighbouring boundaries)
CLONE_CPU, CLONE_MEM = 1, 1


def least_requested(requested, capacity):
    if capacity == 0:
        return 0
    if requested > capacity:
        return 0
    return ((capacity - requested) * 100) // capacity        # both operands >= 0: floor == Go's truncation


def least_score(a_cpu, a_mem, q_cpu, q_mem, w_cpu, w_mem):
    node_score = weight_sum = 0
    for a, q, w in ((a_cpu, q_cpu, w_cpu), (a_mem, q_mem, w_mem)):
        if a == 0:
            continue
        node_score += least_requested(q, a) * w
        weight_sum += w
    if weight_sum == 0:
        return 0
    return node_score // weight_sum


def balanced_score(a_cpu, a_mem, q_cpu, q_mem):
    fr = []
    for a, q in ((a_cpu, q_cpu), (a_mem, q_mem)):
        if a == 0:
            continue
        f = float(q) / float(a)
        if f > 1:
            f = 1.0
        fr.append(f)
    std = abs((fr[0] - fr[1]) / 2) if len(fr) == 2 else 0.0
    return int((1 - std) * 100.0)


def boundary_requests(c):
    """Requests on every quotient boundary of capacity c, +-1 and +-2, and requested == capacity, capacity + 1, 0."""
    out = {0, c, c + 1}
    for q in range(101):
        r0 = c - (-(-q * c // 100))          # the largest request whose free part still gives quotient >= q
        for d in (-2, -1, 0, 1, 2):
            if 0 <= r0 + d <= c + 1:
                out.add(r0 + d)
    return sorted(out)


@functools.lru_cache(maxsize=None)
def edge_rows():
    """(a_cpu, a_mem, req_cpu, req_mem) rows, >= 10^5 of them. NonZeroRequested equals Requested on every row."""
    rng = np.random.default_rng(20261017)
    pairs = [(c, r) for c in CAPACITIES for r in boundary_requests(c)]
    rows = []
    n = len(pairs)
    for mult, off in ((1, 0), (7, 13), (31, 101), (113, 7), (257, 999), (1021, 4242)):
        for i, (c, r) in enumerate(pairs):
            c2, r2 = pairs[(i * mult + off) % n]
            rows.append((c, c2, r, r2))
    for c, r in pairs:                       # allocatable 0 on one resource (its fraction / quotient is left out)
        rows.append((c, 0, r, r % 5))
        rows.append((0, c, r % 3, r))
    # balanced values within a hair of an integer: cpu fraction ~ k/50 next to a zero memory request (680/1000 -> 65.999...),
    # and two fractions whose difference is ~ 2k/100
    for c0 in CAPACITIES + [3, 50, 300, 3000, 10**6, 999983]:
        for k in range(51):
            base = (k * c0 + 25) // 50
            for d in (-2, -1, 0, 1, 2):
                r0 = base + d
                if r0 < 0:
                    continue
                for c1 in (1000, 7, 1 << 40, CAP_MAX):
                    rows.append((c0, c1, r0, 0))
                for r1n, r1d in ((1, 3), (1, 7), (2, 5), (17, 64)):
                    r1 = c0 * r1n // r1d
                    rows.append((c0, c0, r1 + r0, r1))
    for r, c in FP32_REPAIR_CASES:
        rows.append((c, 1000, r, 680))
        rows.append((1000, c, 680, r))
    rows.append((1000, 1000, 680, 0))
    # more rows like FP32_REPAIR_CASES: large capacities, free part next to a quotient boundary, where a correctly rounded fp32
    # quotient (the device's approximate one is within 2 ulp of it) is one below or one above the truth
    found = {-1: 0, 1: 0}
    while min(found.values()) < 150:
        c = int(2 ** rng.uniform(25, 56.3))
        x = -(-int(rng.integers(1, 100)) * c // 100) + int(rng.integers(-3, 3))
        e = int(np.float32(np.float32(x * 100) / np.float32(c)))
        s = (e > x * 100 // c) - (e < x * 100 // c)
        if s and found[s] < 150:
            found[s] += 1
            rows.append((c, c, c - x, int(rng.integers(0, c + 1))))
    # clipped fractions (requested > allocatable) and operands above 2^53
    for c in CAPACITIES:
        for r in (c + 1, 2 * c, c + (1 << 53)):
            if r < INT64_MAX // 2:
                rows.append((c, CAPACITIES[int(rng.integers(len(CAPACITIES)))], r, 0))
    big = [1 << 53, (1 << 53) + 1, (1 << 60) // 100, CAP_MAX, CAP_MAX - 1]
    for c in big:
        for _ in range(200):
            rows.append((c, big[int(rng.integers(len(big)))], int(rng.integers(0, c + 2)), int(rng.integers(1 << 52, 1 << 56))))
    # random fill: log-uniform capacities, requests up to 1.2x
    while len(rows) < 100_000 + 5000:
        c0, c1 = (int(min(CAP_MAX, 2 ** rng.uniform(0, 56.3))) for _ in range(2))
        rows.append((c0, c1, int(rng.integers(0, c0 * 6 // 5 + 2)), int(rng.integers(0, c1 * 6 // 5 + 2))))
    return rows


def edge_snapshot(alloc_pods=None, npods=None, taint_mask=None, taint_nosched=(), topo=()):
    rows = edge_rows()
    n = len(rows)
    a = np.array(rows, dtype=np.int64)
    return abi.Snapshot(n, a[:, 0], a[:, 1], np.full(n, 110, np.int32) if alloc_pods is None else alloc_pods,
                        req_cpu=a[:, 2], req_mem=a[:, 3], npods=npods, taint_mask=taint_mask, taint_nosched=taint_nosched, topo=topo)


def probe_template(weights):
    """Scorer-only template: the pod adds CLONE_CPU / CLONE_MEM per clone, its least / balanced requests are 0, every other
    score weight is 0."""
    w_fit, w_bal, w_cpu, w_mem = weights
    t = abi.default_template(CLONE_CPU, CLONE_MEM)
    t.least_cpu = t.least_mem = t.bal_cpu = t.bal_mem = 0
    t.w_taint = t.w_node_affinity = t.w_pts = t.w_ipa = t.w_image = 0
    t.w_fit, t.w_balanced, t.least_w_cpu, t.least_w_mem = w_fit, w_bal, w_cpu, w_mem
    return t


def reference_scores(weights, clones, rows=None):
    """(total, least, balanced) of every row after `clones` clones of probe_template(weights), in Python arithmetic."""
    w_fit, w_bal, w_cpu, w_mem = weights
    tot, lst, bal = [], [], []
    for a_cpu, a_mem, r_cpu, r_mem in (edge_rows() if rows is None else rows):
        q_cpu, q_mem = r_cpu + clones * CLONE_CPU, r_mem + clones * CLONE_MEM
        ls = least_score(a_cpu, a_mem, q_cpu, q_mem, w_cpu, w_mem)
        bs = balanced_score(a_cpu, a_mem, q_cpu, q_mem)
        lst.append(ls)
        bal.append(bs)
        tot.append(w_fit * ls + w_bal * bs)
    return np.array(tot, np.int64), np.array(lst, np.int64), np.array(bal, np.int64)
