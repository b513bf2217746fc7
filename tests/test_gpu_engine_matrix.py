"""GPU: every instantiation of the wave kernel, at the values and sizes where its shortcuts matter, against the CPU oracle.

- The device scorer (ccsim_debug_node_scores: score_node, the function every wave kernel scores with) against the Python
  restatement of the reference's arithmetic on the edge table of tests/score_edges.py.
- The kernel matrix: each of the ten instantiations (run_stats()["kernel"] says which one ran) on a cluster built from the edge
  table, with the default score weights and with score-weight sums of 40 (every bit of the 12-bit packed score field).
- Tile geometry: chunks (nodes per CTA) around one node per thread of the lean kernels, the multi-commit limit, the streaming
  stage ring and the largest chunk the resident-column streaming mode takes; the generic kernel above the resident tile.
- Wraps: the 19-bit memo generation of the resident-column streaming mode, the 8-bit run epoch of a handle.
Every run compares the pod -> node sequence, the stop code, the FitError histogram and the preemption counts with the oracle.
"""
import importlib
import threading

import numpy as np
import pytest

import score_edges as se
from oracle import binding as oracle

abi = importlib.import_module("cluster-capacity_b200._abi")
synth = importlib.import_module("cluster-capacity_b200.synth")

pytestmark = pytest.mark.gpu
MiB = 1 << 20


@pytest.fixture(scope="module")
def engine(built):
    return importlib.import_module("cluster-capacity_b200.engine")


@pytest.fixture(scope="module")
def sm_count(engine):
    with engine.Engine(device=0) as e:
        return e.device_info()["sm_count"]


@pytest.fixture(scope="module")
def limit(sm_count):
    """Pods per run: a few waves per CTA of a full grid, cheap for the oracle."""
    return 3 * sm_count + 17


_ORACLE = {}


def oracle_run(key, snap, tmpl, ctr, lim, mode=0):
    if key not in _ORACLE:
        _ORACLE[key] = oracle.run(snap, tmpl, ctr, max_pods=lim, mode=mode, threads=4, memo=True)
    return _ORACLE[key]


def assert_same(got, want, what):
    assert got.placed == want.placed and got.stop_code == want.stop_code, (what, got.placed, want.placed, got.stop_code, want.stop_code)
    if not np.array_equal(got.pod_node, want.pod_node):
        k = int(np.nonzero(got.pod_node != want.pod_node)[0][0])
        pytest.fail("%s: pod %d went to node %d, the oracle says %d" % (what, k, got.pod_node[k], want.pod_node[k]))
    assert np.array_equal(got.reason_hist, want.reason_hist), what
    assert (got.preempt_no_victims, got.preempt_not_helpful) == (want.preempt_no_victims, want.preempt_not_helpful), what


def run_one(engine, snap, tmpl, ctr, lim, kind=abi.ENGINE_AUTO, sampling=abi.SAMPLING_CANONICAL):
    with engine.Engine(device=0, engine=kind, sampling=sampling) as eng:
        eng.load_nodes(snap)
        eng.set_templates(tmpl, ctr)
        got = eng.run(lim)
        return got, eng.run_stats()


def run_sharded(engine, snap, tmpl, ctr, limits, world=2):
    """All ranks on device 0, wired by pointer, one host thread per rank (like tests/test_gpu_sharded_one_gpu.py). Yields, per
    limit, the per-rank results and run_stats."""
    engs = [engine.Engine(device=0, rank=r, world=world) for r in range(world)]
    try:
        for e in engs:
            e.load_nodes(snap)
            e.set_templates(tmpl, ctr)
        engine.Engine.connect_local(engs)
        for lim in limits:
            for e in engs:
                e.prepare(lim)
            res, errs = [None] * world, []

            def work(r):
                try:
                    res[r] = engs[r].run(lim)
                except Exception as ex:       # noqa: BLE001
                    errs.append(ex)
            th = [threading.Thread(target=work, args=(r,)) for r in range(world)]
            for t in th:
                t.start()
            for t in th:
                t.join(timeout=120)
            assert not errs, errs
            assert all(r is not None for r in res), "a rank did not finish"
            yield res, [e.run_stats() for e in engs]
    finally:
        for e in engs:
            e.close()


def assert_sharded_same(res, want, what):
    for r in res:
        assert r.placed == want.placed and r.stop_code == want.stop_code, what
        assert np.array_equal(r.pod_node, want.pod_node), what
    assert np.array_equal(sum(r.reason_hist for r in res), want.reason_hist), what
    assert sum(r.preempt_no_victims for r in res) == want.preempt_no_victims, what
    assert sum(r.preempt_not_helpful for r in res) == want.preempt_not_helpful, what


# ---- 1. the device scorer against the Python reference --------------------------------------------------------------------
@pytest.mark.parametrize("weights", se.WEIGHTS)
def test_device_scores_match_python_reference(engine, weights):
    snap = se.edge_snapshot()
    with engine.Engine(device=0) as eng:
        eng.load_nodes(snap)
        eng.set_templates([se.probe_template(weights)])
        for clones in se.CLONES:
            got = eng.debug_node_scores(0, clones)
            want = se.reference_scores(weights, clones)
            for name, g, w in zip(("total", "least", "balanced"), got, want):
                bad = np.nonzero(g != w)[0]
                assert len(bad) == 0, "clones %d: %s differs on %d rows, first (a_cpu, a_mem, req_cpu, req_mem) = %s: device %d, reference %d" % (
                    clones, name, len(bad), se.edge_rows()[bad[0]], g[bad[0]], w[bad[0]])


# ---- 2. the kernel matrix ---------------------------------------------------------------------------------------------------
WEIGHT_SETS = {"edge": (1, 1, 3, 7), "w40": (20, 20, 1, 1)}
KERNELS = ["batched", "lean/canonical", "lean/reference", "generic/resident", "generic/streamed", "multi/1gpu", "multi/shards",
           "stream/mode0", "stream/mode1", "stream/mode2"]


def edge_case(kernel, weights):
    """The edge-table cluster set up so that `kernel` runs: (snapshot, templates, counters, env overrides, engine kind, sampling)."""
    n_all = len(se.edge_rows())
    rows = n_all if kernel != "multi/shards" else 20_000          # (two ranks share one GPU: each rank's grid must stay small)
    a = np.array(se.edge_rows()[:rows], dtype=np.int64)
    n = len(a)
    topo, taint, nosched = (), None, ()
    if kernel.startswith("multi"):
        topo = [(np.arange(n) % 7).astype(np.int32)]
    if kernel == "stream/mode1":                                   # a NoSchedule taint the templates do not tolerate
        taint = ((np.arange(n) % 10) == 3).astype(np.uint64).reshape(1, n)
        nosched = [1]
    snap = abi.Snapshot(n, a[:, 0], a[:, 1], np.full(n, 110, np.int32), req_cpu=a[:, 2], req_mem=a[:, 3], topo=topo,
                        taint_mask=taint, taint_nosched=nosched)
    t = se.probe_template(weights)
    tmpl, ctr, env, kind, sampling = [t], [], {}, abi.ENGINE_AUTO, abi.SAMPLING_CANONICAL
    if kernel.startswith("multi"):
        ctr = [abi.make_counter(0, np.zeros(7, np.int32), inc=1)]
        t.n_pts, t.pts[0].counter, t.pts[0].max_skew, t.pts[0].self_match = 1, 0, 2, 1
    if kernel.startswith("stream"):
        t2 = se.probe_template(weights)
        t2.req_cpu = t2.nz_cpu = 3
        t2.req_mem = t2.nz_mem = 2
        tmpl.append(t2)
    if kernel == "stream/mode0":
        env["CCSIM_STREAM_ALL"] = "1"
    if kernel == "lean/canonical":
        kind = abi.ENGINE_SEQUENTIAL
    if kernel == "lean/reference":
        sampling = abi.SAMPLING_REFERENCE
    if kernel.startswith("generic"):
        env["CCSIM_FORCE_GENERIC"] = "1"
    if kernel == "generic/streamed":
        env["CCSIM_FORCE_STREAMING"] = "1"
    return snap, tmpl, ctr, env, kind, sampling


@pytest.mark.parametrize("weights", sorted(WEIGHT_SETS))
@pytest.mark.parametrize("kernel", KERNELS)
def test_kernel_matrix_on_edge_cluster(engine, monkeypatch, limit, kernel, weights):
    snap, tmpl, ctr, env, kind, sampling = edge_case(kernel, WEIGHT_SETS[weights])
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    mode = 1 if sampling == abi.SAMPLING_REFERENCE else 0
    want = oracle_run(("edge", kernel, weights), snap, tmpl, ctr, limit, mode=mode)
    if kernel == "multi/shards":
        for res, stats in run_sharded(engine, snap, tmpl, ctr, [limit]):
            assert [s["kernel"] for s in stats] == [kernel] * 2
            assert_sharded_same(res, want, kernel)
        return
    got, stats = run_one(engine, snap, tmpl, ctr, limit, kind=kind, sampling=sampling)
    assert stats["kernel"] == kernel
    assert_same(got, want, kernel)


def test_score_weight_sum_above_40_is_refused(engine):
    snap = se.edge_snapshot()
    with engine.Engine(device=0) as eng:
        eng.load_nodes(snap)
        eng.set_templates([se.probe_template((20, 20, 1, 1))])
        with pytest.raises(engine.EngineError, match="sum of score weights 41 too large for the packed key"):
            eng.set_templates([se.probe_template((20, 21, 1, 1))])


# ---- 3. tile geometry -------------------------------------------------------------------------------------------------------
def node_local(n, n_templates=1, taint=False, coupled=False):
    """C2-like nodes; one template (or several podspecs for the streaming kernel); optionally a taint on 10% of the nodes that the
    templates do not tolerate, or a zone spread constraint (multi-commit / lean)."""
    rng = np.random.default_rng(n)
    a_cpu = rng.choice([4, 8, 16, 32, 64], n).astype(np.int64) * 1000
    a_mem = a_cpu * int(rng.choice([2, 4])) * MiB
    req_cpu = (rng.random(n) * 0.7 * a_cpu).astype(np.int64) // 10 * 10
    req_mem = (rng.random(n) * 0.7 * a_mem).astype(np.int64)
    kw = {}
    if taint:
        kw = dict(taint_mask=(rng.random(n) < 0.1).astype(np.uint64).reshape(1, n), taint_nosched=[1])
    if coupled:
        kw["topo"] = [rng.integers(0, 16, n).astype(np.int32)]
    snap = abi.Snapshot(n, a_cpu, a_mem, np.full(n, 110, np.int32), req_cpu=req_cpu, req_mem=req_mem,
                        npods=rng.integers(0, 60, n).astype(np.int32), **kw)
    tmpl = [abi.default_template(int(rng.integers(50, 2001)), int(rng.integers(64, 4097)) * MiB) for _ in range(n_templates)]
    ctr = []
    if coupled:
        ctr = [abi.make_counter(0, rng.integers(0, 3, 16).astype(np.int32), inc=1)]
        tmpl[0].n_pts, tmpl[0].pts[0].counter, tmpl[0].pts[0].max_skew, tmpl[0].pts[0].self_match = 1, 0, 2, 1
    return snap, tmpl, ctr


def n_for_chunk(chunk, S):
    """Node count whose grid (min(S, ceil(N / 512)) CTAs) gives `chunk` nodes per CTA, with the fullest grid that does."""
    grid = min(S, -(-chunk * S // 512))
    return chunk * grid if chunk > 512 else chunk


def chunk_of(n, S):
    grid = max(1, min(S, -(-n // 512)))
    return -(-n // grid), grid


def check_geometry(engine, n_label, snap, tmpl, ctr, lim, kind, kernel, env=(), monkeypatch=None):
    for k, v in env:
        monkeypatch.setenv(k, v)
    want = oracle_run(("geo", n_label, snap.n, len(tmpl), len(ctr), bool(snap.taint_mask.any())), snap, tmpl, ctr, lim)
    got, stats = run_one(engine, snap, tmpl, ctr, lim, kind=kind)
    assert stats["kernel"] == kernel, (snap.n, stats["kernel"], stats["grid"])
    assert_same(got, want, "%s n=%d grid=%d" % (kernel, snap.n, stats["grid"]))
    return stats


def lean_geometries(S):
    short = 769 * (S - 1) + (769 - S + 1)               # the smallest last CTA a chunk of 769 can have on S CTAs
    return {"chunk768": 768 * S, "chunk769": 768 * S + 1, "chunk1537": 1536 * S + 1, "n512": 512, "n513": 513, "short_last": short}


@pytest.mark.parametrize("geo", ["chunk768", "chunk769", "chunk1537", "n512", "n513", "short_last"])
def test_lean_and_batched_tile_geometry(engine, sm_count, limit, geo):
    S = sm_count
    n = lean_geometries(S)[geo]
    chunk, grid = chunk_of(n, S)
    if geo == "short_last":
        assert chunk == 769 and n - chunk * (grid - 1) < chunk
    snap, tmpl, ctr = node_local(n)
    for kind, kernel in ((abi.ENGINE_AUTO, "batched"), (abi.ENGINE_SEQUENTIAL, "lean/canonical")):
        st = check_geometry(engine, geo, snap, tmpl, ctr, limit, kind, kernel)
        assert st["grid"] == grid
    if geo in ("chunk768", "chunk769"):     # a coupled template: multi-commit up to 768 nodes per CTA (one per thread), lean beyond
        snap, tmpl, ctr = node_local(n, coupled=True)
        check_geometry(engine, geo + "c", snap, tmpl, ctr, limit, abi.ENGINE_AUTO, "multi/1gpu" if chunk <= 768 else "lean/canonical")
        check_geometry(engine, geo + "c", snap, tmpl, ctr, limit, abi.ENGINE_SEQUENTIAL, "lean/canonical")


@pytest.mark.parametrize("chunk", [1024, 1025, 4096, 4097])
def test_streaming_tile_geometry(engine, sm_count, limit, chunk):
    n = chunk * sm_count
    snap, tmpl, ctr = node_local(n, n_templates=2)
    check_geometry(engine, "s", snap, tmpl, ctr, limit, abi.ENGINE_AUTO, "stream/mode2")


def test_streaming_mask_columns_and_forced_mode0_past_the_stage_ring(engine, monkeypatch, sm_count, limit):
    """Chunks of 5 tiles: more tiles than the 4 stages of the ring (stage reuse within a pass, the winner's row patched into a
    stage that already landed), with the mask columns (MODE 1) and with every column streamed (MODE 0, forced)."""
    n = 4097 * sm_count
    snap, tmpl, ctr = node_local(n, n_templates=2, taint=True)
    check_geometry(engine, "m1", snap, tmpl, ctr, limit, abi.ENGINE_AUTO, "stream/mode1")
    snap, tmpl, ctr = node_local(n, n_templates=2)
    check_geometry(engine, "s", snap, tmpl, ctr, limit, abi.ENGINE_AUTO, "stream/mode0", env=[("CCSIM_STREAM_ALL", "1")], monkeypatch=monkeypatch)


def test_streaming_largest_resident_chunk(engine, sm_count, limit):
    """The largest chunk MODE 2 takes (8 tiles, or fewer when the resident columns and the template table outgrow shared memory),
    found from the kernel that runs; that chunk in MODE 2 and one node more in MODE 0."""
    largest = 0
    for tiles in range(1, 9):
        snap, tmpl, ctr = node_local(tiles * 1024 * sm_count, n_templates=2)
        _, stats = run_one(engine, snap, tmpl, ctr, 1)
        if stats["kernel"] == "stream/mode2":
            largest = tiles * 1024
        else:
            assert stats["kernel"] == "stream/mode0"
    assert largest >= 4096
    for chunk, kernel in ((largest, "stream/mode2"), (largest + 1, "stream/mode0")):
        snap, tmpl, ctr = node_local(chunk * sm_count, n_templates=2)
        check_geometry(engine, "s", snap, tmpl, ctr, limit, abi.ENGINE_AUTO, kernel)


def test_generic_streamed_tile_natural(engine, sm_count, limit):
    """Required pod affinity (no lean / streaming kernel takes it) on a cluster whose tiles do not fit in shared memory."""
    n = 4096 * sm_count
    rng = np.random.default_rng(7)
    snap, tmpl, _ = node_local(n)
    snap.topo = [rng.integers(0, 32, n).astype(np.int32)]
    init = np.zeros(32, np.int32)
    init[[3, 11, 20]] = 1
    ctr = [abi.make_counter(0, init, inc=1)]
    t = tmpl[0]
    t.n_aff, t.aff_counter[0], t.aff_total_init = 1, 0, 3
    check_geometry(engine, "aff", snap, tmpl, ctr, limit, abi.ENGINE_AUTO, "generic/streamed")


# ---- 4. wraps ---------------------------------------------------------------------------------------------------------------
def test_stream_memo_generation_wraps(engine):
    """MODE 2 keeps a 19-bit generation per node (the memo entry of a template is valid while it stands). Two nodes take ~600k
    best-effort clones each, alternating as their scores step down: both pass 2^19 commits."""
    n = 4
    a_cpu = np.array([100 * 700_000, 100 * 700_000 + 31, 4000, 4000], np.int64)
    a_mem = a_cpu * (2 * MiB)
    snap = abi.Snapshot(n, a_cpu, a_mem, np.array([600_000, 600_000, 0, 0], np.int32))
    tmpl = [abi.default_template(0, 0), abi.default_template(0, 0, nz_cpu=130, nz_mem=150 * MiB)]
    want = oracle.run(snap, tmpl, [], max_pods=0, threads=1, memo=True)
    assert np.bincount(want.pod_node, minlength=2)[:2].min() > (1 << 19)
    got, stats = run_one(engine, snap, tmpl, [], 0)
    assert stats["kernel"] == "stream/mode2"
    assert_same(got, want, "memo generation wrap")


def epoch_case(kernel):
    snap, tmpl, ctr = node_local(1200, n_templates=2 if kernel == "stream/mode2" else 1, coupled=kernel.startswith("multi"))
    rng = np.random.default_rng(3)
    snap.alloc_pods = (snap.npods + rng.integers(0, 3, snap.n)).astype(np.int32)     # room for 0..2 pods: small unbounded runs
    return snap, tmpl, ctr


@pytest.mark.parametrize("kernel", ["lean/canonical", "multi/1gpu", "stream/mode2", "multi/shards"])
def test_run_epoch_wraps(engine, kernel):
    """300 runs of one handle (the 8-bit run epoch, which keeps words of earlier runs from validating, wraps after 255), limits
    cycling over 1, 2 and unbounded; every run equals the oracle."""
    snap, tmpl, ctr = epoch_case(kernel)
    limits = [1, 2, 0] * 100
    wants = {lim: oracle.run(snap, tmpl, ctr, max_pods=lim, threads=4, memo=True) for lim in (1, 2, 0)}
    assert wants[0].placed > 100
    if kernel == "multi/shards":
        for i, (res, stats) in enumerate(run_sharded(engine, snap, tmpl, ctr, limits)):
            assert [s["kernel"] for s in stats] == [kernel] * 2
            assert_sharded_same(res, wants[limits[i]], "run %d" % i)
        return
    kind = abi.ENGINE_SEQUENTIAL if kernel == "lean/canonical" else abi.ENGINE_AUTO
    with engine.Engine(device=0, engine=kind) as eng:
        eng.load_nodes(snap)
        eng.set_templates(tmpl, ctr)
        for i, lim in enumerate(limits):
            got = eng.run(lim)
            assert eng.run_stats()["kernel"] == kernel
            assert_same(got, wants[lim], "run %d" % i)
