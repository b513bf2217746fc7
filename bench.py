#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the cluster-capacity hot path.

One "step" = one complete capacity analysis (ClusterCapacity.Run: place clones of the podspec until one does not fit)
of the synthetic BASELINE config C4: 100 000 nodes, 3 DoNotSchedule topology-spread constraints (zone/rack/region) +
required hostname anti-affinity, 200 000 pre-existing pods (cluster-capacity_b200/synth.py, seed 3).

  value     predicate-evals/s with the snapshot already resident in HBM (ccsim_run only). Evals are counted as SURVEY.md
            §8(d) defines them — one per (pod attempt, node) of the reference loop, (placed+1) x N for a run that ends
            Unschedulable — which is also exactly what the CPU arm executes; `physical_evals_per_sec` is what the kernel
            actually pushed through the fused Filter pass (the multi-commit engine decides several cycles per pass)
  e2e       the same metric through the C-ABI with HOST buffers: ccsim_load_nodes (H2D from pinned memory) +
            ccsim_set_templates + ccsim_run + result read-back inside the timed region
  roofline  algorithmic bytes (SURVEY.md §8d: 96 B per predicate-eval for C4) / wave-kernel time vs the measured HBM peak
  cpu_baseline / --impl reference: the CPU oracle (a port of the reference's loop; no Go toolchain exists to run the
            reference itself) on the box's host cores, on a bounded prefix of the same workload.

N > 1 (torchrun): node-sharded run (SURVEY.md §8e), weak scaling: the cluster grows to N x 100k nodes (racks x N), rank r owns
a contiguous block of the node axis, the per-wave exchange of shard winners happens inside the persistent kernel over peer
memory (NVLink), torch.distributed (NCCL) only carries the IPC handles and the final small reductions. value = evals of the
whole job / max-over-ranks time. `--mode replicas` runs N independent single-GPU analyses instead (no data-path collective).

--dump-outputs DIR: after the timed steps, the result of the last timed step (what a caller of ccsim_run receives: pod -> node
sequence, FitError histogram, placed count, stop code, preemption counts) is written as DIR/<name>.npy in float64. The
workloads are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree as the build left it (it may be read-only)

import numpy as np  # noqa: E402

abi = importlib.import_module("cluster-capacity_b200._abi")
synth = importlib.import_module("cluster-capacity_b200.synth")

# workload -> (description, algorithmic bytes per predicate-eval (SURVEY.md §8d), --max-limit of a step, generator(world))
WORKLOADS = {
    "c4": ("C4: 100k nodes, 3x PodTopologySpread(DoNotSchedule zone/rack/region) + hostname anti-affinity, 200k existing pods", 96, 0,
           lambda w: synth.c4() if w == 1 else synth.c4(n=100_000 * w, n_existing=200_000 * w, racks=1024 * w)),
    # BASELINE config C5 (1M nodes x 64 podspecs round-robin): strong scaling over node shards, 100 rounds of the 64 podspecs per step
    "c5": ("C5: 1M nodes, 64 distinct podspecs (cpu 50..2000m, mem 64..4096Mi) placed round-robin, NodeResourcesFit + LeastAllocated + BalancedAllocation, --max-limit 6400",
           72, 6400, lambda w: synth.c5()),
}
WKEY = "c4"
WORKLOAD, B_EVAL, MAX_LIMIT, MAKE = WORKLOADS[WKEY]


def select_workload(key):
    global WKEY, WORKLOAD, B_EVAL, MAX_LIMIT, MAKE
    WKEY = key
    WORKLOAD, B_EVAL, MAX_LIMIT, MAKE = WORKLOADS[key]


def profiled_traffic():
    """dram__bytes_read+write per launch of the wave kernel from the committed ncu --set full capture (profiles/)."""
    # (C5: the capture is of an earlier build of the streaming kernel — 53 ms per launch — with the same DRAM-side behaviour: the
    #  4-byte memo column of the wave's template, 4 MB, comes from HBM every wave because the 64 columns, 256 MB, do not fit the L2)
    for name in ("r2_wave_%s_traffic.json" % WKEY, "r2_stream_%s_traffic.json" % WKEY, "r1_wave_c4_traffic.json" if WKEY == "c4" else ""):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return float(json.load(f)["traffic_bytes_per_launch"])
        except Exception:
            pass
    return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i] == "Active"})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def usable_cores():
    """Host threads this process may really use: min(cpu_count, affinity mask, cgroup cpu quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def calibrate_oracle(snap, tmpl, ctr):
    """The OpenMP node-axis split is calibrated first (the reference's own default is 16 goroutines,
    KS:apis/config/v1/defaults.go:108-110): the best of a few thread counts up to the usable cores is used, so that the
    CPU arm is as strong as this host allows. Returns (threads, evals/s estimate, usable cores)."""
    from oracle import binding as oracle
    cores = usable_cores()
    cand = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores} | {min(cores, 16)})
    best, best_rate = cand[0], 0.0
    for c in cand:
        oracle.run(snap, tmpl, ctr, max_pods=4, threads=c)
        t0 = time.perf_counter()
        r = oracle.run(snap, tmpl, ctr, max_pods=24, threads=c)
        rate = r.evals / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = c, rate
    return best, best_rate, cores


def cpu_oracle_rate(snap, tmpl, ctr, budget_s=20.0, calib=None):
    """Times the CPU oracle on the workload, bounded by a time budget: the first K placements with K = budget x calibrated
    rate / nodes. When the analysis ends (Unschedulable) before K, this IS the whole run. Returns
    (result, seconds, threads, usable cores, K or 0 for a whole run)."""
    from oracle import binding as oracle
    best, best_rate, cores = calib or calibrate_oracle(snap, tmpl, ctr)
    pods = int(max(50, budget_s * best_rate / max(1, snap.n)))
    whole = False
    if MAX_LIMIT and pods >= MAX_LIMIT:       # the step itself is limited (--max-limit): the oracle runs the same limit
        pods, whole = MAX_LIMIT, True
    t0 = time.perf_counter()
    r = oracle.run(snap, tmpl, ctr, max_pods=pods, threads=best)
    dt = time.perf_counter() - t0
    if whole or r.stop_code == abi.STOP_UNSCHEDULABLE:
        pods = 0
    return r, dt, best, cores, pods


def parity_block(got, want, pods):
    """Bit-exact comparison of the GPU result (dict: placed, stop_code, pod_node, reason_hist, preempt_no_victims) with the
    oracle's. pods == 0: the oracle ran to the end -> everything is compared; else the first `pods` placements."""
    gp = np.asarray(got["pod_node"])
    wp = np.asarray(want.pod_node)
    if pods == 0:
        ok = (got["placed"] == want.placed and got["stop_code"] == want.stop_code and np.array_equal(gp, wp)
              and np.array_equal(np.asarray(got["reason_hist"]), want.reason_hist)
              and got["preempt_no_victims"] == want.preempt_no_victims)
        k = int(want.placed)
    else:
        k = int(min(pods, want.placed))
        ok = got["placed"] >= k and np.array_equal(gp[:k], wp[:k])
    first_bad = None
    if not ok:
        m = min(len(gp), len(wp))
        d = np.nonzero(gp[:m] != wp[:m])[0]
        first_bad = int(d[0]) if len(d) else m
    return {"ok": bool(ok), "checked_placements": k, "full_run": pods == 0,
            "compared": "pod->node sequence" + (", placed, stop code, FitError histogram, preemption counts" if pods == 0 else " (prefix)"),
            "against": "oracle/ccsim_oracle.c (canonical mode), same snapshot", "first_mismatch": first_bad}


DUMP_MAX_POD_NODE = 3 << 20    # float64 values + positions of a sampled pod -> node sequence stay under 64 MB in all


def dump_outputs(out_dir, r):
    """Writes a run result (dict: placed, stop_code, pod_node, reason_hist, preempt_no_victims, preempt_not_helpful) as
    <out_dir>/<name>.npy in float64 (exact for these integer outputs). A pod -> node sequence longer than DUMP_MAX_POD_NODE is
    replaced by a fixed seeded sample of its positions, written alongside as pod_node_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    out = {k: np.asarray(r[k], np.float64) for k in ("placed", "stop_code", "reason_hist", "preempt_no_victims", "preempt_not_helpful")}
    pod_node = np.asarray(r["pod_node"], np.float64)
    if len(pod_node) > DUMP_MAX_POD_NODE:
        idx = np.sort(np.random.default_rng(0).choice(len(pod_node), DUMP_MAX_POD_NODE, replace=False))
        pod_node = pod_node[idx]
        out["pod_node_index"] = idx.astype(np.float64)
    out["pod_node"] = pod_node
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def objects_leg(flat, device, steps):
    """e2e through the reference-facing API (include/cchost.h = pkg/framework's New / SyncWithClient / Run / Report): the C4
    cluster as v1.Node / v1.Pod JSON in host memory (what SyncWithClient LISTs, simulator.go:176-295) -> C++ ingest + NodeInfo
    aggregation + encoding -> H2D -> wave kernel -> D2H -> ClusterCapacityReview JSON. Everything inside the timed region;
    the JSON text is built before it. The placement sequence must equal the flat-array run's (same cluster, same node order)."""
    import ctypes as C
    fw = importlib.import_module("cluster-capacity_b200.framework")
    nodes, pods, tmpl = synth.c4_objects()
    nj, pj, tj = json.dumps(nodes).encode(), json.dumps(pods).encode(), json.dumps(tmpl).encode()
    del nodes, pods
    L = fw.lib()
    parts = [0.0, 0.0, 0.0, 0.0]
    wall = []
    same = True
    placed = 0
    for it in range(steps + 1):
        h = C.c_void_p()
        t0 = time.perf_counter()
        rc = L.cc_new(None, tj, 0, b"", device, C.byref(h))
        t1 = time.perf_counter()
        rc = rc or L.cc_sync_with_objects(h, nj, pj, b"[]")
        t2 = time.perf_counter()
        rc = rc or L.cc_run(h)
        t3 = time.perf_counter()
        rep = L.cc_report_json(h) if not rc else None
        t4 = time.perf_counter()
        if rc or rep is None:
            raise RuntimeError("e2e_objects: rc=%s %s" % (rc, L.cc_last_error(h).decode()))
        if it > 0:        # the first iteration warms the allocators / page cache
            wall.append(t4 - t0)
            for q, d in enumerate((t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                parts[q] += d
        placed = int(L.cc_scheduled_count(h))
        if it == steps:   # parity (outside the timed region): count, and every pod's node
            want = flat["pod_node"]
            same = placed == flat["placed"] and all(L.cc_scheduled_node(h, k) == b"node-%06d" % want[k] for k in range(0, placed, 1))
            review = json.loads(rep.decode())
            same = same and review["status"]["replicas"] == placed
        L.cc_close(h)
    evals = (placed + 1) * 100_000
    t = sum(wall)
    return {"value": evals * steps / t, "unit": "evals/s", "ms_per_step": t / steps * 1e3, "steps": steps, "json_bytes_per_step": len(nj) + len(pj) + len(tj),
            "ingest_mb_per_s": (len(nj) + len(pj)) / 1e6 / (parts[1] / steps),
            "breakdown_ms_per_step": {"cc_new": parts[0] / steps * 1e3, "cc_sync_with_objects (JSON -> object model)": parts[1] / steps * 1e3,
                                      "cc_run (NodeInfo aggregation + encode + H2D + wave kernel + D2H)": parts[2] / steps * 1e3,
                                      "cc_report_json": parts[3] / steps * 1e3},
            "same_sequence_as_flat_run": bool(same), "placed": placed}


def latency_block(st, kernel_ms, sm_mhz):
    """What actually bounds the wave kernel: it is latency-bound (dependent instruction issue, L2 round trips of the exchange),
    not bandwidth-bound. Cycle split of CTA 0 from the kernel's own clock64 phase timers (multi-commit engine)."""
    w = max(1, st["waves"])
    out = {"engine": st["engine"], "waves": st["waves"], "us_per_wave": kernel_ms * 1e3 / w, "placements_per_wave": st["placed"] / w,
           "grid": st["grid"], "block": st["block"], "dynamic_smem_bytes": st["smem_bytes"]}
    if st["engine"] == "multi-commit":
        names = ("scan_filter_score_top8", "barrier_wait", "merge_publish", "gather_exchange_compact", "replay", "row_updates")
        cyc = {n: st["phase_cycles"][i] / w for i, n in enumerate(names)}
        out.update({"candidates_replayed_per_wave": st["candidates"] / w, "waves_that_raised_the_bar": st["bar_raised_waves"],
                    "cycles_per_wave_cta0": cyc, "cycles_per_wave_total": sum(cyc.values()),
                    "us_per_wave_from_cycles": (sum(cyc.values()) / (sm_mhz or 1965)) if sm_mhz else None})
    elif st["engine"].startswith("streaming"):
        names = ("scan_mbarrier_wait_filter_argmax", "barriers_prefetch_issue_block_argmax", "exchange_l2_round_trip", "commit_barrier")
        cyc = {n: st["phase_cycles"][i] / w for i, n in enumerate(names)}
        out.update({"stale_memo_rescored_per_wave_cta0": st["candidates"] / w, "cycles_per_wave_cta0": cyc, "cycles_per_wave_total": sum(cyc.values()),
                    "us_per_wave_from_cycles": (sum(cyc.values()) / (sm_mhz or 1965)) if sm_mhz else None})
    return out


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def run_reference(args):
    """--impl reference: the reference's own CPU implementation is Go (no toolchain here), so this arm times the CPU
    oracle port of the same loop with all host threads on a bounded prefix of the same workload. Rank 0 only."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    snap, tmpl, ctr = MAKE(world if args.mode == "sharded" else 1)     # the same workload as our arm at this N
    steps = args.steps
    evals = placed = 0
    dt = 0.0
    threads = cores = pods = 0
    calib = calibrate_oracle(snap, tmpl, ctr)
    for _ in range(steps):   # the whole analysis when it ends within ~30 s on this host, else the first K placements
        r, d, threads, cores, pods = cpu_oracle_rate(snap, tmpl, ctr, budget_s=30.0, calib=calib)
        evals += r.evals
        placed += r.placed
        dt += d
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, vars(r))
    val = evals / dt
    line = {
        "impl": "reference", "metric": "predicate-evals/sec", "value": val, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": 1, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "nodes": snap.n, "sample": ("first %d placements of the run" % pods) if pods else "the whole run (%d placements)" % (placed // steps),
                   "note": "no Go toolchain: the CPU oracle (C port of the reference loop, canonical mode) stands in for the reference"},
        "placements_per_sec": placed / dt,
        "cpu_baseline": {"value": val, "unit": "evals/s", "cores": threads, "kind": "port", "usable_cores": cores,
                         "sample": "%s (%d evals) per step; C port of the reference loop (not the Go reference), OpenMP over the node axis for filter, "
                                   "score and arg-max, thread count calibrated" % (("first %d placements" % pods) if pods else "the whole run", evals // steps),
                         "dram_gbs_algorithmic": val * B_EVAL / 1e9},
        "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def ref_equivalent_evals(res):
    """Predicate-evals as SURVEY.md §8(d) counts them: one per (pod attempt, node) of the reference loop in canonical mode,
    (placed [+1 for the attempt that did not fit]) x nodes of this rank. The sequential engines run exactly that many fused
    Filter evaluations; the multi-commit engine decides several reference cycles per pass over the nodes (res.evals is the
    physical count, reported separately and used for the roofline)."""
    n_local = res.evals // max(1, res.waves)
    return (res.placed + (1 if res.stop_code == abi.STOP_UNSCHEDULABLE else 0)) * n_local


def pinned_snapshot(snap):
    """Copy the snapshot's arrays into pinned host memory (torch) so that the e2e H2D copies are real DMA transfers."""
    import torch
    keep = []

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        keep.append(t)
        return t.numpy()

    s2 = abi.Snapshot(snap.n, pin(snap.alloc_cpu), pin(snap.alloc_mem), pin(snap.alloc_pods), alloc_eph=pin(snap.alloc_eph),
                      req_cpu=pin(snap.req_cpu), req_mem=pin(snap.req_mem), req_eph=pin(snap.req_eph), npods=pin(snap.npods),
                      nz_cpu=pin(snap.nz_cpu), nz_mem=pin(snap.nz_mem), taint_mask=pin(snap.taint_mask),
                      taint_nosched=snap.taint_nosched, taint_prefer=snap.taint_prefer,
                      static_mask=pin(snap.static_mask) if snap.static_words else None, topo=[pin(t) for t in snap.topo])
    s2._pins = keep
    nbytes = sum(t.numel() * t.element_size() for t in keep)
    return s2, nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-parity", "--no-cpu-baseline", dest="no_parity", action="store_true",
                    help="skip the oracle run (parity check of the timed configuration + cpu_baseline)")
    ap.add_argument("--no-objects", action="store_true", help="skip the e2e_objects leg (plugin call from Node/Pod JSON)")
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS), help="c4 (default: the metric's 100k-node configuration) or c5 (1M nodes x 64 podspecs)")
    ap.add_argument("--mode", default="sharded", choices=["sharded", "replicas"], help="N>1: node-sharded run or independent replicas")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    select_workload(args.workload)
    if args.impl == "reference":
        return run_reference(args)

    rank, world, local = dist_env()
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    engine = importlib.import_module("cluster-capacity_b200.engine")

    sharded_run = world > 1 and args.mode == "sharded"
    sharded = importlib.import_module("cluster-capacity_b200.sharded")
    # C4: weak scaling (world x 100k nodes, hierarchy kept: racks scale with the node count); C5: the 1M-node cluster is split
    snap, tmpl, ctr = MAKE(world if sharded_run else 1)
    psnap, h2d_bytes = pinned_snapshot(snap)
    ctr_bytes = sum(c.n_domains * 4 for c in ctr)
    warm = max(3, args.warmup)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = engine.Engine(device=local, rank=rank if sharded_run else 0, world=world if sharded_run else 1)
    eng.load_nodes(psnap)
    eng.set_templates(tmpl, ctr)
    if sharded_run:
        eng.connect_peers(dist)
        lo_, hi_ = sharded.shard_bounds(snap.n, world, rank)
        h2d_bytes = int(h2d_bytes * (hi_ - lo_) / snap.n)
    for _ in range(warm):
        res = eng.run(MAX_LIMIT)
    sampler = ClockSampler(local)
    sampler.start()
    # ---- resident-input arm: K steps, L2 flushed (untimed) between steps, each step bracketed by a synchronize ----
    launches0 = eng.kernel_launches()
    step_wall = []
    kernel_ms = 0.0
    evals = placed = waves = ref_evals = 0
    barrier()
    for _ in range(args.steps):
        eng.flush_l2()
        torch.cuda.synchronize()
        if sharded_run:
            dist.barrier()
        t0 = time.perf_counter()
        res = eng.run(MAX_LIMIT)
        torch.cuda.synchronize()
        step_wall.append(time.perf_counter() - t0)
        kernel_ms += res.run_ms
        evals += res.evals            # physical: fused Filter passes the kernel ran x nodes of this rank
        placed += res.placed
        waves += res.waves
        ref_evals += ref_equivalent_evals(res)
    stats = eng.run_stats()            # latency anatomy of the last timed run (CTA 0's clock cycles per phase, candidates, ...)
    barrier()
    # the result the parity check compares (sharded: per-shard histograms summed, replicated parts cross-checked between ranks)
    if sharded_run:
        last_result = sharded.merge_results(dist, res)
    else:
        last_result = {"placed": res.placed, "stop_code": res.stop_code, "pod_node": res.pod_node, "reason_hist": res.reason_hist,
                       "preempt_no_victims": res.preempt_no_victims, "preempt_not_helpful": res.preempt_not_helpful}
    flushes = args.steps
    launches = eng.kernel_launches() - launches0 - flushes
    t_total = sum(step_wall)
    # ---- end-to-end arm: host buffers -> C-ABI -> results on the host, everything inside the timed region ----
    e2e_wall = []
    e2e_parts = [0.0, 0.0, 0.0]
    e2e_evals = 0
    d2h = 0
    for it in range(args.steps + 1):
        torch.cuda.synchronize()
        if sharded_run:
            dist.barrier()
        t0 = time.perf_counter()
        eng.load_nodes(psnap)          # H2D of every column of this rank's shard (pinned source)
        ta = time.perf_counter()
        eng.set_templates(tmpl, ctr)   # H2D of the template table + per-domain counters
        tb = time.perf_counter()
        r2 = eng.run(MAX_LIMIT)                # run + D2H of pod->node, histogram, counters
        torch.cuda.synchronize()
        if it > 0:                     # first iteration warms the allocator
            e2e_wall.append(time.perf_counter() - t0)
            e2e_parts[0] += ta - t0; e2e_parts[1] += tb - ta; e2e_parts[2] += time.perf_counter() - tb
            e2e_evals += ref_equivalent_evals(r2)
            d2h = r2.placed * 4 + abi.C.sizeof(abi.Result)
    barrier()
    sampler.stop_flag.set()
    sampler.join(timeout=2)

    # max over ranks of the timed regions, sum of the work
    vals = torch.tensor([t_total, sum(e2e_wall), kernel_ms], dtype=torch.float64, device="cuda")
    work = torch.tensor([float(ref_evals), float(placed), float(e2e_evals), float(evals)], dtype=torch.float64, device="cuda")
    if sharded_run:
        work[1] = work[1] / world      # placements are replicated on every rank of a sharded run; evals are per shard
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(work, op=dist.ReduceOp.SUM)
    t_total, t_e2e, kernel_ms_max = [float(x) for x in vals.tolist()]
    evals_all, placed_all, e2e_evals_all, phys_all = [float(x) for x in work.tolist()]

    parity_ok = True
    if rank == 0:
        peak, peak_kind = measured_peak()
        # SURVEY.md §8(d): algorithmic bytes of a canonical run = (placed+1) x N x B_eval — every pod attempt streams every node row
        # once. `achieved` follows that definition; `achieved_physical` counts the passes the kernel really made over its tile.
        achieved = (ref_evals * B_EVAL) / (kernel_ms * 1e-3) / 1e9       # this rank's kernel (its shard)
        achieved_phys = (evals * B_EVAL) / (kernel_ms * 1e-3) / 1e9
        line = {
            "metric": "predicate-evals/sec", "value": evals_all / t_total, "unit": "evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": t_total / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak" if WKEY == "c4" else "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "nodes": snap.n, "templates": len(tmpl), "max_limit": MAX_LIMIT, "mode": "canonical (percentageOfNodesToScore=100)",
                       "parallelism": ("node-sharded x%d (in-kernel peer-memory exchange per wave)" % world if sharded_run else "replicas x%d" % world) if world > 1 else "single GPU",
                       "l2": "flushed between timed steps (2x L2 write, untimed)",
                       "bytes_per_eval_algorithmic": B_EVAL, "placed_per_step": int(placed / args.steps),
                       "waves_per_step": int(waves / args.steps),
                       "evals": "reference-equivalent: (placed+1) x nodes per step (SURVEY.md §8d), the count the CPU arm executes"},
            "placements_per_sec": placed_all / t_total,
            "physical_evals_per_sec": phys_all / t_total,
            "kernel_ms_per_step": kernel_ms / args.steps,
            "e2e": {"value": e2e_evals_all / t_e2e, "unit": "evals/s", "h2d_bytes_per_step": int(h2d_bytes + ctr_bytes + len(tmpl) * abi.C.sizeof(abi.Template)),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": t_e2e / args.steps * 1e3,
                    "breakdown_ms_per_step": {"ccsim_load_nodes": e2e_parts[0] / args.steps * 1e3, "ccsim_set_templates": e2e_parts[1] / args.steps * 1e3,
                                              "ccsim_run": e2e_parts[2] / args.steps * 1e3}},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": profiled_traffic() if world == 1 else None, "peak_kind": peak_kind,
                         "algorithmic_bytes_per_launch": ref_evals * B_EVAL / args.steps,
                         "achieved_physical": achieved_phys, "frac_physical": achieved_phys / peak,
                         "physical_bytes_per_launch": evals * B_EVAL / args.steps,
                         "latency": latency_block(stats, kernel_ms / args.steps, sampler.summary().get("sm_mhz")),
                         "note": "bound: the wave kernel is LATENCY-bound (see `latency`): `frac` is the SURVEY.md §8d figure — algorithmic bytes = "
                                 "(placed+1) x N x %d B (every pod attempt of the reference loop streams every node row) over the wave kernel's CUDA-event "
                                 "time vs the measured HBM copy peak — and may exceed 1: the multi-commit engine decides ~placed/waves reference cycles per "
                                 "pass over the (shared-memory resident) node tile and the streaming engine reads 24 B of the 72 B row; achieved_physical "
                                 "counts one row per node and PASS actually made; `traffic` is ncu's dram bytes per launch (profiles/)" % B_EVAL},
        }
        # ---- parity on the timed configuration (and the CPU baseline: the same oracle run serves both) ----
        # N=1: the oracle runs the WHOLE analysis of the timed snapshot when that fits ~40 s (C4: ~18 s on 16 threads) and
        # everything is compared; N>1 (weak-scaled clusters): the first K placements within the budget are compared.
        line["cpu_baseline"] = None
        if not args.no_parity:
            rc, dtc, threads, cores, pods = cpu_oracle_rate(snap, tmpl, ctr, budget_s=40.0 if world == 1 else 25.0)
            line["parity"] = parity_block(last_result, rc, pods)
            parity_ok = line["parity"]["ok"]
            if world == 1:
                line["cpu_baseline"] = {"value": rc.evals / dtc, "unit": "evals/s", "cores": threads, "kind": "port", "usable_cores": cores,
                                        "sample": "%s of the same snapshot (%d evals, %.1f s); C port of the reference loop (not the Go reference), "
                                                  "OpenMP over the node axis for filter, score and arg-max, thread count calibrated"
                                                  % ("the whole run" if pods == 0 else "first %d placements" % pods, rc.evals, dtc),
                                        "dram_gbs_algorithmic": rc.evals / dtc * B_EVAL / 1e9}
        else:
            line["parity"] = None
        # ---- the reference-facing plugin call: framework.New + SyncWithClient + Run + Report from Node / Pod JSON in host memory ----
        if WKEY == "c4" and world == 1 and not args.no_objects:
            line["e2e_objects"] = objects_leg(last_result, local, args.steps)
            parity_ok = parity_ok and line["e2e_objects"]["same_sequence_as_flat_run"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_result)
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and not parity_ok:
        sys.stderr.write("bench.py: PARITY MISMATCH against the oracle on the timed configuration\n")
        sys.exit(3)


if __name__ == "__main__":
    main()
