"""ctypes binding of libccsim.so — the CUDA hot path behind include/ccsim.h.

There is NO CPU fallback: if the shared object is missing, or no CUDA device is visible, every entry point raises.
(The CPU oracle under oracle/ is test infrastructure and is never imported from here.)
"""
import ctypes as C
import os

import numpy as np

from . import _abi as abi

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("CCSIM_SO") or os.path.join(_HERE, "libccsim.so")   # CCSIM_SO: kernel-variant experiments only
_lib = None

EXPORTS = ["ccsim_create", "ccsim_destroy", "ccsim_last_error", "ccsim_abi_version", "ccsim_load_nodes",
           "ccsim_set_templates", "ccsim_run", "ccsim_prepare", "ccsim_node_counts", "ccsim_peer_export", "ccsim_peer_import",
           "ccsim_device_info", "ccsim_kernel_launches", "ccsim_flush_l2", "ccsim_run_stats", "ccsim_peer_local", "ccsim_peer_import_local",
           "ccsim_debug_node_scores"]


class EngineError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise EngineError("libccsim.so not built (%s): run __graft_entry__.build(); there is no CPU fallback" % SO_PATH)
        L = C.CDLL(SO_PATH)
        L.ccsim_create.restype = C.c_int
        L.ccsim_create.argtypes = [C.POINTER(abi.Config), C.POINTER(C.c_void_p)]
        L.ccsim_destroy.restype = None
        L.ccsim_destroy.argtypes = [C.c_void_p]
        L.ccsim_last_error.restype = C.c_char_p
        L.ccsim_last_error.argtypes = [C.c_void_p]
        L.ccsim_abi_version.restype = C.c_int
        L.ccsim_load_nodes.restype = C.c_int
        L.ccsim_load_nodes.argtypes = [C.c_void_p, C.POINTER(abi.Nodes)]
        L.ccsim_set_templates.restype = C.c_int
        L.ccsim_set_templates.argtypes = [C.c_void_p, C.c_int32, C.POINTER(abi.Template), C.c_int32, C.POINTER(abi.Counter)]
        L.ccsim_prepare.restype = C.c_int
        L.ccsim_prepare.argtypes = [C.c_void_p, C.c_int64]
        L.ccsim_run.restype = C.c_int
        L.ccsim_run.argtypes = [C.c_void_p, C.c_int64, C.POINTER(abi.Result)]
        L.ccsim_node_counts.restype = C.c_int
        L.ccsim_node_counts.argtypes = [C.c_void_p, C.c_int32, abi.P32, abi.P64]
        L.ccsim_device_info.restype = C.c_int
        L.ccsim_device_info.argtypes = [C.c_void_p, abi.P32, abi.P32, abi.P32, abi.P64]
        L.ccsim_kernel_launches.restype = C.c_int64
        L.ccsim_kernel_launches.argtypes = [C.c_void_p]
        L.ccsim_flush_l2.restype = C.c_int
        L.ccsim_flush_l2.argtypes = [C.c_void_p]
        L.ccsim_peer_local.restype = C.c_int
        L.ccsim_peer_local.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.ccsim_peer_import_local.restype = C.c_int
        L.ccsim_peer_import_local.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]
        L.ccsim_run_stats.restype = C.c_int
        L.ccsim_run_stats.argtypes = [C.c_void_p, abi.P64]
        L.ccsim_debug_node_scores.restype = C.c_int
        L.ccsim_debug_node_scores.argtypes = [C.c_void_p, C.c_int32, C.c_int32, abi.P64, abi.P64, abi.P64]
        L.ccsim_peer_export.restype = C.c_int
        L.ccsim_peer_export.argtypes = [C.c_void_p, abi.PU8]
        L.ccsim_peer_import.restype = C.c_int
        L.ccsim_peer_import.argtypes = [C.c_void_p, C.c_int32, abi.PU8]
        _lib = L
    return _lib


class RunResult:
    def __init__(self, res):
        self.placed = int(res.placed)
        self.stop_code = int(res.stop_code)
        self.n_nodes = int(res.n_nodes)
        self.waves = int(res.waves)
        self.evals = int(res.evals)
        self.examined = int(res.examined)
        self.run_ms = float(res.run_ms)
        self.reason_hist = np.array(res.reason_hist[:], dtype=np.int64)
        self.preempt_no_victims = int(res.preempt_no_victims)
        self.preempt_not_helpful = int(res.preempt_not_helpful)
        if self.placed:
            self.pod_node = np.ctypeslib.as_array(res.pod_node, shape=(self.placed,)).copy()
        else:
            self.pod_node = np.zeros(0, np.int32)


class Engine:
    """One ccsim handle (one GPU / one node-axis shard)."""

    def __init__(self, device=0, engine=abi.ENGINE_AUTO, rank=0, world=1, sampling=abi.SAMPLING_CANONICAL, pct_nodes_to_score=0):
        cfg = abi.Config()
        cfg.abi_version = abi.ABI_VERSION
        cfg.device, cfg.engine, cfg.rank, cfg.world = device, engine, rank, world
        cfg.sampling, cfg.pct_nodes_to_score = sampling, pct_nodes_to_score
        self._h = C.c_void_p()
        rc = lib().ccsim_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise EngineError("ccsim_create rc=%d: %s" % (rc, lib().ccsim_last_error(None).decode()))
        self._keep = None

    def _check(self, rc, what):
        if rc != 0:
            raise EngineError("%s rc=%d: %s" % (what, rc, lib().ccsim_last_error(self._h).decode()))

    def load_nodes(self, snapshot):
        nd = snapshot.c_struct()
        self._check(lib().ccsim_load_nodes(self._h, C.byref(nd)), "ccsim_load_nodes")
        self._n = snapshot.n

    def set_templates(self, templates, counters=()):
        T = (abi.Template * len(templates))(*templates)
        Cn = (abi.Counter * max(1, len(counters)))(*counters)
        self._check(lib().ccsim_set_templates(self._h, len(templates), T, len(counters), Cn), "ccsim_set_templates")

    def prepare(self, max_pods=0):
        """The allocation / restore half of run(max_pods); see ccsim_prepare."""
        self._check(lib().ccsim_prepare(self._h, max_pods), "ccsim_prepare")

    def run(self, max_pods=0):
        res = abi.Result()
        self._check(lib().ccsim_run(self._h, max_pods, C.byref(res)), "ccsim_run")
        return RunResult(res)

    def connect_peers(self, dist):
        """Node-sharded multi-GPU run: all-gather the CUDA IPC handles of the exchange buffers over torch.distributed
        and map every peer's buffer (the per-wave exchange itself then happens inside the persistent kernel)."""
        import torch
        mine = np.zeros(64, np.uint8)
        self._check(lib().ccsim_peer_export(self._h, mine.ctypes.data_as(abi.PU8)), "ccsim_peer_export")
        world = dist.get_world_size()
        dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
        t = torch.from_numpy(mine).to(dev)
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        allh = np.concatenate([o.cpu().numpy() for o in out]).astype(np.uint8)
        self._check(lib().ccsim_peer_import(self._h, world, allh.ctypes.data_as(abi.PU8)), "ccsim_peer_import")

    @staticmethod
    def connect_local(engines):
        """All ranks live in this process (rank r = engines[r]): hand every engine the others' exchange-buffer pointers. The
        runs must then be started concurrently (one host thread per rank): the persistent kernels talk to each other."""
        ptrs = (C.c_void_p * len(engines))()
        for r, e in enumerate(engines):
            p = C.c_void_p()
            e._check(lib().ccsim_peer_local(e._h, C.byref(p)), "ccsim_peer_local")
            ptrs[r] = p
        for e in engines:
            e._check(lib().ccsim_peer_import_local(e._h, len(engines), ptrs), "ccsim_peer_import_local")

    def node_counts(self, t=0):
        counts = np.zeros(max(1, self._n), np.int32)
        first = np.zeros(max(1, self._n), np.int64)
        self._check(lib().ccsim_node_counts(self._h, t, counts.ctypes.data_as(abi.P32), first.ctypes.data_as(abi.P64)),
                    "ccsim_node_counts")
        return counts[: self._n], first[: self._n]

    def device_info(self):
        sm, grid, block, l2 = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        lib().ccsim_device_info(self._h, C.byref(sm), C.byref(grid), C.byref(block), C.byref(l2))
        return dict(sm_count=sm.value, grid=grid.value, block=block.value, l2_bytes=l2.value)

    ENGINE_NAMES = ("generic", "lean sequential", "tie-run batching", "multi-commit", "streaming (TMA)")

    @staticmethod
    def kernel_name(code):
        """The wave kernel instantiation behind ccsim_run_stats out[0]: generic/resident, generic/streamed, lean/canonical,
        lean/reference, batched, multi/1gpu, multi/shards, stream/mode0, stream/mode1 or stream/mode2."""
        engine = code & abi.KV_ENGINE_MASK
        if engine == 0:
            return "generic/resident" if code & abi.KV_RESIDENT else "generic/streamed"
        if engine == 1:
            return "lean/reference" if code & abi.KV_REFERENCE_SAMPLING else "lean/canonical"
        if engine == 2:
            return "batched"
        if engine == 3:
            return "multi/shards" if code & abi.KV_CROSS_GPU else "multi/1gpu"
        return "stream/mode%d" % ((code >> abi.KV_STREAM_MODE_SHIFT) & 3)

    def run_stats(self):
        """Latency anatomy of the last run (see ccsim_run_stats in include/ccsim.h). "replay_rounds" was called "smem_bytes" (the
        slot once held the shared-memory size); the old key stays for existing readers."""
        v = np.zeros(16, np.int64)
        self._check(lib().ccsim_run_stats(self._h, v.ctypes.data_as(abi.P64)), "ccsim_run_stats")
        code = int(v[0])
        return {"engine": self.ENGINE_NAMES[code & abi.KV_ENGINE_MASK], "kernel": self.kernel_name(code), "waves": int(v[1]), "placed": int(v[2]),
                "candidates": int(v[3]), "bar_raised_waves": int(v[4]), "grid": int(v[5]), "block": int(v[6]),
                "replay_rounds": int(v[7]), "smem_bytes": int(v[7]), "phase_cycles": [int(x) for x in v[8:16]]}

    def debug_node_scores(self, t, clones=0):
        """Device scores of every node for template t after `clones` commits of it (see ccsim_debug_node_scores):
        (total, least, balanced) int64 arrays of this handle's nodes."""
        n = max(1, self._n)
        total, least, balanced = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int64)
        self._check(lib().ccsim_debug_node_scores(self._h, t, clones, total.ctypes.data_as(abi.P64), least.ctypes.data_as(abi.P64),
                                                  balanced.ctypes.data_as(abi.P64)), "ccsim_debug_node_scores")
        return total[: self._n], least[: self._n], balanced[: self._n]

    def kernel_launches(self):
        return int(lib().ccsim_kernel_launches(self._h))

    def flush_l2(self):
        self._check(lib().ccsim_flush_l2(self._h), "ccsim_flush_l2")

    def close(self):
        if self._h:
            lib().ccsim_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
