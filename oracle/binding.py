"""ctypes binding of the CPU oracle (oracle/ccsim_oracle.c). TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs — never from the
product package. The shared object is built by `make -C oracle` (also done by __graft_entry__.build()).
"""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np

_abi = importlib.import_module("cluster-capacity_b200._abi")
_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libccsim_oracle.so")
_lib = None


def build(force=False):
    src = os.path.join(_HERE, "ccsim_oracle.c")
    hdr = os.path.join(_HERE, "..", "include", "ccsim.h")
    if os.environ.get("CCSIM_NO_REBUILD") and os.path.exists(_SO) and not force:
        return _SO
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.ccsim_oracle_run.restype = C.c_int
        _lib.ccsim_oracle_run.argtypes = [C.POINTER(_abi.Nodes), C.c_int32, C.POINTER(_abi.Template), C.c_int32,
                                          C.POINTER(_abi.Counter), C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                          C.POINTER(_abi.Result), _abi.P32, C.c_int64]
        _lib.ccsim_oracle_run_ex.restype = C.c_int
        _lib.ccsim_oracle_run_ex.argtypes = [C.POINTER(_abi.Nodes), C.c_int32, C.POINTER(_abi.Template), C.c_int32,
                                             C.POINTER(_abi.Counter), C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                             C.POINTER(_abi.Result), _abi.P32, C.c_int64]
        _lib.ccsim_oracle_node_score.restype = C.c_int64
        _lib.ccsim_oracle_node_score.argtypes = [C.POINTER(_abi.Nodes), C.POINTER(_abi.Template), C.c_int32, C.c_int32,
                                                 _abi.P64, _abi.P64]
    return _lib


class OracleResult:
    def __init__(self, res, pod_node):
        self.placed = int(res.placed)
        self.stop_code = int(res.stop_code)
        self.waves = int(res.waves)
        self.evals = int(res.evals)
        self.examined = int(res.examined)
        self.reason_hist = np.array(res.reason_hist[:], dtype=np.int64)
        self.preempt_no_victims = int(res.preempt_no_victims)
        self.preempt_not_helpful = int(res.preempt_not_helpful)
        self.pod_node = pod_node[: self.placed].copy()


def run(snapshot, templates, counters=(), max_pods=0, mode=0, pct=0, threads=1, cap=None, memo=False):
    """Run the oracle loop. mode 0 = canonical, 1 = faithful (adaptive sampling + rotation). memo=True memoises the node-local
    score per (template, node) until that node is committed (identical results, for full-size parity runs; never for timing)."""
    nd = snapshot.c_struct()
    T = (_abi.Template * len(templates))(*templates)
    Cn = (_abi.Counter * max(1, len(counters)))(*counters)
    if cap is None:
        cap = max_pods if max_pods > 0 else int(snapshot.alloc_pods.astype(np.int64).sum()) + 1
    buf = np.zeros(max(1, cap), np.int32)
    res = _abi.Result()
    rc = lib().ccsim_oracle_run_ex(C.byref(nd), len(templates), T, len(counters), Cn, max_pods, mode, pct, threads, 1 if memo else 0,
                                   C.byref(res), buf.ctypes.data_as(_abi.P32), cap)
    if rc != 0:
        raise RuntimeError("oracle rc=%d" % rc)
    return OracleResult(res, buf)


def node_score(snapshot, template, i, clones):
    nd = snapshot.c_struct()
    l, b = C.c_int64(), C.c_int64()
    tot = lib().ccsim_oracle_node_score(C.byref(nd), C.byref(template), i, clones, C.byref(l), C.byref(b))
    return int(tot), int(l.value), int(b.value)


def node_scores(snapshot, template, clones):
    """node_score of every node: (total, least, balanced) int64 arrays."""
    nd = snapshot.c_struct()
    f = lib().ccsim_oracle_node_score
    l, b = C.c_int64(), C.c_int64()
    out = np.zeros((3, snapshot.n), np.int64)
    for i in range(snapshot.n):
        out[0, i] = f(C.byref(nd), C.byref(template), i, clones, C.byref(l), C.byref(b))
        out[1, i], out[2, i] = l.value, b.value
    return out[0], out[1], out[2]
