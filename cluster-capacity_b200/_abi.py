"""ctypes mirror of include/ccsim.h (the C-ABI of the hot path).

Only plain data: the same structs are handed to libccsim.so (product, CUDA) and — from tests/bench only — to the
CPU oracle. Field order and limits must match include/ccsim.h exactly; tests/test_abi.py checks sizeof().
"""
import ctypes as C
import numpy as np

ABI_VERSION = 3
MAX_TAINT_WORDS = 4
MAX_STATIC_WORDS = 4
MAX_SCALARS = 4
MAX_AFF_TERMS = 8
MAX_PTS = 8
MAX_IPA = 8
MAX_TOPO_COLS = 16
MAX_COUNTERS = 24
MAX_TEMPLATES = 64
MAX_CLASSES = 8
TAINT_UNSCHEDULABLE_BIT = 63

OK, EINVAL, ENOMEM, ECUDA, EUNSUPPORTED, ESTATE, ENCCL = 0, -1, -2, -3, -4, -5, -6

TF_TOLERATES_UNSCHEDULABLE = 1 << 0
TF_HAS_NODE_SELECTOR = 1 << 1
TF_HAS_AFFINITY_TERMS = 1 << 2
TF_HAS_HOST_PORTS = 1 << 3
TF_FIT_ALL_ZERO = 1 << 4
TF_BALANCED_SKIP = 1 << 5
TF_AFF_SELF_MATCH_ALL = 1 << 6
TF_PREFILTER_NODES = 1 << 7

PL_NODE_UNSCHEDULABLE = 1 << 0
PL_NODE_NAME = 1 << 1
PL_TAINT_TOLERATION = 1 << 2
PL_NODE_AFFINITY = 1 << 3
PL_NODE_PORTS = 1 << 4
PL_FIT = 1 << 5
PL_POD_TOPOLOGY_SPREAD = 1 << 6
PL_INTER_POD_AFFINITY = 1 << 7
PL_BALANCED = 1 << 8
PL_IMAGE_LOCALITY = 1 << 9
PL_ALL = 0x3FF

(R_UNSCHEDULABLE, R_NODE_NAME, R_NODE_AFFINITY, R_NODE_PORTS, R_TOO_MANY_PODS, R_INSUFFICIENT_CPU,
 R_INSUFFICIENT_MEMORY, R_INSUFFICIENT_EPHEMERAL, R_PTS_MISSING_LABEL, R_PTS_SKEW, R_IPA_AFFINITY,
 R_IPA_ANTI_AFFINITY, R_IPA_EXISTING_ANTI, R_PREFILTER_NODES, R_FIXED_COUNT) = range(15)
R_SCALAR0 = R_FIXED_COUNT
R_TAINT0 = R_SCALAR0 + MAX_SCALARS
R_TOTAL = R_TAINT0 + 64 * MAX_TAINT_WORDS

# reason strings, in the reference's own words (files cited in include/ccsim.h)
REASON_TEXT = {
    R_UNSCHEDULABLE: "node(s) were unschedulable",
    R_NODE_NAME: "node(s) didn't match the requested node name",
    R_NODE_AFFINITY: "node(s) didn't match Pod's node affinity/selector",
    R_NODE_PORTS: "node(s) didn't have free ports for the requested pod ports",
    R_TOO_MANY_PODS: "Too many pods",
    R_INSUFFICIENT_CPU: "Insufficient cpu",
    R_INSUFFICIENT_MEMORY: "Insufficient memory",
    R_INSUFFICIENT_EPHEMERAL: "Insufficient ephemeral-storage",
    R_PTS_MISSING_LABEL: "node(s) didn't match pod topology spread constraints (missing required label)",
    R_PTS_SKEW: "node(s) didn't match pod topology spread constraints",
    R_IPA_AFFINITY: "node(s) didn't match pod affinity rules",
    R_IPA_ANTI_AFFINITY: "node(s) didn't match pod anti-affinity rules",
    R_IPA_EXISTING_ANTI: "node(s) didn't satisfy existing pods anti-affinity rules",
    R_PREFILTER_NODES: "node(s) didn't satisfy plugin(s) [NodeAffinity]",
}

STOP_UNSCHEDULABLE, STOP_LIMIT_REACHED = 0, 1
ENGINE_AUTO, ENGINE_SEQUENTIAL, ENGINE_BATCHED = 0, 1, 2
SAMPLING_CANONICAL, SAMPLING_REFERENCE = 0, 1
# ccsim_run_stats out[0]: engine code in the low byte, the wave kernel's instantiation above it
KV_ENGINE_MASK = 0xFF
KV_RESIDENT = 1 << 8
KV_STREAM_MODE_SHIFT = 9
KV_REFERENCE_SAMPLING = 1 << 11
KV_CROSS_GPU = 1 << 12

P64 = C.POINTER(C.c_int64)
P32 = C.POINTER(C.c_int32)
PU64 = C.POINTER(C.c_uint64)
PU8 = C.POINTER(C.c_uint8)


class Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("engine", C.c_int32),
                ("rank", C.c_int32), ("world", C.c_int32), ("sampling", C.c_int32), ("pct_nodes_to_score", C.c_int32),
                ("reserved", C.c_int32 * 1)]


class Nodes(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_int32), ("n_scalars", C.c_int32), ("taint_words", C.c_int32),
        ("static_words", C.c_int32), ("n_topo_cols", C.c_int32), ("has_placed_mask", C.c_int32),
        ("alloc_cpu", P64), ("alloc_mem", P64), ("alloc_eph", P64), ("alloc_pods", P32),
        ("req_cpu", P64), ("req_mem", P64), ("req_eph", P64), ("npods", P32),
        ("nz_cpu", P64), ("nz_mem", P64),
        ("alloc_scalar", P64 * MAX_SCALARS), ("req_scalar", P64 * MAX_SCALARS),
        ("taint_mask", PU64), ("static_mask", PU64),
        ("topo", P32 * MAX_TOPO_COLS),
        ("taint_nosched", C.c_uint64 * MAX_TAINT_WORDS), ("taint_prefer", C.c_uint64 * MAX_TAINT_WORDS),
        ("taint_list_off", P32), ("taint_list", PU8),
    ]


class Counter(C.Structure):
    _fields_ = [("topo_col", C.c_int32), ("n_domains", C.c_int32), ("n_present", C.c_int32),
                ("inc", C.c_int32), ("elig_bit", C.c_int32), ("pad", C.c_int32), ("init", P32)]


class Pts(C.Structure):
    _fields_ = [("counter", C.c_int32), ("max_skew", C.c_int32), ("self_match", C.c_int32),
                ("min_zero", C.c_int32)]


class Spts(C.Structure):
    _fields_ = [("counter", C.c_int32), ("max_skew", C.c_int32), ("hostname", C.c_int32),
                ("has_key_bit", C.c_int32)]


class Template(C.Structure):
    _fields_ = [
        ("req_cpu", C.c_int64), ("req_mem", C.c_int64), ("req_eph", C.c_int64),
        ("req_scalar", C.c_int64 * MAX_SCALARS),
        ("nz_cpu", C.c_int64), ("nz_mem", C.c_int64),
        ("least_cpu", C.c_int64), ("least_mem", C.c_int64),
        ("bal_cpu", C.c_int64), ("bal_mem", C.c_int64),
        ("flags", C.c_uint32), ("filter_enable", C.c_uint32), ("score_enable", C.c_uint32),
        ("nodename_idx", C.c_int32),
        ("w_taint", C.c_int32), ("w_node_affinity", C.c_int32), ("w_fit", C.c_int32), ("w_pts", C.c_int32),
        ("w_ipa", C.c_int32), ("w_balanced", C.c_int32), ("w_image", C.c_int32),
        ("least_w_cpu", C.c_int32), ("least_w_mem", C.c_int32),
        ("tol_nosched", C.c_uint64 * MAX_TAINT_WORDS), ("tol_prefer", C.c_uint64 * MAX_TAINT_WORDS),
        ("sel_mask", C.c_uint64 * MAX_STATIC_WORDS),
        ("n_aff_terms", C.c_int32), ("prefilter_bit", C.c_int32),
        ("aff_term_mask", (C.c_uint64 * MAX_STATIC_WORDS) * MAX_AFF_TERMS),
        ("port_static_mask", C.c_uint64 * MAX_STATIC_WORDS), ("port_tmpl_conflict", C.c_uint64),
        ("existing_anti_mask", C.c_uint64 * MAX_STATIC_WORDS),
        ("n_pts", C.c_int32), ("pts", Pts * MAX_PTS),
        ("n_aff", C.c_int32), ("aff_counter", C.c_int32 * MAX_IPA),
        ("n_anti", C.c_int32), ("anti_counter", C.c_int32 * MAX_IPA),
        ("aff_total_init", C.c_int64),
        ("n_pref_terms", C.c_int32), ("pref_weight", C.c_int32 * MAX_AFF_TERMS), ("pad_pref", C.c_int32),
        ("pref_mask", (C.c_uint64 * MAX_STATIC_WORDS) * MAX_AFF_TERMS),
        ("n_spts", C.c_int32), ("spts_ignored_bit", C.c_int32), ("spts", Spts * MAX_PTS),
        ("n_ipa_score", C.c_int32), ("ipa_score_counter", C.c_int32 * MAX_IPA), ("pad_soft", C.c_int32),
        ("image_score", C.POINTER(C.c_uint8)),
    ]


class Result(C.Structure):
    _fields_ = [
        ("placed", C.c_int64), ("stop_code", C.c_int32), ("n_nodes", C.c_int32),
        ("waves", C.c_int64), ("evals", C.c_int64), ("examined", C.c_int64),
        ("reason_hist", C.c_int64 * R_TOTAL),
        ("preempt_no_victims", C.c_int64), ("preempt_not_helpful", C.c_int64),
        ("run_ms", C.c_double), ("pod_node", P32),
    ]


def _ptr(a, ty):
    return a.ctypes.data_as(ty) if a is not None else ty()


class Snapshot:
    """Numpy-backed flat snapshot (A1 of SURVEY.md §8a): keeps the arrays alive and builds the ccsim_nodes view."""

    def __init__(self, n, alloc_cpu, alloc_mem, alloc_pods, alloc_eph=None, req_cpu=None, req_mem=None, req_eph=None,
                 npods=None, nz_cpu=None, nz_mem=None, scalars=(), taint_mask=None, taint_nosched=(), taint_prefer=(),
                 static_mask=None, topo=(), has_placed_mask=False, taint_lists=None, names=None):
        i64 = lambda a: np.ascontiguousarray(np.zeros(n, np.int64) if a is None else a, dtype=np.int64)
        i32 = lambda a: np.ascontiguousarray(np.zeros(n, np.int32) if a is None else a, dtype=np.int32)
        self.n = int(n)
        self.alloc_cpu, self.alloc_mem, self.alloc_eph = i64(alloc_cpu), i64(alloc_mem), i64(alloc_eph)
        self.alloc_pods = i32(alloc_pods)
        self.req_cpu, self.req_mem, self.req_eph = i64(req_cpu), i64(req_mem), i64(req_eph)
        self.npods = i32(npods)
        self.nz_cpu = i64(self.req_cpu if nz_cpu is None else nz_cpu)
        self.nz_mem = i64(self.req_mem if nz_mem is None else nz_mem)
        self.scalars = [(i64(a), i64(r)) for a, r in scalars]
        if taint_mask is None:
            taint_mask = np.zeros((1, n), np.uint64)
        self.taint_mask = np.ascontiguousarray(taint_mask, dtype=np.uint64).reshape(-1, n) if n else np.zeros((1, 0), np.uint64)
        self.taint_words = self.taint_mask.shape[0]
        self.taint_nosched = list(taint_nosched) + [0] * (MAX_TAINT_WORDS - len(taint_nosched))
        self.taint_prefer = list(taint_prefer) + [0] * (MAX_TAINT_WORDS - len(taint_prefer))
        if static_mask is None:
            self.static_mask = np.zeros((0, n), np.uint64)
        else:
            self.static_mask = np.ascontiguousarray(static_mask, dtype=np.uint64).reshape(-1, n)
        self.static_words = self.static_mask.shape[0]
        self.topo = [i32(t) for t in topo]
        self.has_placed_mask = bool(has_placed_mask)
        self.names = names
        if taint_lists is not None:
            off = np.zeros(n + 1, np.int32)
            flat = []
            for i, l in enumerate(taint_lists):
                flat.extend(l)
                off[i + 1] = len(flat)
            self.taint_list_off = off
            self.taint_list = np.asarray(flat if flat else [0], dtype=np.uint8)
        else:
            self.taint_list_off = None
            self.taint_list = None
        assert len(self.scalars) <= MAX_SCALARS and len(self.topo) <= MAX_TOPO_COLS
        assert self.taint_words <= MAX_TAINT_WORDS and self.static_words <= MAX_STATIC_WORDS

    def c_struct(self):
        nd = Nodes()
        nd.n_nodes = self.n
        nd.n_scalars = len(self.scalars)
        nd.taint_words = self.taint_words
        nd.static_words = self.static_words
        nd.n_topo_cols = len(self.topo)
        nd.has_placed_mask = int(self.has_placed_mask)
        for f in ("alloc_cpu", "alloc_mem", "alloc_eph", "req_cpu", "req_mem", "req_eph", "nz_cpu", "nz_mem"):
            setattr(nd, f, _ptr(getattr(self, f), P64))
        nd.alloc_pods = _ptr(self.alloc_pods, P32)
        nd.npods = _ptr(self.npods, P32)
        for k, (a, r) in enumerate(self.scalars):
            nd.alloc_scalar[k] = _ptr(a, P64)
            nd.req_scalar[k] = _ptr(r, P64)
        nd.taint_mask = _ptr(self.taint_mask, PU64)
        nd.static_mask = _ptr(self.static_mask, PU64) if self.static_words else PU64()
        for k, t in enumerate(self.topo):
            nd.topo[k] = _ptr(t, P32)
        for w in range(MAX_TAINT_WORDS):
            nd.taint_nosched[w] = self.taint_nosched[w]
            nd.taint_prefer[w] = self.taint_prefer[w]
        if self.taint_list_off is not None:
            nd.taint_list_off = _ptr(self.taint_list_off, P32)
            nd.taint_list = _ptr(self.taint_list, PU8)
        return nd

    def core_bytes_per_node(self):
        """Algorithmic bytes one predicate-eval must read (SURVEY.md §8d accounting): the SoA row of this snapshot."""
        b = 72 + 16 * len(self.scalars) + 8 * self.taint_words + 8 * self.static_words
        return b


def default_template(cpu_milli=0, mem=0, eph=0, nz_cpu=None, nz_mem=None, fit_only=False):
    """Template with the default profile's plugin set and weights (default_plugins.go:30-58; defaults.go:229-245).

    nz_* default to the pod's own requests when > 0, else the scheduler's 100m / 200Mi non-zero defaults
    (util/pod_resources.go:29,31) — the single-container case of types.go:700-734.
    """
    t = Template()
    t.req_cpu, t.req_mem, t.req_eph = int(cpu_milli), int(mem), int(eph)
    t.nz_cpu = int(nz_cpu if nz_cpu is not None else (cpu_milli if cpu_milli > 0 else 100))
    t.nz_mem = int(nz_mem if nz_mem is not None else (mem if mem > 0 else 200 * 1024 * 1024))
    t.least_cpu, t.least_mem = t.nz_cpu, t.nz_mem
    t.bal_cpu, t.bal_mem = int(cpu_milli), int(mem)
    t.flags = 0
    if cpu_milli == 0 and mem == 0 and eph == 0:
        t.flags |= TF_FIT_ALL_ZERO
    if cpu_milli == 0 and mem == 0:
        t.flags |= TF_BALANCED_SKIP
    t.filter_enable = PL_FIT if fit_only else PL_ALL
    t.score_enable = (PL_FIT | PL_BALANCED) if fit_only else PL_ALL
    t.nodename_idx = -1
    t.prefilter_bit = -1
    t.spts_ignored_bit = -1
    t.w_taint, t.w_node_affinity, t.w_fit, t.w_pts, t.w_ipa, t.w_balanced, t.w_image = 3, 2, 1, 2, 2, 1, 1
    t.least_w_cpu, t.least_w_mem = 1, 1
    return t


def make_counter(topo_col, init, n_present=None, inc=0, elig_bit=-1):
    init = np.ascontiguousarray(init, dtype=np.int32)
    c = Counter()
    c.topo_col = topo_col
    c.n_domains = len(init)
    c.n_present = len(init) if n_present is None else n_present
    c.inc = inc
    c.elig_bit = elig_bit
    c.init = _ptr(init, P32)
    c._keep = init
    return c


def fit_error_message(n_nodes, hist, no_victims, not_helpful, reason_text):
    """FitError.Error() + DefaultPreemption suffix (framework/types.go:787-838; defaultpreemption/default_preemption.go:138-141;
    preemption/preemption.go:262-277). `hist` maps reason id -> count; reason_text(id) gives the string."""
    def one(n, items):
        msg = "0/%d nodes are available:" % n
        strs = sorted("%d %s" % (v, k) for k, v in items if v)
        if strs:
            msg += " %s." % ", ".join(strs)
        return msg
    msg = one(n_nodes, [(reason_text(r), c) for r, c in hist.items()])
    post = one(n_nodes, [("No preemption victims found for incoming pod", no_victims),
                         ("Preemption is not helpful for scheduling", not_helpful)])
    return msg + " preemption: " + post
