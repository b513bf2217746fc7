/*
 * ccsim.h — C-ABI of the B200 cluster-capacity hot path ("libccsim.so").
 *
 * This is the drop-in boundary of SURVEY.md §8(b): plain pointers and sizes, no torch / C++ types.
 * It replaces, for the simulated pod stream, what the reference drives through the embedded
 * kube-scheduler:
 *
 *   ccsim_load_nodes      <- NodeInfo / Resource built by SetNode + AddPodInfo/update
 *                            (vendor/k8s.io/kubernetes/pkg/scheduler/framework/types.go:160-200,333-343,409-427,461-465)
 *                            in nodeTree.list() order (backend/cache/node_tree.go:119-143)
 *   ccsim_set_templates   <- per-pod PreFilter/PreScore state (noderesources/fit.go:224-233,
 *                            resource_allocation.go:118-140, tainttoleration, nodeaffinity, nodeports,
 *                            podtopologyspread/filtering.go:235-308, interpodaffinity/filtering.go:274-309)
 *   ccsim_run             <- ClusterCapacity.Run: the ScheduleOne loop
 *                            (pkg/framework/simulator.go:356-381; scheduler/schedule_one.go:66-148,430-478),
 *                            the ClusterCapacityBinder commit (pkg/framework/plugins/clustercapacitybinder/plugin.go:34-53)
 *                            and the postBindHook limit check (pkg/framework/simulator.go:297-312)
 *   ccsim_result          <- Status{Pods, StopReason} (pkg/framework/simulator.go:90-93) + the FitError
 *                            reason histogram (framework/types.go:787-838) + the preemption suffix counts
 *                            (framework/preemption/preemption.go:234-279)
 *
 * All strings (node names, label keys, reasons) stay on the host: the device sees ids and bitmasks only.
 * The host side that produces these arrays from Node/Pod objects is include/cchost.h.
 *
 * Conventions: every function returns 0 on success or a negative CCSIM_E* code; ccsim_last_error(h)
 * gives text. A handle is not thread-safe (one Run at a time, like the reference). Input arrays are
 * caller-owned HOST memory and are copied (H2D) before the call returns. No exceptions cross the ABI.
 */
#ifndef CCSIM_H
#define CCSIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCSIM_ABI_VERSION 3

/* ---- limits (compile-time, shared by host encoder, oracle and kernels) ---- */
#define CCSIM_MAX_TAINT_WORDS   4   /* 64-bit words of the taint dictionary mask per node  */
#define CCSIM_MAX_STATIC_WORDS  4   /* 64-bit words of static node-predicate bits per node */
#define CCSIM_MAX_SCALARS       4   /* extended/scalar resources referenced by templates    */
#define CCSIM_MAX_AFF_TERMS     8   /* required nodeAffinity terms (ORed)                   */
#define CCSIM_MAX_PTS           8   /* hard topology-spread constraints                     */
#define CCSIM_MAX_IPA           8   /* distinct topology keys of required (anti-)affinity   */
#define CCSIM_MAX_TOPO_COLS     16  /* topology domain-id columns                           */
#define CCSIM_MAX_COUNTERS      24  /* per-domain counters (PTS + IPA)                      */
#define CCSIM_MAX_TEMPLATES     64
#define CCSIM_MAX_CLASSES       8   /* distinct PreferNoSchedule intolerable-taint counts   */

/* bit 63 of taint word 0 is node.Spec.Unschedulable (nodeunschedulable/node_unschedulable.go:133-150) */
#define CCSIM_TAINT_UNSCHEDULABLE_BIT 63

/* ---- error codes ---- */
#define CCSIM_OK             0
#define CCSIM_EINVAL        -1
#define CCSIM_ENOMEM        -2
#define CCSIM_ECUDA         -3
#define CCSIM_EUNSUPPORTED  -4
#define CCSIM_ESTATE        -5
#define CCSIM_ENCCL         -6

/* ---- template flags ---- */
#define CCSIM_TF_TOLERATES_UNSCHEDULABLE  (1u << 0)  /* pod tolerates node.kubernetes.io/unschedulable:NoSchedule */
#define CCSIM_TF_HAS_NODE_SELECTOR        (1u << 1)  /* NodeAffinity filter not skipped (node_affinity.go:147-155) */
#define CCSIM_TF_HAS_AFFINITY_TERMS       (1u << 2)  /* spec.affinity.nodeAffinity.required present                */
#define CCSIM_TF_HAS_HOST_PORTS           (1u << 3)  /* NodePorts not skipped (node_ports.go:68-76)                */
#define CCSIM_TF_FIT_ALL_ZERO             (1u << 4)  /* cpu=mem=eph=0 and no scalars: fit.go:578-583 early-out     */
#define CCSIM_TF_BALANCED_SKIP            (1u << 5)  /* best-effort pod: BalancedAllocation PreScore Skip (:68-73) */
#define CCSIM_TF_AFF_SELF_MATCH_ALL       (1u << 6)  /* pod matches all of its own required affinity terms          */
#define CCSIM_TF_PREFILTER_NODES          (1u << 7)  /* NodeAffinity PreFilterResult.NodeNames (node_affinity.go:164-194) */

/* ---- plugin enable bits (filter_enable / score_enable); default profile = all ---- */
#define CCSIM_PL_NODE_UNSCHEDULABLE (1u << 0)
#define CCSIM_PL_NODE_NAME          (1u << 1)
#define CCSIM_PL_TAINT_TOLERATION   (1u << 2)
#define CCSIM_PL_NODE_AFFINITY      (1u << 3)
#define CCSIM_PL_NODE_PORTS         (1u << 4)
#define CCSIM_PL_FIT                (1u << 5)
#define CCSIM_PL_POD_TOPOLOGY_SPREAD (1u << 6)
#define CCSIM_PL_INTER_POD_AFFINITY (1u << 7)
#define CCSIM_PL_BALANCED           (1u << 8)   /* score only */
#define CCSIM_PL_IMAGE_LOCALITY     (1u << 9)   /* score only; contributes weight*0 on snapshots without images */
#define CCSIM_PL_ALL                0x3ffu

/* ---- FitError reason ids (framework/types.go:787-838 builds "<count> <reason>" from these) ---- */
enum {
  CCSIM_R_UNSCHEDULABLE = 0,      /* "node(s) were unschedulable"                                      */
  CCSIM_R_NODE_NAME,              /* "node(s) didn't match the requested node name"                    */
  CCSIM_R_NODE_AFFINITY,          /* "node(s) didn't match Pod's node affinity/selector"               */
  CCSIM_R_NODE_PORTS,             /* "node(s) didn't have free ports for the requested pod ports"      */
  CCSIM_R_TOO_MANY_PODS,          /* "Too many pods"                                                   */
  CCSIM_R_INSUFFICIENT_CPU,       /* "Insufficient cpu"                                                */
  CCSIM_R_INSUFFICIENT_MEMORY,    /* "Insufficient memory"                                             */
  CCSIM_R_INSUFFICIENT_EPHEMERAL, /* "Insufficient ephemeral-storage"                                  */
  CCSIM_R_PTS_MISSING_LABEL,      /* "node(s) didn't match pod topology spread constraints (missing required label)" */
  CCSIM_R_PTS_SKEW,               /* "node(s) didn't match pod topology spread constraints"            */
  CCSIM_R_IPA_AFFINITY,           /* "node(s) didn't match pod affinity rules"                         */
  CCSIM_R_IPA_ANTI_AFFINITY,      /* "node(s) didn't match pod anti-affinity rules"                    */
  CCSIM_R_IPA_EXISTING_ANTI,      /* "node(s) didn't satisfy existing pods anti-affinity rules"        */
  CCSIM_R_PREFILTER_NODES,        /* "node(s) didn't satisfy plugin(s) [NodeAffinity]"                 */
  CCSIM_R_FIXED_COUNT,
  /* then CCSIM_MAX_SCALARS entries "Insufficient <scalar name>", then one per taint-dictionary id:
     "node(s) had untolerated taint {key: value}" */
  CCSIM_R_SCALAR0 = CCSIM_R_FIXED_COUNT,
  CCSIM_R_TAINT0  = CCSIM_R_SCALAR0 + CCSIM_MAX_SCALARS,
  CCSIM_R_TOTAL   = CCSIM_R_TAINT0 + 64 * CCSIM_MAX_TAINT_WORDS
};

/* stop codes: pkg/framework/simulator.go:300-305 (LimitReached) and :327-342 (Unschedulable) */
#define CCSIM_STOP_UNSCHEDULABLE 0
#define CCSIM_STOP_LIMIT_REACHED 1

/* sampling: CANONICAL = percentageOfNodesToScore 100 (every node filtered every cycle, start index fixed);
 * REFERENCE = the default profile's sampling as a deterministic sequential scan: stop at the numFeasibleNodesToFind-th
 * feasible node in rotated order, nextStartNodeIndex advances by the nodes examined (schedule_one.go:538-539,610-723).
 * Ties -> first maximum in (rotated) scan order in both. */
#define CCSIM_SAMPLING_CANONICAL 0
#define CCSIM_SAMPLING_REFERENCE 1

/* engine selection */
#define CCSIM_ENGINE_AUTO        0  /* batched tie-run waves when provably order-equivalent, else sequential */
#define CCSIM_ENGINE_SEQUENTIAL  1  /* one winner per wave (always valid; evals = (placed+1)*N)               */
#define CCSIM_ENGINE_BATCHED     2  /* error if the templates are not eligible                               */

typedef struct ccsim_config {
  int32_t abi_version;      /* CCSIM_ABI_VERSION */
  int32_t device;           /* CUDA device ordinal */
  int32_t engine;           /* CCSIM_ENGINE_* */
  int32_t rank, world;      /* node-axis shard of a multi-GPU run; world=1 for a single GPU */
  int32_t sampling;         /* CCSIM_SAMPLING_*: which valid execution of the (non-deterministic) reference loop is reproduced */
  int32_t pct_nodes_to_score; /* percentageOfNodesToScore for CCSIM_SAMPLING_REFERENCE (0 = adaptive, schedule_one.go:697-723) */
  int32_t reserved[1];
} ccsim_config;

/*
 * Node columns (SoA), all length n_nodes, in nodeTree.list() order. A1 of SURVEY.md §8(a).
 * Bitmask columns are word-major: word w of node i is mask[w * n_nodes + i] (coalesced per word).
 */
typedef struct ccsim_nodes {
  int32_t n_nodes;
  int32_t n_scalars;        /* <= CCSIM_MAX_SCALARS */
  int32_t taint_words;      /* 1..CCSIM_MAX_TAINT_WORDS (word 0 always present: carries the unschedulable bit) */
  int32_t static_words;     /* 0..CCSIM_MAX_STATIC_WORDS */
  int32_t n_topo_cols;      /* <= CCSIM_MAX_TOPO_COLS */
  int32_t has_placed_mask;  /* 1 if any template has hostPorts: engine keeps a per-node "templates placed here" mask */
  /* Allocatable (types.go:461-465) */
  const int64_t *alloc_cpu, *alloc_mem, *alloc_eph;
  const int32_t *alloc_pods;
  /* Requested / NonZeroRequested / len(Pods) (types.go:409-427) */
  const int64_t *req_cpu, *req_mem, *req_eph;
  const int32_t *npods;
  const int64_t *nz_cpu, *nz_mem;
  const int64_t *alloc_scalar[CCSIM_MAX_SCALARS];
  const int64_t *req_scalar[CCSIM_MAX_SCALARS];
  /* taint dictionary mask: bit t of word w <=> node carries taint id 64*w+t (any effect); bit 63 of word 0 = Spec.Unschedulable */
  const uint64_t *taint_mask;
  /* static node-predicate bits (label requirements, existing hostPort conflicts, existing-pod anti-affinity, ...) */
  const uint64_t *static_mask;
  /* topology domain ids per column: >=0 domain id, -1 = node lacks the key */
  const int32_t *topo[CCSIM_MAX_TOPO_COLS];
  /* taint-dictionary effect masks (global, taint_words each): NoSchedule|NoExecute and PreferNoSchedule entries */
  uint64_t taint_nosched[CCSIM_MAX_TAINT_WORDS];
  uint64_t taint_prefer[CCSIM_MAX_TAINT_WORDS];
  /* per node: taint ids in node.Spec.Taints list order, CSR, used only by the terminal diagnosis pass
     (FindMatchingUntoleratedTaint returns the FIRST untolerated taint: component-helpers/scheduling/corev1/helpers.go:78-101) */
  const int32_t *taint_list_off;  /* n_nodes+1 */
  const uint8_t *taint_list;      /* taint ids (<256) */
} ccsim_nodes;

/* One per-domain counter of the (single) template: a PTS constraint or an IPA topology key. */
typedef struct ccsim_counter {
  int32_t topo_col;      /* index into ccsim_nodes.topo, or -1: node-local (every node its own domain, e.g. unique hostnames) */
  int32_t n_domains;     /* D; for node-local counters = n_nodes */
  int32_t n_present;     /* PTS only: domains [0,n_present) are in TpValueToMatchNum (take part in the global min) */
  int32_t inc;           /* added to the winner's domain at every commit (self-match count; signed for score counters) */
  int32_t elig_bit;      /* static bit a node must carry for its commits to count (soft PTS: "has every constraint key and
                            passes the node-inclusion policies", scoring.go:157-186); -1 = every node */
  int32_t pad;
  const int32_t *init;   /* [n_domains] counts from pre-existing pods */
} ccsim_counter;

/* One ScheduleAnyway / system-default topology-spread constraint (PL:podtopologyspread/scoring.go:60-265). */
typedef struct ccsim_spts {
  int32_t counter;       /* matching pods per domain (node-local column when hostname != 0) */
  int32_t max_skew;
  int32_t hostname;      /* 1: topologyKey == kubernetes.io/hostname: per-node count, weight from the number of scored nodes */
  int32_t has_key_bit;   /* hostname constraints: static bit "node carries the key", -1 = every node does.
                            Other keys: the topology column says -1 where the key is missing */
} ccsim_spts;

typedef struct ccsim_pts {
  int32_t counter;       /* index into counters */
  int32_t max_skew;
  int32_t self_match;    /* 1 if the pod's own labels match the constraint selector (filtering.go:341-344) */
  int32_t min_zero;      /* 1 if #domains < minDomains: global minimum treated as 0 (filtering.go:56-69) */
} ccsim_pts;

typedef struct ccsim_template {
  /* A2: request vectors (fit.go:224-233; types.go:700-734; resource_allocation.go:118-140) */
  int64_t req_cpu, req_mem, req_eph;
  int64_t req_scalar[CCSIM_MAX_SCALARS];
  int64_t nz_cpu, nz_mem;         /* Non0CPU / Non0Mem added to NonZeroRequested at commit */
  int64_t least_cpu, least_mem;   /* LeastAllocated pod request (useRequested=false)        */
  int64_t bal_cpu, bal_mem;       /* BalancedAllocation pod request (useRequested=true)     */
  uint32_t flags;                 /* CCSIM_TF_*  */
  uint32_t filter_enable;         /* CCSIM_PL_*  */
  uint32_t score_enable;          /* CCSIM_PL_*  */
  int32_t nodename_idx;           /* -1: spec.nodeName empty (always, for generated pods: podgenerator.go:31) */
  /* weights (default_plugins.go:38-50) */
  int32_t w_taint, w_node_affinity, w_fit, w_pts, w_ipa, w_balanced, w_image;
  int32_t least_w_cpu, least_w_mem;  /* NodeResourcesFitArgs.ScoringStrategy.Resources weights (defaults.go:229-245) */
  /* TaintToleration */
  uint64_t tol_nosched[CCSIM_MAX_TAINT_WORDS];  /* dictionary taints (NoSchedule/NoExecute) tolerated by the pod */
  uint64_t tol_prefer[CCSIM_MAX_TAINT_WORDS];   /* PreferNoSchedule taints tolerated (taint_toleration.go:129-137) */
  /* NodeAffinity: nodeSelector AND (OR over terms); static bits */
  uint64_t sel_mask[CCSIM_MAX_STATIC_WORDS];
  int32_t n_aff_terms;
  int32_t prefilter_bit;          /* static bit "node name is in PreFilterResult.NodeNames", -1 none */
  uint64_t aff_term_mask[CCSIM_MAX_AFF_TERMS][CCSIM_MAX_STATIC_WORDS];
  /* NodePorts */
  uint64_t port_static_mask[CCSIM_MAX_STATIC_WORDS]; /* static bits: an existing pod on the node conflicts with a wanted hostPort */
  uint64_t port_tmpl_conflict;    /* templates whose hostPorts conflict with this one's (bit = template index) */
  /* InterPodAffinity: static bit(s) "an existing pod's required anti-affinity term matches this pod in one of the node's topology pairs" */
  uint64_t existing_anti_mask[CCSIM_MAX_STATIC_WORDS];
  /* PodTopologySpread hard constraints, in spec order */
  int32_t n_pts;
  ccsim_pts pts[CCSIM_MAX_PTS];
  /* InterPodAffinity required terms, grouped by topology key */
  int32_t n_aff;                  /* affinity keys  */
  int32_t aff_counter[CCSIM_MAX_IPA];
  int32_t n_anti;                 /* anti-affinity keys */
  int32_t anti_counter[CCSIM_MAX_IPA];
  int64_t aff_total_init;         /* sum of all affinity counts (len(affinityCounts)==0 test, filtering.go:396-405) */
  /* NodeAffinity preferredDuringScheduling terms (node_affinity.go:241-290): raw score = sum of the weights of the
   * matching terms (static bits), normalised per cycle to 100*raw/max over the feasible nodes (normalize_score.go:28-56) */
  int32_t n_pref_terms;
  int32_t pref_weight[CCSIM_MAX_AFF_TERMS];
  int32_t pad_pref;
  uint64_t pref_mask[CCSIM_MAX_AFF_TERMS][CCSIM_MAX_STATIC_WORDS];
  /* PodTopologySpread score (scoring.go:60-265): soft constraints in spec order (or the two system defaults when a
   * Service/RC/RS/StatefulSet selects the pod, plugin.go:48-59, helper/spread.go:40-93). Per cycle: weight_c =
   * log(size_c + 2) with size_c = distinct domains (hostname: nodes) among the feasible non-ignored nodes; node raw =
   * Round(sum_c cnt_c(node) * weight_c + (maxSkew_c - 1)); normalised 100*(max+min-raw)/max over the same nodes. */
  int32_t n_spts;
  int32_t spts_ignored_bit;       /* static bit "node misses one of the constraint keys" (IgnoredNodes, only when the
                                     constraints come from the podspec); -1: no node is ignored */
  ccsim_spts spts[CCSIM_MAX_PTS];
  /* InterPodAffinity score (interpodaffinity/scoring.go:51-295): per topology key a counter of signed weights
   * (preferred terms of the pod vs existing pods, existing pods' required*hardPodAffinityWeight / preferred terms vs the
   * pod); node raw = sum over keys the node carries; normalised int64(100 * float64(raw-min)/float64(max-min)). */
  int32_t n_ipa_score;
  int32_t ipa_score_counter[CCSIM_MAX_IPA];
  int32_t pad_soft;
  /* ImageLocality (imagelocality/image_locality.go:54-131): the score is static per node and template (image states do
   * not change when pods are assumed); [n_nodes] values 0..100 or NULL (all 0). Host memory at ccsim_set_templates. */
  const uint8_t *image_score;
} ccsim_template;

typedef struct ccsim_result {
  int64_t placed;                 /* len(status.Pods) */
  int32_t stop_code;              /* CCSIM_STOP_* */
  int32_t n_nodes;
  int64_t waves;                  /* grid-wide waves executed */
  int64_t evals;                  /* (pod attempt, node) pairs pushed through the fused Filter pass on the device */
  int64_t examined;               /* nodes the reference would have examined (== evals unless CCSIM_SAMPLING_REFERENCE) */
  int64_t reason_hist[CCSIM_R_TOTAL]; /* terminal FitError histogram (zero when stop_code == LIMIT_REACHED) */
  int64_t preempt_no_victims;     /* nodes whose terminal status code is Unschedulable ("No preemption victims found for incoming pod") */
  int64_t preempt_not_helpful;    /* the rest ("Preemption is not helpful for scheduling") */
  double  run_ms;                 /* device time of the run (CUDA events on the engine stream) */
  const int32_t *pod_node;        /* [placed] node index of pod k, host memory owned by the handle until the next run/destroy */
} ccsim_result;

typedef struct ccsim_handle ccsim_handle;

/* lifecycle */
int  ccsim_create(const ccsim_config *cfg, ccsim_handle **out);
void ccsim_destroy(ccsim_handle *h);
const char *ccsim_last_error(const ccsim_handle *h);  /* h may be NULL: last create error */
int  ccsim_abi_version(void);

/* snapshot upload (H2D inside the call) */
int  ccsim_load_nodes(ccsim_handle *h, const ccsim_nodes *nodes);
int  ccsim_set_templates(ccsim_handle *h, int32_t n_templates, const ccsim_template *templates,
                         int32_t n_counters, const ccsim_counter *counters);

/* Run: place pods k = 0,1,2,... (template k % n_templates) until one does not fit or max_pods (>0) are placed.
 * Restores the loaded snapshot first, so it can be called repeatedly. Blocking. */
int  ccsim_run(ccsim_handle *h, int64_t max_pods, ccsim_result *out);
/* Optional: everything ccsim_run(h, max_pods) does BEFORE the wave kernel starts (buffers, restoring the snapshot, engine choice),
 * synchronously. A host that drives several ranks from one process calls it on every handle, then starts the ccsim_run calls
 * concurrently: no rank's persistent kernel then waits for a peer that is still inside a (device-synchronising) allocation. */
int  ccsim_prepare(ccsim_handle *h, int64_t max_pods);

/* per-node number of placed pods of template t after the last run (device histogram; report.go:146-180 without the O(P*nodes) scan)
 * and the index of the first pod placed on each node (-1 none): ReplicasOnNodes is ordered by first placement. */
int  ccsim_node_counts(ccsim_handle *h, int32_t t, int32_t *counts /*[n_nodes]*/, int64_t *first_pod /*[n_nodes]*/);

/* multi-GPU (node-axis shards, SURVEY.md §8(e)): one process per GPU, rank r owns nodes [r*ceil(N/W), ...).
 * The per-wave exchange of the shard winners happens INSIDE the persistent kernel through peer memory (NVLink/NVSwitch):
 * every rank exports the CUDA IPC handle of its exchange buffer, the caller all-gathers the handles (torch.distributed)
 * and every rank imports its peers' buffers. Results: placed / stop_code / pod_node are identical on every rank;
 * reason_hist, preempt_* and evals are per shard and must be summed by the caller (one small all-reduce). */
#define CCSIM_IPC_HANDLE_BYTES 64
#define CCSIM_MAX_WORLD 8
int  ccsim_peer_export(ccsim_handle *h, uint8_t handle_out[CCSIM_IPC_HANDLE_BYTES]);
int  ccsim_peer_import(ccsim_handle *h, int32_t world, const uint8_t *handles /* world x CCSIM_IPC_HANDLE_BYTES, rank order */);

/* Peers inside ONE process (a host that drives its GPUs from one process; the single-GPU tests of the sharded engines, where all
 * ranks share device 0): the exchange buffer's device pointer instead of an IPC handle. Ranks on different devices need peer
 * access enabled by the caller (cudaDeviceEnablePeerAccess). */
int  ccsim_peer_local(ccsim_handle *h, void **ptr_out);
int  ccsim_peer_import_local(ccsim_handle *h, int32_t world, void *const *ptrs /* world pointers, rank order */);

/* introspection for tests / bench */
int  ccsim_device_info(ccsim_handle *h, int32_t *sm_count, int32_t *grid, int32_t *block, int64_t *l2_bytes);
int64_t ccsim_kernel_launches(const ccsim_handle *h);  /* kernels launched by this handle so far */
int  ccsim_flush_l2(ccsim_handle *h);                  /* writes a buffer larger than L2 (bench hygiene) */
/* latency anatomy of the last run (bench.py's roofline block): [0] engine in the low byte (0 generic, 1 lean sequential, 2 tie-run
 * batching, 3 multi-commit, 4 streaming), CCSIM_KV_* bits above it [1] waves [2] placed [3] multi-commit: candidates replayed, summed
 * over waves [4] multi-commit: waves that raised the candidate bar [5] grid [6] block [7] multi-commit: replay rounds, summed over
 * waves [8..15] CTA 0's clock cycles per phase, summed over waves (multi-commit: scan, barrier, merge+publish, gather, replay, row
 * updates+recount; 0 for the other engines) */
int  ccsim_run_stats(const ccsim_handle *h, int64_t out[16]);
/* which instantiation of the engine's wave kernel ran (ccsim_run_stats out[0]) */
#define CCSIM_KV_ENGINE_MASK          0xffll
#define CCSIM_KV_RESIDENT             (1ll << 8)   /* generic kernel: the node tile stays in shared memory (else columns are re-read from L2) */
#define CCSIM_KV_STREAM_MODE_SHIFT    9            /* streaming kernel: 2 bits, MODE 0 (every column streamed), 1 (+ taint/static words),
                                                      2 (free columns resident, only the score memo streamed) */
#define CCSIM_KV_REFERENCE_SAMPLING   (1ll << 11)  /* lean kernel in CCSIM_SAMPLING_REFERENCE mode */
#define CCSIM_KV_CROSS_GPU            (1ll << 12)  /* multi-commit kernel of a node-sharded run (world > 1) */

/* Scores node i of the loaded snapshot (this handle's shard, [n] entries each) for template t as if `clones` pods of t had been
 * committed to it, with the device function every wave kernel scores with: total = NodeResourcesFit (LeastAllocated) * w_fit +
 * BalancedAllocation * w_balanced as enabled by the template, least / balanced = the unweighted plugin scores. The other plugins'
 * shares (TaintToleration, NodeAffinity, ...) are not part of it. Needs ccsim_set_templates; does not touch the run state. */
int  ccsim_debug_node_scores(ccsim_handle *h, int32_t t, int32_t clones, int64_t *total, int64_t *least, int64_t *balanced);

#ifdef __cplusplus
}
#endif
#endif /* CCSIM_H */
