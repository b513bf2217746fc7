// ccsim_engine.cu — libccsim.so: the B200 cluster-capacity hot path behind the C-ABI of include/ccsim.h.
//
// Replaces the reference's sequential schedule-one-pod-then-update loop
// (pkg/framework/simulator.go:356-381 driving vendor/k8s.io/kubernetes/pkg/scheduler/schedule_one.go:66-148) by ONE
// persistent cooperative kernel per Run:
//
//   wave k (pod k, template k % M):
//     every CTA owns a contiguous tile of nodes and pushes each through the fused Filter+Score pass (eval_node),
//     warp-shuffle + shared-memory arg-max over packed (score, ~index) keys,
//     all-to-all exchange of one 64-bit tagged key per CTA (and per normalisation class) through L2 — this is the
//     only grid-wide synchronisation of the wave (no atomics, no fences: the tag makes each word self-validating),
//     every CTA redundantly reduces the 148 keys, the owner CTA commits the winner row (NodeInfo.update,
//     framework/types.go:409-427), every CTA updates its replica of the per-domain counters.
//
// The node state is mutated in place in HBM/L2; only the owner CTA ever reads or writes a given row, so no
// inter-CTA ordering is needed beyond the key exchange.
#include <cuda_runtime.h>
#include <algorithm>
#include <climits>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdarg.h>
#include <dlfcn.h>
#include <map>
#include <string>
#include <vector>
#include "ccsim_device.cuh"
#ifdef CCSIM_PHASE_TIMERS
#define PH_START() do { if (cta == 0 && tid == 0) tc0 = clock64(); } while (0)
#define PH_MARK(i) do { if (cta == 0 && tid == 0) { tc1 = clock64(); ph[i] += tc1 - tc0; tc0 = tc1; } } while (0)
#else
#define PH_START() do {} while (0)
#define PH_MARK(i) do {} while (0)
#endif
#include "ccsim_lean.cuh"
#include "ccsim_batched.cuh"
#include "ccsim_multi.cuh"
#include "ccsim_stream.cuh"

#define BLOCK_THREADS 512
#define MAX_WARPS (BLOCK_THREADS / 32)
#define SMEM_CNT_MAX_INTS 16384      /* 64 KB of replicated counters in shared memory; above that: global replicas */
#define WATCHDOG_SPINS (1u << 24)

struct __align__(16) WaveShared {
  ccsim_template tmpl;                              // current template
  FilterConsts fc;                                  // folded per-wave constants of the Filter pass
  unsigned long long warp_best[MAX_WARPS][CCSIM_MAX_CLASSES];
  const int32_t *topo_ptr[CCSIM_MAX_TOPO_COLS];     // topology columns as this CTA indexes them (pre-offset)
  int32_t *cnt_ptr[CCSIM_MAX_COUNTERS];             // counter bases (shared replica / global replica / node-local column)
  int32_t ptsmin[CCSIM_MAX_PTS];
  int32_t ptsnum[CCSIM_MAX_PTS];
  long long aff_total;
  int32_t winner;        // global node index, -1 = none
  int32_t stop;          // 0 continue, 1 unschedulable, 2 limit, 3 error
  int32_t dirty;         // FilterConsts must be rebuilt before the next scan
  // normalised soft scorers (multi-phase waves): extrema of the raw scores over the feasible nodes of this wave
  long long na_max, spts_min, spts_max, ipa_min, ipa_max;
  long long spts_scored;                 // feasible nodes that are not in IgnoredNodes
  double spts_w[CCSIM_MAX_PTS];          // topologyNormalizingWeight per soft constraint
  long long red[MAX_WARPS][6];           // block reductions of the above
  ScoreWeights sw;       // scalar copy of the template's score configuration (passed by value to score_node)
  CommitInfo cinfo[CCSIM_MAX_COUNTERS];   // what a commit does to each counter under the current template
  int32_t scratch[MAX_WARPS];
};

// Statically allocated so that every access is a direct LDS/STS with a compile-time offset (a reference obtained by
// casting the dynamic shared array makes nvcc re-derive the generic window base — S2UR SR_CgaCtaId — at each use).
__shared__ WaveShared ws;

// recount of a PTS constraint's minimum and its multiplicity over the present domains (all threads of the CTA)
__device__ void pts_recount(const DevParams &p, int c) {
  const ccsim_pts &pc = ws.tmpl.pts[c];
  const DevCounter &dc = p.counters[pc.counter];
  const int32_t *cnt = ws.cnt_ptr[pc.counter];
  int32_t m = INT32_MAX;
  for (int d = threadIdx.x; d < dc.n_present; d += blockDim.x) m = min(m, cnt[d]);
  for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) ws.scratch[threadIdx.x >> 5] = m;
  __syncthreads();
  m = INT32_MAX;
  for (int w = 0; w < (int)(blockDim.x >> 5); w++) m = min(m, ws.scratch[w]);
  __syncthreads();
  int32_t num = 0;
  for (int d = threadIdx.x; d < dc.n_present; d += blockDim.x) num += (cnt[d] == m);
  for (int o = 16; o > 0; o >>= 1) num += __shfl_xor_sync(0xffffffffu, num, o);
  if ((threadIdx.x & 31) == 0) ws.scratch[threadIdx.x >> 5] = num;
  __syncthreads();
  if (threadIdx.x == 0) {
    int32_t s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += ws.scratch[w];
    ws.ptsmin[c] = pc.min_zero ? 0 : m;    // filtering.go:56-69: fewer domains than minDomains -> global minimum 0
    ws.ptsnum[c] = s;
    ws.dirty = 1;
  }
  __syncthreads();
}

// PodTopologySpread.Score of a node that is not in IgnoredNodes, with this wave's weights (scoring.go:192-224,302-304)
__device__ __forceinline__ long long spts_raw(const DevParams &p, const ccsim_template &t, int32_t i) {
  double score = 0.0;
  for (int c = 0; c < t.n_spts; c++) {
    const ccsim_spts sc = t.spts[c];
    long long cnt;
    if (sc.hostname) {
      if (sc.has_key_bit >= 0 && !static_bit(p, i, sc.has_key_bit)) continue;
      cnt = ws.cnt_ptr[sc.counter][i];
    } else {
      const int32_t dom = ws.topo_ptr[p.counters[sc.counter].topo_col][i];
      if (dom < 0) continue;
      cnt = ws.cnt_ptr[sc.counter][dom];
    }
    score = __dadd_rn(score, __dadd_rn(__dmul_rn((double)cnt, ws.spts_w[c]), (double)(sc.max_skew - 1)));
  }
  return __double2ll_rn(round(score)) ;   // math.Round: half away from zero (round() already yields an integer value)
}

// InterPodAffinity.Score (interpodaffinity/scoring.go:236-256)
__device__ __forceinline__ long long ipa_raw(const DevParams &p, const ccsim_template &t, int32_t i) {
  long long sc = 0;
  for (int k = 0; k < t.n_ipa_score; k++) {
    const int j = t.ipa_score_counter[k];
    const int32_t tc = p.counters[j].topo_col;
    const int32_t dom = tc < 0 ? i : ws.topo_ptr[tc][i];
    if (dom >= 0) sc += ws.cnt_ptr[j][dom];
  }
  return sc;
}

// ------------------------------------------------------------------------------------------------------------------
// The persistent wave kernel (sequential engine: one winner per wave; always a valid execution of the reference loop)
//   RESIDENT: the CTA's node tile (every column the Filter/Score pass reads) is staged into shared memory once and
//             stays there for all waves; commits write through to the global columns (read by the diagnosis pass).
//   streaming: tiles too large for shared memory are re-read from global memory (L2) every wave.
// ------------------------------------------------------------------------------------------------------------------
template <bool RESIDENT>
__global__ void __launch_bounds__(BLOCK_THREADS, 1) ccsim_wave_kernel(const DevParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t *smem_cnt = reinterpret_cast<int32_t *>(smem_raw);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cta = blockIdx.x;
  const int32_t lo = min(p.n, cta * p.chunk), hi = min(p.n, lo + p.chunk);
  const int ncls = p.n_classes;
  const bool use_cache = (p.n_templates == 1);

  // ---- tile: shared-memory columns (pre-offset by -lo) or the global columns themselves ----
  Tile tl;
  int32_t *tile_topo = nullptr, *tile_local = nullptr;
  if (RESIDENT) {
    const size_t cp = (size_t)p.chunk_pad;
    unsigned char *base = smem_raw + (((size_t)p.smem_cnt_ints * 4 + 15) & ~(size_t)15);
    unsigned long long *q8 = reinterpret_cast<unsigned long long *>(base);
    unsigned long long *s_taint = q8;            q8 += cp;
    unsigned long long *s_static = q8;           if (p.static_words > 0) q8 += cp;
    long long *s_acpu = (long long *)q8;         q8 += cp;
    long long *s_amem = (long long *)q8;         q8 += cp;
    long long *s_rcpu = (long long *)q8;         q8 += cp;
    long long *s_rmem = (long long *)q8;         q8 += cp;
    long long *s_zcpu = (long long *)q8;         q8 += cp;
    long long *s_zmem = (long long *)q8;         q8 += cp;
    long long *s_fcpu = (long long *)q8;         q8 += cp;
    long long *s_fmem = (long long *)q8;         q8 += cp;
    int32_t *q4 = reinterpret_cast<int32_t *>(q8);
    int32_t *s_fpods = q4;                       q4 += cp;
    int32_t *s_apods = q4;                       q4 += cp;
    int32_t *s_npods = q4;                       q4 += cp;
    int32_t *s_score = q4;                       q4 += cp;
    tile_topo = q4;                              q4 += cp * p.n_topo;
    tile_local = q4;
    for (int32_t i = lo + tid; i < hi; i += blockDim.x) {
      const int32_t j = i - lo;
      s_taint[j] = p.taint_mask[i];
      if (p.static_words > 0) s_static[j] = p.static_mask[i];
      s_acpu[j] = p.alloc_cpu[i]; s_amem[j] = p.alloc_mem[i];
      s_rcpu[j] = p.req_cpu[i];   s_rmem[j] = p.req_mem[i];
      s_zcpu[j] = p.nz_cpu[i];    s_zmem[j] = p.nz_mem[i];
      s_apods[j] = p.alloc_pods[i]; s_npods[j] = p.npods[i];
      s_fcpu[j] = s_acpu[j] - s_rcpu[j]; s_fmem[j] = s_amem[j] - s_rmem[j]; s_fpods[j] = s_apods[j] - s_npods[j];
      s_score[j] = -1;
      for (int c = 0; c < p.n_topo; c++) tile_topo[(size_t)c * cp + j] = p.topo[c][i];
    }
    tl.taint0 = s_taint - lo; tl.static0 = s_static - lo;
    tl.alloc_cpu = s_acpu - lo; tl.alloc_mem = s_amem - lo; tl.req_cpu = s_rcpu - lo; tl.req_mem = s_rmem - lo;
    tl.nz_cpu = s_zcpu - lo; tl.nz_mem = s_zmem - lo;
    tl.alloc_pods = s_apods - lo; tl.npods = s_npods - lo; tl.score = s_score - lo;
    tl.free_cpu = s_fcpu - lo; tl.free_mem = s_fmem - lo; tl.free_pods = s_fpods - lo;
  } else {
    tl.taint0 = (const unsigned long long *)p.taint_mask; tl.static0 = (const unsigned long long *)p.static_mask;
    tl.alloc_cpu = (const long long *)p.alloc_cpu; tl.alloc_mem = (const long long *)p.alloc_mem;
    tl.req_cpu = (long long *)p.req_cpu; tl.req_mem = (long long *)p.req_mem;
    tl.nz_cpu = (long long *)p.nz_cpu; tl.nz_mem = (long long *)p.nz_mem;
    tl.alloc_pods = p.alloc_pods; tl.npods = p.npods; tl.score = p.score_cache;
    tl.free_cpu = nullptr; tl.free_mem = nullptr; tl.free_pods = nullptr;
    for (int32_t i = lo + tid; i < hi; i += blockDim.x) p.score_cache[i] = -1;
  }

  // ---- prologue: template 0, replicated counters, pointer tables, PTS minima ----
  for (int k = tid; k < (int)(sizeof(ccsim_template) / 8); k += blockDim.x)
    reinterpret_cast<unsigned long long *>(&ws.tmpl)[k] = reinterpret_cast<const unsigned long long *>(&p.templates[0])[k];
  {
    int nl = 0;
    for (int j = 0; j < p.n_counters; j++) {
      const DevCounter &dc = p.counters[j];
      if (dc.topo_col < 0) {   // node-local column (restored by the host before the launch)
        int32_t *col = dc.work;
        if (RESIDENT) {
          int32_t *sc = tile_local + (size_t)nl * p.chunk_pad;
          for (int32_t i = lo + tid; i < hi; i += blockDim.x) sc[i - lo] = dc.work[i];
          col = sc - lo;
        }
        if (tid == 0) ws.cnt_ptr[j] = col;
        nl++;
        continue;
      }
      int32_t *dst = dc.smem_off >= 0 ? smem_cnt + dc.smem_off : dc.work + (size_t)cta * dc.n_domains;
      for (int d = tid; d < dc.n_domains; d += blockDim.x) dst[d] = dc.init[d];
      if (tid == 0) ws.cnt_ptr[j] = dst;
    }
  }
  if (tid == 0) {
    for (int c = 0; c < p.n_topo; c++) ws.topo_ptr[c] = RESIDENT ? (tile_topo + (size_t)c * p.chunk_pad - lo) : p.topo[c];
    ws.aff_total = p.templates[0].aff_total_init; ws.winner = -1; ws.stop = 0; ws.dirty = 1;
  }
  __syncthreads();
  for (int c = 0; c < ws.tmpl.n_pts; c++) pts_recount(p, c);

#ifdef CCSIM_PHASE_TIMERS
  long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tc0 = 0, tc1 = 0;
#endif
  long long k = 0;
  bool limit_hit = false;   // postBindHook's limit (simulator.go:300-305)
  uint32_t wtag = 1;         // 1..4095; waves k and k+2 (same parity buffer) always differ
  uint32_t tag = (p.epoch << 12) | wtag;
  int32_t ti = 0;            // template of pod k = k % n_templates (report.go:160)
  for (;; k++) {
    PH_START();
    // postBindHook limit (pkg/framework/simulator.go:300-305): checked after the k-th pod was bound
    if (p.max_pods > 0 && k >= p.max_pods) { limit_hit = true; break; }   // uniform; no shared write (slower threads may still be reading ws.stop)
    if (k > p.pod_cap) { if (tid == 0) ws.stop = 3; __syncthreads(); break; }   // cannot happen (pod_cap bounds every run): never spin forever
    if (p.n_templates > 1) {
      const ccsim_template *src = &p.templates[ti];
      for (int q = tid; q < (int)(sizeof(ccsim_template) / 8); q += blockDim.x)
        reinterpret_cast<unsigned long long *>(&ws.tmpl)[q] = reinterpret_cast<const unsigned long long *>(src)[q];
      if (tid == 0) ws.dirty = 1;
      __syncthreads();
    }
    const ccsim_template &t = ws.tmpl;
    if (ws.dirty) {    // uniform: written before the last barrier
      if (tid == 0) {
        build_filter_consts(p, t, ti, ws.topo_ptr, ws.cnt_ptr, ws.ptsmin, ws.aff_total, ws.fc);
        ws.sw.w_fit = (t.score_enable & CCSIM_PL_FIT) ? t.w_fit : 0;
        ws.sw.w_balanced = ((t.score_enable & CCSIM_PL_BALANCED) && !(t.flags & CCSIM_TF_BALANCED_SKIP)) ? t.w_balanced : 0;
        ws.sw.least_w_cpu = t.least_w_cpu; ws.sw.least_w_mem = t.least_w_mem;
        for (int j = 0; j < p.n_counters; j++) {
          const DevCounter &dc = p.counters[j];
          CommitInfo &ci = ws.cinfo[j];
          const bool skip = (dc.inc == 0) || (dc.is_aff && !(t.flags & CCSIM_TF_AFF_SELF_MATCH_ALL));
          ci.inc = skip ? 0 : dc.inc;
          ci.local = dc.topo_col < 0; ci.is_aff = dc.is_aff; ci.n_present = dc.n_present; ci.elig_bit = dc.elig_bit;
          ci.gtopo = dc.topo_col < 0 ? nullptr : p.topo_full[dc.topo_col];
          ci.ltopo = dc.topo_col < 0 ? nullptr : ws.topo_ptr[dc.topo_col];
          ci.pts_idx = -1;
          for (int c = 0; c < t.n_pts; c++) if (t.pts[c].counter == j && !t.pts[c].min_zero) ci.pts_idx = c;
        }
      }
      __syncthreads();
      if (tid == 0) ws.dirty = 0;    // cleared only after every thread has read it
    }
    const FilterConsts &fc = ws.fc;
    const HotConsts hc = load_hot(fc);

    // ---- fused Filter pass over this CTA's tile (+ memoised node-local score of the feasible nodes) ----
    unsigned long long best[CCSIM_MAX_CLASSES];
    #pragma unroll
    for (int c = 0; c < CCSIM_MAX_CLASSES; c++) best[c] = 0ull;
    // Normalised soft scorers (NodeAffinity preferred terms, PodTopologySpread ScheduleAnyway/system defaults, InterPodAffinity
    // score) need extrema of their raw scores over the FEASIBLE nodes of this cycle before any node's total is known
    // (helper/normalize_score.go:28-56; podtopologyspread/scoring.go:226-265; interpodaffinity/scoring.go:258-290): such
    // templates take up to three passes over the tile with one or two extra grid-wide exchanges per wave.
    const bool na_on = (t.n_pref_terms > 0) && (t.score_enable & CCSIM_PL_NODE_AFFINITY);
    const bool spts_on = (t.n_spts > 0) && (t.score_enable & CCSIM_PL_POD_TOPOLOGY_SPREAD);
    const bool ipa_on = (t.n_ipa_score > 0) && (t.score_enable & CCSIM_PL_INTER_POD_AFFINITY);
    const bool soft = na_on || spts_on || ipa_on;
    const int32_t w_image = ((t.score_enable & CCSIM_PL_IMAGE_LOCALITY) && t.image_score) ? t.w_image : 0;
    const uint32_t stamp_now = (uint32_t)(k + 1);
    long long na_local = 0, ipa_lo = LLONG_MAX, ipa_hi = LLONG_MIN, scored_local = 0;
    for (int32_t i = lo + tid; i < hi; i += blockDim.x) {
      int cls;
      const bool ok = filter_node<RESIDENT>(p, hc, fc, tl, i, cls);
      if (soft) p.feas[i] = ok ? 1 : 0;
      if (ok) {
        int32_t sc = use_cache ? tl.score[i] : -1;
        if (sc < 0) {
          sc = score_node(tl.alloc_cpu[i], tl.alloc_mem[i], tl.nz_cpu[i] + t.least_cpu, tl.nz_mem[i] + t.least_mem,
                          tl.req_cpu[i] + t.bal_cpu, tl.req_mem[i] + t.bal_mem, ws.sw);
          if (w_image) sc += w_image * (int32_t)t.image_score[i];
          if (use_cache || soft) tl.score[i] = sc;
        }
        if (soft) {
          if (na_on) na_local = max(na_local, (long long)node_affinity_raw(p, t, i));
          if (ipa_on) { const long long r = ipa_raw(p, t, i); ipa_lo = min(ipa_lo, r); ipa_hi = max(ipa_hi, r); }
          if (spts_on && !(t.spts_ignored_bit >= 0 && static_bit(p, i, t.spts_ignored_bit))) {
            scored_local++;
            for (int c = 0; c < t.n_spts; c++) {
              if (t.spts[c].hostname) continue;
              const DevCounter &dc = p.counters[t.spts[c].counter];
              const int32_t dom = ws.topo_ptr[dc.topo_col][i];
              __stcg(&p.stamp[c][dom < 0 ? dc.n_domains : dom], stamp_now);   // a missing key reads as the value ""
            }
          }
          continue;
        }
        const unsigned long long key = pack_key(sc, (uint32_t)(p.node_base + i));
        if (ncls == 1) best[0] = key > best[0] ? key : best[0];
        else {
          #pragma unroll
          for (int c = 0; c < CCSIM_MAX_CLASSES; c++) if (c == cls) best[c] = key > best[c] ? key : best[c];
        }
      }
    }
    if (soft) {
      long long spts_lo = LLONG_MAX, spts_hi = 0;
      if (spts_on) {
        // ---- PreScore: sizes of the topologies among the scored nodes -> weights (scoring.go:60-116,294-296) ----
        for (int o = 16; o > 0; o >>= 1) scored_local += __shfl_xor_sync(0xffffffffu, scored_local, o);
        if (lane == 0) ws.red[warp][0] = scored_local;
        __syncthreads();
        if (warp == 0) {
          long long m = (lane < (int)(blockDim.x >> 5)) ? ws.red[lane][0] : 0;
          for (int o = 16; o > 0; o >>= 1) m += __shfl_xor_sync(0xffffffffu, m, o);
          bool dead = false;
          const unsigned long long g = exchange_sum_fenced(p, k, tag, CCSIM_MAX_CLASSES, (unsigned long long)m, lane, cta, dead);
          if (lane == 0) { ws.spts_scored = (long long)g; if (dead) ws.stop = 3; }
        }
        __syncthreads();
        for (int c = 0; c < t.n_spts; c++) {
          long long size = ws.spts_scored;
          if (!t.spts[c].hostname) {
            const int nd1 = p.counters[t.spts[c].counter].n_domains + 1;
            int32_t cnt = 0;
            for (int d = tid; d < nd1; d += blockDim.x) cnt += (__ldcg(&p.stamp[c][d]) == stamp_now);
            for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            if (lane == 0) ws.scratch[warp] = cnt;
            __syncthreads();
            size = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); w++) size += ws.scratch[w];
          }
          if (tid == 0) ws.spts_w[c] = go_log((double)(size + 2));
          __syncthreads();
        }
        for (int32_t i = lo + tid; i < hi; i += blockDim.x) {
          if (!p.feas[i] || (t.spts_ignored_bit >= 0 && static_bit(p, i, t.spts_ignored_bit))) continue;
          const long long r = spts_raw(p, t, i);
          spts_lo = min(spts_lo, r); spts_hi = max(spts_hi, r);
        }
      }
      // ---- extrema over the feasible nodes: block reduction, then one grid-wide exchange of five words ----
      {
        long long v[5] = {na_local, spts_hi, spts_lo == LLONG_MAX ? LLONG_MIN : -spts_lo, ipa_hi, ipa_lo == LLONG_MAX ? LLONG_MIN : -ipa_lo};
        #pragma unroll
        for (int q = 0; q < 5; q++) {
          for (int o = 16; o > 0; o >>= 1) { const long long u = __shfl_xor_sync(0xffffffffu, v[q], o); v[q] = u > v[q] ? u : v[q]; }
          if (lane == 0) ws.red[warp][q] = v[q];
        }
      }
      __syncthreads();
      if (warp == 0) {
        const long long IPA_BIAS = 1ll << 40;
        long long v[5];
        #pragma unroll
        for (int q = 0; q < 5; q++) {
          long long m = (q == 0 || q == 1) ? 0 : LLONG_MIN;
          if (lane < (int)(blockDim.x >> 5)) m = ws.red[lane][q];
          for (int o = 16; o > 0; o >>= 1) { const long long u = __shfl_xor_sync(0xffffffffu, m, o); m = u > m ? u : m; }
          v[q] = m;
        }
        // encode as non-zero unsigned maxima (0 = this CTA has no feasible node)
        unsigned long long e[5];
        e[0] = (unsigned long long)(v[0] + 1);
        e[1] = (v[2] == LLONG_MIN) ? 0ull : (unsigned long long)(v[1] + 1);
        e[2] = (v[2] == LLONG_MIN) ? 0ull : (unsigned long long)((1ll << 43) + v[2]);       // 2^43 - min
        e[3] = (v[4] == LLONG_MIN) ? 0ull : (unsigned long long)(v[3] + IPA_BIAS);
        e[4] = (v[4] == LLONG_MIN) ? 0ull : (unsigned long long)(v[4] + IPA_BIAS);          // bias - min
        bool dead = false;
        exchange_max_n<5>(p, k, tag, CCSIM_MAX_CLASSES + 1, e, lane, cta, dead);
        if (lane == 0) {
          ws.na_max = e[0] ? (long long)e[0] - 1 : 0;
          ws.spts_max = e[1] ? (long long)e[1] - 1 : 0;
          ws.spts_min = e[2] ? (1ll << 43) - (long long)e[2] : LLONG_MAX;
          ws.ipa_max = e[3] ? (long long)e[3] - IPA_BIAS : LLONG_MIN;
          ws.ipa_min = e[4] ? IPA_BIAS - (long long)e[4] : LLONG_MAX;
          if (dead) ws.stop = 3;
        }
      }
      __syncthreads();
      const long long na_max = ws.na_max, pmin = ws.spts_min, pmax = ws.spts_max, imin = ws.ipa_min, imax = ws.ipa_max;
      for (int32_t i = lo + tid; i < hi; i += blockDim.x) {
        if (!p.feas[i]) continue;
        long long total = tl.score[i];
        if (na_on) {
          const long long raw = node_affinity_raw(p, t, i);
          total += (long long)t.w_node_affinity * (na_max == 0 ? raw : 100 * raw / na_max);
        }
        if (spts_on && !(t.spts_ignored_bit >= 0 && static_bit(p, i, t.spts_ignored_bit))) {
          const long long r = spts_raw(p, t, i);
          total += (long long)t.w_pts * (pmax == 0 ? 100 : 100 * (pmax + pmin - r) / pmax);
        }
        if (ipa_on && imax > imin) {
          const long long r = ipa_raw(p, t, i);
          const double f = __dmul_rn(100.0, __ddiv_rn((double)(r - imin), (double)(imax - imin)));
          total += (long long)t.w_ipa * __double2ll_rz(f);
        }
        const unsigned long long key = pack_key(total, (uint32_t)(p.node_base + i));
        if (ncls == 1) best[0] = key > best[0] ? key : best[0];
        else {
          const int cls = __popcll(tl.taint0[i] & hc.prefer0);
          #pragma unroll
          for (int c = 0; c < CCSIM_MAX_CLASSES; c++) if (c == cls) best[c] = key > best[c] ? key : best[c];
        }
      }
    }
    for (int c = 0; c < ncls; c++) {
      unsigned long long v = 0ull;
      #pragma unroll
      for (int q = 0; q < CCSIM_MAX_CLASSES; q++) if (q == c) v = best[q];
      v = warp_max_u64(v);
      if (lane == 0) ws.warp_best[warp][c] = v;
    }
    PH_MARK(0);
    __syncthreads();                                                    // S1
    PH_MARK(1);

    if (warp == 0) {
      const unsigned long long tagbits = (unsigned long long)tag << KEY_TAG_SHIFT;
      unsigned long long *myslots = p.slots + ((size_t)(k & 1) * CCSIM_MAX_GRID + cta) * SLOT_STRIDE;
      // CTA arg-max per class, published as one tagged word each
      for (int c = 0; c < ncls; c++) {
        unsigned long long v = (lane < (int)(blockDim.x >> 5)) ? ws.warp_best[lane][c] : 0ull;
        v = warp_max_u64(v);
        if (lane == 0) st_slot(&myslots[c], v | tagbits);
      }
      PH_MARK(2);
      // gather every CTA's word: all of a lane's loads are in flight together; retry until every tag is this wave's
      const unsigned long long *all = p.slots + (size_t)(k & 1) * CCSIM_MAX_GRID * SLOT_STRIDE;
      unsigned long long cbest[CCSIM_MAX_CLASSES];
      bool dead = false;
      for (int c = 0; c < ncls; c++) {
        unsigned long long v[CCSIM_MAX_GRID / 32];
        unsigned spins = 0;
        bool pending;
        do {
          pending = false;
          #pragma unroll
          for (int q = 0; q < CCSIM_MAX_GRID / 32; q++) {
            const int b = lane + 32 * q;
            v[q] = (b < p.grid) ? ld_slot(&all[(size_t)b * SLOT_STRIDE + c]) : tagbits;
          }
          #pragma unroll
          for (int q = 0; q < CCSIM_MAX_GRID / 32; q++) pending |= ((uint32_t)(v[q] >> KEY_TAG_SHIFT) != tag);
          if (++spins > WATCHDOG_SPINS) { dead = true; break; }
        } while (__any_sync(0xffffffffu, pending));
        unsigned long long m = 0ull;
        #pragma unroll
        for (int q = 0; q < CCSIM_MAX_GRID / 32; q++) { const unsigned long long b = v[q] & KEY_BODY_MASK; m = b > m ? b : m; }
        cbest[c] = warp_max_u64(m);
      }
      dead = __any_sync(0xffffffffu, dead);
      if (p.world > 1 && !dead) dead = cross_gpu_exchange(p, k, tag, ncls, cbest, lane, cta);
      PH_MARK(3);
      // prioritizeNodes + selectHost over the class winners (schedule_one.go:776-941)
      unsigned long long wkey = cbest[0];
      if (ncls > 1 || (t.score_enable & CCSIM_PL_TAINT_TOLERATION)) {
        int maxraw = 0;
        for (int c = 0; c < ncls; c++) if (cbest[c] != 0ull) maxraw = c;
        wkey = 0ull;
        for (int c = 0; c < ncls; c++) {
          if (cbest[c] == 0ull) continue;
          int64_t total = key_score(cbest[c]);
          if (t.score_enable & CCSIM_PL_TAINT_TOLERATION) total += (int64_t)t.w_taint * taint_norm(c, maxraw);
          const unsigned long long kk = pack_key(total, key_index(cbest[c]));
          wkey = kk > wkey ? kk : wkey;
        }
      }
      if (lane == 0) {
        if (dead) { ws.stop = 3; ws.winner = -1; }
        else if (wkey == 0ull) { ws.stop = 1; ws.winner = -1; }
        else ws.winner = (int32_t)key_index(wkey);
      }
      // ---- commit (assume -> AssumePod -> NodeInfo.update(+1): schedule_one.go:967-984, types.go:409-427) ----
      if (!dead && wkey != 0ull) {
        const int32_t g = (int32_t)key_index(wkey);
        const int32_t w = g - p.node_base;
        const bool mine = (w >= lo && w < hi);
        if (mine && lane == 31) {
          const long long rc = tl.req_cpu[w] + t.req_cpu, rm = tl.req_mem[w] + t.req_mem;
          const long long zc = tl.nz_cpu[w] + t.nz_cpu, zm = tl.nz_mem[w] + t.nz_mem;
          const int32_t np = tl.npods[w] + 1;
          tl.req_cpu[w] = rc; tl.req_mem[w] = rm; tl.nz_cpu[w] = zc; tl.nz_mem[w] = zm; tl.npods[w] = np;
          tl.score[w] = -1;    // this node's NodeInfo generation changed
          if (RESIDENT) {      // write through: the global columns stay the authoritative snapshot-after-run
            tl.free_cpu[w] = tl.alloc_cpu[w] - rc; tl.free_mem[w] = tl.alloc_mem[w] - rm; tl.free_pods[w] = tl.alloc_pods[w] - np;
            p.req_cpu[w] = rc; p.req_mem[w] = rm; p.nz_cpu[w] = zc; p.nz_mem[w] = zm; p.npods[w] = np;
          }
          if (t.req_eph != 0) p.req_eph[w] += t.req_eph;
          for (int q = 0; q < p.n_scalars; q++) if (t.req_scalar[q] != 0) p.req_scalar[q][w] += t.req_scalar[q];
          if (p.placed_mask) p.placed_mask[w] |= 1ull << ti;
          // ClusterCapacityBinder.Bind + postBindHook: record pod k -> node (plugin.go:34-53; simulator.go:297-312)
          if (k < p.pod_cap) p.pod_node[k] = g; else ws.stop = 3;
        }
        if (p.world > 1 && !mine && cta == 0 && lane == 31) {   // sharded run: every rank keeps the whole pod -> node sequence
          const bool local = (w >= 0 && w < p.n);
          if (!local) { if (k < p.pod_cap) p.pod_node[k] = g; else ws.stop = 3; }
        }
        // per-domain counters: every CTA applies the same update to its own replica, one lane per counter
        // (the next cycle's PreFilter recount would see this clone: podtopologyspread/filtering.go:255-289,
        //  interpodaffinity/filtering.go:234-271)
        if (lane < p.n_counters) {
          const int j = lane;
          const CommitInfo ci = ws.cinfo[j];
          if (ci.inc && !(ci.elig_bit >= 0 && !static_bit(p, w, ci.elig_bit))) {   // elig_bit only exists on single-GPU runs: w is a local index
            if (ci.local) {
              if (mine) {
                const int32_t nv = ws.cnt_ptr[j][w] + ci.inc;
                ws.cnt_ptr[j][w] = nv;
                if (RESIDENT) p.counters[j].work[w] = nv;
              }
              if (ci.is_aff) { atomicAdd((unsigned long long *)&ws.aff_total, (unsigned long long)ci.inc); ws.dirty = 1; }
            } else {
              // the winner's domain id: from this CTA's tile if it owns the node, else from the global column (L2)
              const int32_t dom = mine ? ci.ltopo[w] : ci.gtopo[g];   // gtopo: whole-cluster column, global index
              if (dom >= 0) {
                int32_t *cnt = ws.cnt_ptr[j];
                const int32_t old = cnt[dom];
                cnt[dom] = old + ci.inc;
                if (ci.is_aff) { atomicAdd((unsigned long long *)&ws.aff_total, (unsigned long long)ci.inc); ws.dirty = 1; }
                if (ci.pts_idx >= 0 && dom < ci.n_present && old == ws.ptsmin[ci.pts_idx]) ws.ptsnum[ci.pts_idx] -= 1;
              }
            }
          }
        }
      }
    }
    PH_MARK(4);
    __syncthreads();                                                    // S2
    PH_MARK(5);
    if (ws.stop) break;
    // a PTS minimum whose last domain moved up: recount (rare: once per n_present commits at that level)
    for (int c = 0; c < t.n_pts; c++)
      if (!t.pts[c].min_zero && ws.ptsnum[c] <= 0 && p.counters[t.pts[c].counter].n_present > 0) pts_recount(p, c);
    wtag = (wtag == 4095u) ? 1u : wtag + 1u;
    tag = (p.epoch << 12) | wtag;
    ti = (ti + 1 == p.n_templates) ? 0 : ti + 1;
  }

  // ---- epilogue ----
  if (cta == 0) {
    for (int j = 0; j < p.n_counters; j++) {
      const DevCounter &dc = p.counters[j];
      if (dc.topo_col < 0) continue;
      const int32_t *src = ws.cnt_ptr[j];
      for (int d = tid; d < dc.n_domains; d += blockDim.x) p.final_cnt[p.final_off[j] + d] = src[d];
    }
    if (tid == 0) {
      DevOut *o = p.out;
      o->placed = k;
      o->stop_code = limit_hit ? CCSIM_STOP_LIMIT_REACHED : CCSIM_STOP_UNSCHEDULABLE;
      o->error = (ws.stop == 3) ? 1 : 0;
      o->waves = limit_hit ? k : k + 1;
      o->evals = o->waves * (long long)p.n;
      for (int c = 0; c < CCSIM_MAX_PTS; c++) o->ptsmin[c] = ws.ptsmin[c];
      o->aff_total = ws.aff_total;
#ifdef CCSIM_PHASE_TIMERS
      for (int q = 0; q < 8; q++) o->phase_cycles[q] = ph[q];
#endif
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Terminal diagnosis: FitError histogram of the pod that did not fit (framework/types.go:787-838) and the status codes
// the DefaultPreemption PostFilter groups nodes by (preemption/preemption.go:309-331). Runs once per Run.
// ------------------------------------------------------------------------------------------------------------------
__global__ void ccsim_diag_kernel(const DevParams p, int tmpl_index) {
  const ccsim_template &t = p.templates[tmpl_index];
  DevOut *o = p.out;
  const int32_t n = p.n;
  for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int st = ST_OK;
    int reasons[8 + CCSIM_MAX_SCALARS]; int nr = 0;
    const uint64_t taint0 = p.taint_mask[i];
    do {
      if ((t.flags & CCSIM_TF_PREFILTER_NODES) && t.prefilter_bit >= 0) {
        const int b = t.prefilter_bit;
        if (!((p.static_mask[(size_t)(b >> 6) * n + i] >> (b & 63)) & 1ull)) { reasons[nr++] = CCSIM_R_PREFILTER_NODES; st = ST_UNRESOLVABLE; break; }
      }
      if ((t.filter_enable & CCSIM_PL_NODE_UNSCHEDULABLE) && ((taint0 >> CCSIM_TAINT_UNSCHEDULABLE_BIT) & 1ull) &&
          !(t.flags & CCSIM_TF_TOLERATES_UNSCHEDULABLE)) { reasons[nr++] = CCSIM_R_UNSCHEDULABLE; st = ST_UNRESOLVABLE; break; }
      if ((t.filter_enable & CCSIM_PL_NODE_NAME) && t.nodename_idx >= 0 && t.nodename_idx != p.node_base + i) {
        reasons[nr++] = CCSIM_R_NODE_NAME; st = ST_UNRESOLVABLE; break; }
      if (t.filter_enable & CCSIM_PL_TAINT_TOLERATION) {
        uint64_t untol_any = 0; int low = -1;
        for (int w = 0; w < p.taint_words; w++) {
          const uint64_t m = p.taint_mask[(size_t)w * n + i] & p.taint_nosched[w] & ~t.tol_nosched[w];
          if (m && low < 0) low = 64 * w + __ffsll((long long)m) - 1;
          untol_any |= m;
        }
        if (untol_any) {
          int id = -1;
          if (p.taint_list_off) {   // first untolerated taint in node.Spec.Taints order (corev1/helpers.go:78-101)
            for (int32_t q = p.taint_list_off[i]; q < p.taint_list_off[i + 1]; q++) {
              const int tid = p.taint_list[q];
              if (((p.taint_nosched[tid >> 6] >> (tid & 63)) & 1ull) && !((t.tol_nosched[tid >> 6] >> (tid & 63)) & 1ull)) { id = tid; break; }
            }
          }
          if (id < 0) id = low;
          reasons[nr++] = CCSIM_R_TAINT0 + id; st = ST_UNRESOLVABLE; break;
        }
      }
      uint64_t sw[CCSIM_MAX_STATIC_WORDS];
      for (int w = 0; w < CCSIM_MAX_STATIC_WORDS; w++) sw[w] = (w < p.static_words) ? p.static_mask[(size_t)w * n + i] : 0ull;
      if ((t.filter_enable & CCSIM_PL_NODE_AFFINITY) && (t.flags & (CCSIM_TF_HAS_NODE_SELECTOR | CCSIM_TF_HAS_AFFINITY_TERMS))) {
        bool m = true;
        for (int w = 0; w < CCSIM_MAX_STATIC_WORDS; w++) m &= ((sw[w] & t.sel_mask[w]) == t.sel_mask[w]);
        if (m && (t.flags & CCSIM_TF_HAS_AFFINITY_TERMS)) {
          bool any = false;
          for (int k = 0; k < t.n_aff_terms; k++) {
            bool tm = true;
            for (int w = 0; w < CCSIM_MAX_STATIC_WORDS; w++) tm &= ((sw[w] & t.aff_term_mask[k][w]) == t.aff_term_mask[k][w]);
            any |= tm;
          }
          m = any;
        }
        if (!m) { reasons[nr++] = CCSIM_R_NODE_AFFINITY; st = ST_UNRESOLVABLE; break; }
      }
      if ((t.filter_enable & CCSIM_PL_NODE_PORTS) && (t.flags & CCSIM_TF_HAS_HOST_PORTS)) {
        uint64_t c = 0;
        for (int w = 0; w < CCSIM_MAX_STATIC_WORDS; w++) c |= sw[w] & t.port_static_mask[w];
        if (p.placed_mask && (p.placed_mask[i] & t.port_tmpl_conflict)) c = 1;
        if (c) { reasons[nr++] = CCSIM_R_NODE_PORTS; st = ST_UNSCHEDULABLE; break; }
      }
      if (t.filter_enable & CCSIM_PL_FIT) {
        bool fail = false, unres = false;
        if (p.npods[i] + 1 > p.alloc_pods[i]) { fail = true; reasons[nr++] = CCSIM_R_TOO_MANY_PODS; }
        if (!(t.flags & CCSIM_TF_FIT_ALL_ZERO)) {
          if (t.req_cpu > 0 && t.req_cpu > p.alloc_cpu[i] - p.req_cpu[i]) { fail = true; unres |= t.req_cpu > p.alloc_cpu[i]; reasons[nr++] = CCSIM_R_INSUFFICIENT_CPU; }
          if (t.req_mem > 0 && t.req_mem > p.alloc_mem[i] - p.req_mem[i]) { fail = true; unres |= t.req_mem > p.alloc_mem[i]; reasons[nr++] = CCSIM_R_INSUFFICIENT_MEMORY; }
          if (t.req_eph > 0 && t.req_eph > p.alloc_eph[i] - p.req_eph[i]) { fail = true; unres |= t.req_eph > p.alloc_eph[i]; reasons[nr++] = CCSIM_R_INSUFFICIENT_EPHEMERAL; }
          for (int k = 0; k < p.n_scalars; k++) {
            const int64_t q = t.req_scalar[k];
            if (q == 0) continue;
            if (q > p.alloc_scalar[k][i] - p.req_scalar[k][i]) { fail = true; unres |= q > p.alloc_scalar[k][i]; reasons[nr++] = CCSIM_R_SCALAR0 + k; }
          }
        }
        if (fail) { st = unres ? ST_UNRESOLVABLE : ST_UNSCHEDULABLE; break; }
      }
      if (t.filter_enable & CCSIM_PL_POD_TOPOLOGY_SPREAD) {
        bool done = false;
        for (int c = 0; c < t.n_pts && !done; c++) {
          const ccsim_pts &pc = t.pts[c];
          const DevCounter &dc = p.counters[pc.counter];
          const int32_t dom = dc.topo_col < 0 ? i : p.topo[dc.topo_col][i];
          if (dom < 0) { reasons[nr++] = CCSIM_R_PTS_MISSING_LABEL; st = ST_UNRESOLVABLE; done = true; break; }
          const int32_t cv = dc.topo_col < 0 ? dc.work[i] : p.final_cnt[p.final_off[pc.counter] + dom];
          const long long skew = (long long)cv + pc.self_match - (long long)o->ptsmin[c];
          if (skew > pc.max_skew) { reasons[nr++] = CCSIM_R_PTS_SKEW; st = ST_UNSCHEDULABLE; done = true; }
        }
        if (done) break;
      }
      if (t.filter_enable & CCSIM_PL_INTER_POD_AFFINITY) {
        bool pods_exist = true, missing = false;
        for (int a = 0; a < t.n_aff; a++) {
          const DevCounter &dc = p.counters[t.aff_counter[a]];
          const int32_t dom = dc.topo_col < 0 ? i : p.topo[dc.topo_col][i];
          if (dom < 0) { missing = true; break; }
          const int32_t cv = dc.topo_col < 0 ? dc.work[i] : p.final_cnt[p.final_off[t.aff_counter[a]] + dom];
          if (cv <= 0) pods_exist = false;
        }
        if (t.n_aff > 0 && (missing || (!pods_exist && !(o->aff_total == 0 && (t.flags & CCSIM_TF_AFF_SELF_MATCH_ALL))))) {
          reasons[nr++] = CCSIM_R_IPA_AFFINITY; st = ST_UNRESOLVABLE; break; }
        bool anti = false;
        for (int a = 0; a < t.n_anti; a++) {
          const DevCounter &dc = p.counters[t.anti_counter[a]];
          const int32_t dom = dc.topo_col < 0 ? i : p.topo[dc.topo_col][i];
          if (dom < 0) continue;
          const int32_t cv = dc.topo_col < 0 ? dc.work[i] : p.final_cnt[p.final_off[t.anti_counter[a]] + dom];
          if (cv > 0) anti = true;
        }
        if (anti) { reasons[nr++] = CCSIM_R_IPA_ANTI_AFFINITY; st = ST_UNSCHEDULABLE; break; }
        uint64_t c = 0;
        for (int w = 0; w < CCSIM_MAX_STATIC_WORDS; w++) c |= sw[w] & t.existing_anti_mask[w];
        if (c) { reasons[nr++] = CCSIM_R_IPA_EXISTING_ANTI; st = ST_UNSCHEDULABLE; break; }
      }
    } while (0);
    for (int q = 0; q < nr; q++) atomicAdd(&o->reason_hist[reasons[q]], 1ull);
    if (st == ST_UNSCHEDULABLE) atomicAdd(&o->preempt_no_victims, 1ull);
    atomicAdd(&o->n_diag, 1ull);
  }
}

// per-node replica counts of template t and first-placement index (report.go:146-180 without the O(P*nodes) scan)
__global__ void ccsim_count_kernel(const int32_t *pod_node, long long placed, int n_templates, int t,
                                   int32_t *counts, unsigned long long *first) {
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < placed; k += (long long)gridDim.x * blockDim.x) {
    if ((int)(k % n_templates) != t) continue;
    const int32_t w = pod_node[k];
    atomicAdd(&counts[w], 1);
    atomicMin(&first[w], (unsigned long long)k);
  }
}

// ccsim_debug_node_scores: score_node (and its two parts) of every node, `clones` pods of the template after the snapshot
__global__ void ccsim_debug_score_kernel(int32_t n, const int64_t *a_cpu, const int64_t *a_mem, const int64_t *r_cpu, const int64_t *r_mem,
                                         const int64_t *z_cpu, const int64_t *z_mem, const ccsim_template t, ScoreWeights sw, int64_t clones,
                                         int64_t *total, int64_t *least, int64_t *balanced) {
  for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int64_t lq_cpu = z_cpu[i] + clones * t.nz_cpu + t.least_cpu, lq_mem = z_mem[i] + clones * t.nz_mem + t.least_mem;
    const int64_t bq_cpu = r_cpu[i] + clones * t.req_cpu + t.bal_cpu, bq_mem = r_mem[i] + clones * t.req_mem + t.bal_mem;
    total[i] = score_node(a_cpu[i], a_mem[i], lq_cpu, lq_mem, bq_cpu, bq_mem, sw);
    least[i] = score_least(a_cpu[i], a_mem[i], lq_cpu, lq_mem, sw.least_w_cpu, sw.least_w_mem);
    balanced[i] = score_balanced(a_cpu[i], a_mem[i], bq_cpu, bq_mem);
  }
}

__global__ void ccsim_flush_kernel(unsigned long long *buf, size_t n, unsigned long long v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) buf[i] = v + i;
}

// ------------------------------------------------------------------------------------------------------------------
// host side of the C-ABI
// ------------------------------------------------------------------------------------------------------------------
struct RunPlan {      // what run_prepare decided, consumed by the launch
  bool valid = false, empty = false;
  int64_t max_pods = 0;
  DevParams p; LeanParams lp; MultiParams mp; StreamParams sp;
  const void *kern = nullptr; int grid = 0, block = 0; size_t smem = 0;
  bool stream = false, multi = false, batched = false, lean = false, resident = false;
  int64_t variant = 0;   // CCSIM_KV_* bits of the instantiation (ccsim_run_stats out[0] above the engine code)
};

struct ccsim_handle {
  ccsim_config cfg;
  int sm_count = 0;
  size_t l2_bytes = 0;
  size_t smem_optin = 0;
  int last_resident = 0;
  int last_lean = 0;
  int last_batched = 0;
  int last_multi = 0;
  int last_stream = 0;
  std::vector<void *> stream_allocs;                    // padded streaming columns + per-template score memo (ccsim_stream.cuh)
  uint64_t taint_or0 = 0;                               // OR over the nodes of taint word 0
  std::vector<std::pair<void *, size_t>> block_cache;   // freed device blocks kept for reuse (exact size match)
  std::map<void *, size_t> block_bytes;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;
  int64_t launches = 0;
  // snapshot
  bool have_nodes = false, have_templates = false;
  int32_t n = 0, n_global = 0, node_base = 0;
  ccsim_nodes meta;            // scalar members only
  std::vector<void *> allocs;  // every device allocation, freed in destroy / reload
  std::vector<void *> tmpl_allocs;
  // device columns: snapshot copies and working copies of the mutable ones
  int64_t *d_alloc_cpu = nullptr, *d_alloc_mem = nullptr, *d_alloc_eph = nullptr;
  int32_t *d_alloc_pods = nullptr;
  int64_t *d_alloc_scalar[CCSIM_MAX_SCALARS] = {};
  uint64_t *d_taint = nullptr, *d_static = nullptr;
  int32_t *d_topo[CCSIM_MAX_TOPO_COLS] = {};
  int64_t *s_req_cpu = nullptr, *s_req_mem = nullptr, *s_req_eph = nullptr, *s_nz_cpu = nullptr, *s_nz_mem = nullptr;
  int32_t *s_npods = nullptr;
  int64_t *s_req_scalar[CCSIM_MAX_SCALARS] = {};
  int64_t *w_req_cpu = nullptr, *w_req_mem = nullptr, *w_req_eph = nullptr, *w_nz_cpu = nullptr, *w_nz_mem = nullptr;
  int32_t *w_npods = nullptr;
  int64_t *w_req_scalar[CCSIM_MAX_SCALARS] = {};
  uint64_t *w_placed = nullptr;
  int32_t *w_score = nullptr;
  uint8_t *w_feas = nullptr;
  uint32_t *d_stamp[CCSIM_MAX_PTS] = {nullptr};
  size_t stamp_len[CCSIM_MAX_PTS] = {0};
  int32_t *d_taint_off = nullptr; uint8_t *d_taint_list = nullptr;
  int64_t pod_bound = 0;       // sum over nodes of max(0, alloc_pods - npods): no run can place more
  int max_prefer_pop = 0;      // max over nodes of popcount(taint & prefer): number of normalisation classes - 1
  // templates
  int32_t n_templates = 0, n_counters = 0;
  std::vector<ccsim_template> h_templates;
  ccsim_template *d_templates = nullptr;
  DevCounter counters[CCSIM_MAX_COUNTERS];
  int32_t *d_final_cnt = nullptr; int32_t final_off[CCSIM_MAX_COUNTERS] = {}; int32_t final_total = 0;
  int32_t smem_cnt_ints = 0;
  // run state
  int grid = 0;
  unsigned long long *d_slots = nullptr;
  unsigned long long *d_xslots = nullptr;                 // cross-GPU exchange buffer (exported over CUDA IPC)
  unsigned long long *x_peer[CCSIM_MAX_WORLD] = {};       // every rank's buffer as mapped here
  bool peers_ready = false;
  bool peers_local = false;                               // peers are plain pointers of this process (nothing to close)
  uint32_t epoch = 0;
  uint32_t xwave0 = 0;                                    // exchanges of earlier sharded runs (buffer parity continues across runs)
  int64_t last_stat[16] = {};                             // ccsim_run_stats
  RunPlan plan;
  int32_t *d_topo_full[CCSIM_MAX_TOPO_COLS] = {};
  int32_t *d_pod_node = nullptr; int64_t pod_cap = 0;
  std::vector<int32_t> h_pod_node;
  DevOut *d_out = nullptr;
  DevParams *d_params = nullptr;
  int64_t last_placed = 0;
  void *d_flush = nullptr; size_t flush_bytes = 0;
};

static std::string g_create_err;

static int fail(ccsim_handle *h, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  if (h) h->err = buf; else g_create_err = buf;
  return code;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(h, CCSIM_ECUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

// Device blocks are recycled per handle: ccsim_load_nodes / ccsim_set_templates are called once per analysis by the host side,
// usually with the same shapes as the last time, and cudaMalloc/cudaFree are slow, synchronising driver calls.
template <typename T> static int dev_alloc(ccsim_handle *h, std::vector<void *> &pool, T **out, size_t count) {
  void *p = nullptr;
  size_t bytes = (count ? count : 1) * sizeof(T);
  for (size_t i = 0; i < h->block_cache.size(); i++)
    if (h->block_cache[i].second == bytes) { p = h->block_cache[i].first; h->block_cache.erase(h->block_cache.begin() + i); break; }
  if (!p) {
    // stream-ordered allocation: no device-wide synchronisation (a host that drives several ranks from one process may have a
    // peer's persistent kernel running, waiting for this rank's kernel to start)
    cudaError_t e = cudaMallocAsync(&p, bytes, h->stream);
    if (e != cudaSuccess) return fail(h, CCSIM_ENOMEM, "cudaMallocAsync(%zu): %s", bytes, cudaGetErrorString(e));
  }
  pool.push_back(p);
  h->block_bytes[p] = bytes;
  *out = (T *)p;
  return 0;
}
template <typename T> static int dev_upload(ccsim_handle *h, std::vector<void *> &pool, T **out, const T *src, size_t count) {
  int rc = dev_alloc(h, pool, out, count);
  if (rc) return rc;
  if (count) CK(cudaMemcpyAsync(*out, src, count * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  return 0;
}
// blocks of a pool go back to the handle's cache (the stream is drained first: they may still be in use)
static void free_pool(ccsim_handle *h, std::vector<void *> &pool) {
  if (pool.empty()) return;
  cudaStreamSynchronize(h->stream);
  size_t cached = 0;
  for (auto &b : h->block_cache) cached += b.second;
  for (void *p : pool) {
    const size_t bytes = h->block_bytes[p];
    if (cached + bytes <= ((size_t)1 << 31)) { h->block_cache.push_back({p, bytes}); cached += bytes; }   // keep at most 2 GiB around
    else { cudaFreeAsync(p, h->stream); h->block_bytes.erase(p); }
  }
  pool.clear();
}
static void drop_cache(ccsim_handle *h) {
  for (auto &b : h->block_cache) cudaFreeAsync(b.first, h->stream);
  cudaStreamSynchronize(h->stream);
  h->block_cache.clear(); h->block_bytes.clear();
}

extern "C" int ccsim_abi_version(void) { return CCSIM_ABI_VERSION; }

extern "C" const char *ccsim_last_error(const ccsim_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

extern "C" int ccsim_create(const ccsim_config *cfg, ccsim_handle **out) {
  ccsim_handle *h = nullptr;
  if (!cfg || !out) return fail(h, CCSIM_EINVAL, "null argument");
  if (cfg->abi_version != CCSIM_ABI_VERSION) return fail(h, CCSIM_EINVAL, "abi_version %d != %d", cfg->abi_version, CCSIM_ABI_VERSION);
  if (cfg->world < 1 || cfg->world > CCSIM_MAX_WORLD || cfg->rank < 0 || cfg->rank >= cfg->world) return fail(h, CCSIM_EINVAL, "bad rank/world");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(h, CCSIM_ECUDA, "no CUDA device: %s (libccsim has no CPU fallback)", cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(h, CCSIM_EINVAL, "device %d out of range (%d)", cfg->device, ndev);
  h = new ccsim_handle();
  h->cfg = *cfg;
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(cfg->device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess) {
    fail(nullptr, CCSIM_ECUDA, "cudaSetDevice/GetDeviceProperties: %s", cudaGetErrorString(e));
    delete h; return CCSIM_ECUDA;
  }
  if (!prop.cooperativeLaunch) { fail(nullptr, CCSIM_EUNSUPPORTED, "device lacks cooperative launch"); delete h; return CCSIM_EUNSUPPORTED; }
  h->sm_count = prop.multiProcessorCount;
  h->l2_bytes = (size_t)prop.l2CacheSize;
  {   // the stream-ordered allocator keeps what it has mapped (default: everything goes back to the driver at the next synchronize,
      // and every analysis would map its snapshot's memory again)
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, cfg->device) == cudaSuccess) { uint64_t keep = UINT64_MAX; cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep); }
  }
  cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  cudaEventCreate(&h->ev0); cudaEventCreate(&h->ev1);
  cudaMalloc((void **)&h->d_out, sizeof(DevOut));
  cudaMalloc((void **)&h->d_params, sizeof(DevParams));
  cudaMalloc((void **)&h->d_slots, sizeof(unsigned long long) * 2 * CCSIM_MAX_GRID * SLOT_STRIDE);
  cudaMalloc((void **)&h->d_xslots, sizeof(unsigned long long) * XSLOTS_TOTAL_WORDS);     // winner words (lean kernel) + candidate lines (multi-commit)
  cudaMemset(h->d_xslots, 0, sizeof(unsigned long long) * XSLOTS_TOTAL_WORDS);
  h->x_peer[cfg->rank] = h->d_xslots;
  h->smem_optin = (size_t)prop.sharedMemPerBlockOptin;
  cudaFuncSetAttribute(ccsim_wave_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)(h->smem_optin - sizeof(WaveShared) - 1024));
  cudaFuncSetAttribute(ccsim_wave_lean_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)(h->smem_optin - sizeof(LeanShared) - 1024));
  cudaFuncSetAttribute(ccsim_wave_lean_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)(h->smem_optin - sizeof(LeanShared) - 1024));
  cudaFuncSetAttribute(ccsim_wave_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)(h->smem_optin - sizeof(LeanShared) - sizeof(BatchShared) - 1024));
  cudaFuncSetAttribute(ccsim_wave_multi_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)(h->smem_optin - sizeof(LeanShared) - sizeof(MultiShared) - 1024));
  cudaFuncSetAttribute(ccsim_wave_multi_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)(h->smem_optin - sizeof(LeanShared) - sizeof(MultiShared) - 1024));
  cudaFuncSetAttribute(ccsim_wave_stream_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(STREAM_STAGES * STREAM_TILE * 24 + 128));
  cudaFuncSetAttribute(ccsim_wave_stream_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(STREAM_STAGES * STREAM_TILE * 40 + 128));
  cudaFuncSetAttribute(ccsim_wave_stream_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(h->smem_optin - sizeof(StreamShared) - 1024));
  cudaFuncSetAttribute(ccsim_wave_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)(SMEM_CNT_MAX_INTS * sizeof(int32_t) + 16));
  *out = h;
  return CCSIM_OK;
}

extern "C" void ccsim_destroy(ccsim_handle *h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  cudaStreamSynchronize(h->stream);
  free_pool(h, h->allocs); free_pool(h, h->tmpl_allocs); free_pool(h, h->stream_allocs); drop_cache(h);
  for (int r = 0; r < CCSIM_MAX_WORLD; r++) if (h->x_peer[r] && r != h->cfg.rank && !h->peers_local) cudaIpcCloseMemHandle(h->x_peer[r]);
  cudaFree(h->d_xslots);
  if (h->d_pod_node) { cudaFreeAsync(h->d_pod_node, h->stream); cudaStreamSynchronize(h->stream); }
  cudaFree(h->d_out); cudaFree(h->d_params); cudaFree(h->d_slots); cudaFree(h->d_flush);
  cudaEventDestroy(h->ev0); cudaEventDestroy(h->ev1);
  cudaStreamDestroy(h->stream);
  delete h;
}

extern "C" int ccsim_load_nodes(ccsim_handle *h, const ccsim_nodes *nd) {
  if (!h || !nd) return fail(h, CCSIM_EINVAL, "null argument");
  if (nd->n_nodes < 0 || nd->n_scalars < 0 || nd->n_scalars > CCSIM_MAX_SCALARS || nd->taint_words < 1 ||
      nd->taint_words > CCSIM_MAX_TAINT_WORDS || nd->static_words < 0 || nd->static_words > CCSIM_MAX_STATIC_WORDS ||
      nd->n_topo_cols < 0 || nd->n_topo_cols > CCSIM_MAX_TOPO_COLS)
    return fail(h, CCSIM_EINVAL, "ccsim_nodes dimensions out of range");
  CK(cudaSetDevice(h->cfg.device));
  free_pool(h, h->allocs);
  h->have_nodes = false; h->have_templates = false; h->plan.valid = false;
  const int32_t N = nd->n_nodes;
  // node-axis shard of this rank (SURVEY.md §8e): contiguous block of the nodeTree order
  const int32_t per = (N + h->cfg.world - 1) / h->cfg.world;
  const int32_t lo = std::min<int64_t>((int64_t)per * h->cfg.rank, N), hi = std::min<int64_t>((int64_t)lo + per, N);
  const int32_t n = hi - lo;
  // every rank of a sharded run takes part in the per-wave exchange: a rank without nodes would never launch the kernel and its
  // peers would wait for its words forever
  if (h->cfg.world > 1 && N > 0 && (int64_t)per * (h->cfg.world - 1) >= N)
    return fail(h, CCSIM_EUNSUPPORTED, "sharded run: %d nodes over %d ranks leaves a rank without nodes (use fewer ranks)", N, h->cfg.world);
  h->n = n; h->n_global = N; h->node_base = lo;
  h->meta = *nd;
  int rc;
#define UP(dst, src, T) if ((rc = dev_upload<T>(h, h->allocs, &h->dst, (src) ? (src) + lo : (const T *)nullptr, (src) ? (size_t)n : 0))) return rc
  if (N > 0 && (!nd->alloc_cpu || !nd->alloc_mem || !nd->alloc_eph || !nd->alloc_pods || !nd->req_cpu || !nd->req_mem ||
                !nd->req_eph || !nd->npods || !nd->nz_cpu || !nd->nz_mem || !nd->taint_mask))
    return fail(h, CCSIM_EINVAL, "null core column");
  UP(d_alloc_cpu, nd->alloc_cpu, int64_t); UP(d_alloc_mem, nd->alloc_mem, int64_t); UP(d_alloc_eph, nd->alloc_eph, int64_t);
  UP(d_alloc_pods, nd->alloc_pods, int32_t);
  UP(s_req_cpu, nd->req_cpu, int64_t); UP(s_req_mem, nd->req_mem, int64_t); UP(s_req_eph, nd->req_eph, int64_t);
  UP(s_nz_cpu, nd->nz_cpu, int64_t); UP(s_nz_mem, nd->nz_mem, int64_t); UP(s_npods, nd->npods, int32_t);
  for (int k = 0; k < nd->n_scalars; k++) {
    if (!nd->alloc_scalar[k] || !nd->req_scalar[k]) return fail(h, CCSIM_EINVAL, "null scalar column %d", k);
    UP(d_alloc_scalar[k], nd->alloc_scalar[k], int64_t); UP(s_req_scalar[k], nd->req_scalar[k], int64_t);
  }
#undef UP
  // word-major bitmask columns: copy the shard slice of each word
  if ((rc = dev_alloc(h, h->allocs, &h->d_taint, (size_t)nd->taint_words * n))) return rc;
  for (int w = 0; w < nd->taint_words && n; w++)
    CK(cudaMemcpyAsync(h->d_taint + (size_t)w * n, nd->taint_mask + (size_t)w * N + lo, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
  if ((rc = dev_alloc(h, h->allocs, &h->d_static, (size_t)nd->static_words * n))) return rc;
  if (nd->static_words && N > 0 && !nd->static_mask) return fail(h, CCSIM_EINVAL, "null static_mask");
  for (int w = 0; w < nd->static_words && n; w++)
    CK(cudaMemcpyAsync(h->d_static + (size_t)w * n, nd->static_mask + (size_t)w * N + lo, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
  for (int k = 0; k < nd->n_topo_cols; k++) {
    if (!nd->topo[k] && N > 0) return fail(h, CCSIM_EINVAL, "null topo column %d", k);
    if ((rc = dev_upload<int32_t>(h, h->allocs, &h->d_topo[k], nd->topo[k] ? nd->topo[k] + lo : nullptr, (size_t)n))) return rc;
    h->d_topo_full[k] = h->d_topo[k];
    if (h->cfg.world > 1)   // winners of other shards: their domain ids are looked up in the whole-cluster column
      if ((rc = dev_upload<int32_t>(h, h->allocs, &h->d_topo_full[k], nd->topo[k], (size_t)N))) return rc;
  }
  // working copies
#define WK(dst, T) if ((rc = dev_alloc<T>(h, h->allocs, &h->dst, (size_t)n))) return rc
  WK(w_req_cpu, int64_t); WK(w_req_mem, int64_t); WK(w_req_eph, int64_t); WK(w_nz_cpu, int64_t); WK(w_nz_mem, int64_t); WK(w_npods, int32_t);
  for (int k = 0; k < nd->n_scalars; k++) WK(w_req_scalar[k], int64_t);
  h->w_placed = nullptr;
  if (nd->has_placed_mask) WK(w_placed, uint64_t);
  WK(w_score, int32_t);
  WK(w_feas, uint8_t);
#undef WK
  h->d_taint_off = nullptr; h->d_taint_list = nullptr;
  if (nd->taint_list_off && nd->taint_list && n > 0) {
    std::vector<int32_t> off(n + 1);
    const int32_t base = nd->taint_list_off[lo];
    for (int32_t i = 0; i <= n; i++) off[i] = nd->taint_list_off[lo + i] - base;
    if ((rc = dev_upload<int32_t>(h, h->allocs, &h->d_taint_off, off.data(), (size_t)n + 1))) return rc;
    if ((rc = dev_upload<uint8_t>(h, h->allocs, &h->d_taint_list, nd->taint_list + base, (size_t)off[n]))) return rc;
    CK(cudaStreamSynchronize(h->stream));   // off[] is a local
  }
  // host-side bounds used to size outputs / classes
  int64_t bound = 0; int maxpop = 0;
  for (int32_t i = 0; i < N; i++) {
    const int64_t free_pods = (int64_t)nd->alloc_pods[i] - nd->npods[i];
    if (free_pods > 0) bound += free_pods;
    int pc = 0;
    for (int w = 0; w < nd->taint_words; w++) pc += __builtin_popcountll(nd->taint_mask[(size_t)w * N + i] & nd->taint_prefer[w]);
    if (pc > maxpop) maxpop = pc;
  }
  h->pod_bound = bound; h->max_prefer_pop = maxpop;
  h->taint_or0 = 0;
  for (int32_t i = 0; i < N; i++) h->taint_or0 |= nd->taint_mask[i];
  CK(cudaStreamSynchronize(h->stream));
  h->have_nodes = true;
  return CCSIM_OK;
}

extern "C" int ccsim_set_templates(ccsim_handle *h, int32_t n_templates, const ccsim_template *templates,
                                   int32_t n_counters, const ccsim_counter *counters) {
  if (!h || !templates) return fail(h, CCSIM_EINVAL, "null argument");
  if (!h->have_nodes) return fail(h, CCSIM_ESTATE, "ccsim_load_nodes must come first");
  if (n_templates < 1 || n_templates > CCSIM_MAX_TEMPLATES) return fail(h, CCSIM_EINVAL, "n_templates out of range");
  if (n_counters < 0 || n_counters > CCSIM_MAX_COUNTERS || (n_counters && !counters)) return fail(h, CCSIM_EINVAL, "n_counters out of range");
  if (n_templates > 1 && n_counters > 0)
    return fail(h, CCSIM_EUNSUPPORTED, "PodTopologySpread/InterPodAffinity templates are single-template only");
  CK(cudaSetDevice(h->cfg.device));
  free_pool(h, h->tmpl_allocs);
  h->have_templates = false; h->plan.valid = false;
  const ccsim_nodes &nd = h->meta;
  for (int t = 0; t < n_templates; t++) {
    const ccsim_template &T = templates[t];
    if (T.n_pref_terms < 0 || T.n_pref_terms > CCSIM_MAX_AFF_TERMS) return fail(h, CCSIM_EINVAL, "template %d: n_pref_terms", t);
    if (T.n_pts < 0 || T.n_pts > CCSIM_MAX_PTS || T.n_aff < 0 || T.n_aff > CCSIM_MAX_IPA || T.n_anti < 0 || T.n_anti > CCSIM_MAX_IPA ||
        T.n_aff_terms < 0 || T.n_aff_terms > CCSIM_MAX_AFF_TERMS)
      return fail(h, CCSIM_EINVAL, "template %d: term counts out of range", t);
    for (int c = 0; c < T.n_pts; c++) {
      if (T.pts[c].counter < 0 || T.pts[c].counter >= n_counters) return fail(h, CCSIM_EINVAL, "template %d: pts counter index", t);
      if (counters[T.pts[c].counter].topo_col < 0)
        return fail(h, CCSIM_EUNSUPPORTED, "topology spread over a node-local (hostname) domain is not supported yet");
    }
    for (int a = 0; a < T.n_aff; a++) if (T.aff_counter[a] < 0 || T.aff_counter[a] >= n_counters) return fail(h, CCSIM_EINVAL, "aff counter index");
    for (int a = 0; a < T.n_anti; a++) if (T.anti_counter[a] < 0 || T.anti_counter[a] >= n_counters) return fail(h, CCSIM_EINVAL, "anti counter index");
    if ((T.flags & CCSIM_TF_PREFILTER_NODES) && (T.prefilter_bit < 0 || T.prefilter_bit >= 64 * nd.static_words))
      return fail(h, CCSIM_EINVAL, "template %d: prefilter_bit", t);
    if (T.n_spts < 0 || T.n_spts > CCSIM_MAX_PTS || T.n_ipa_score < 0 || T.n_ipa_score > CCSIM_MAX_IPA)
      return fail(h, CCSIM_EINVAL, "template %d: soft term counts out of range", t);
    if (T.spts_ignored_bit >= 64 * nd.static_words) return fail(h, CCSIM_EINVAL, "template %d: spts_ignored_bit", t);
    for (int c = 0; c < T.n_spts; c++) {
      const ccsim_spts &sc = T.spts[c];
      if (sc.counter < 0 || sc.counter >= n_counters) return fail(h, CCSIM_EINVAL, "template %d: spts counter index", t);
      if ((sc.hostname != 0) != (counters[sc.counter].topo_col < 0)) return fail(h, CCSIM_EINVAL, "template %d: spts %d: hostname constraints use node-local counters (and only they)", t, c);
      if (sc.has_key_bit >= 64 * nd.static_words) return fail(h, CCSIM_EINVAL, "template %d: spts has_key_bit", t);
    }
    for (int a = 0; a < T.n_ipa_score; a++) if (T.ipa_score_counter[a] < 0 || T.ipa_score_counter[a] >= n_counters) return fail(h, CCSIM_EINVAL, "ipa score counter index");
  }
  for (int j = 0; j < n_counters; j++) if (counters[j].elig_bit >= 64 * nd.static_words) return fail(h, CCSIM_EINVAL, "counter %d: elig_bit", j);
  for (int t = 0; t < n_templates; t++) {
    const ccsim_template &T = templates[t];
    const long long wsum = (long long)abs(T.w_taint) + abs(T.w_node_affinity) + abs(T.w_fit) + abs(T.w_pts) + abs(T.w_ipa) + abs(T.w_balanced) + abs(T.w_image);
    if (wsum * 100 >= 4095) return fail(h, CCSIM_EUNSUPPORTED, "template %d: sum of score weights %lld too large for the packed key", t, wsum);
  }
  if (h->max_prefer_pop + 1 > CCSIM_MAX_CLASSES)
    return fail(h, CCSIM_EUNSUPPORTED, "a node carries %d PreferNoSchedule taints (max %d)", h->max_prefer_pop, CCSIM_MAX_CLASSES - 1);
  h->h_templates.assign(templates, templates + n_templates);
  int rc;
  {
    // ImageLocality columns: this shard's slice goes to the device, the device copy of the template points at it
    std::vector<ccsim_template> dev_t(templates, templates + n_templates);
    for (int t = 0; t < n_templates; t++)
      if (templates[t].image_score) {
        uint8_t *d = nullptr;
        if ((rc = dev_upload<uint8_t>(h, h->tmpl_allocs, &d, templates[t].image_score + h->node_base, (size_t)h->n))) return rc;
        dev_t[t].image_score = d;
      }
    if ((rc = dev_upload<ccsim_template>(h, h->tmpl_allocs, &h->d_templates, dev_t.data(), (size_t)n_templates))) return rc;
    CK(cudaStreamSynchronize(h->stream));   // dev_t is about to go out of scope
  }
  for (int c = 0; c < CCSIM_MAX_PTS; c++) { h->d_stamp[c] = nullptr; h->stamp_len[c] = 0; }
  for (int c = 0; c < templates[0].n_spts; c++)
    if (!templates[0].spts[c].hostname) {
      h->stamp_len[c] = (size_t)counters[templates[0].spts[c].counter].n_domains + 1;
      if ((rc = dev_alloc<uint32_t>(h, h->tmpl_allocs, &h->d_stamp[c], h->stamp_len[c]))) return rc;
    }
  // counters: small domain sets live replicated in shared memory, large ones as per-CTA replicas in global memory
  h->smem_cnt_ints = 0; h->final_total = 0;
  const int grid_max = std::min(h->sm_count, CCSIM_MAX_GRID);
  for (int j = 0; j < n_counters; j++) {
    const ccsim_counter &c = counters[j];
    DevCounter &d = h->counters[j];
    d.topo_col = c.topo_col; d.inc = c.inc; d.n_present = c.n_present; d.is_aff = 0; d.smem_off = -1; d.work = nullptr; d.elig_bit = c.elig_bit; d.pad = 0;
    for (int a = 0; a < templates[0].n_aff; a++) if (templates[0].aff_counter[a] == j) d.is_aff = 1;
    if (c.topo_col >= nd.n_topo_cols) return fail(h, CCSIM_EINVAL, "counter %d: topo_col", j);
    if (c.topo_col < 0) {
      // node-local: init is a whole-cluster column; keep this shard's slice
      if (c.n_domains != h->n_global) return fail(h, CCSIM_EINVAL, "counter %d: node-local counter needs n_domains == n_nodes", j);
      d.n_domains = h->n;
      if ((rc = dev_upload<int32_t>(h, h->tmpl_allocs, &d.init, c.init + h->node_base, (size_t)h->n))) return rc;
      if ((rc = dev_alloc<int32_t>(h, h->tmpl_allocs, &d.work, (size_t)h->n))) return rc;
    } else {
      if (c.n_domains < 0 || c.n_present < 0 || c.n_present > c.n_domains) return fail(h, CCSIM_EINVAL, "counter %d: domains", j);
      d.n_domains = c.n_domains;
      if ((rc = dev_upload<int32_t>(h, h->tmpl_allocs, &d.init, c.init, (size_t)c.n_domains))) return rc;
      if (h->smem_cnt_ints + c.n_domains <= SMEM_CNT_MAX_INTS) { d.smem_off = h->smem_cnt_ints; h->smem_cnt_ints += c.n_domains; }
      else if ((rc = dev_alloc<int32_t>(h, h->tmpl_allocs, &d.work, (size_t)grid_max * c.n_domains))) return rc;
      h->final_off[j] = h->final_total; h->final_total += c.n_domains;
    }
  }
  if ((rc = dev_alloc<int32_t>(h, h->tmpl_allocs, &h->d_final_cnt, (size_t)h->final_total))) return rc;
  h->n_templates = n_templates; h->n_counters = n_counters;
  CK(cudaStreamSynchronize(h->stream));
  h->have_templates = true;
  return CCSIM_OK;
}

static void fill_params(ccsim_handle *h, DevParams &p, int64_t max_pods) {
  memset(&p, 0, sizeof(p));
  const ccsim_nodes &nd = h->meta;
  p.n = h->n; p.n_global = h->n_global; p.node_base = h->node_base;
  p.n_scalars = nd.n_scalars; p.taint_words = nd.taint_words; p.static_words = nd.static_words; p.n_topo = nd.n_topo_cols;
  p.n_templates = h->n_templates; p.n_counters = h->n_counters;
  p.n_classes = h->max_prefer_pop + 1;
  p.rank = h->cfg.rank; p.world = h->cfg.world;
  p.alloc_cpu = h->d_alloc_cpu; p.alloc_mem = h->d_alloc_mem; p.alloc_eph = h->d_alloc_eph; p.alloc_pods = h->d_alloc_pods;
  for (int k = 0; k < nd.n_scalars; k++) { p.alloc_scalar[k] = h->d_alloc_scalar[k]; p.req_scalar[k] = h->w_req_scalar[k]; }
  p.taint_mask = h->d_taint; p.static_mask = h->d_static;
  for (int k = 0; k < nd.n_topo_cols; k++) { p.topo[k] = h->d_topo[k]; p.topo_full[k] = h->d_topo_full[k]; }
  for (int r = 0; r < CCSIM_MAX_WORLD; r++) p.xslots_peer[r] = h->x_peer[r];
  p.req_cpu = h->w_req_cpu; p.req_mem = h->w_req_mem; p.req_eph = h->w_req_eph; p.nz_cpu = h->w_nz_cpu; p.nz_mem = h->w_nz_mem;
  p.npods = h->w_npods; p.placed_mask = h->w_placed; p.score_cache = h->w_score; p.feas = h->w_feas;
  for (int c = 0; c < CCSIM_MAX_PTS; c++) p.stamp[c] = h->d_stamp[c];
  for (int w = 0; w < CCSIM_MAX_TAINT_WORDS; w++) { p.taint_nosched[w] = nd.taint_nosched[w]; p.taint_prefer[w] = nd.taint_prefer[w]; }
  p.templates = h->d_templates;
  for (int j = 0; j < h->n_counters; j++) { p.counters[j] = h->counters[j]; p.final_off[j] = h->final_off[j]; }
  p.final_cnt = h->d_final_cnt;
  p.slots = h->d_slots;
  p.pod_node = h->d_pod_node; p.pod_cap = h->pod_cap; p.max_pods = max_pods;
  p.out = h->d_out;
  p.taint_list_off = h->d_taint_off; p.taint_list = h->d_taint_list;
}

// Everything a Run does before the wave kernel starts: output / streaming buffers, restoring the working columns, choosing the
// engine, uploading the parameters. Kept apart from the launch (ccsim_prepare) for hosts that drive several ranks from one
// process: every rank must be past its allocations before any rank's persistent kernel starts waiting for its peers.
static int run_prepare(ccsim_handle *h, int64_t max_pods) {
  if (!h->have_nodes || !h->have_templates) return fail(h, CCSIM_ESTATE, "load_nodes and set_templates must come first");
  if (h->cfg.world > 1 && !h->peers_ready) return fail(h, CCSIM_ESTATE, "sharded run: ccsim_peer_import must come first");
  CK(cudaSetDevice(h->cfg.device));
  RunPlan &pl = h->plan;
  pl.valid = false; pl.empty = false; pl.max_pods = max_pods;
  const int32_t n = h->n;
  // output capacity: no run can place more than sum(max(0, alloc_pods - npods)) pods (fit.go:567-576)
  int64_t cap = h->pod_bound + 1;
  // ("Too many pods" bounds a run only while NodeResourcesFit filters: with the plugin disabled through --default-config an
  //  unlimited run never ends in the reference either)
  if (max_pods <= 0)
    for (const ccsim_template &T : h->h_templates)
      if (!(T.filter_enable & CCSIM_PL_FIT))
        return fail(h, CCSIM_EUNSUPPORTED, "NodeResourcesFit is disabled for a template: the run is unbounded, --max-limit is required");
  if (max_pods > 0 && (max_pods < cap || [&] { for (const ccsim_template &T : h->h_templates) if (!(T.filter_enable & CCSIM_PL_FIT)) return true; return false; }())) cap = max_pods;
  if (cap > h->pod_cap) {
    if (h->d_pod_node) cudaFreeAsync(h->d_pod_node, h->stream);
    h->d_pod_node = nullptr; h->pod_cap = 0;
    CK(cudaMallocAsync((void **)&h->d_pod_node, (size_t)cap * sizeof(int32_t), h->stream));
    h->pod_cap = cap;
  }
  // restore the working copies of the mutable columns from the snapshot (a Run never changes the loaded snapshot)
  cudaStream_t s = h->stream;
  if (n) {
    CK(cudaMemcpyAsync(h->w_req_cpu, h->s_req_cpu, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(h->w_req_mem, h->s_req_mem, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(h->w_req_eph, h->s_req_eph, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(h->w_nz_cpu, h->s_nz_cpu, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(h->w_nz_mem, h->s_nz_mem, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(h->w_npods, h->s_npods, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
    for (int k = 0; k < h->meta.n_scalars; k++)
      CK(cudaMemcpyAsync(h->w_req_scalar[k], h->s_req_scalar[k], (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    if (h->w_placed) CK(cudaMemsetAsync(h->w_placed, 0, (size_t)n * 8, s));
    for (int j = 0; j < h->n_counters; j++)
      if (h->counters[j].topo_col < 0)
        CK(cudaMemcpyAsync(h->counters[j].work, h->counters[j].init, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
  }
  for (int c = 0; c < CCSIM_MAX_PTS; c++) if (h->d_stamp[c]) CK(cudaMemsetAsync(h->d_stamp[c], 0, h->stamp_len[c] * 4, s));
  CK(cudaMemsetAsync(h->d_out, 0, sizeof(DevOut), s));
  CK(cudaMemsetAsync(h->d_slots, 0, sizeof(unsigned long long) * 2 * CCSIM_MAX_GRID * SLOT_STRIDE, s));
  // (the cross-GPU buffer is NOT cleared here: peers may already be writing wave 0 of this run; stale words are
  //  harmless because runs advance a per-handle epoch that is folded into the tag)

  if (n == 0) {   // ErrNoNodesAvailable (scheduler.go:68): nothing to evaluate; the host formats the message
    CK(cudaStreamSynchronize(s));
    pl.empty = true; pl.valid = true;
    return CCSIM_OK;
  }
  // grid: one persistent CTA per SM (fewer for tiny clusters: the exchange cost grows with the CTA count)
  int grid = std::min(h->sm_count, CCSIM_MAX_GRID);
  // (node-sharded runs: every rank sizes the grid from the largest shard, so that all ranks launch the same grid and every
  //  rank knows how many candidate lines its peers publish)
  const int32_t n_grid = h->cfg.world > 1 ? (h->n_global + h->cfg.world - 1) / h->cfg.world : n;
  const int want = (n_grid + BLOCK_THREADS - 1) / BLOCK_THREADS;
  if (want < grid) grid = want;
  if (grid < 1) grid = 1;
  h->grid = grid;
  DevParams p;
  fill_params(h, p, max_pods);
  p.grid = grid;
  p.chunk = (n + grid - 1) / grid;
  h->epoch = (h->epoch % 255u) + 1u;     // every rank of a sharded run calls ccsim_run the same number of times
  p.epoch = h->epoch;
  p.xwave0 = h->xwave0;
  p.debug_flags = getenv("CCSIM_DEBUG_FLAGS") ? (uint32_t)atoi(getenv("CCSIM_DEBUG_FLAGS")) : 0u;
  // resident mode: every column the Filter/Score pass reads is staged into shared memory once
  int n_local = 0;
  for (int j = 0; j < h->n_counters; j++) if (h->counters[j].topo_col < 0) n_local++;
  p.n_local = n_local;
  p.chunk_pad = (p.chunk + 3) & ~3;
  p.smem_cnt_ints = h->smem_cnt_ints;
  const size_t cnt_bytes = ((size_t)h->smem_cnt_ints * 4 + 15) & ~(size_t)15;
  const size_t per_node = 8 * (9 + (h->meta.static_words > 0 ? 1 : 0)) + 4 * (4 + h->meta.n_topo_cols + n_local);
  const size_t smem_res = cnt_bytes + per_node * (size_t)p.chunk_pad;
  const size_t smem_str = cnt_bytes;
  const bool resident = smem_res + sizeof(WaveShared) + 1024 <= h->smem_optin && !getenv("CCSIM_FORCE_STREAMING");
  p.tile_resident = resident ? 1 : 0;
  h->last_resident = p.tile_resident;
  size_t smem = resident ? smem_res : smem_str;
  const void *kern = resident ? (const void *)ccsim_wave_kernel<true> : (const void *)ccsim_wave_kernel<false>;
  int block = BLOCK_THREADS;
  // lean resident kernel: the common case (see ccsim_lean.cuh for the eligibility rules)
  // reference sampling mode (ccsim_config.sampling): numFeasibleNodesToFind (schedule_one.go:697-723)
  const bool faithful = h->cfg.sampling == CCSIM_SAMPLING_REFERENCE;
  {
    const long long N = h->n_global;
    long long pct = h->cfg.pct_nodes_to_score, kf = N;
    if (N >= 100) {
      if (pct == 0) { pct = 50 - N / 125; if (pct < 5) pct = 5; }
      kf = N * pct / 100;
      if (kf < 100) kf = 100;
    }
    p.sample_k = kf;
  }
  LeanParams lp; memset(&lp, 0, sizeof(lp));
  // measured on B200 (profiles/r1_kernel_variants.md): at 768 threads the lean kernel beats the generic resident kernel on
  // every eligible workload (C2 2.50 vs 2.67, C3 2.64 vs 2.84, C4 4.27 vs 4.95 us/wave); CCSIM_FORCE_GENERIC overrides.
  // normalised soft scorers / ImageLocality columns run in the generic kernel only (multi-phase waves)
  bool has_pref = false, has_soft = false;
  for (auto &T : h->h_templates) {
    if (T.n_pref_terms > 0 && (T.score_enable & CCSIM_PL_NODE_AFFINITY)) has_soft = true;
    if (T.n_spts > 0 && (T.score_enable & CCSIM_PL_POD_TOPOLOGY_SPREAD)) has_soft = true;
    if (T.n_ipa_score > 0 && (T.score_enable & CCSIM_PL_INTER_POD_AFFINITY)) has_soft = true;
    if (T.image_score && (T.score_enable & CCSIM_PL_IMAGE_LOCALITY)) has_pref = true;
  }
  for (int j = 0; j < h->n_counters; j++) if (h->counters[j].elig_bit >= 0) has_soft = true;
  if (has_soft && (h->cfg.world > 1 || h->n_templates > 1))
    return fail(h, CCSIM_EUNSUPPORTED, "normalised soft scorers (preferred nodeAffinity, ScheduleAnyway spreading, pod-affinity scoring): single template, single GPU only");
  has_pref = has_pref || has_soft;
  bool lean = resident && !has_pref && h->n_templates == 1 && h->meta.taint_words == 1 && h->meta.static_words <= 1 && !getenv("CCSIM_FORCE_GENERIC");
  if (lean) {
    const ccsim_template &T = h->h_templates[0];
    const bool nzfit = (T.filter_enable & CCSIM_PL_FIT) && !(T.flags & CCSIM_TF_FIT_ALL_ZERO);
    if (nzfit && T.req_eph > 0) lean = false;
    if (nzfit) for (int k = 0; k < h->meta.n_scalars; k++) if (T.req_scalar[k] != 0) lean = false;
    if ((T.filter_enable & CCSIM_PL_NODE_AFFINITY) && (T.flags & CCSIM_TF_HAS_AFFINITY_TERMS)) lean = false;
    if ((T.filter_enable & CCSIM_PL_NODE_NAME) && T.nodename_idx >= 0) lean = false;
    if (T.flags & CCSIM_TF_PREFILTER_NODES) lean = false;
    if ((T.filter_enable & CCSIM_PL_NODE_PORTS) && (T.flags & CCSIM_TF_HAS_HOST_PORTS) && h->w_placed) lean = false;
    if (T.n_pts + T.n_aff + T.n_anti > LEAN_MAX_TERMS) lean = false;
    int ns = 0;
    for (int j = 0; j < h->n_counters && lean; j++) {
      const DevCounter &dc = h->counters[j];
      if (dc.topo_col >= 0 && dc.smem_off < 0) { lean = false; break; }
      int slot = -1;
      if (dc.topo_col >= 0) for (int q = 0; q < ns; q++) if (lp.slot_topo[q] == dc.topo_col) slot = q;
      if (slot < 0) {
        if (ns >= LEAN_MAX_SLOTS) { lean = false; break; }
        slot = ns++;
        lp.slot_topo[slot] = dc.topo_col >= 0 ? dc.topo_col : -1;
        lp.slot_counter[slot] = dc.topo_col >= 0 ? -1 : j;
      }
      lp.counter_slot[j] = slot;
    }
    if (lean) {
      lp.n_slots = ns;
      int units = (10 + ns + 3) / 4;
      if ((units & 1) == 0) units++;
      lp.stride_u = units;
      const int want1024 = (n + LEAN_THREADS - 1) / LEAN_THREADS;
      (void)want1024;
      lp.rec_bytes_total = (uint32_t)((size_t)units * 16 * p.chunk_pad);
      const size_t smem_lean = cnt_bytes + lp.rec_bytes_total + (size_t)p.chunk_pad * (6 * 8 + 2 * 4 + (faithful ? 8 : 0));
      if (smem_lean + sizeof(LeanShared) + 1024 > h->smem_optin) lean = false;
      else { smem = smem_lean; kern = faithful ? (const void *)ccsim_wave_lean_kernel<true> : (const void *)ccsim_wave_lean_kernel<false>; block = LEAN_THREADS; }
    }
  }
  h->last_lean = lean ? 1 : 0;
  if (faithful && (!lean || h->cfg.world > 1))
    return fail(h, CCSIM_EUNSUPPORTED, "reference sampling mode needs the lean resident kernel on a single GPU (one template, <=1 taint/static word, no extras)");
  // batched tie-run engine (ccsim_batched.cuh): one template, node-local predicates and scorers only
  bool batched = lean && !faithful && h->n_counters == 0 && h->max_prefer_pop == 0 && h->cfg.world == 1 &&
                 h->cfg.engine != CCSIM_ENGINE_SEQUENTIAL && !getenv("CCSIM_FORCE_SEQUENTIAL");
  if (batched) {
    const size_t smem_b = smem + (size_t)p.chunk_pad * 12;
    if (smem_b + sizeof(LeanShared) + sizeof(BatchShared) + 1024 > h->smem_optin) batched = false;
    else { smem = smem_b; kern = (const void *)ccsim_wave_batched_kernel; }
  }
  if (h->cfg.engine == CCSIM_ENGINE_BATCHED && !batched)
    return fail(h, CCSIM_EUNSUPPORTED, "batched engine needs one template with node-local predicates only, no PreferNoSchedule taints, a resident tile and a single GPU");
  h->last_batched = batched ? 1 : 0;
  // multi-commit waves (ccsim_multi.cuh): one template coupled through per-domain counters, one node per thread
  MultiParams mp; memset(&mp, 0, sizeof(mp));
  bool multi = lean && !faithful && !batched && h->n_counters > 0 && h->max_prefer_pop == 0 &&
               h->cfg.engine == CCSIM_ENGINE_AUTO && !getenv("CCSIM_FORCE_SEQUENTIAL") && h->h_templates[0].n_aff == 0 &&
               p.chunk <= LEAN_THREADS && h->n_global < (1 << MULTI_IDX_BITS);
  if (multi) {
    for (int j = 0; j < h->n_counters; j++) if (h->counters[j].inc < 0) multi = false;   // feasibility must be monotone within a wave
    {
      const ccsim_template &T = h->h_templates[0];
      int gt = 0;
      if (T.filter_enable & CCSIM_PL_POD_TOPOLOGY_SPREAD) for (int c = 0; c < T.n_pts; c++) if (h->counters[T.pts[c].counter].topo_col >= 0) gt++;
      if (T.filter_enable & CCSIM_PL_INTER_POD_AFFINITY) for (int a = 0; a < T.n_anti; a++) if (h->counters[T.anti_counter[a]].topo_col >= 0) gt++;
      if (gt > MULTI_GT) multi = false;
      // (a committed node may win again inside a wave: every candidate carries its key after one more clone, MULTI_NEXT_SHIFT)
      // the replay updates counters term by term: every incremented replicated counter must be read by exactly one Filter term
      for (int j = 0; j < h->n_counters; j++) {
        if (h->counters[j].topo_col < 0 || h->counters[j].inc == 0) continue;
        int refs = 0;
        if (T.filter_enable & CCSIM_PL_POD_TOPOLOGY_SPREAD) for (int c = 0; c < T.n_pts; c++) if (T.pts[c].counter == j) refs++;
        if (T.filter_enable & CCSIM_PL_INTER_POD_AFFINITY) for (int a = 0; a < T.n_anti; a++) if (T.anti_counter[a] == j) refs++;
        if (refs != 1) multi = false;
      }
    }
    uint32_t shift = 0;
    for (int sl = 0; sl < lp.n_slots && multi; sl++) {
      if (lp.slot_topo[sl] < 0) continue;
      int maxd = 1;
      for (int j = 0; j < h->n_counters; j++) if (lp.counter_slot[j] == sl && h->counters[j].topo_col >= 0) maxd = std::max(maxd, h->counters[j].n_domains);
      uint32_t bits = 0; while ((1u << bits) <= (uint32_t)maxd) bits++;        // values 0..maxd (dom + 1)
      if (shift + bits > MULTI_PAY_BITS) { multi = false; break; }
      mp.pay_shift[sl] = shift; mp.pay_mask[sl] = (1u << bits) - 1u; shift += bits;
    }
    const size_t smem_m = smem + (size_t)p.chunk_pad * 8 + 16;     // + the per-node payload column
    if (smem_m + sizeof(LeanShared) + sizeof(MultiShared) + 1024 > h->smem_optin) multi = false;
    if (multi) { kern = h->cfg.world > 1 ? (const void *)ccsim_wave_multi_kernel<true> : (const void *)ccsim_wave_multi_kernel<false>; smem = smem_m; }
  }
  h->last_multi = multi ? 1 : 0;
  // streaming engine (ccsim_stream.cuh): node-local templates when the tile is not resident, or several templates; the node
  // tiles go through shared memory with bulk-async copies (TMA) and the score is memoised per (template, node)
  StreamParams sp; memset(&sp, 0, sizeof(sp));
  int stream_mode = 0;
  bool stream = !lean && !has_pref && h->n_counters == 0 && h->max_prefer_pop == 0 && !faithful &&
                h->meta.taint_words == 1 && h->meta.static_words <= 1 && !getenv("CCSIM_FORCE_GENERIC");
  if (stream)
    for (const ccsim_template &T : h->h_templates) {
      const bool nzfit = (T.filter_enable & CCSIM_PL_FIT) && !(T.flags & CCSIM_TF_FIT_ALL_ZERO);
      if (nzfit && T.req_eph > 0) stream = false;
      if (nzfit) for (int k = 0; k < h->meta.n_scalars; k++) if (T.req_scalar[k] != 0) stream = false;
      if ((T.filter_enable & CCSIM_PL_NODE_AFFINITY) && (T.flags & CCSIM_TF_HAS_AFFINITY_TERMS)) stream = false;
      if ((T.filter_enable & CCSIM_PL_NODE_NAME) && T.nodename_idx >= 0) stream = false;
      if (T.flags & CCSIM_TF_PREFILTER_NODES) stream = false;
      if ((T.filter_enable & CCSIM_PL_NODE_PORTS) && (T.flags & CCSIM_TF_HAS_HOST_PORTS) && h->w_placed) stream = false;
      if (T.n_pts || T.n_aff || T.n_anti) stream = false;
    }
  if (stream) {
    free_pool(h, h->stream_allocs);
    bool masks = false;
    for (const ccsim_template &T : h->h_templates) {
      uint64_t tb = 0;
      if (T.filter_enable & CCSIM_PL_TAINT_TOLERATION) tb |= h->meta.taint_nosched[0] & ~T.tol_nosched[0] & ~(1ull << CCSIM_TAINT_UNSCHEDULABLE_BIT);
      if ((T.filter_enable & CCSIM_PL_NODE_UNSCHEDULABLE) && !(T.flags & CCSIM_TF_TOLERATES_UNSCHEDULABLE)) tb |= 1ull << CCSIM_TAINT_UNSCHEDULABLE_BIT;
      if (tb & h->taint_or0) masks = true;
      if (h->meta.static_words > 0) {
        if ((T.filter_enable & CCSIM_PL_NODE_AFFINITY) && (T.flags & CCSIM_TF_HAS_NODE_SELECTOR) && T.sel_mask[0]) masks = true;
        if ((T.filter_enable & CCSIM_PL_NODE_PORTS) && (T.flags & CCSIM_TF_HAS_HOST_PORTS) && T.port_static_mask[0]) masks = true;
        if ((T.filter_enable & CCSIM_PL_INTER_POD_AFFINITY) && T.existing_anti_mask[0]) masks = true;
      }
    }
    sp.use_masks = masks ? 1 : 0;
    sp.chunk_pad = ((p.chunk + STREAM_TILE - 1) / STREAM_TILE) * STREAM_TILE;
    sp.tiles = sp.chunk_pad / STREAM_TILE;
    sp.n_pad = (long long)grid * sp.chunk_pad;
    int rc2;
    unsigned long long *mt = nullptr, *mst = nullptr;
    if ((rc2 = dev_alloc<long long>(h, h->stream_allocs, &sp.f_cpu, (size_t)sp.n_pad))) return rc2;
    if ((rc2 = dev_alloc<long long>(h, h->stream_allocs, &sp.f_mem, (size_t)sp.n_pad))) return rc2;
    if ((rc2 = dev_alloc<int32_t>(h, h->stream_allocs, &sp.f_pods, (size_t)sp.n_pad))) return rc2;
    if (masks) {
      if ((rc2 = dev_alloc<unsigned long long>(h, h->stream_allocs, &mt, (size_t)sp.n_pad))) return rc2;
      if ((rc2 = dev_alloc<unsigned long long>(h, h->stream_allocs, &mst, (size_t)sp.n_pad))) return rc2;
    }
    sp.m_taint = mt; sp.m_static = mst;
    if ((rc2 = dev_alloc<int32_t>(h, h->stream_allocs, &sp.memo, (size_t)sp.n_pad * h->n_templates))) return rc2;
    CK(cudaMemsetAsync(sp.memo, 0xFF, (size_t)sp.n_pad * h->n_templates * 4, s));
    ccsim_stream_prep_kernel<<<std::min<long long>(8LL * h->sm_count, (sp.n_pad + 255) / 256), 256, 0, s>>>(p, sp);
    h->launches++;
    CK(cudaGetLastError());
    // resident free_* columns when the chunk fits next to the memo ring (24 B per node: up to ~8k nodes per SM)
    const size_t smem_resf = (size_t)STREAM_STAGES_RES * STREAM_TILE * 4 + (size_t)sp.chunk_pad * 24 + 128;
    stream_mode = masks ? 1 : ((smem_resf + sizeof(StreamShared) + 1024 <= h->smem_optin && sp.tiles <= STREAM_STAGES_RES && !getenv("CCSIM_STREAM_ALL")) ? 2 : 0);
    kern = stream_mode == 1 ? (const void *)ccsim_wave_stream_kernel<1> : stream_mode == 2 ? (const void *)ccsim_wave_stream_kernel<2> : (const void *)ccsim_wave_stream_kernel<0>;
    smem = stream_mode == 2 ? smem_resf : (size_t)STREAM_STAGES * STREAM_TILE * (masks ? 40 : 24) + 128;
    block = STREAM_BLOCK;
  }
  h->last_stream = stream ? 1 : 0;
  p.self = h->d_params;
  CK(cudaMemcpyAsync(h->d_params, &p, sizeof(DevParams), cudaMemcpyHostToDevice, s));
  int occ = 0;
  if (stream && stream_mode == 1) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_stream_kernel<1>, block, smem));
  else if (stream && stream_mode == 2) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_stream_kernel<2>, block, smem));
  else if (stream) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_stream_kernel<0>, block, smem));
  else if (multi && h->cfg.world > 1) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_multi_kernel<true>, block, smem));
  else if (multi) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_multi_kernel<false>, block, smem));
  else if (batched) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_batched_kernel, block, smem));
  else if (lean && faithful) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_lean_kernel<true>, block, smem));
  else if (lean) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_lean_kernel<false>, block, smem));
  else if (resident) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_kernel<true>, block, smem));
  else CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ccsim_wave_kernel<false>, block, smem));
  if (occ < 1 || occ * h->sm_count < grid) return fail(h, CCSIM_ECUDA, "persistent grid %d does not fit (occupancy %d x %d SMs)", grid, occ, h->sm_count);
  pl.p = p; pl.lp = lp; pl.mp = mp; pl.sp = sp; pl.kern = kern; pl.grid = grid; pl.block = block; pl.smem = smem;
  pl.stream = stream; pl.multi = multi; pl.batched = batched; pl.lean = lean; pl.resident = resident;
  pl.variant = (!stream && !lean && resident ? CCSIM_KV_RESIDENT : 0) | (stream ? (int64_t)stream_mode << CCSIM_KV_STREAM_MODE_SHIFT : 0) |
               (lean && faithful ? CCSIM_KV_REFERENCE_SAMPLING : 0) | (multi && h->cfg.world > 1 ? CCSIM_KV_CROSS_GPU : 0);
  pl.valid = true;
  return CCSIM_OK;
}

extern "C" int ccsim_prepare(ccsim_handle *h, int64_t max_pods) {
  if (!h) return fail(h, CCSIM_EINVAL, "null argument");
  int rc = run_prepare(h, max_pods);
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->stream));     // allocations and restores are done when this returns
  return CCSIM_OK;
}

extern "C" int ccsim_run(ccsim_handle *h, int64_t max_pods, ccsim_result *out) {
  if (!h || !out) return fail(h, CCSIM_EINVAL, "null argument");
  if (!(h->plan.valid && h->plan.max_pods == max_pods)) { int rc = run_prepare(h, max_pods); if (rc) return rc; }
  RunPlan &pl = h->plan;
  pl.valid = false;                          // one launch per preparation: the working columns are consumed by the run
  memset(out, 0, sizeof(*out));
  out->n_nodes = h->n_global;
  if (pl.empty) { out->placed = 0; out->stop_code = CCSIM_STOP_UNSCHEDULABLE; out->pod_node = nullptr; return CCSIM_OK; }
  CK(cudaSetDevice(h->cfg.device));
  const int32_t n = h->n;
  cudaStream_t s = h->stream;
  DevParams &p = pl.p; LeanParams &lp = pl.lp; MultiParams &mp = pl.mp; StreamParams &sp = pl.sp;
  const void *kern = pl.kern; const int grid = pl.grid, block = pl.block; const size_t smem = pl.smem;
  const bool stream = pl.stream, multi = pl.multi, batched = pl.batched, lean = pl.lean, resident = pl.resident;
  (void)resident;
  void *args[] = { (void *)&p, stream ? (void *)&sp : (void *)&lp, (void *)&mp };
  CK(cudaEventRecord(h->ev0, s));
  // Cooperative launch = the driver guarantees that the whole persistent grid is co-resident (the kernels never use grid.sync()).
  // Ranks that share a process (ccsim_peer_import_local) may share a device; cooperative launches of different streams are not
  // run concurrently there, so those ranks use a plain launch: the occupancy check above still holds for each grid on its own.
  if (h->peers_local) CK(cudaLaunchKernel(kern, dim3(grid), dim3(block), args, smem, s));
  else CK(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(block), args, smem, s));
  h->launches++;
  CK(cudaEventRecord(h->ev1, s));
  DevOut ho;
  CK(cudaMemcpyAsync(&ho, h->d_out, sizeof(DevOut), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (ho.error) return fail(h, CCSIM_ECUDA, "wave kernel aborted (error %d: %s)", ho.error, ho.error == 1 ? "exchange watchdog / output overflow" : "?");
  float ms = 0.f; CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  if (stream && (p.debug_flags & 8u) && h->cfg.world == 1 && ho.waves > 0) {     // per-CTA cycle split of the streaming kernel (kernel experiments)
    std::vector<unsigned long long> d((size_t)grid * 4);
    CK(cudaMemcpy(d.data(), h->d_xslots + XLINES_OFF, d.size() * 8, cudaMemcpyDeviceToHost));
    const char *nm[4] = {"mbarrier wait", "scan", "exchange", "rest"};
    for (int q = 0; q < 4; q++) {
      double mn = 1e30, mx = 0, sum = 0; int amx = 0, amn = 0;
      for (int c = 0; c < grid; c++) { const double v = (double)d[(size_t)c * 4 + q] / (double)ho.waves; sum += v; if (v > mx) { mx = v; amx = c; } if (v < mn) { mn = v; amn = c; } }
      fprintf(stderr, "[ccsim stream per-CTA cycles/wave] %-14s min %.0f (CTA %d)  mean %.0f  max %.0f (CTA %d)\n", nm[q], mn, amn, sum / grid, mx, amx);
    }
  }
#ifdef CCSIM_PHASE_TIMERS
  fprintf(stderr, "[ccsim %s tile %zu B smem] ", multi ? "multi" : batched ? "batched" : (lean ? "lean" : (resident ? "resident" : "streaming")), smem);
  fprintf(stderr, "[ccsim phases, CTA0 cycles/wave] scan=%.0f S1=%.0f publish=%.0f gather=%.0f commit=%.0f S2=%.0f (waves=%lld, %.3f ms)\n",
          (double)ho.phase_cycles[0] / ho.waves, (double)ho.phase_cycles[1] / ho.waves, (double)ho.phase_cycles[2] / ho.waves,
          (double)ho.phase_cycles[3] / ho.waves, (double)ho.phase_cycles[4] / ho.waves, (double)ho.phase_cycles[5] / ho.waves,
          (long long)ho.waves, ms);
  fprintf(stderr, "[ccsim phases 6/7] %.0f %.0f\n", (double)ho.phase_cycles[6] / ho.waves, (double)ho.phase_cycles[7] / ho.waves);
#endif
  if (h->cfg.world > 1) h->xwave0 += (uint32_t)ho.waves;    // identical on every rank: the engines run the same waves everywhere
  h->last_stat[0] = (stream ? 4 : multi ? 3 : batched ? 2 : lean ? 1 : 0) | pl.variant; h->last_stat[1] = ho.waves; h->last_stat[2] = ho.placed;
  h->last_stat[3] = ho.stat[0]; h->last_stat[4] = ho.stat[1]; h->last_stat[5] = grid; h->last_stat[6] = block;
  h->last_stat[7] = ho.stat[2];   // multi-commit replay rounds
  for (int q = 0; q < 8; q++) h->last_stat[8 + q] = ho.phase_cycles[q];
  out->placed = ho.placed; out->stop_code = ho.stop_code; out->waves = ho.waves; out->evals = ho.evals; out->run_ms = ms;
  out->examined = ho.examined ? ho.examined : ho.evals;
  h->last_placed = ho.placed;
  if (ho.stop_code == CCSIM_STOP_UNSCHEDULABLE) {
    const int ti = (int)(ho.placed % h->n_templates);
    ccsim_diag_kernel<<<std::min(4 * h->sm_count, (n + 255) / 256), 256, 0, s>>>(p, ti);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&ho, h->d_out, sizeof(DevOut), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (int r = 0; r < CCSIM_R_TOTAL; r++) out->reason_hist[r] = (int64_t)ho.reason_hist[r];
    out->preempt_no_victims = (int64_t)ho.preempt_no_victims;
    out->preempt_not_helpful = (int64_t)h->n - (int64_t)ho.preempt_no_victims;   // per shard, like reason_hist: sums to N - no_victims
  }
  h->h_pod_node.resize((size_t)ho.placed);
  if (ho.placed) CK(cudaMemcpyAsync(h->h_pod_node.data(), h->d_pod_node, (size_t)ho.placed * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  out->pod_node = h->h_pod_node.data();
  return CCSIM_OK;
}

extern "C" int ccsim_node_counts(ccsim_handle *h, int32_t t, int32_t *counts, int64_t *first_pod) {
  if (!h || !counts || !first_pod) return fail(h, CCSIM_EINVAL, "null argument");
  if (!h->have_templates || t < 0 || t >= h->n_templates) return fail(h, CCSIM_EINVAL, "template index");
  CK(cudaSetDevice(h->cfg.device));
  const int32_t N = h->n_global;
  int32_t *d_counts = nullptr; unsigned long long *d_first = nullptr;
  CK(cudaMalloc((void **)&d_counts, (size_t)(N ? N : 1) * 4));
  CK(cudaMalloc((void **)&d_first, (size_t)(N ? N : 1) * 8));
  CK(cudaMemsetAsync(d_counts, 0, (size_t)N * 4, h->stream));
  CK(cudaMemsetAsync(d_first, 0xFF, (size_t)N * 8, h->stream));
  if (h->last_placed > 0) {
    ccsim_count_kernel<<<std::min<long long>(4 * h->sm_count, (h->last_placed + 255) / 256), 256, 0, h->stream>>>(
        h->d_pod_node, h->last_placed, h->n_templates, t, d_counts, d_first);
    h->launches++;
  }
  CK(cudaMemcpyAsync(counts, d_counts, (size_t)N * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(first_pod, d_first, (size_t)N * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  cudaFree(d_counts); cudaFree(d_first);
  return CCSIM_OK;
}

extern "C" int ccsim_device_info(ccsim_handle *h, int32_t *sm_count, int32_t *grid, int32_t *block, int64_t *l2_bytes) {
  if (!h) return CCSIM_EINVAL;
  if (sm_count) *sm_count = h->sm_count;
  if (grid) *grid = h->grid;
  if (block) *block = BLOCK_THREADS;
  if (l2_bytes) *l2_bytes = (int64_t)h->l2_bytes;
  return CCSIM_OK;
}

extern "C" int64_t ccsim_kernel_launches(const ccsim_handle *h) { return h ? h->launches : 0; }

extern "C" int ccsim_run_stats(const ccsim_handle *h, int64_t out[16]) {
  if (!h || !out) return CCSIM_EINVAL;
  memcpy(out, h->last_stat, sizeof(h->last_stat));
  return CCSIM_OK;
}

extern "C" int ccsim_debug_node_scores(ccsim_handle *h, int32_t t, int32_t clones, int64_t *total, int64_t *least, int64_t *balanced) {
  if (!h || !total || !least || !balanced) return fail(h, CCSIM_EINVAL, "null argument");
  if (!h->have_templates || t < 0 || t >= h->n_templates) return fail(h, CCSIM_EINVAL, "template index");
  if (clones < 0) return fail(h, CCSIM_EINVAL, "clones < 0");
  CK(cudaSetDevice(h->cfg.device));
  const int32_t n = h->n;
  if (n == 0) return CCSIM_OK;
  const ccsim_template &T = h->h_templates[t];
  ScoreWeights sw;      // as the wave kernels fold it (lean_build_consts)
  sw.w_fit = (T.score_enable & CCSIM_PL_FIT) ? T.w_fit : 0;
  sw.w_balanced = ((T.score_enable & CCSIM_PL_BALANCED) && !(T.flags & CCSIM_TF_BALANCED_SKIP)) ? T.w_balanced : 0;
  sw.least_w_cpu = T.least_w_cpu; sw.least_w_mem = T.least_w_mem;
  int64_t *d = nullptr;
  CK(cudaMalloc((void **)&d, (size_t)n * 3 * sizeof(int64_t)));
  ccsim_debug_score_kernel<<<std::min(4 * h->sm_count, (n + 255) / 256), 256, 0, h->stream>>>(
      n, h->d_alloc_cpu, h->d_alloc_mem, h->s_req_cpu, h->s_req_mem, h->s_nz_cpu, h->s_nz_mem, T, sw, clones, d, d + n, d + 2 * (size_t)n);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(total, d, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(least, d + n, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(balanced, d + 2 * (size_t)n, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(d);
  if (e != cudaSuccess) return fail(h, CCSIM_ECUDA, "ccsim_debug_node_scores: %s", cudaGetErrorString(e));
  return CCSIM_OK;
}

extern "C" int ccsim_flush_l2(ccsim_handle *h) {
  if (!h) return CCSIM_EINVAL;
  CK(cudaSetDevice(h->cfg.device));
  const size_t bytes = std::max<size_t>(2 * h->l2_bytes, (size_t)256 << 20);
  if (h->flush_bytes < bytes) {
    cudaFree(h->d_flush); h->d_flush = nullptr; h->flush_bytes = 0;
    CK(cudaMalloc(&h->d_flush, bytes));
    h->flush_bytes = bytes;
  }
  ccsim_flush_kernel<<<h->sm_count * 4, 512, 0, h->stream>>>((unsigned long long *)h->d_flush, bytes / 8, (unsigned long long)h->launches);
  h->launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  return CCSIM_OK;
}

extern "C" int ccsim_peer_export(ccsim_handle *h, uint8_t handle_out[CCSIM_IPC_HANDLE_BYTES]) {
  if (!h || !handle_out) return fail(h, CCSIM_EINVAL, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  cudaIpcMemHandle_t mh;
  CK(cudaIpcGetMemHandle(&mh, h->d_xslots));
  static_assert(sizeof(mh) == CCSIM_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
  memcpy(handle_out, &mh, sizeof(mh));
  return CCSIM_OK;
}

extern "C" int ccsim_peer_local(ccsim_handle *h, void **ptr_out) {
  if (!h || !ptr_out) return fail(h, CCSIM_EINVAL, "null argument");
  *ptr_out = h->d_xslots;
  return CCSIM_OK;
}

extern "C" int ccsim_peer_import_local(ccsim_handle *h, int32_t world, void *const *ptrs) {
  if (!h || !ptrs) return fail(h, CCSIM_EINVAL, "null argument");
  if (world != h->cfg.world) return fail(h, CCSIM_EINVAL, "world %d != configured %d", world, h->cfg.world);
  for (int r = 0; r < world; r++) {
    if (!ptrs[r]) return fail(h, CCSIM_EINVAL, "null peer pointer %d", r);
    h->x_peer[r] = r == h->cfg.rank ? h->d_xslots : (unsigned long long *)ptrs[r];
  }
  h->peers_local = true;
  h->peers_ready = true;
  return CCSIM_OK;
}

extern "C" int ccsim_peer_import(ccsim_handle *h, int32_t world, const uint8_t *handles) {
  if (!h || !handles) return fail(h, CCSIM_EINVAL, "null argument");
  if (world != h->cfg.world) return fail(h, CCSIM_EINVAL, "world %d != configured %d", world, h->cfg.world);
  CK(cudaSetDevice(h->cfg.device));
  for (int r = 0; r < world; r++) {
    if (r == h->cfg.rank) { h->x_peer[r] = h->d_xslots; continue; }
    cudaIpcMemHandle_t mh;
    memcpy(&mh, handles + (size_t)r * CCSIM_IPC_HANDLE_BYTES, sizeof(mh));
    void *ptr = nullptr;
    CK(cudaIpcOpenMemHandle(&ptr, mh, cudaIpcMemLazyEnablePeerAccess));
    h->x_peer[r] = (unsigned long long *)ptr;
  }
  h->peers_ready = true;
  return CCSIM_OK;
}
