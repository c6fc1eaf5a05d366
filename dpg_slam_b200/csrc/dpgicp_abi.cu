/*
 * dpgicp_abi.cu — host side of the C ABI declared in include/dpgicp.h.
 *
 * Thin by design: argument validation, host<->device copies, kernel launches.  All arithmetic of
 * the path runs in the sm_100a kernels of dpgicp_kernels.cuh; there is no CPU implementation
 * behind these entry points (dpgicp_create fails without a CUDA device).
 */
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>      /* header-only; ranges show the batch phases in Nsight timelines, no-ops otherwise */

#include <algorithm>
#include <cmath>
#include <map>
#include <mutex>
#include <tuple>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <set>
#include <string>
#include <utility>
#include <vector>

#include "dpgicp.h"
#include "dpgicp_kernels.cuh"

using namespace dpg;

namespace {

struct NvtxRange {                 /* scoped NVTX range */
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

std::string g_create_error;
std::mutex g_optin_mutex;
std::map<std::pair<int, const void *>, size_t> g_smem_optin;   /* (device, kernel) -> dynamic shared memory opted in */

/* Device memory (cudaMalloc) or page-locked host memory (cudaMallocHost), freed by its owner.  An owner whose memory a
 * stream may still read lets it go only after that stream has drained. */
template <cudaError_t (*Alloc)(void **, size_t), cudaError_t (*Free)(void *)>
struct Buf {
  void *p = nullptr;
  size_t cap = 0;
  Buf() = default;
  Buf(const Buf &) = delete;
  Buf &operator=(const Buf &) = delete;
  Buf &operator=(Buf &&o) noexcept { release(); std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
  ~Buf() { release(); }
  void release() {
    if (p) Free(p);
    p = nullptr; cap = 0;
  }
  cudaError_t alloc(size_t bytes) {      /* exactly `bytes`; the old buffer is freed first */
    release();
    void *q = nullptr;
    const cudaError_t e = Alloc(&q, bytes);
    if (e == cudaSuccess) { p = q; cap = bytes; }
    return e;
  }
};
using DevBuf = Buf<cudaMalloc, cudaFree>;
using HostBuf = Buf<cudaMallocHost, cudaFreeHost>;

/* a CUDA event or stream, destroyed by its owner */
template <class T, cudaError_t (*Destroy)(T)>
struct Handle {
  T h = nullptr;
  Handle() = default;
  Handle(const Handle &) = delete;
  Handle &operator=(const Handle &) = delete;
  ~Handle() { reset(); }
  void reset() {
    if (h) Destroy(h);
    h = nullptr;
  }
  operator T() const { return h; }
};
using Event = Handle<cudaEvent_t, cudaEventDestroy>;
using Stream = Handle<cudaStream_t, cudaStreamDestroy>;

/* padded rows + counts on the device, counts mirrored on the host.  A write of the scan store fills the rows behind
 * n_scans and only then advances it (commit_rows). */
struct Store {
  DevBuf rows, count;
  int32_t pitch = 0, n_scans = 0, max_count = 0;
  std::vector<int32_t> h_count;
};

struct Batch {
  DevBuf tasks, results, order;
  bool has_order = false;
  HostBuf h_tasks;               /* PairTask staging of set_pairs */
  Event h_tasks_free;            /* recorded after the H2D copy out of h_tasks: the buffer may be rewritten */
  int64_t n_pairs = 0;
  int32_t max_scan = -1;         /* device-enumerated lists: highest scan (= node) index used; -1 = validated on the host */
};

struct StageTarget { int warps, csize; };      /* of the stage chain: warps per CTA, CTAs per cluster */

struct Nodes {                   /* pose-graph node estimates on the device (dpgicp_set_nodes, dpgicp_update_nodes) */
  DevBuf xy, aux, pass;          /* float2 (x, y); float4 (theta, cosf(-theta), sinf(-theta), 0); int32 pass */
  DevBuf boxes;                  /* index-order box hierarchy, levels back to back, each sized for `cap` nodes */
  int32_t n = 0, cap = 0;        /* nodes in the table; nodes the buffers hold (grows by doubling) */
  int levels = 0;                /* levels and level_cnt follow n; level_off follows cap, so growth below cap moves no level */
  int64_t level_off[8] = {0}, level_cnt[8] = {0};
  HostBuf h_rows;                /* dpgicp_update_nodes: the listed rows and dirty leaves, staged for one copy */
  DevBuf d_rows;
  Event rows_free;               /* recorded after the last kernel that reads d_rows: both staging buffers may be rewritten */
};

}  // namespace

/* One pair batch of a context and the per-run cells of its stage chain.  The context holds the default slot (the batch of
 * dpgicp_set_pairs / dpgicp_run / dpgicp_fetch_*), which runs on the context's stream; dpgicp_slot_create adds slots with
 * a stream of their own, so several batches can be in flight over the one scan store.  Its members free themselves: a
 * slot is deleted only after its stream has drained. */
struct dpgicp_slot {
  dpgicp_ctx *ctx = nullptr;
  Stream own;                                /* null: the default slot, on the context's stream */
  Batch batch;
  DevBuf state[2], susp[2];                  /* suspended-pair state slots + pair lists, ping-pong between stages */
  DevBuf d_queue;                            /* unsigned long long [0..4] stage queue heads, [6],[7] suspended counts, [8..15] counters, [16..23] development phase timers, [24..28] pairs finished per stage */
  Event stage_ev[9];
  bool stage_timing = false;
  int last_stages = 0;
};

/* Its members free themselves: a context is deleted only after its slots are destroyed and its stream has drained. */
struct dpgicp_ctx {
  int device = 0;
  int sm_count = 148;
  Stream own_stream;                         /* the stream the context made; null while a caller's stream is in use */
  cudaStream_t stream = nullptr;             /* the stream in use: own_stream or the one of dpgicp_set_stream */
  Store store, scratch_store;
  dpgicp_slot main;                          /* the default slot */
  std::vector<dpgicp_slot *> slots;          /* the live slots of dpgicp_slot_create */
  Event written;                             /* recorded on the context's stream behind every write a later slot run reads
                                              * (store rows and counts, an enumerated pair list): slot streams wait on it */
  Batch scratch_batch;
  Nodes nodes;                               /* dpgicp_set_nodes: the table of dpgicp_enumerate_pairs_device */
  Nodes list_nodes;                          /* dpgicp_enumerate_pairs: its own positions-only table */
  DevBuf enum_amb;                           /* enumeration: pairs whose guess the host re-derives */
  DevBuf stage, offsets, misc, corr, trig, enum_cnt;
  /* per (kernel, warps, shared memory): resident CTAs per SM or clusters per device — queried once, not on every run */
  std::map<std::tuple<const void *, int, size_t>, int> occupancy;
  HostBuf h_pair;                            /* scratch of the single-pair call shapes */
  int gather_root_only = 0;
  bool gather_local = false;                 /* peers attached by dpgicp_gather_attach_local (no IPC mappings to close) */
  int trig_n = 0;
  float trig_min = 0.f, trig_inc = 0.f;
  DevBuf gather;                             /* this rank's copy of the whole batch's records (fused gather)  */
  int64_t gather_n = 0;
  int gather_world = 0, gather_rank = 0;
  void *gather_peer[DPGICP_MAX_GATHER_RANKS] = {nullptr};
  StageTarget chain[5];                      /* DPGICP_CHAIN: target warps (and "x<cluster size>") per stage (development knob) */
  int n_chain = 0;
  DevBuf d_bad;                              /* int: range flag of the store writes */
  HostBuf h_stage;                           /* staging for subset uploads from pageable memory */
  double handover_factor = 2.0;              /* DPGICP_HANDOVER="f[,fc]": a stage hands over once at most f x (CTAs of the next stage) pairs are */
  double handover_cluster = 1.0;             /* left; fc x (clusters) when the next stage runs clusters (development knob; 0 = plain queue-dry rule) */
  uint64_t launches = 0;
  std::string err;
};

namespace {

int fail(dpgicp_ctx *ctx, int code, const std::string &msg) {
  if (ctx) ctx->err = msg; else g_create_error = msg;
  return code;
}

#define CU_TRY(ctx, expr)                                                                         \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess) {                                                                     \
      return fail(ctx, e__ == cudaErrorMemoryAllocation ? DPGICP_E_NOMEM : DPGICP_E_CUDA,         \
                  std::string(#expr) + ": " + cudaGetErrorString(e__));                           \
    }                                                                                             \
  } while (0)

cudaStream_t stream_of(const dpgicp_slot *s) { return s->own ? s->own.h : s->ctx->stream; }

/* a buffer the runs of every slot may read is about to be overwritten or freed: wait until the slots' streams have
 * drained (the default slot's runs are ordered on the context's stream) */
int drain_slots(dpgicp_ctx *ctx) {
  for (dpgicp_slot *s : ctx->slots) CU_TRY(ctx, cudaStreamSynchronize(s->own));
  return DPGICP_OK;
}

/* the store is about to be replaced (make_room): every slot's runs have read it, and every batch is emptied (its indices
 * referred to the old store) */
int replace_store(dpgicp_ctx *ctx) {
  int rc = drain_slots(ctx);
  if (rc) return rc;
  ctx->main.batch.n_pairs = 0;
  for (dpgicp_slot *s : ctx->slots) s->batch.n_pairs = std::min<int64_t>(s->batch.n_pairs, 0);
  return DPGICP_OK;
}

/* the context's stream has written what a slot's later runs read (store rows and counts, an enumerated list) */
int mark_written(dpgicp_ctx *ctx) {
  CU_TRY(ctx, cudaEventRecord(ctx->written, ctx->stream));
  return DPGICP_OK;
}

/* at least `bytes` in b, its contents not kept; a pinned buffer's caller first waits for any copy still queued out of it */
template <class B>
int reserve(dpgicp_ctx *ctx, B &b, size_t bytes) {
  if (bytes <= b.cap) return DPGICP_OK;
  CU_TRY(ctx, b.alloc(std::max(bytes, (size_t)256)));
  return DPGICP_OK;
}

int check_params(dpgicp_ctx *ctx, const dpgicp_params *p) {
  if (!p) return fail(ctx, DPGICP_E_INVALID, "params is NULL");
  if (p->max_iterations < 1) return fail(ctx, DPGICP_E_INVALID, "max_iterations must be >= 1");
  if (p->downsample_divisor < 1) return fail(ctx, DPGICP_E_INVALID, "downsample_divisor must be >= 1");
  if (!(p->max_correspondence_distance > 0.0) || !std::isfinite(p->max_correspondence_distance))
    return fail(ctx, DPGICP_E_INVALID, "max_correspondence_distance must be positive and finite");
  if (p->max_correspondence_distance > 30.0)      /* sum of d^2 * 2^40 over 8192 pairs must fit int64 (arithmetic contract) */
    return fail(ctx, DPGICP_E_INVALID, "max_correspondence_distance must be <= 30 m");
  if (!(p->transformation_epsilon >= 0.0)) return fail(ctx, DPGICP_E_INVALID, "transformation_epsilon must be >= 0");
  if (p->metric != DPGICP_METRIC_POINT_TO_POINT && p->metric != DPGICP_METRIC_POINT_TO_LINE)
    return fail(ctx, DPGICP_E_INVALID, "metric must be DPGICP_METRIC_POINT_TO_POINT or DPGICP_METRIC_POINT_TO_LINE");
  if (p->search != DPGICP_SEARCH_BRUTE && p->search != DPGICP_SEARCH_PRUNED && p->search != DPGICP_SEARCH_PROJECTIVE)
    return fail(ctx, DPGICP_E_INVALID, "search must be DPGICP_SEARCH_BRUTE, DPGICP_SEARCH_PRUNED or DPGICP_SEARCH_PROJECTIVE");
  if (p->search == DPGICP_SEARCH_PROJECTIVE) {
    if (p->projective_window < 1 || p->projective_window > 1024)
      return fail(ctx, DPGICP_E_INVALID, "projective_window must be in 1..1024");
    if (!std::isfinite(p->sensor_x) || !std::isfinite(p->sensor_y) || std::fabs(p->sensor_x) > DPGICP_MAX_ABS_COORD ||
        std::fabs(p->sensor_y) > DPGICP_MAX_ABS_COORD)
      return fail(ctx, DPGICP_E_INVALID, "sensor_x / sensor_y must be finite and within DPGICP_MAX_ABS_COORD");
  }
  if (p->cov_mode < DPGICP_COV_REFERENCE_LIVE || p->cov_mode > DPGICP_COV_CENSI_CORR)
    return fail(ctx, DPGICP_E_INVALID, "cov_mode out of range");
  if (p->cov_cap < 0) return fail(ctx, DPGICP_E_INVALID, "cov_cap must be >= 0");
  if (p->outlier_mode != DPGICP_OUTLIER_NONE && p->outlier_mode != DPGICP_OUTLIER_TRIMMED && p->outlier_mode != DPGICP_OUTLIER_MEDIAN)
    return fail(ctx, DPGICP_E_INVALID, "outlier_mode must be DPGICP_OUTLIER_NONE, _TRIMMED or _MEDIAN");
  if (p->outlier_mode == DPGICP_OUTLIER_TRIMMED && !(p->outlier_param > 0.0 && p->outlier_param <= 1.0))
    return fail(ctx, DPGICP_E_INVALID, "outlier_param (overlap ratio) must be in (0, 1] for DPGICP_OUTLIER_TRIMMED");
  if (p->outlier_mode == DPGICP_OUTLIER_MEDIAN && !(p->outlier_param > 0.0 && std::isfinite(p->outlier_param)))
    return fail(ctx, DPGICP_E_INVALID, "outlier_param (median factor) must be positive and finite for DPGICP_OUTLIER_MEDIAN");
  return DPGICP_OK;
}

/* largest binary32 <= max_correspondence_distance^2 (binary64): same predicate as PCL's
 * `float_distance > double_threshold` */
float gate_threshold(const dpgicp_params *p) {
  const double d = p->max_correspondence_distance * p->max_correspondence_distance;
  float f = (float)d;
  if ((double)f > d) f = std::nextafterf(f, -INFINITY);
  return f;
}

using IcpKernel = void (*)(KernelParams);

/* the icp_pairs_kernel instantiation of a stage: nw warps per CTA run on the one with the next power-of-two register
 * budget; clusters (the last stage only) use the 16-warp budget */
template <int SEARCH>
IcpKernel icp_kernel_w(int nw, int csize, bool resume) {
  /* first stage of large scans: 12 warps with the 80-register budget so that two CTAs share an SM */
  if (csize == 1 && !resume && nw > 8 && nw <= 12) return icp_pairs_kernel<12, SEARCH, 1>;
  if (csize == 2) return icp_pairs_kernel<16, SEARCH, 2>;
  if (csize == 4) return icp_pairs_kernel<16, SEARCH, 4>;
  if (nw <= 1) return icp_pairs_kernel<1, SEARCH, 1>;
  if (nw <= 2) return icp_pairs_kernel<2, SEARCH, 1>;
  if (nw <= 4) return icp_pairs_kernel<4, SEARCH, 1>;
  if (nw <= 8) return icp_pairs_kernel<8, SEARCH, 1>;
  return icp_pairs_kernel<16, SEARCH, 1>;
}

IcpKernel icp_kernel(int search, int nw, int csize, bool resume) {
  if (search == DPGICP_SEARCH_PROJECTIVE) return icp_kernel_w<DPGICP_SEARCH_PROJECTIVE>(nw, csize, resume);
  if (search == DPGICP_SEARCH_PRUNED) return icp_kernel_w<DPGICP_SEARCH_PRUNED>(nw, csize, resume);
  if (search == kSearchPrunedFlat) return icp_kernel_w<kSearchPrunedFlat>(nw, csize, resume);
  if (search == kSearchPrunedStock) return icp_kernel_w<kSearchPrunedStock>(nw, csize, resume);
  if (search == kSearchPrunedFlatStock) return icp_kernel_w<kSearchPrunedFlatStock>(nw, csize, resume);
  return icp_kernel_w<DPGICP_SEARCH_BRUTE>(nw, csize, resume);
}

/* one stage of the chain: a persistent grid of `units` CTAs (csize 1) or clusters of csize CTAs, `warps` warps each */
struct Stage {
  IcpKernel kern;
  int warps, csize;
  size_t smem;
  int64_t units;
  long long handover;      /* KernelParams::handover (0 on the last stage, which never suspends) */
};

cudaLaunchConfig_t launch_config(const Stage &s, int64_t grid, cudaStream_t stream, cudaLaunchAttribute *cluster) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid, 1, 1);
  cfg.blockDim = dim3((unsigned)s.warps * 32, 1, 1);
  cfg.dynamicSmemBytes = s.smem;
  cfg.stream = stream;
  cluster->id = cudaLaunchAttributeClusterDimension;
  cluster->val.clusterDim.x = s.csize; cluster->val.clusterDim.y = 1; cluster->val.clusterDim.z = 1;
  cfg.attrs = cluster;
  cfg.numAttrs = s.csize > 1 ? 1 : 0;
  return cfg;
}

/* resident CTAs (csize 1) or clusters of stage s's kernel on the whole device.  The dynamic shared-memory opt-in and the
 * occupancy of a shape do not change between runs: set / queried once. */
int units(dpgicp_ctx *ctx, const Stage &s, int64_t *out) {
  const void *kfn = reinterpret_cast<const void *>(s.kern);
  {
    /* the attribute belongs to (device, function), not to a context: several contexts of one process share it, so it is
     * tracked process-wide and only ever raised */
    std::lock_guard<std::mutex> lock(g_optin_mutex);
    size_t &have = g_smem_optin[std::make_pair(ctx->device, kfn)];
    if (have < s.smem) {
      CU_TRY(ctx, cudaFuncSetAttribute(s.kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s.smem));
      have = s.smem;
    }
  }
  const auto key = std::make_tuple(kfn, s.warps, s.smem);
  auto occ = ctx->occupancy.find(key);
  if (occ == ctx->occupancy.end()) {
    int n = 0;
    if (s.csize > 1) {
      cudaLaunchAttribute cluster;
      const cudaLaunchConfig_t cfg = launch_config(s, (ctx->sm_count / s.csize) * s.csize, nullptr, &cluster);
      CU_TRY(ctx, cudaOccupancyMaxActiveClusters(&n, s.kern, &cfg));
      if (n < 1) return fail(ctx, DPGICP_E_TOOBIG, "no cluster of this shape fits the device");
    } else {
      CU_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, s.kern, s.warps * 32, s.smem));
      if (n < 1) return fail(ctx, DPGICP_E_TOOBIG, "scan too large for one CTA's shared memory");
      n *= ctx->sm_count;
    }
    occ = ctx->occupancy.emplace(key, n).first;
  }
  *out = occ->second;
  return DPGICP_OK;
}

int launch(dpgicp_ctx *ctx, cudaStream_t stream, const Stage &s, const KernelParams &kp) {
  cudaLaunchAttribute cluster;
  const cudaLaunchConfig_t cfg = launch_config(s, s.units * s.csize, stream, &cluster);
  CU_TRY(ctx, cudaLaunchKernelEx(&cfg, s.kern, kp));
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return DPGICP_OK;
}

/* warps per CTA close to `target` that split `tiles` 32-point tiles evenly (every warp gets
 * ceil(tiles / nw) or one fewer): 34 tiles -> 4, 7, 12, 17 for targets 4, 8, 16, 32 */
int balanced_warps(int tiles, int target, int csize = 1) {
  target = std::max(1, std::min(16, target));
  const int slots = target * csize;
  const int per_warp = (tiles + slots - 1) / slots;
  const int warps_total = (tiles + per_warp - 1) / per_warp;
  return std::max(1, (warps_total + csize - 1) / csize);
}

/* st[0 .. *n_stages) = the stage chain of `count` pairs of n_cap-point clouds.  trim: a rejector runs (its block-wide
 * select does not span a cluster); one_stage: the correspondences hook. */
int plan_stages(dpgicp_ctx *ctx, int search, int n_cap, int64_t count, bool trim, bool one_stage, Stage (&st)[5],
                int *n_stages) {
  const int tiles = n_cap / kTile;
  /* 34 tiles (1081 beams) -> 4, 7, 12 warps per CTA, then clusters of 4 CTAs x 9 warps (one tile per warp on four
   * SMs) for the last pairs: measured per-pass latency of one pair 28.7 / 17.9 / 11.4 / 6.3 us */
  const int w0 = n_cap <= 512 ? 2 : (n_cap <= 2048 ? 4 : 12);
  const StageTarget defaults[4] = {{w0, 1}, {std::min(16, 2 * w0), 1}, {16, 1}, {16, 4}};
  const StageTarget *targets = ctx->n_chain ? ctx->chain : defaults;
  const int n_targets = ctx->n_chain ? ctx->n_chain : (tiles >= 16 && !trim) ? 4 : 3;
  /* widths balanced against the tile count, a cluster only on the last stage (it never suspends), each wider than the
   * one before: narrow CTAs for the bulk of the batch, wider ones for the pairs still running when a queue runs dry */
  int n = 0;
  for (int k = 0; k < (one_stage ? 1 : n_targets); ++k) {
    const int cs = k > 0 && k + 1 == n_targets && !trim ? targets[k].csize : 1;
    const int w = balanced_warps(tiles, targets[k].warps, cs);
    if (n == 0 || w * cs > st[n - 1].warps * st[n - 1].csize)
      st[n++] = {icp_kernel(search, w, cs, k > 0), w, cs, smem_bytes(n_cap, search == DPGICP_SEARCH_PROJECTIVE, trim, w), 0, 0};
  }
  /* the hand-over bound towards stage s of cap units: DPGICP_HANDOVER's factor x its clusters (default 1) or CTAs
   * (default 2; the next stage's own queue-dry rule then takes over).  Factor 0: the plain queue-dry rule, no drop. */
  const auto bound = [&](const Stage &s, int64_t cap) {
    if (ctx->handover_factor <= 0.0) return (long long)1 << 40;
    return (long long)std::ceil((s.csize > 1 ? ctx->handover_cluster : ctx->handover_factor) * (double)cap);
  };
  int64_t cap;
  /* Small batches (the online caller's handful of pairs, a single runIcp-shaped call): a stage whose WHOLE batch is within
   * the hand-over bound towards the next stage would see its queue dry at once and suspend every pair after its first
   * pass — a launch, a state round trip through HBM and a re-staging for nothing.  Start the chain at the first stage that
   * would keep its pairs (the last one at the latest). */
  while (n > 1 && ctx->handover_factor > 0.0) {
    if (const int rc = units(ctx, st[1], &cap)) return rc;
    if (count > bound(st[1], cap)) break;
    std::copy(st + 1, st + n, st);
    --n;
  }
  st[0].kern = icp_kernel(search, st[0].warps, st[0].csize, false);      /* the first stage takes fresh pairs */
  /* persistent grids, never more than work items: stage 0's pairs, then the pairs the stage before can suspend */
  for (int k = 0; k < n; ++k) {
    if (const int rc = units(ctx, st[k], &cap)) return rc;
    if (k > 0) st[k - 1].handover = bound(st[k], cap);
    st[k].units = std::max<int64_t>(1, std::min(cap, k > 0 ? st[k - 1].units : count));
  }
  *n_stages = n;
  return DPGICP_OK;
}

/* the stage chain of batch b over store st, on slot s's stream with s's queue cells and state buffers (b is s's batch, or
 * the context's scratch batch for the single-pair shapes on the default slot) */
int launch_icp(dpgicp_slot *s, const Store &st, const Batch &b, const dpgicp_params *p, int32_t *corr_out,
               float *corr_d2, const int32_t *corr_seed = nullptr, int32_t *corr_nn_out = nullptr, int64_t first = 0,
               int64_t count = -1) {
  NvtxRange range("dpgicp: ICP + covariance stage chain");
  dpgicp_ctx *ctx = s->ctx;
  cudaStream_t stream = stream_of(s);
  const int div = p->downsample_divisor;
  int n_max = (st.max_count + div - 1) / div;
  int n_cap = ((std::max(n_max, 1) + kTile - 1) / kTile) * kTile;
  if (n_cap > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "scan exceeds DPGICP_MAX_POINTS");
  KernelParams kp;
  std::memset(&kp, 0, sizeof(kp));
  kp.store.pts = (const float2 *)st.rows.p;
  kp.store.count = (const int32_t *)st.count.p;
  kp.store.pitch = st.pitch;
  kp.store.n_scans = st.n_scans;
  if (count < 0) count = b.n_pairs - first;
  const bool whole = first == 0 && count == b.n_pairs;
  kp.tasks = (const PairTask *)b.tasks.p + first;
  kp.order = (b.has_order && whole) ? (const long long *)b.order.p : nullptr;
  kp.results = (dpgicp_result *)b.results.p + first;
  kp.pair_base = first;
  unsigned long long *const q = (unsigned long long *)s->d_queue.p;
  kp.counters = q + 8;
  kp.n_pairs = count;
  kp.n_cap = n_cap;
  kp.max_iterations = p->max_iterations;
  kp.use_reciprocal = p->use_reciprocal;
  kp.divisor = div;
  kp.metric = p->metric;
  kp.cov_mode = p->cov_mode;
  kp.cov_cap = p->cov_cap;
  kp.gate = gate_threshold(p);
  kp.one = 1.0f;
  kp.eps = p->transformation_epsilon;
  kp.rot_thr = 1.0 - p->transformation_epsilon;
  kp.sensor_var = p->cov_sensor_variance;
  kp.live[0] = p->laser_x_variance; kp.live[1] = p->laser_y_variance; kp.live[2] = p->laser_theta_variance;
  kp.corr_out = corr_out;
  kp.corr_d2_out = corr_d2;
  kp.corr_seed = corr_seed;
  kp.corr_nn_out = corr_nn_out;
  kp.outlier_mode = p->outlier_mode;
  kp.outlier_param = p->outlier_param;
  kp.slot_bytes = (long long)kStateHeader + 12ll * n_cap;
  if (ctx->gather_world > 1 && corr_out == nullptr && &b == &ctx->main.batch) {
    if ((b.n_pairs - 1) * (int64_t)ctx->gather_world + ctx->gather_rank >= ctx->gather_n)
      return fail(ctx, DPGICP_E_STATE, "the attached gather buffers are too small for this shard");
    kp.gather_world = ctx->gather_world;
    kp.gather_rank = ctx->gather_rank;
    kp.gather_fanout = ctx->gather_root_only ? 1 : ctx->gather_world;
    kp.gather_slots = ctx->gather_n;
    for (int g = 0; g < ctx->gather_world; ++g) kp.gather_peer[g] = (dpgicp_result *)ctx->gather_peer[g];
  }
  kp.proj_window = p->projective_window;
  kp.sensor_x = p->sensor_x;
  kp.sensor_y = p->sensor_y;
  const bool trim = p->outlier_mode != DPGICP_OUTLIER_NONE;
  /* clouds of at most 32 groups: the pruned search's flat instantiation (one candidate round, no upper box level) */
  int search = p->search;
  if (search == DPGICP_SEARCH_PRUNED) {
    /* ... and the stock configuration's: point-to-point, no rejector, no parity hook */
    const bool stock = p->metric == DPGICP_METRIC_POINT_TO_POINT && !trim && corr_out == nullptr && corr_seed == nullptr;
    const bool flat = n_cap / kGroup <= kFlatMaxGroups;
    search = stock ? (flat ? kSearchPrunedFlatStock : kSearchPrunedStock) : (flat ? kSearchPrunedFlat : DPGICP_SEARCH_PRUNED);
  }
  Stage stages[5];
  int n_stages = 0;
  int rc = plan_stages(ctx, search, n_cap, count, trim, corr_out != nullptr, stages, &n_stages);
  if (rc) return rc;
  CU_TRY(ctx, cudaMemsetAsync(q, 0, 32 * sizeof(unsigned long long), stream));
  const bool timing = s->stage_timing && corr_out == nullptr;
  if (timing) { s->last_stages = n_stages; CU_TRY(ctx, cudaEventRecord(s->stage_ev[0], stream)); }
  if (n_stages > 1) {
    /* every stage can suspend at most one pair per CTA: size the state slots for stage 0's grid */
    kp.slot_cap = stages[0].units;
    for (int k = 0; k < 2; ++k) {
      if ((rc = reserve(ctx, s->state[k], (size_t)kp.slot_cap * (size_t)kp.slot_bytes))) return rc;
      if ((rc = reserve(ctx, s->susp[k], (size_t)kp.slot_cap * sizeof(long long)))) return rc;
    }
  }
  for (int sidx = 0; sidx < n_stages; ++sidx) {
    KernelParams ks = kp;
    ks.queue = q + sidx;
    ks.resume = sidx > 0 ? 1 : 0;
    if (sidx > 0) {
      ks.in_count = reinterpret_cast<const unsigned int *>(q + 6 + ((sidx - 1) & 1));
      ks.susp_in = (const long long *)s->susp[(sidx - 1) & 1].p;
      ks.state_in = (const unsigned char *)s->state[(sidx - 1) & 1].p;
    }
    ks.finished = q + 24 + sidx;
    ks.handover = stages[sidx].handover;
    if (sidx + 1 < n_stages) {
      ks.out_count = reinterpret_cast<unsigned int *>(q + 6 + (sidx & 1));
      ks.susp_out = (long long *)s->susp[sidx & 1].p;
      ks.state_out = (unsigned char *)s->state[sidx & 1].p;
      if (sidx >= 2)      /* the count cell is reused by stage sidx: clear it after stage sidx-1 consumed it */
        CU_TRY(ctx, cudaMemsetAsync(q + 6 + (sidx & 1), 0, sizeof(unsigned long long), stream));
    }
    if ((rc = launch(ctx, stream, stages[sidx], ks))) return rc;
    if (timing) CU_TRY(ctx, cudaEventRecord(s->stage_ev[sidx + 1], stream));
  }
  return DPGICP_OK;
}

/* arguments of a range-scan write (dpgicp_upload_ranges, _upload_ranges_subset, _append_ranges, _convert_ranges_device) */
int check_ranges(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans, int32_t n_beams) {
  if (n_scans < 0 || n_beams < 2 || (n_scans > 0 && !ranges)) return fail(ctx, DPGICP_E_INVALID, "bad range-scan arguments");
  if (n_beams > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "n_beams exceeds DPGICP_MAX_POINTS");
  return DPGICP_OK;
}

/* arguments of a ragged cloud upload (dpgicp_upload_scans / dpgicp_append_scans): the largest scan and the point total */
int check_clouds(dpgicp_ctx *ctx, const void *points, size_t stride, const int64_t *offsets, int32_t n_scans,
                 int64_t *max_count, int64_t *total) {
  if (n_scans < 0 || (n_scans > 0 && (!offsets))) return fail(ctx, DPGICP_E_INVALID, "bad scan arguments");
  if (stride < 8 || (stride % 4) != 0) return fail(ctx, DPGICP_E_INVALID, "stride_bytes must be >= 8 and a multiple of 4");
  int64_t maxc = 0;
  for (int k = 0; k < n_scans; ++k) {
    const int64_t c = offsets[k + 1] - offsets[k];
    if (c < 0 || offsets[k] < 0) return fail(ctx, DPGICP_E_INVALID, "offsets must be non-negative and non-decreasing");
    maxc = std::max(maxc, c);
  }
  if (maxc > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "a scan has more than DPGICP_MAX_POINTS points");
  *max_count = maxc;
  *total = n_scans > 0 ? offsets[n_scans] : 0;
  if (*total > 0 && !points) return fail(ctx, DPGICP_E_INVALID, "points is NULL");
  return DPGICP_OK;
}

int set_pairs_into(dpgicp_ctx *ctx, cudaStream_t stream, const Store &st, Batch &b, const int32_t *src, const int32_t *tgt,
                   const float *guess, const float *T_direct, int64_t n) {
  if (n < 0 || (n > 0 && (!src || !tgt || (!guess && !T_direct))))
    return fail(ctx, DPGICP_E_INVALID, "bad pair arguments");
  if (st.n_scans <= 0 && n > 0) return fail(ctx, DPGICP_E_STATE, "no scans uploaded");
  /* dpgicp_run is asynchronous: the previous list's H2D copy out of the pinned staging buffer may still be queued
   * behind a running kernel; wait for it before the buffer is rewritten (or freed) */
  if (b.h_tasks_free) CU_TRY(ctx, cudaEventSynchronize(b.h_tasks_free));
  else CU_TRY(ctx, cudaEventCreateWithFlags(&b.h_tasks_free.h, cudaEventDisableTiming));
  int rc;
  if ((rc = reserve(ctx, b.h_tasks, sizeof(PairTask) * (size_t)n))) return rc;
  PairTask *h_tasks = (PairTask *)b.h_tasks.p;
  /* host threads share the loop (the libm cos/sin of the guesses is the bulk of it); the first offending pair is
   * reported, as the serial loop would */
  int64_t bad_index = n, bad_guess = n;
#pragma omp parallel for schedule(static) reduction(min : bad_index, bad_guess) if (n >= 4096)
  for (int64_t k = 0; k < n; ++k) {
    if (src[k] < 0 || src[k] >= st.n_scans || tgt[k] < 0 || tgt[k] >= st.n_scans) { if (k < bad_index) bad_index = k; continue; }
    PairTask t;
    t.src = src[k]; t.tgt = tgt[k];
    if (T_direct) {
      t.c = T_direct[4 * k]; t.s = T_direct[4 * k + 1]; t.tx = T_direct[4 * k + 2]; t.ty = T_direct[4 * k + 3];
    } else {
      /* Matrix4f guess of runIcp (dpg_slam.cc:374-378): cos/sin of the float angle, binary64 libm
       * rounded to binary32 (computed on the host so device and CPU agree bit for bit) */
      const float g0 = guess[3 * k], g1 = guess[3 * k + 1], g2 = guess[3 * k + 2];
      if (!std::isfinite(g0) || !std::isfinite(g1) || !std::isfinite(g2)) { if (k < bad_guess) bad_guess = k; continue; }
      t.c = (float)std::cos((double)g2); t.s = (float)std::sin((double)g2); t.tx = g0; t.ty = g1;
    }
    h_tasks[k] = t;
  }
  if (bad_index < n && bad_index <= bad_guess)
    return fail(ctx, DPGICP_E_INVALID, "pair index out of range at pair " + std::to_string(bad_index));
  if (bad_guess < n) return fail(ctx, DPGICP_E_RANGE, "non-finite guess at pair " + std::to_string(bad_guess));
  if ((rc = reserve(ctx, b.tasks, sizeof(PairTask) * (size_t)std::max<int64_t>(n, 1)))) return rc;
  if ((rc = reserve(ctx, b.results, sizeof(dpgicp_result) * (size_t)std::max<int64_t>(n, 1)))) return rc;
  if (n > 0)
    CU_TRY(ctx, cudaMemcpyAsync(b.tasks.p, h_tasks, sizeof(PairTask) * (size_t)n, cudaMemcpyHostToDevice, stream));
  CU_TRY(ctx, cudaEventRecord(b.h_tasks_free, stream));
  b.n_pairs = n;
  b.has_order = false;
  b.max_scan = -1;
  return DPGICP_OK;
}

/* cos/sin of every beam direction angle_i = angle_inc * i + angle_min (binary32, as createNode computes it,
 * dpg_slam.cc:497-504), evaluated in binary64 by the host's libm like the reference's double overloads
 * (dpg_measurement.h:102-104); uploaded once per scanner geometry */
int ensure_trig(dpgicp_ctx *ctx, int n_beams, float angle_min, float angle_inc) {
  if (ctx->trig_n == n_beams && ctx->trig_min == angle_min && ctx->trig_inc == angle_inc && ctx->trig.p) return DPGICP_OK;
  std::vector<double> t((size_t)n_beams * 2);
  for (int i = 0; i < n_beams; ++i) {
    const float angle = angle_inc * (float)i + angle_min;
    t[2 * (size_t)i] = std::cos((double)angle);
    t[2 * (size_t)i + 1] = std::sin((double)angle);
  }
  int rc;
  if ((rc = reserve(ctx, ctx->trig, sizeof(double) * t.size()))) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(ctx->trig.p, t.data(), sizeof(double) * t.size(), cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));      /* t goes out of scope */
  ctx->trig_n = n_beams; ctx->trig_min = angle_min; ctx->trig_inc = angle_inc;
  return DPGICP_OK;
}

/* close the peer mappings of the fused gather */
int gather_close(dpgicp_ctx *ctx) {
  for (int g = 0; g < ctx->gather_world; ++g) {
    if (!ctx->gather_local && g != ctx->gather_rank && ctx->gather_peer[g]) cudaIpcCloseMemHandle(ctx->gather_peer[g]);
    ctx->gather_peer[g] = nullptr;
  }
  ctx->gather_world = 0;
  ctx->gather_local = false;
  return DPGICP_OK;
}

/* The two clouds of a single-pair call (runIcp / calculate_ICP_COV shapes) as a two-row scratch store.  This is the
 * latency path: the rows are laid out on the host in a page-locked buffer (range check included — the counts are
 * known, so nothing has to come back from the device) and go up in one asynchronous copy; no kernel, no
 * synchronisation. */
int two_cloud_store(dpgicp_ctx *ctx, const void *a, int na, const void *b, int nb, size_t stride) {
  if (na < 0 || nb < 0 || (na > 0 && !a) || (nb > 0 && !b)) return fail(ctx, DPGICP_E_INVALID, "bad cloud arguments");
  if (stride < 8 || (stride % 4) != 0) return fail(ctx, DPGICP_E_INVALID, "stride_bytes must be >= 8 and a multiple of 4");
  if (na > DPGICP_MAX_POINTS || nb > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "a scan has more than DPGICP_MAX_POINTS points");
  Store &st = ctx->scratch_store;
  const int pitch = std::max(2, (std::max(na, nb) + 1) & ~1);
  const size_t row_bytes = sizeof(float2) * (size_t)pitch, blob = 2 * row_bytes + 16;
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));         /* a previous call's copy out of the buffer (already done: every
                                                            * single-pair call ends with a synchronisation) */
  int rc;
  if ((rc = reserve(ctx, ctx->h_pair, blob))) return rc;
  float *rows = (float *)ctx->h_pair.p;
  const void *src[2] = {a, b};
  const int cnt[2] = {na, nb};
  for (int r = 0; r < 2; ++r) {
    float *row = rows + (size_t)r * pitch * 2;
    const unsigned char *p = (const unsigned char *)src[r];
    for (int k = 0; k < cnt[r]; ++k) {
      const float *f = (const float *)(p + (size_t)k * stride);
      const float x = f[0], y = f[1];
      if (!(std::fabs(x) <= DPGICP_MAX_ABS_COORD) || !(std::fabs(y) <= DPGICP_MAX_ABS_COORD)) {
        st.n_scans = 0;
        return fail(ctx, DPGICP_E_RANGE, "scan store holds a non-finite point or |coordinate| > DPGICP_MAX_ABS_COORD");
      }
      row[2 * k] = x; row[2 * k + 1] = y;
    }
    std::memset(row + 2 * (size_t)cnt[r], 0, sizeof(float) * 2 * (size_t)(pitch - cnt[r]));
  }
  int32_t *h_cnt = (int32_t *)((char *)ctx->h_pair.p + 2 * row_bytes);
  h_cnt[0] = na; h_cnt[1] = nb;
  if ((rc = reserve(ctx, st.rows, 2 * row_bytes))) return rc;
  if ((rc = reserve(ctx, st.count, 2 * sizeof(int32_t)))) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(st.rows.p, rows, 2 * row_bytes, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(st.count.p, h_cnt, 2 * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  st.pitch = pitch;
  st.n_scans = 2;
  st.max_count = std::max(na, nb);
  st.h_count.assign({na, nb});
  return DPGICP_OK;
}

/* box levels over n >= 1 nodes: L = 1 boxes of 32 nodes, L + 1 boxes of 32 level-L boxes, until one warp can test the
 * top level at once; cnt[L - 1] = boxes of level L */
struct Levels {
  int levels = 0;
  int64_t cnt[kEnumMaxLevels] = {0};
};
Levels box_levels(int64_t n) {
  Levels lv;
  int64_t c = n;
  do {
    c = (c + kEnumFan - 1) / kEnumFan;
    lv.cnt[lv.levels++] = c;
  } while (c > kEnumFan && lv.levels < kEnumMaxLevels);
  return lv;
}

void set_levels(Nodes &N, const Levels &lv) {
  N.levels = lv.levels;
  for (int L = 0; L < lv.levels; ++L) N.level_cnt[L] = lv.cnt[L];
}

/* every box level above the leaves, from the leaves up (at most n / 1024 boxes), in the layout `off` */
void refit_upper_levels(dpgicp_ctx *ctx, NodeBox *bx, const int64_t *off, const Levels &lv) {
  for (int L = 1; L < lv.levels; ++L) {
    const int nb = (int)lv.cnt[L], blocks = (nb + 3) / 4;
    node_boxes_up_kernel<<<blocks, 128, 0, ctx->stream>>>(bx + off[L - 1], (int)lv.cnt[L - 1], bx + off[L], nb);
    ctx->launches++;
  }
}

/* the node row of one estimate: position, and theta with the cos / sin of -theta from the host's libm
 * (Eigen::Rotation2Df(-theta_1), math_utils.cc:28), which the enumeration's guesses take bit for bit */
inline void node_row(float x, float y, float th, float2 &xy, float4 &aux) {
  const float ang = -th;
  xy = make_float2(x, y);
  aux = make_float4(th, cosf(ang), sinf(ang), 0.f);
}

/* Room for n nodes in N.  Capacity grows by doubling and the box levels are laid out for the capacity, so a table that
 * grows one node at a time reallocates O(log n) times and keeps every level in place in between.  keep: the current
 * N.n nodes move to the new buffers (rows and leaf boxes device to device, upper levels refit in the new layout), so
 * the grown table is complete for N.n; the old buffers are freed only after the context's stream has drained.  The
 * level counts stay those of N.n: the caller sets them with the new count.  On failure N is as it was. */
int node_room(dpgicp_ctx *ctx, Nodes &N, int32_t n, bool keep) {
  const Levels lv = box_levels(n);
  if (lv.cnt[lv.levels - 1] > kEnumFan) return fail(ctx, DPGICP_E_TOOBIG, "too many nodes");
  if (n <= N.cap) return DPGICP_OK;
  const int32_t cap = (int32_t)std::min<int64_t>(INT32_MAX, std::max<int64_t>(n, 2 * (int64_t)N.cap));
  const Levels cap_lv = box_levels(cap);
  int64_t off[8] = {0}, total = 0;
  for (int L = 0; L < cap_lv.levels; ++L) { off[L] = total; total += cap_lv.cnt[L]; }
  DevBuf xy, aux, pass, boxes;
  CU_TRY(ctx, xy.alloc(sizeof(float2) * (size_t)cap));
  CU_TRY(ctx, aux.alloc(sizeof(float4) * (size_t)cap));
  CU_TRY(ctx, pass.alloc(sizeof(int32_t) * (size_t)cap));
  CU_TRY(ctx, boxes.alloc(sizeof(NodeBox) * (size_t)total));
  cudaError_t e = cudaSuccess;
  if (keep && N.n > 0) {
    const size_t m = (size_t)N.n;
    Levels old;
    old.levels = N.levels;
    for (int L = 0; L < N.levels; ++L) old.cnt[L] = N.level_cnt[L];
    e = cudaMemcpyAsync(xy.p, N.xy.p, sizeof(float2) * m, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(aux.p, N.aux.p, sizeof(float4) * m, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(pass.p, N.pass.p, sizeof(int32_t) * m, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(boxes.p, N.boxes.p, sizeof(NodeBox) * (size_t)old.cnt[0], cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) {
      refit_upper_levels(ctx, (NodeBox *)boxes.p, off, old);
      e = cudaGetLastError();
    }
  }
  const cudaError_t s = cudaStreamSynchronize(ctx->stream);   /* before the new buffers or the old ones are freed: an
                                                               * enqueued kernel may still read the old ones */
  CU_TRY(ctx, e);
  CU_TRY(ctx, s);
  N.xy = std::move(xy); N.aux = std::move(aux); N.pass = std::move(pass); N.boxes = std::move(boxes);
  N.cap = cap;
  for (int L = 0; L < 8; ++L) N.level_off[L] = off[L];
  return DPGICP_OK;
}

/* node estimates -> node table N on the device, plus the index-order box hierarchy the enumeration walks */
int set_nodes_impl(dpgicp_ctx *ctx, Nodes &N, const float *pose, const int32_t *pass, int32_t n, bool pose_is_xy) {
  N.n = 0;
  if (n == 0) return DPGICP_OK;
  std::vector<float2> xy((size_t)n);
  std::vector<float4> aux((size_t)n);
  const int stride = pose_is_xy ? 2 : 3;
  for (int32_t k = 0; k < n; ++k) {
    const float x = pose[(size_t)stride * k], y = pose[(size_t)stride * k + 1], th = pose_is_xy ? 0.0f : pose[(size_t)stride * k + 2];
    if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(th))
      return fail(ctx, DPGICP_E_RANGE, "non-finite node estimate at node " + std::to_string(k));
    node_row(x, y, th, xy[(size_t)k], aux[(size_t)k]);
  }
  int rc;
  if ((rc = node_room(ctx, N, n, false))) return rc;
  const Levels lv = box_levels(n);
  CU_TRY(ctx, cudaMemcpyAsync(N.xy.p, xy.data(), sizeof(float2) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(N.aux.p, aux.data(), sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(N.pass.p, pass, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  {
    const int nb = (int)lv.cnt[0], blocks = (nb + 3) / 4;
    node_boxes_leaf_kernel<<<blocks, 128, 0, ctx->stream>>>((const float2 *)N.xy.p, (const int32_t *)N.pass.p, n,
                                                            (NodeBox *)N.boxes.p, nb);
    ctx->launches++;
  }
  refit_upper_levels(ctx, (NodeBox *)N.boxes.p, N.level_off, lv);
  CU_TRY(ctx, cudaGetLastError());
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));         /* the host staging vectors go out of scope */
  set_levels(N, lv);
  N.n = n;
  return DPGICP_OK;
}

/* dpgicp_update_nodes on the context's table: the listed rows and the leaf boxes that hold them, then the upper levels.
 * Everything is checked on the host before the first device write; host work and copies scale with n_ids.  A CUDA
 * error once the device work has been enqueued empties the table, as a failed set_nodes_impl does. */
int update_nodes_impl(dpgicp_ctx *ctx, Nodes &N, int32_t n, const int32_t *ids, const float *pose, const int32_t *pass,
                      int32_t n_ids) {
  if (n_ids < 0 || (n_ids > 0 && (!ids || !pose || !pass))) return fail(ctx, DPGICP_E_INVALID, "bad node arguments");
  if (n < N.n) return fail(ctx, DPGICP_E_INVALID, "n_nodes is below the current node count: the table does not shrink");
  if (n_ids == 0 && n == N.n) return DPGICP_OK;
  std::vector<int32_t> copy;                /* ascending ids (what a diff of the estimate vector gives) are used as they are */
  const int32_t *sorted = ids, *sorted_end = ids + n_ids;
  if (!std::is_sorted(ids, ids + n_ids)) {
    copy.assign(ids, ids + n_ids);
    std::sort(copy.begin(), copy.end());
    sorted = copy.data(); sorted_end = sorted + n_ids;
  }
  if (n_ids > 0 && (sorted[0] < 0 || sorted_end[-1] >= n))
    return fail(ctx, DPGICP_E_INVALID, "node id out of range [0, n_nodes)");
  if (std::adjacent_find(sorted, sorted_end) != sorted_end) return fail(ctx, DPGICP_E_INVALID, "duplicate node id");
  const int64_t listed_new = sorted_end - std::lower_bound(sorted, sorted_end, N.n);
  if (listed_new != (int64_t)n - N.n) return fail(ctx, DPGICP_E_INVALID, "every new node id in [old count, n_nodes) must be listed");
  for (int32_t k = 0; k < n_ids; ++k)
    if (!std::isfinite(pose[3 * (size_t)k]) || !std::isfinite(pose[3 * (size_t)k + 1]) || !std::isfinite(pose[3 * (size_t)k + 2]))
      return fail(ctx, DPGICP_E_RANGE, "non-finite node estimate at node " + std::to_string(ids[k]));
  /* dirty leaves: the leaf of every listed id, ascending, once each */
  std::vector<int32_t> leaves;
  for (const int32_t *q = sorted; q != sorted_end; ++q)
    if (leaves.empty() || leaves.back() != *q / kEnumFan) leaves.push_back(*q / kEnumFan);
  /* staging: aux (float4) | xy (float2) | ids | pass | leaves */
  const size_t m = (size_t)n_ids, bytes = 32 * m + 4 * leaves.size();
  if (N.rows_free) CU_TRY(ctx, cudaEventSynchronize(N.rows_free));
  else CU_TRY(ctx, cudaEventCreateWithFlags(&N.rows_free.h, cudaEventDisableTiming));
  int rc;
  if ((rc = reserve(ctx, N.h_rows, std::max(bytes, bytes > N.h_rows.cap ? 2 * N.h_rows.cap : 0)))) return rc;
  if ((rc = reserve(ctx, N.d_rows, std::max(bytes, bytes > N.d_rows.cap ? 2 * N.d_rows.cap : 0)))) return rc;
  if ((rc = node_room(ctx, N, n, true))) return rc;
  const Levels lv = box_levels(n);
  char *h = (char *)N.h_rows.p;
  float4 *h_aux = (float4 *)h;
  float2 *h_xy = (float2 *)(h + 16 * m);
  std::memcpy(h + 24 * m, ids, 4 * m);
  std::memcpy(h + 28 * m, pass, 4 * m);
  std::memcpy(h + 32 * m, leaves.data(), 4 * leaves.size());
  for (size_t k = 0; k < m; ++k) node_row(pose[3 * k], pose[3 * k + 1], pose[3 * k + 2], h_xy[k], h_aux[k]);
  const char *d = (const char *)N.d_rows.p;
  cudaError_t e = cudaMemcpyAsync(N.d_rows.p, h, bytes, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) {
    node_rows_scatter_kernel<<<(n_ids + 127) / 128, 128, 0, ctx->stream>>>(
        (const int32_t *)(d + 24 * m), (const float2 *)(d + 16 * m), (const float4 *)d, (const int32_t *)(d + 28 * m), n_ids,
        (float2 *)N.xy.p, (float4 *)N.aux.p, (int32_t *)N.pass.p);
    const int nl = (int)leaves.size();
    node_boxes_refit_kernel<<<(nl + 3) / 4, 128, 0, ctx->stream>>>((const float2 *)N.xy.p, (const int32_t *)N.pass.p, n,
                                                                   (const int32_t *)(d + 32 * m), nl, (NodeBox *)N.boxes.p);
    ctx->launches += 2;
    refit_upper_levels(ctx, (NodeBox *)N.boxes.p, N.level_off, lv);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaEventRecord(N.rows_free, ctx->stream);
  if (e != cudaSuccess) N.n = 0;
  CU_TRY(ctx, e);
  set_levels(N, lv);
  N.n = n;
  return DPGICP_OK;
}

/* the caller's pair list of `mode` over node table N built on the device into batch b (this shard's part); host learns
 * the counts */
int enumerate_into(dpgicp_ctx *ctx, const Nodes &N, Batch &b, int mode, float r_same, float r_other, int rank, int world,
                   int64_t *n_total, int64_t *n_local) {
  if (n_total) *n_total = 0;
  if (n_local) *n_local = 0;
  b.n_pairs = 0; b.has_order = false; b.max_scan = -1;
  if (N.n < 2) return DPGICP_OK;
  const int n = N.n;
  const int n_chunks = mode == DPGICP_ENUM_ONLINE ? std::max(1, (n - 3 + 31) / 32) : n;
  int rc;
  if ((rc = reserve(ctx, ctx->enum_cnt, sizeof(unsigned long long) * ((size_t)n_chunks + 2)))) return rc;
  if ((rc = reserve(ctx, ctx->enum_amb, sizeof(AmbPair) * 4096))) return rc;
  EnumParams E;
  std::memset(&E, 0, sizeof(E));
  E.xy = (const float2 *)N.xy.p; E.pass = (const int32_t *)N.pass.p; E.aux = (const float4 *)N.aux.p;
  E.boxes = (const NodeBox *)N.boxes.p;
  for (int L = 0; L < N.levels; ++L) { E.level_off[L] = N.level_off[L]; E.level_cnt[L] = (int32_t)N.level_cnt[L]; }
  E.levels = N.levels; E.n = n; E.r_same = r_same; E.r_other = r_other;
  E.cnt = (unsigned long long *)ctx->enum_cnt.p;
  E.amb_count = E.cnt + n_chunks + 1;
  E.amb_list = (AmbPair *)ctx->enum_amb.p;
  E.amb_cap = (long long)(ctx->enum_amb.cap / sizeof(AmbPair));
  E.rank = rank; E.world = world;
  const int blocks = (n_chunks + 3) / 4;
  if (mode == DPGICP_ENUM_ONLINE) enumerate_online_kernel<false><<<blocks, 128, 0, ctx->stream>>>(E, n_chunks);
  else enumerate_reopt_kernel<false><<<blocks, 128, 0, ctx->stream>>>(E);
  scan_u64_kernel<<<1, 1024, 0, ctx->stream>>>(E.cnt, n_chunks);
  ctx->launches += 2;
  CU_TRY(ctx, cudaGetLastError());
  unsigned long long total = 0;
  CU_TRY(ctx, cudaMemcpyAsync(&total, E.cnt + n_chunks, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaMemsetAsync(E.amb_count, 0, sizeof(*E.amb_count), ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const int64_t local = (int64_t)total > rank ? ((int64_t)total - rank + world - 1) / world : 0;
  if (n_total) *n_total = (int64_t)total;
  if (n_local) *n_local = local;
  if ((rc = reserve(ctx, b.tasks, sizeof(PairTask) * (size_t)std::max<int64_t>(local, 1)))) return rc;
  if ((rc = reserve(ctx, b.results, sizeof(dpgicp_result) * (size_t)std::max<int64_t>(local, 1)))) return rc;
  E.tasks = (PairTask *)b.tasks.p;
  E.n_local = local;
  /* pairs whose cos/sin of the guess angle sit within a few binary64 ulps of a binary32 rounding boundary (about one
   * in 10^7 for random headings, but every pair of a recurring boundary heading difference): the device's libm and the
   * host's are not guaranteed to round them alike, so the host — whose libm defines the guess matrix everywhere else
   * (set_pairs) — re-derives them.  The fill pass lists them with their angles; when the list overflows, it grows to
   * the count and the (deterministic) fill pass runs again.  Then one copy down, host libm, one copy up and a scatter:
   * the number of synchronisations does not depend on the number of listed pairs. */
  unsigned long long amb = 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    if (mode == DPGICP_ENUM_ONLINE) enumerate_online_kernel<true><<<blocks, 128, 0, ctx->stream>>>(E, n_chunks);
    else enumerate_reopt_kernel<true><<<blocks, 128, 0, ctx->stream>>>(E);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaMemcpyAsync(&amb, E.amb_count, sizeof(amb), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (amb <= (unsigned long long)E.amb_cap) break;
    if ((rc = reserve(ctx, ctx->enum_amb, sizeof(AmbPair) * (size_t)amb))) return rc;
    E.amb_list = (AmbPair *)ctx->enum_amb.p;
    E.amb_cap = (long long)(ctx->enum_amb.cap / sizeof(AmbPair));
    CU_TRY(ctx, cudaMemsetAsync(E.amb_count, 0, sizeof(*E.amb_count), ctx->stream));
  }
  if (amb > (unsigned long long)E.amb_cap)        /* the second fill pass lists exactly the pairs the first one counted */
    return fail(ctx, DPGICP_E_STATE, "the guess re-derivation list changed between two identical fill passes");
  if (amb > 0) {
    std::vector<AmbPair> list(amb);
    CU_TRY(ctx, cudaMemcpyAsync(list.data(), E.amb_list, sizeof(AmbPair) * amb, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (AmbPair &p : list) {
      const float g2 = p.a;                      /* AngleMod of the pair, as dpgicp_relative_guess computes it */
      p.a = (float)std::cos((double)g2); p.b = (float)std::sin((double)g2);
    }
    CU_TRY(ctx, cudaMemcpyAsync(E.amb_list, list.data(), sizeof(AmbPair) * amb, cudaMemcpyHostToDevice, ctx->stream));
    amb_scatter_kernel<<<(unsigned)((amb + 255) / 256), 256, 0, ctx->stream>>>(E.amb_list, (long long)amb, E.tasks);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));   /* `list` goes out of scope */
  }
  b.n_pairs = local;
  b.max_scan = n - 1;
  return DPGICP_OK;
}

/* the pair list of a batch back on the host */
int fetch_pairs_from(dpgicp_ctx *ctx, cudaStream_t stream, const Batch &b, int32_t *src, int32_t *tgt, float *T, int64_t n) {
  if (n < 0 || n > b.n_pairs) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (n == 0) return DPGICP_OK;
  int rc;
  if ((rc = reserve(ctx, ctx->stage, (size_t)n * 24 + 64))) return rc;
  int32_t *d_src = (int32_t *)ctx->stage.p, *d_tgt = d_src + n;
  float4 *d_T = (float4 *)((char *)ctx->stage.p + (((size_t)n * 8 + 15) & ~(size_t)15));
  const int threads = 256;
  const long long blocks = (n + threads - 1) / threads;
  unpack_tasks_kernel<<<(unsigned)blocks, threads, 0, stream>>>((const PairTask *)b.tasks.p, (long long)n, src ? d_src : nullptr,
                                                                   tgt ? d_tgt : nullptr, T ? d_T : nullptr);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  if (src) CU_TRY(ctx, cudaMemcpyAsync(src, d_src, (size_t)n * 4, cudaMemcpyDeviceToHost, stream));
  if (tgt) CU_TRY(ctx, cudaMemcpyAsync(tgt, d_tgt, (size_t)n * 4, cudaMemcpyDeviceToHost, stream));
  if (T) CU_TRY(ctx, cudaMemcpyAsync(T, d_T, (size_t)n * 16, cudaMemcpyDeviceToHost, stream));
  CU_TRY(ctx, cudaStreamSynchronize(stream));
  return DPGICP_OK;
}

/* Room for n_new more rows of at least need_pitch (even) points behind the rows of the store, every existing row kept
 * (make_room of an append).  Rows and counts grow by doubling, so n one-scan appends copy O(n) rows in total; a scan longer
 * than the pitch re-pitches the kept rows on the device.  A buffer that moves is freed only after the context's stream
 * and every slot's stream have drained: the copy out of it, and any run enqueued before the append, read it.  On failure the store is as
 * it was. */
int grow_store(dpgicp_ctx *ctx, Store &st, int n_new, int need_pitch) {
  const int n_old = st.n_scans;
  const int64_t rows = (int64_t)n_old + n_new;
  const int pitch = n_old > 0 ? std::max(st.pitch, need_pitch) : need_pitch;
  const size_t row_bytes = sizeof(float2) * (size_t)pitch;
  const bool move_rows = (n_old > 0 && pitch != st.pitch) || (size_t)rows * row_bytes > st.rows.cap;
  const bool move_count = (size_t)rows * sizeof(int32_t) > st.count.cap;
  DevBuf nr, nc;            /* on failure freed on return, after the context's stream has drained the copies into them */
  auto cuda = [&](cudaError_t e, const char *what) {
    return e == cudaSuccess ? (int)DPGICP_OK
                            : fail(ctx, e == cudaErrorMemoryAllocation ? DPGICP_E_NOMEM : DPGICP_E_CUDA,
                                   std::string(what) + ": " + cudaGetErrorString(e));
  };
  int rc = DPGICP_OK;
  if (move_rows) {
    int64_t cap = st.pitch > 0 ? (int64_t)(st.rows.cap / (sizeof(float2) * (size_t)st.pitch)) : 0;
    if (rows > cap) cap = std::max(rows, 2 * cap);
    rc = cuda(nr.alloc((size_t)cap * row_bytes), "cudaMalloc (scan store growth)");
    if (!rc && n_old > 0 && pitch == st.pitch)
      rc = cuda(cudaMemcpyAsync(nr.p, st.rows.p, (size_t)n_old * row_bytes, cudaMemcpyDeviceToDevice, ctx->stream),
                "cudaMemcpyAsync (scan rows)");
    if (!rc && n_old > 0 && pitch != st.pitch) {
      const int threads = 128, blocks = (n_old + threads / 32 - 1) / (threads / 32);
      repitch_rows_kernel<<<blocks, threads, 0, ctx->stream>>>((const float4 *)st.rows.p, n_old, st.pitch, pitch, (float4 *)nr.p);
      ctx->launches++;
      rc = cuda(cudaGetLastError(), "repitch_rows_kernel");
    }
  }
  if (!rc && move_count) {
    const int64_t cap = std::max(rows, 2 * (int64_t)(st.count.cap / sizeof(int32_t)));
    rc = cuda(nc.alloc((size_t)cap * sizeof(int32_t)), "cudaMalloc (scan store growth)");
    if (!rc && n_old > 0)
      rc = cuda(cudaMemcpyAsync(nc.p, st.count.p, (size_t)n_old * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream),
                "cudaMemcpyAsync (scan counts)");
  }
  if (!rc && (move_rows || move_count)) rc = cuda(cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize");
  if (!rc && (move_rows || move_count)) rc = drain_slots(ctx);
  if (rc) {
    cudaStreamSynchronize(ctx->stream);
    return rc;
  }
  if (move_rows) st.rows = std::move(nr);       /* the old buffers go: nothing queued reads them any more */
  if (move_count) st.count = std::move(nc);
  st.pitch = pitch;
  return DPGICP_OK;
}

/* ---- the write path of the scan store ---------------------------------------------------------------------------
 * dpgicp_upload_scans, _upload_ranges, _upload_ranges_subset and _convert_ranges_device replace the store;
 * dpgicp_append_ranges and _append_scans append to it.  Each one checks its arguments before it touches anything (store,
 * batches, slots), then calls make_room, stages its input, converts into the rows behind n_scans (convert_ranges or
 * pack_clouds) and calls commit_rows.  From make_room on, a replace that fails for any reason leaves an empty store and
 * an append that fails leaves the store as it was. */

/* the row pitch for scans of at most n points: even, so that every row is 16-byte aligned */
int row_pitch(int64_t n) { return (int)std::max<int64_t>(2, (n + 1) & ~(int64_t)1); }

/* Room for n rows of at least `pitch` points behind n_scans, and the range flag cleared.
 * Replace: the slots drain and every batch empties (replace_store), and the store is emptied before any allocation.
 * Rows and counts are then reserved at exactly the size needed, the old buffers freed first, so a re-upload never holds
 * two copies of the store (3.5 GB at config 5).
 * Append: the row count must fit int32; then grow_store.  An empty append touches nothing. */
int make_room(dpgicp_ctx *ctx, bool append, int32_t n, int pitch) {
  Store &st = ctx->store;
  int rc;
  if (append) {
    if ((int64_t)st.n_scans + n > INT32_MAX) return fail(ctx, DPGICP_E_INVALID, "the store would hold more than 2^31 - 1 scans");
    if (n == 0) return DPGICP_OK;
    if ((rc = grow_store(ctx, st, n, pitch))) return rc;
  } else {
    if ((rc = replace_store(ctx))) return rc;
    st.n_scans = 0;
    st.max_count = 0;
    st.h_count.clear();
    if ((rc = reserve(ctx, st.rows, sizeof(float2) * (size_t)pitch * (size_t)std::max(n, 1)))) return rc;
    if ((rc = reserve(ctx, st.count, sizeof(int32_t) * (size_t)std::max(n, 1)))) return rc;
    st.pitch = pitch;
  }
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_bad.p, 0, sizeof(int), ctx->stream));
  return DPGICP_OK;
}

/* n range scans of n_beams beams in device memory -> the n rows behind n_scans (with d_ids: scan k is row d_ids[k] of
 * d_in).  The conversion of createNode (dpg_slam.cc:488-513) + getCachedPointCloudFromNode (dpg_node.cc:8-26); every
 * range-scan writer converts here, so an appended row is bit for bit the row one upload of the same scans holds. */
int convert_ranges(dpgicp_ctx *ctx, const float *d_in, const int32_t *d_ids, int32_t n, int32_t n_beams, float angle_min,
                   float angle_max, float range_max, float lx, float ly, float ltheta) {
  /* createNode dpg_slam.cc:497: angle_inc = (max - min) / (n - 1.0), stored as float */
  const float angle_inc = (float)(((double)(float)(angle_max - angle_min)) / ((double)n_beams - 1.0));
  const float lc = cosf(ltheta), ls = sinf(ltheta);       /* Eigen::Rotation2Df(ltheta), host libm */
  int rc;
  if ((rc = ensure_trig(ctx, n_beams, angle_min, angle_inc))) return rc;
  const Store &st = ctx->store;
  const int threads = 128, warps_per_block = threads / 32;
  const int blocks = (n + warps_per_block - 1) / warps_per_block;
  ranges_to_rows_kernel<<<blocks, threads, 0, ctx->stream>>>(d_in, d_ids, n, n_beams, (const double2 *)ctx->trig.p, range_max,
                                                            lx, ly, lc, ls, st.pitch, (float2 *)st.rows.p + (size_t)st.n_scans * st.pitch,
                                                            (int32_t *)st.count.p + st.n_scans, (int *)ctx->d_bad.p);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return DPGICP_OK;
}

/* n ragged host clouds (the layout of dpgicp_upload_scans, `total` points) -> the n rows behind n_scans */
int pack_clouds(dpgicp_ctx *ctx, const void *points, size_t stride, const int64_t *offsets, int32_t n, int64_t total) {
  int rc;
  if ((rc = reserve(ctx, ctx->stage, (size_t)total * stride + 16))) return rc;
  if ((rc = reserve(ctx, ctx->offsets, sizeof(int64_t) * ((size_t)n + 1)))) return rc;
  if (total > 0)
    CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, points, (size_t)total * stride, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(ctx->offsets.p, offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice,
                              ctx->stream));
  const Store &st = ctx->store;
  pack_rows_kernel<<<n, 256, 0, ctx->stream>>>((const unsigned char *)ctx->stage.p, stride, (const long long *)ctx->offsets.p,
                                               n, st.pitch, (float2 *)st.rows.p + (size_t)st.n_scans * st.pitch,
                                               (int32_t *)st.count.p + st.n_scans, (int *)ctx->d_bad.p);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return DPGICP_OK;
}

/* the counts of the n rows just written behind n_scans back to the host (only those) + the range flag.  The store takes
 * the rows only when every point is in range; otherwise n_scans stays where make_room left it: an append keeps its old
 * rows and count, a replace leaves an empty store. */
int commit_rows(dpgicp_ctx *ctx, int32_t n) {
  Store &st = ctx->store;
  const size_t first = (size_t)st.n_scans;
  st.h_count.resize(first + (size_t)n);
  int bad = 0;
  CU_TRY(ctx, cudaMemcpyAsync(st.h_count.data() + first, (const int32_t *)st.count.p + first, sizeof(int32_t) * (size_t)n,
                              cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(&bad, ctx->d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (bad) {
    st.h_count.resize(first);
    return fail(ctx, DPGICP_E_RANGE, "the scans hold a non-finite point or |coordinate| > DPGICP_MAX_ABS_COORD and were not "
                                     "stored (an append leaves the store as it was, a full upload leaves it empty)");
  }
  for (size_t k = first; k < st.h_count.size(); ++k) st.max_count = std::max(st.max_count, st.h_count[k]);
  st.n_scans = (int32_t)st.h_count.size();
  return mark_written(ctx);
}

/* the device cells and events of a slot (own_stream: a stream of its own, else the context's); on failure, deleting the
 * slot frees what was made */
cudaError_t slot_init(dpgicp_slot *s, dpgicp_ctx *ctx, bool own_stream) {
  s->ctx = ctx;
  cudaError_t e = s->d_queue.alloc(32 * sizeof(unsigned long long));
  for (Event &ev : s->stage_ev)
    if (e == cudaSuccess) e = cudaEventCreate(&ev.h);
  if (e == cudaSuccess && own_stream) e = cudaStreamCreateWithFlags(&s->own.h, cudaStreamNonBlocking);
  return e;
}

/* slot handles a caller holds: a destroyed (or never created) handle is refused, not followed */
std::mutex g_slots_mutex;
std::set<const dpgicp_slot *> g_slots;

dpgicp_slot *live(dpgicp_slot *s) {
  std::lock_guard<std::mutex> lock(g_slots_mutex);
  return s && g_slots.count(s) ? s : nullptr;
}

}  // namespace

/* ================================================================================================
 * exported C ABI
 * ============================================================================================== */
extern "C" {

int dpgicp_abi_version(void) { return DPGICP_ABI_VERSION; }

int dpgicp_default_params(dpgicp_params *p) {
  if (!p) return DPGICP_E_INVALID;
  std::memset(p, 0, sizeof(*p));
  p->max_iterations = 500;                  /* parameters.h:146 */
  p->use_reciprocal = 1;                    /* parameters.h:201 */
  p->ransac_iterations = 50;                /* parameters.h:191 */
  p->downsample_divisor = 5;                /* parameters.h:402 */
  p->metric = DPGICP_METRIC_POINT_TO_POINT;
  p->search = DPGICP_SEARCH_PRUNED;
  p->cov_mode = DPGICP_COV_REFERENCE_LIVE;  /* cov.h:572-575 */
  p->cov_cap = 200;                         /* cov.h:307 */
  p->transformation_epsilon = 5e-9;         /* parameters.h:159 */
  p->max_correspondence_distance = 0.6;     /* parameters.h:173 */
  p->cov_sensor_variance = 0.01;            /* cov.h:554 */
  p->laser_x_variance = 0.5f;               /* parameters.h:374 */
  p->laser_y_variance = 0.5f;               /* parameters.h:385 */
  p->laser_theta_variance = 0.3f;           /* parameters.h:396 */
  p->projective_window = 8;                 /* DPGICP_SEARCH_PROJECTIVE only */
  p->sensor_x = 0.2f;                       /* parameters.h:319-339: laser at (0.2, 0, 0) in base_link */
  p->sensor_y = 0.0f;
  return DPGICP_OK;
}

int dpgicp_create(int device, dpgicp_ctx **out) {
  if (!out) return fail(nullptr, DPGICP_E_INVALID, "out_ctx is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(nullptr, DPGICP_E_NODEVICE,
                std::string("no CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "count = 0") +
                    "); this library has no CPU fallback");
  if (device < 0 || device >= n) return fail(nullptr, DPGICP_E_NODEVICE, "device ordinal out of range");
  dpgicp_ctx *ctx = new (std::nothrow) dpgicp_ctx();
  if (!ctx) return fail(nullptr, DPGICP_E_NOMEM, "out of host memory");
  ctx->device = device;
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    delete ctx;
    return fail(nullptr, DPGICP_E_CUDA, cudaGetErrorString(e));
  }
  if (prop.major < 10) {
    delete ctx;
    return fail(nullptr, DPGICP_E_NODEVICE, "device is not sm_100 class; this library is built for sm_100a only");
  }
  ctx->sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->own_stream.h, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = ctx->d_bad.alloc(sizeof(int))) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->written.h, cudaEventDisableTiming)) != cudaSuccess ||
      (e = slot_init(&ctx->main, ctx, false)) != cudaSuccess) {
    delete ctx;                               /* frees what was made */
    return fail(nullptr, DPGICP_E_CUDA, cudaGetErrorString(e));
  }
  ctx->stream = ctx->own_stream;
  if (const char *c = std::getenv("DPGICP_HANDOVER")) {
    ctx->handover_factor = std::max(0.0, std::atof(c));
    if (const char *q = std::strchr(c, ',')) ctx->handover_cluster = std::max(0.0, std::atof(q + 1));
  }
  if (const char *c = std::getenv("DPGICP_CHAIN")) {
    for (const char *q = c; *q && ctx->n_chain < 5;) {      /* e.g. "4,8,16,9x2": the last stage as clusters of 2 CTAs x 9 warps */
      const int w = std::max(1, std::atoi(q));
      int cs = 1;
      while (*q && *q != ',') { if (*q == 'x') cs = std::atoi(q + 1); ++q; }
      ctx->chain[ctx->n_chain++] = {w, cs == 2 || cs == 4 ? cs : 1};
      if (*q == ',') ++q;
    }
  }
  *out = ctx;
  return DPGICP_OK;
}

void dpgicp_destroy(dpgicp_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  while (!ctx->slots.empty()) dpgicp_slot_destroy(ctx->slots.back());
  cudaStreamSynchronize(ctx->stream);         /* the members, which the stream's work may read, go only after it drained */
  gather_close(ctx);
  delete ctx;
}

const char *dpgicp_last_error(const dpgicp_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int dpgicp_set_stream(dpgicp_ctx *ctx, void *stream) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (stream) {
    ctx->own_stream.reset();                  /* the context's own stream goes; the caller's is never destroyed */
    ctx->stream = (cudaStream_t)stream;
  } else if (!ctx->own_stream) {
    CU_TRY(ctx, cudaStreamCreateWithFlags(&ctx->own_stream.h, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
  }
  return DPGICP_OK;
}

int dpgicp_synchronize(dpgicp_ctx *ctx) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

/* the scan-store writers: argument checks, then the write path above */
static int write_scans(dpgicp_ctx *ctx, bool append, const void *points, size_t stride, const int64_t *offsets,
                       int32_t n_scans) {
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int64_t maxc = 0, total = 0;
  int rc = check_clouds(ctx, points, stride, offsets, n_scans, &maxc, &total);
  if (rc || (rc = make_room(ctx, append, n_scans, row_pitch(maxc))) || n_scans == 0) return rc;
  if ((rc = pack_clouds(ctx, points, stride, offsets, n_scans, total))) return rc;
  return commit_rows(ctx, n_scans);
}

/* host ranges, converted on the device */
static int write_ranges(dpgicp_ctx *ctx, bool append, const float *ranges, int32_t n_scans, int32_t n_beams,
                        float angle_min, float angle_max, float range_max, float lx, float ly, float ltheta) {
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_ranges(ctx, ranges, n_scans, n_beams);
  if (rc || (rc = make_room(ctx, append, n_scans, row_pitch(n_beams))) || n_scans == 0) return rc;
  if ((rc = reserve(ctx, ctx->stage, sizeof(float) * (size_t)n_scans * (size_t)n_beams + 16))) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, ranges, sizeof(float) * (size_t)n_scans * (size_t)n_beams,
                              cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = convert_ranges(ctx, (const float *)ctx->stage.p, nullptr, n_scans, n_beams, angle_min, angle_max, range_max,
                           lx, ly, ltheta)))
    return rc;
  return commit_rows(ctx, n_scans);
}

int dpgicp_upload_scans(dpgicp_ctx *ctx, const void *points, size_t stride, const int64_t *offsets, int32_t n_scans) {
  if (!ctx) return DPGICP_E_INVALID;
  return write_scans(ctx, false, points, stride, offsets, n_scans);
}

int dpgicp_upload_ranges(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans, int32_t n_beams, float angle_min,
                         float angle_max, float range_max, float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: upload ranges + scan->cloud");
  return write_ranges(ctx, false, ranges, n_scans, n_beams, angle_min, angle_max, range_max, lx, ly, ltheta);
}

int dpgicp_upload_ranges_subset(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans_total, int32_t n_beams,
                                const int32_t *scan_ids, int32_t n_ids, float angle_min, float angle_max, float range_max,
                                float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_scans_total < 0 || (n_ids > 0 && !scan_ids)) return fail(ctx, DPGICP_E_INVALID, "bad range-scan arguments");
  int rc = check_ranges(ctx, ranges, n_ids, n_beams);
  if (rc) return rc;
  for (int32_t k = 0; k < n_ids; ++k)
    if (scan_ids[k] < 0 || scan_ids[k] >= n_scans_total)
      return fail(ctx, DPGICP_E_INVALID, "scan id out of range at position " + std::to_string(k));
  if ((rc = make_room(ctx, false, n_ids, row_pitch(n_beams))) || n_ids == 0) return rc;
  /* page-locked input: the kernel reads the selected rows straight from host memory, so only they cross the
   * bus and nothing is staged; pageable input: gather the rows through a pinned buffer and copy them */
  cudaPointerAttributes attr;
  const bool mapped = cudaPointerGetAttributes(&attr, ranges) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
                      attr.devicePointer != nullptr;
  cudaGetLastError();
  const float *d_in = nullptr;
  const int32_t *d_ids = nullptr;
  if (mapped) {
    if ((rc = reserve(ctx, ctx->offsets, sizeof(int32_t) * (size_t)n_ids))) return rc;
    CU_TRY(ctx, cudaMemcpyAsync(ctx->offsets.p, scan_ids, sizeof(int32_t) * (size_t)n_ids, cudaMemcpyHostToDevice, ctx->stream));
    d_in = (const float *)attr.devicePointer;
    d_ids = (const int32_t *)ctx->offsets.p;
  } else {
    const size_t bytes = sizeof(float) * (size_t)n_ids * (size_t)n_beams;
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));       /* the buffer may still feed a previous copy */
    if ((rc = reserve(ctx, ctx->h_stage, bytes))) return rc;
    for (int32_t k = 0; k < n_ids; ++k)
      std::memcpy((float *)ctx->h_stage.p + (size_t)k * n_beams, ranges + (size_t)scan_ids[k] * n_beams, sizeof(float) * (size_t)n_beams);
    if ((rc = reserve(ctx, ctx->stage, bytes + 16))) return rc;
    CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, ctx->h_stage.p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    d_in = (const float *)ctx->stage.p;
  }
  if ((rc = convert_ranges(ctx, d_in, d_ids, n_ids, n_beams, angle_min, angle_max, range_max, lx, ly, ltheta))) return rc;
  return commit_rows(ctx, n_ids);
}

int dpgicp_append_ranges(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans, int32_t n_beams, float angle_min,
                         float angle_max, float range_max, float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: append ranges + scan->cloud");
  return write_ranges(ctx, true, ranges, n_scans, n_beams, angle_min, angle_max, range_max, lx, ly, ltheta);
}

int dpgicp_append_scans(dpgicp_ctx *ctx, const void *points, size_t stride, const int64_t *offsets, int32_t n_scans) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: append clouds");
  return write_scans(ctx, true, points, stride, offsets, n_scans);
}

int dpgicp_scan_count(const dpgicp_ctx *ctx) { return ctx ? ctx->store.n_scans : DPGICP_E_INVALID; }

int dpgicp_download_scan(dpgicp_ctx *ctx, int32_t scan, float *xy, int32_t *n_points) {
  if (!ctx || !n_points) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const Store &st = ctx->store;
  if (scan < 0 || scan >= st.n_scans) return fail(ctx, DPGICP_E_INVALID, "scan index out of range");
  const int n = st.h_count[(size_t)scan];
  if (*n_points < n || (n > 0 && !xy)) { *n_points = n; return fail(ctx, DPGICP_E_TOOBIG, "output capacity too small"); }
  *n_points = n;
  if (n > 0) {
    CU_TRY(ctx, cudaMemcpyAsync(xy, (const float2 *)st.rows.p + (size_t)scan * st.pitch, sizeof(float2) * (size_t)n,
                                cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return DPGICP_OK;
}

static int set_pairs_slot(dpgicp_slot *s, const int32_t *src, const int32_t *tgt, const float *guess, int64_t n) {
  dpgicp_ctx *ctx = s->ctx;
  NvtxRange range("dpgicp: pair list");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  return set_pairs_into(ctx, stream_of(s), ctx->store, s->batch, src, tgt, guess, nullptr, n);
}

int dpgicp_set_pairs(dpgicp_ctx *ctx, const int32_t *src, const int32_t *tgt, const float *guess, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  return set_pairs_slot(&ctx->main, src, tgt, guess, n);
}

static int set_pair_cost_hints_slot(dpgicp_slot *s, const float *hints, int64_t n) {
  dpgicp_ctx *ctx = s->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  Batch &b = s->batch;
  if (!hints) { b.has_order = false; return DPGICP_OK; }
  if (n != b.n_pairs) return fail(ctx, DPGICP_E_INVALID, "hint count differs from the pair list");
  if (n == 0) return DPGICP_OK;
  for (int64_t k = 0; k < n; ++k)       /* a NaN would break the strict weak ordering the sorts below rely on */
    if (!std::isfinite(hints[k])) return fail(ctx, DPGICP_E_RANGE, "non-finite cost hint at pair " + std::to_string(k));
  /* Only the quarter of the pairs with the largest hints is moved to the front (most expensive first); the rest keep
   * their input order.  A full descending sort would put every pair predicted cheap at the very end — exactly where
   * a mispredicted long alignment hurts most; this way a misprediction starts at an arbitrary time, as without
   * hints, and scan locality of the input order is mostly kept. */
  std::vector<long long> order((size_t)n);
  for (int64_t k = 0; k < n; ++k) order[(size_t)k] = k;
  const int64_t head = std::max<int64_t>(1, n / 4);
  std::nth_element(order.begin(), order.begin() + (head - 1), order.end(),
                   [&](long long a, long long c) { return hints[a] > hints[c] || (hints[a] == hints[c] && a < c); });
  std::sort(order.begin(), order.begin() + head,
            [&](long long a, long long c) { return hints[a] > hints[c] || (hints[a] == hints[c] && a < c); });
  std::sort(order.begin() + head, order.end());
  int rc;
  if ((rc = reserve(ctx, b.order, sizeof(long long) * (size_t)n))) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(b.order.p, order.data(), sizeof(long long) * (size_t)n, cudaMemcpyHostToDevice, stream_of(s)));
  CU_TRY(ctx, cudaStreamSynchronize(stream_of(s)));        /* `order` goes out of scope */
  b.has_order = true;
  return DPGICP_OK;
}

int dpgicp_set_pair_cost_hints(dpgicp_ctx *ctx, const float *hints, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  return set_pair_cost_hints_slot(&ctx->main, hints, n);
}

/* slot s's whole batch, or its pairs [first, first + count); a slot with a stream of its own first waits
 * for the context's writes enqueued before (store, enumerated list) */
static int run_slot(dpgicp_slot *s, const dpgicp_params *params, bool whole, int64_t first, int64_t count) {
  dpgicp_ctx *ctx = s->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const int rc = check_params(ctx, params);
  if (rc) return rc;
  const Batch &b = s->batch;
  if (whole && b.n_pairs == 0) return DPGICP_OK;           /* an empty batch is valid and does nothing */
  if (b.n_pairs < 0) return fail(ctx, DPGICP_E_STATE, "no pair list set");
  if (!whole) {
    if (first < 0 || count < 0 || first + count > b.n_pairs) return fail(ctx, DPGICP_E_INVALID, "pair range outside the batch");
    if (count == 0) return DPGICP_OK;
  }
  if (ctx->store.n_scans <= 0) return fail(ctx, DPGICP_E_STATE, "no scans uploaded");
  if (b.max_scan >= ctx->store.n_scans)
    return fail(ctx, DPGICP_E_STATE, "the enumerated pair list refers to nodes without a scan in the store (node k owns scan k)");
  if (s->own) CU_TRY(ctx, cudaStreamWaitEvent(s->own, ctx->written, 0));
  return whole ? launch_icp(s, ctx->store, b, params, nullptr, nullptr)
               : launch_icp(s, ctx->store, b, params, nullptr, nullptr, nullptr, nullptr, first, count);
}

int dpgicp_run(dpgicp_ctx *ctx, const dpgicp_params *params) {
  if (!ctx) return DPGICP_E_INVALID;
  return run_slot(&ctx->main, params, true, 0, 0);
}

int dpgicp_run_range(dpgicp_ctx *ctx, const dpgicp_params *params, int64_t first, int64_t count) {
  if (!ctx) return DPGICP_E_INVALID;
  return run_slot(&ctx->main, params, false, first, count);
}

static int fetch_results_slot(dpgicp_slot *s, dpgicp_result *out, int64_t first, int64_t count) {
  dpgicp_ctx *ctx = s->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (first < 0 || count < 0 || first + count > s->batch.n_pairs || (count > 0 && !out)) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (count > 0)
    CU_TRY(ctx, cudaMemcpyAsync(out, (const dpgicp_result *)s->batch.results.p + first, sizeof(dpgicp_result) * (size_t)count,
                                cudaMemcpyDeviceToHost, stream_of(s)));
  CU_TRY(ctx, cudaStreamSynchronize(stream_of(s)));
  return DPGICP_OK;
}

int dpgicp_fetch_results_range(dpgicp_ctx *ctx, dpgicp_result *out, int64_t first, int64_t count) {
  if (!ctx) return DPGICP_E_INVALID;
  return fetch_results_slot(&ctx->main, out, first, count);
}

int dpgicp_gather_fetch_range(dpgicp_ctx *ctx, dpgicp_result *out, int64_t first, int64_t count) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (first < 0 || count < 0 || first + count > ctx->gather_n || (count > 0 && !out)) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (sizeof(dpgicp_result) * (size_t)(first + count) > ctx->gather.cap)
    return fail(ctx, DPGICP_E_STATE, "this rank holds no gathered records (root-only gather: fetch from rank 0)");
  if (count > 0)
    CU_TRY(ctx, cudaMemcpyAsync(out, (const dpgicp_result *)ctx->gather.p + first, sizeof(dpgicp_result) * (size_t)count,
                                cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

int dpgicp_fetch_results(dpgicp_ctx *ctx, dpgicp_result *out, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: fetch records");
  return fetch_results_slot(&ctx->main, out, 0, n);
}

static int fetch_factors_slot(dpgicp_slot *s, dpgicp_factor *out, int64_t n) {
  dpgicp_ctx *ctx = s->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n < 0 || n > s->batch.n_pairs || (n > 0 && !out)) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (n == 0) { CU_TRY(ctx, cudaStreamSynchronize(stream_of(s))); return DPGICP_OK; }
  int rc;
  if ((rc = reserve(ctx, ctx->stage, sizeof(dpgicp_factor) * (size_t)n))) return rc;
  const int threads = 128;
  const long long blocks = (n + threads - 1) / threads;
  factors_kernel<<<(unsigned)blocks, threads, 0, stream_of(s)>>>((const dpgicp_result *)s->batch.results.p,
                                                              (const PairTask *)s->batch.tasks.p, (long long)n,
                                                              (dpgicp_factor *)ctx->stage.p);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  CU_TRY(ctx, cudaMemcpyAsync(out, ctx->stage.p, sizeof(dpgicp_factor) * (size_t)n, cudaMemcpyDeviceToHost, stream_of(s)));
  CU_TRY(ctx, cudaStreamSynchronize(stream_of(s)));
  return DPGICP_OK;
}

int dpgicp_fetch_factors(dpgicp_ctx *ctx, dpgicp_factor *out, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  return fetch_factors_slot(&ctx->main, out, n);
}

static int gather_export_impl(dpgicp_ctx *ctx, int64_t n_global, int64_t n_alloc, unsigned char *handle_out) {
  static_assert(sizeof(cudaIpcMemHandle_t) == DPGICP_IPC_HANDLE_BYTES, "IPC handle size");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->gather_world > 0)
    return fail(ctx, DPGICP_E_STATE, "gather buffers are attached (peers may still store into this one): dpgicp_gather_detach on every rank first");
  /* a dedicated cudaMalloc allocation (IPC handles cover whole allocations) */
  ctx->gather.release();
  int rc;
  if ((rc = reserve(ctx, ctx->gather, sizeof(dpgicp_result) * (size_t)std::max<int64_t>(n_alloc, 1)))) return rc;
  CU_TRY(ctx, cudaMemsetAsync(ctx->gather.p, 0, ctx->gather.cap, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->gather_n = n_global;
  cudaIpcMemHandle_t h;
  CU_TRY(ctx, cudaIpcGetMemHandle(&h, ctx->gather.p));
  std::memcpy(handle_out, &h, sizeof(h));
  return DPGICP_OK;
}

int dpgicp_gather_export(dpgicp_ctx *ctx, int64_t n_global, unsigned char handle_out[DPGICP_IPC_HANDLE_BYTES]) {
  if (!ctx || !handle_out || n_global < 0) return DPGICP_E_INVALID;
  return gather_export_impl(ctx, n_global, n_global, handle_out);
}

int dpgicp_gather_declare(dpgicp_ctx *ctx, int64_t n_global, unsigned char handle_out[DPGICP_IPC_HANDLE_BYTES]) {
  if (!ctx || !handle_out || n_global < 0) return DPGICP_E_INVALID;
  return gather_export_impl(ctx, n_global, 1, handle_out);
}

int dpgicp_gather_attach(dpgicp_ctx *ctx, const unsigned char *handles, int32_t world, int32_t rank) {
  if (!ctx || !handles || world < 1 || world > DPGICP_MAX_GATHER_RANKS || rank < 0 || rank >= world) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (!ctx->gather.p) return fail(ctx, DPGICP_E_STATE, "dpgicp_gather_export must be called first");
  gather_close(ctx);
  for (int g = 0; g < world; ++g) {
    if (g == rank) { ctx->gather_peer[g] = ctx->gather.p; continue; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handles + (size_t)g * DPGICP_IPC_HANDLE_BYTES, sizeof(h));
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      ctx->gather_world = g; ctx->gather_rank = rank;       /* so that gather_close releases what was opened */
      gather_close(ctx);
      return fail(ctx, DPGICP_E_CUDA, std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(g) + "): " + cudaGetErrorString(e));
    }
    ctx->gather_peer[g] = p;
  }
  ctx->gather_world = world;
  ctx->gather_rank = rank;
  return DPGICP_OK;
}

int dpgicp_gather_set_root_only(dpgicp_ctx *ctx, int32_t root_only) {
  if (!ctx) return DPGICP_E_INVALID;
  ctx->gather_root_only = root_only != 0;
  return DPGICP_OK;
}

int dpgicp_gather_attach_local(dpgicp_ctx **ctxs, int32_t world, int64_t n_global, int32_t root_only) {
  if (!ctxs || world < 1 || world > DPGICP_MAX_GATHER_RANKS || n_global < 0) return DPGICP_E_INVALID;
  for (int r = 0; r < world; ++r) if (!ctxs[r]) return DPGICP_E_INVALID;
  /* every rank's buffer (rank 0's only when root_only), then peer access between the devices, then the pointers */
  for (int r = 0; r < world; ++r) {
    dpgicp_ctx *ctx = ctxs[r];
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    gather_close(ctx);
    ctx->gather.release();
    const int64_t want = (root_only && r > 0) ? 1 : std::max<int64_t>(n_global, 1);
    int rc;
    if ((rc = reserve(ctx, ctx->gather, sizeof(dpgicp_result) * (size_t)want))) return rc;
    CU_TRY(ctx, cudaMemsetAsync(ctx->gather.p, 0, ctx->gather.cap, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->gather_n = n_global;
    for (int g = 0; g < world; ++g) {
      if (ctxs[g]->device == ctx->device) continue;
      int can = 0;
      CU_TRY(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, ctxs[g]->device));
      if (!can) return fail(ctx, DPGICP_E_CUDA, "no peer access from device " + std::to_string(ctx->device) + " to device " + std::to_string(ctxs[g]->device));
      cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[g]->device, 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) return fail(ctx, DPGICP_E_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
    }
  }
  for (int r = 0; r < world; ++r) {
    dpgicp_ctx *ctx = ctxs[r];
    for (int g = 0; g < world; ++g) ctx->gather_peer[g] = ctxs[g]->gather.p;
    ctx->gather_world = world;
    ctx->gather_rank = r;
    ctx->gather_root_only = root_only != 0;
    ctx->gather_local = true;
  }
  return DPGICP_OK;
}

int dpgicp_gather_detach(dpgicp_ctx *ctx) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return gather_close(ctx);
}

int dpgicp_gather_fetch(dpgicp_ctx *ctx, dpgicp_result *out, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n < 0 || n > ctx->gather_n || (n > 0 && !out)) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (sizeof(dpgicp_result) * (size_t)n > ctx->gather.cap)
    return fail(ctx, DPGICP_E_STATE, "this rank holds no gathered records (root-only gather: fetch from rank 0)");
  if (n > 0)
    CU_TRY(ctx, cudaMemcpyAsync(out, ctx->gather.p, sizeof(dpgicp_result) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

int dpgicp_gather_device_ptr(dpgicp_ctx *ctx, void **out_ptr, int64_t *out_n) {
  if (!ctx || !out_ptr || !out_n) return DPGICP_E_INVALID;
  *out_ptr = ctx->gather.p;
  *out_n = ctx->gather_n;
  return DPGICP_OK;
}

int dpgicp_results_device_ptr(dpgicp_ctx *ctx, void **out_ptr, int64_t *out_n) {
  if (!ctx || !out_ptr || !out_n) return DPGICP_E_INVALID;
  *out_ptr = ctx->main.batch.results.p;
  *out_n = ctx->main.batch.n_pairs;
  return DPGICP_OK;
}

static int last_run_counters_slot(dpgicp_slot *s, uint64_t counters[8]) {
  dpgicp_ctx *ctx = s->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  unsigned long long h[8];
  CU_TRY(ctx, cudaMemcpyAsync(h, (const unsigned long long *)s->d_queue.p + 8, sizeof(h), cudaMemcpyDeviceToHost, stream_of(s)));
  CU_TRY(ctx, cudaStreamSynchronize(stream_of(s)));
  for (int k = 0; k < 8; ++k) counters[k] = h[k];
  counters[4] = ctx->launches;
  return DPGICP_OK;
}

int dpgicp_last_run_counters(dpgicp_ctx *ctx, uint64_t counters[8]) {
  if (!ctx || !counters) return DPGICP_E_INVALID;
  return last_run_counters_slot(&ctx->main, counters);
}

#ifdef DPGICP_PHASE_TIMING
/* development builds only: cycles thread 0 spent in each phase of the pass loop, summed over pairs */
int dpgicp_debug_phase_counters(dpgicp_ctx *ctx, uint64_t out[8]) {
  unsigned long long h[8];
  CU_TRY(ctx, cudaMemcpyAsync(h, (const unsigned long long *)ctx->main.d_queue.p + 16, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 8; ++k) out[k] = h[k];
  return DPGICP_OK;
}
#endif

int dpgicp_submit_pairs(dpgicp_ctx *ctx, const int32_t *src, const int32_t *tgt, const float *guess, int64_t n,
                        const dpgicp_params *params, dpgicp_result *out) {
  int rc;
  if ((rc = dpgicp_set_pairs(ctx, src, tgt, guess, n))) return rc;
  if ((rc = dpgicp_run(ctx, params))) return rc;
  return dpgicp_fetch_results(ctx, out, n);
}

int dpgicp_relative_guess(const float p1[3], const float p2[3], float guess[3]) {
  if (!p1 || !p2 || !guess) return DPGICP_E_INVALID;
  /* translate, rotate by Rotation2Df(-theta_1) (cosf/sinf of the float angle), AngleMod */
  const float tx = p2[0] - p1[0], ty = p2[1] - p1[1];
  const float ang = -p1[2];
  const float c = cosf(ang), s = sinf(ang), ms = -s;
  guess[0] = (c * tx) + (ms * ty);
  guess[1] = (s * tx) + (c * ty);
  double d = (double)(float)(p2[2] - p1[2]);
  d -= (M_PI * 2.0) * rint(d / (M_PI * 2.0));
  guess[2] = (float)d;
  return DPGICP_OK;
}

int dpgicp_single_pair(dpgicp_ctx *ctx, const void *source, int32_t n_source, const void *target, int32_t n_target,
                       size_t stride, const float guess[3], const dpgicp_params *params, dpgicp_result *out) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_params(ctx, params);
  if (rc) return rc;
  if (!guess || !out) return fail(ctx, DPGICP_E_INVALID, "guess/out is NULL");
  if ((rc = two_cloud_store(ctx, source, n_source, target, n_target, stride))) return rc;
  const int32_t s = 0, t = 1;
  if ((rc = set_pairs_into(ctx, ctx->stream, ctx->scratch_store, ctx->scratch_batch, &s, &t, guess, nullptr, 1))) return rc;
  if ((rc = launch_icp(&ctx->main, ctx->scratch_store, ctx->scratch_batch, params, nullptr, nullptr))) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(out, ctx->scratch_batch.results.p, sizeof(dpgicp_result), cudaMemcpyDeviceToHost,
                              ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

int dpgicp_correspondences_seeded(dpgicp_ctx *ctx, const void *source, int32_t n_source, const void *target,
                                  int32_t n_target, size_t stride, const float T[4], const dpgicp_params *params,
                                  const int32_t *prev_nn, int32_t *corr_tgt, float *corr_d2, int32_t *nn_out) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_params(ctx, params);
  if (rc) return rc;
  if (!T || (n_source > 0 && (!corr_tgt || !corr_d2))) return fail(ctx, DPGICP_E_INVALID, "T/corr outputs NULL");
  if (prev_nn)
    for (int32_t i = 0; i < n_source; ++i)
      if (prev_nn[i] < -1 || prev_nn[i] >= n_target) return fail(ctx, DPGICP_E_INVALID, "prev_nn out of range at point " + std::to_string(i));
  if ((rc = two_cloud_store(ctx, source, n_source, target, n_target, stride))) return rc;
  const int32_t s = 0, t = 1;
  if ((rc = set_pairs_into(ctx, ctx->stream, ctx->scratch_store, ctx->scratch_batch, &s, &t, nullptr, T, 1))) return rc;
  const size_t n = (size_t)std::max(n_source, 1);
  if ((rc = reserve(ctx, ctx->corr, n * 16))) return rc;
  dpgicp_params p = *params;
  p.downsample_divisor = 1;          /* the clouds given here are the ICP clouds */
  int32_t *d_corr = (int32_t *)ctx->corr.p;
  float *d_d2 = (float *)((char *)ctx->corr.p + n * 4);
  int32_t *d_seed = (int32_t *)((char *)ctx->corr.p + n * 8);
  int32_t *d_nn = (int32_t *)((char *)ctx->corr.p + n * 12);
  if (prev_nn && n_source > 0)
    CU_TRY(ctx, cudaMemcpyAsync(d_seed, prev_nn, sizeof(int32_t) * (size_t)n_source, cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = launch_icp(&ctx->main, ctx->scratch_store, ctx->scratch_batch, &p, d_corr, d_d2, prev_nn ? d_seed : nullptr, nn_out ? d_nn : nullptr))) return rc;
  if (n_source > 0) {
    CU_TRY(ctx, cudaMemcpyAsync(corr_tgt, d_corr, sizeof(int32_t) * (size_t)n_source, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(corr_d2, d_d2, sizeof(float) * (size_t)n_source, cudaMemcpyDeviceToHost, ctx->stream));
    if (nn_out) CU_TRY(ctx, cudaMemcpyAsync(nn_out, d_nn, sizeof(int32_t) * (size_t)n_source, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

int dpgicp_correspondences(dpgicp_ctx *ctx, const void *source, int32_t n_source, const void *target,
                           int32_t n_target, size_t stride, const float T[4], const dpgicp_params *params,
                           int32_t *corr_tgt, float *corr_d2) {
  return dpgicp_correspondences_seeded(ctx, source, n_source, target, n_target, stride, T, params, nullptr, corr_tgt, corr_d2, nullptr);
}

int dpgicp_cov(dpgicp_ctx *ctx, const void *data_pi, int32_t n_data, const void *model_qi, int32_t n_model,
               size_t stride, const float Tm[16], const dpgicp_params *params, double cov_out[9], uint32_t *status_out) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_params(ctx, params);
  if (rc) return rc;
  if (!Tm || !cov_out) return fail(ctx, DPGICP_E_INVALID, "transform/cov_out is NULL");
  if (params->cov_mode == DPGICP_COV_CENSI_CORR)
    return fail(ctx, DPGICP_E_INVALID, "dpgicp_cov pairs the clouds by index (LIVE or CENSI_INDEXPAIR); "
                                       "CENSI_CORR needs the ICP run (dpgicp_single_pair / submit_pairs)");
  if ((rc = two_cloud_store(ctx, data_pi, n_data, model_qi, n_model, stride))) return rc;
  const Store &st = ctx->scratch_store;
  CovItem it;
  it.p = (const float2 *)st.rows.p;
  it.q = (const float2 *)st.rows.p + st.pitch;
  it.n_p = n_data; it.n_q = n_model;
  it.c = Tm[0];  it.s = Tm[1];      /* column-major Matrix4f: T(0,0) = m[0], T(1,0) = m[1] */
  it.tx = Tm[12]; it.ty = Tm[13];   /* T(0,3) = m[12], T(1,3) = m[13]                      */
  if ((rc = reserve(ctx, ctx->misc, sizeof(CovItem) + 9 * sizeof(double) + 16))) return rc;
  char *base = (char *)ctx->misc.p;
  double *d_cov = (double *)base;
  uint32_t *d_status = (uint32_t *)(base + 9 * sizeof(double));
  CovItem *d_item = (CovItem *)(base + 9 * sizeof(double) + 16);
  CU_TRY(ctx, cudaMemcpyAsync(d_item, &it, sizeof(it), cudaMemcpyHostToDevice, ctx->stream));
  cov_indexpair_kernel<8><<<1, 256, 0, ctx->stream>>>(d_item, 1, params->cov_mode, params->cov_cap,
                                                      params->cov_sensor_variance, params->laser_x_variance,
                                                      params->laser_y_variance, params->laser_theta_variance, d_cov,
                                                      d_status);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  uint32_t status = 0;
  CU_TRY(ctx, cudaMemcpyAsync(cov_out, d_cov, 9 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(&status, d_status, sizeof(status), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (status_out) *status_out = status;
  return DPGICP_OK;
}

int dpgicp_cov_pairs(dpgicp_ctx *ctx, const int32_t *data_idx, const int32_t *model_idx, const float *T, int64_t n,
                     const dpgicp_params *params, double *cov_out, uint32_t *status_out, float *kernel_ms) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_params(ctx, params);
  if (rc) return rc;
  if (n < 0 || n > 0x7fffffff || (n > 0 && (!data_idx || !model_idx || !T || !cov_out || !status_out)))
    return fail(ctx, DPGICP_E_INVALID, "bad covariance batch arguments");
  if (params->cov_mode == DPGICP_COV_CENSI_CORR)
    return fail(ctx, DPGICP_E_INVALID, "dpgicp_cov_pairs pairs the clouds by index (LIVE or CENSI_INDEXPAIR)");
  const Store &st = ctx->store;
  if (n > 0 && st.n_scans <= 0) return fail(ctx, DPGICP_E_STATE, "no scans uploaded");
  if (kernel_ms) *kernel_ms = 0.f;
  if (n == 0) return DPGICP_OK;
  std::vector<CovItem> items((size_t)n);
  for (int64_t k = 0; k < n; ++k) {
    const int a = data_idx[k], b = model_idx[k];
    if (a < 0 || a >= st.n_scans || b < 0 || b >= st.n_scans)
      return fail(ctx, DPGICP_E_INVALID, "scan index out of range at item " + std::to_string(k));
    CovItem &it = items[(size_t)k];
    it.p = (const float2 *)st.rows.p + (size_t)a * st.pitch;
    it.q = (const float2 *)st.rows.p + (size_t)b * st.pitch;
    it.n_p = st.h_count[(size_t)a]; it.n_q = st.h_count[(size_t)b];
    it.c = T[4 * k]; it.s = T[4 * k + 1]; it.tx = T[4 * k + 2]; it.ty = T[4 * k + 3];
  }
  const size_t b_items = sizeof(CovItem) * (size_t)n, b_cov = sizeof(double) * 9 * (size_t)n, b_st = sizeof(uint32_t) * (size_t)n;
  if ((rc = reserve(ctx, ctx->stage, b_items + b_cov + b_st + 64))) return rc;
  char *base = (char *)ctx->stage.p;
  double *d_cov = (double *)base;
  CovItem *d_items = (CovItem *)(base + b_cov);
  uint32_t *d_status = (uint32_t *)(base + b_cov + b_items);
  CU_TRY(ctx, cudaMemcpyAsync(d_items, items.data(), b_items, cudaMemcpyHostToDevice, ctx->stream));
  Event e0, e1;
  CU_TRY(ctx, cudaEventCreate(&e0.h));
  CU_TRY(ctx, cudaEventCreate(&e1.h));
  CU_TRY(ctx, cudaEventRecord(e0, ctx->stream));
  /* one warp per item: no block reduction, the most independent items in flight (measured on B200 with a store larger
   * than L2: 82 % of the measured HBM copy bandwidth with 1 warp per item, 66 / 53 / 33 % with 2 / 4 / 8) */
  int cw = 1;
  if (const char *e = std::getenv("DPGICP_COV_WARPS")) cw = std::atoi(e);     /* development knob */
#define COV_LAUNCH(W)                                                                                              \
  cov_indexpair_kernel<W><<<(unsigned)n, W * 32, 0, ctx->stream>>>(d_items, (int)n, params->cov_mode, params->cov_cap, \
                                                                  params->cov_sensor_variance, params->laser_x_variance, \
                                                                  params->laser_y_variance, params->laser_theta_variance, d_cov, d_status)
  if (cw <= 1) COV_LAUNCH(1); else if (cw == 2) COV_LAUNCH(2); else if (cw <= 4) COV_LAUNCH(4); else COV_LAUNCH(8);
#undef COV_LAUNCH
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  CU_TRY(ctx, cudaEventRecord(e1, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(cov_out, d_cov, b_cov, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(status_out, d_status, b_st, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  if (kernel_ms) *kernel_ms = ms;
  return DPGICP_OK;
}

int dpgicp_enumerate_pairs(dpgicp_ctx *ctx, const float *node_xy, const int32_t *node_pass, int32_t n_nodes,
                           float r_same, float r_other, int32_t *src, int32_t *tgt, int64_t *n_pairs) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_nodes < 0 || !n_pairs || (n_nodes > 0 && (!node_xy || !node_pass)))
    return fail(ctx, DPGICP_E_INVALID, "bad node arguments");
  if (!(r_same >= 0.0f) || !(r_other >= 0.0f)) return fail(ctx, DPGICP_E_INVALID, "radii must be >= 0");
  const int64_t capacity = *n_pairs;
  *n_pairs = 0;
  if (n_nodes < 2) return DPGICP_OK;
  /* the device enumeration with the list copied out: its own positions-only table (theta = 0) and the scratch batch;
   * the node table of dpgicp_set_nodes and the batch stay as they are */
  int rc;
  if ((rc = set_nodes_impl(ctx, ctx->list_nodes, node_xy, node_pass, n_nodes, true))) return rc;
  int64_t total = 0, local = 0;
  rc = enumerate_into(ctx, ctx->list_nodes, ctx->scratch_batch, DPGICP_ENUM_REOPTIMIZE, r_same, r_other, 0, 1, &total, &local);
  if (rc) return rc;
  *n_pairs = total;
  if (total > capacity || (total > 0 && (!src || !tgt))) {
    ctx->scratch_batch.n_pairs = 0;
    return fail(ctx, DPGICP_E_TOOBIG, "pair capacity too small; required count returned in *n_pairs");
  }
  rc = fetch_pairs_from(ctx, ctx->stream, ctx->scratch_batch, src, tgt, nullptr, total);
  ctx->scratch_batch.n_pairs = 0;
  return rc;
}

int dpgicp_set_nodes(dpgicp_ctx *ctx, const float *pose, const int32_t *pass, int32_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n < 0 || (n > 0 && (!pose || !pass))) return fail(ctx, DPGICP_E_INVALID, "bad node arguments");
  return set_nodes_impl(ctx, ctx->nodes, pose, pass, n, false);
}

int dpgicp_update_nodes(dpgicp_ctx *ctx, int32_t n_nodes, const int32_t *ids, const float *pose, const int32_t *pass,
                        int32_t n_ids) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: update nodes");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  return update_nodes_impl(ctx, ctx->nodes, n_nodes, ids, pose, pass, n_ids);
}

/* enumeration into slot s: on the context's stream (synchronous, as the host re-derives guesses), after the slot's own
 * work has drained (its list and records are rewritten); the slot's later runs follow it through ctx->written */
static int enumerate_slot(dpgicp_slot *s, int32_t mode, float r_same, float r_other, int32_t rank, int32_t world,
                          int64_t *n_total, int64_t *n_local) {
  dpgicp_ctx *ctx = s->ctx;
  NvtxRange range("dpgicp: enumerate pairs (device)");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (mode != DPGICP_ENUM_REOPTIMIZE && mode != DPGICP_ENUM_ONLINE) return fail(ctx, DPGICP_E_INVALID, "mode must be DPGICP_ENUM_REOPTIMIZE or DPGICP_ENUM_ONLINE");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, DPGICP_E_INVALID, "bad shard arguments");
  if (!(r_same >= 0.0f) || !(r_other >= 0.0f)) return fail(ctx, DPGICP_E_INVALID, "radii must be >= 0");
  if (s->own) CU_TRY(ctx, cudaStreamSynchronize(s->own));
  if (ctx->nodes.n <= 0) {
    if (n_total) *n_total = 0;
    if (n_local) *n_local = 0;
    s->batch.n_pairs = 0;
    return DPGICP_OK;
  }
  int rc = enumerate_into(ctx, ctx->nodes, s->batch, mode, r_same, r_other, rank, world, n_total, n_local);
  if (rc) return rc;
  return s->own ? mark_written(ctx) : DPGICP_OK;
}

int dpgicp_enumerate_pairs_device(dpgicp_ctx *ctx, int32_t mode, float r_same, float r_other, int32_t rank, int32_t world,
                                  int64_t *n_total, int64_t *n_local) {
  if (!ctx) return DPGICP_E_INVALID;
  return enumerate_slot(&ctx->main, mode, r_same, r_other, rank, world, n_total, n_local);
}

int dpgicp_fetch_pairs(dpgicp_ctx *ctx, int32_t *src, int32_t *tgt, float *T, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  return fetch_pairs_from(ctx, ctx->stream, ctx->main.batch, src, tgt, T, n);
}

int dpgicp_convert_ranges_device(dpgicp_ctx *ctx, const float *d_ranges, int32_t n_scans, int32_t n_beams, float angle_min,
                                 float angle_max, float range_max, float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_ranges(ctx, d_ranges, n_scans, n_beams);
  if (rc || (rc = make_room(ctx, false, n_scans, row_pitch(n_beams))) || n_scans == 0) return rc;
  if ((rc = convert_ranges(ctx, d_ranges, nullptr, n_scans, n_beams, angle_min, angle_max, range_max, lx, ly, ltheta))) return rc;
  return commit_rows(ctx, n_scans);
}

int dpgicp_enable_stage_timing(dpgicp_ctx *ctx, int32_t on) {
  if (!ctx) return DPGICP_E_INVALID;
  ctx->main.stage_timing = on != 0;
  ctx->main.last_stages = 0;
  return DPGICP_OK;
}

int dpgicp_last_run_stage_ms(dpgicp_ctx *ctx, float stage_ms[8], int32_t *n_stages) {
  if (!ctx || !stage_ms || !n_stages) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  *n_stages = 0;
  for (int k = 0; k < 8; ++k) stage_ms[k] = 0.f;
  if (!ctx->main.stage_timing || ctx->main.last_stages <= 0) return fail(ctx, DPGICP_E_STATE, "stage timing is off (dpgicp_enable_stage_timing) or nothing has run");
  CU_TRY(ctx, cudaEventSynchronize(ctx->main.stage_ev[ctx->main.last_stages]));
  for (int k = 0; k < ctx->main.last_stages; ++k) CU_TRY(ctx, cudaEventElapsedTime(&stage_ms[k], ctx->main.stage_ev[k], ctx->main.stage_ev[k + 1]));
  *n_stages = ctx->main.last_stages;
  return DPGICP_OK;
}

int dpgicp_fp32_probe(dpgicp_ctx *ctx, double *mul_add, double *fma) {
  if (!ctx || !mul_add || !fma) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc;
  if ((rc = reserve(ctx, ctx->misc, 256))) return rc;
  Event e0, e1;
  CU_TRY(ctx, cudaEventCreate(&e0.h));
  CU_TRY(ctx, cudaEventCreate(&e1.h));
  const int iters = 1 << 14, blocks = ctx->sm_count * 8, threads = 256;
  double best[2] = {0.0, 0.0};
  for (int mode = 0; mode < 2; ++mode) {
    for (int rep = 0; rep < 4; ++rep) {           /* rep 0 warms up */
      CU_TRY(ctx, cudaEventRecord(e0, ctx->stream));
      if (mode == 0) fp32_probe_kernel<false><<<blocks, threads, 0, ctx->stream>>>((float *)ctx->misc.p, iters, 1.0000001f, 1e-7f);
      else fp32_probe_kernel<true><<<blocks, threads, 0, ctx->stream>>>((float *)ctx->misc.p, iters, 1.0000001f, 1e-7f);
      ctx->launches++;
      CU_TRY(ctx, cudaGetLastError());
      CU_TRY(ctx, cudaEventRecord(e1, ctx->stream));
      CU_TRY(ctx, cudaEventSynchronize(e1));
      float ms = 0.f;
      CU_TRY(ctx, cudaEventElapsedTime(&ms, e0, e1));
      const double ops = (double)blocks * threads * (double)iters * 8.0 * (mode == 0 ? 2.0 : 1.0);
      if (rep > 0 && ms > 0.f) best[mode] = std::max(best[mode], ops / (ms * 1e-3));
    }
  }
  *mul_add = best[0]; *fma = best[1];
  return DPGICP_OK;
}

int dpgicp_fp32x2_probe(dpgicp_ctx *ctx, double *mul_add_packed) {
  if (!ctx || !mul_add_packed) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc;
  if ((rc = reserve(ctx, ctx->misc, 256))) return rc;
  Event e0, e1;
  CU_TRY(ctx, cudaEventCreate(&e0.h));
  CU_TRY(ctx, cudaEventCreate(&e1.h));
  const int iters = 1 << 14, blocks = ctx->sm_count * 8, threads = 256;
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {             /* rep 0 warms up */
    CU_TRY(ctx, cudaEventRecord(e0, ctx->stream));
    fp32x2_probe_kernel<<<blocks, threads, 0, ctx->stream>>>((float *)ctx->misc.p, iters, 1.0000001f, 1e-7f, 1.0f);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaEventRecord(e1, ctx->stream));
    CU_TRY(ctx, cudaEventSynchronize(e1));
    float ms = 0.f;
    CU_TRY(ctx, cudaEventElapsedTime(&ms, e0, e1));
    const double ops = (double)blocks * threads * (double)iters * 8.0 * 4.0;   /* FMUL2 + packed sum = 2 instructions, 4 operations */
    if (rep > 0 && ms > 0.f) best = std::max(best, ops / (ms * 1e-3));
  }
  *mul_add_packed = best;
  return DPGICP_OK;
}

/* ---- batch slots ------------------------------------------------------------------------------------------------ */
int dpgicp_slot_create(dpgicp_ctx *ctx, dpgicp_slot **out) {
  if (!ctx || !out) return DPGICP_E_INVALID;
  *out = nullptr;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  dpgicp_slot *s = new (std::nothrow) dpgicp_slot();
  if (!s) return fail(ctx, DPGICP_E_NOMEM, "out of host memory");
  s->batch.n_pairs = -1;                     /* no pair list yet: a run is refused */
  cudaError_t e = slot_init(s, ctx, true);
  if (e != cudaSuccess) {
    delete s;
    return fail(ctx, e == cudaErrorMemoryAllocation ? DPGICP_E_NOMEM : DPGICP_E_CUDA, std::string("dpgicp_slot_create: ") + cudaGetErrorString(e));
  }
  ctx->slots.push_back(s);
  {
    std::lock_guard<std::mutex> lock(g_slots_mutex);
    g_slots.insert(s);
  }
  *out = s;
  return DPGICP_OK;
}

int dpgicp_slot_destroy(dpgicp_slot *slot) {
  dpgicp_slot *s = live(slot);
  if (!s) return DPGICP_E_INVALID;
  {
    std::lock_guard<std::mutex> lock(g_slots_mutex);
    g_slots.erase(s);
  }
  dpgicp_ctx *ctx = s->ctx;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(s->own);              /* the members, which the slot's work may read, go only after it drained */
  ctx->slots.erase(std::find(ctx->slots.begin(), ctx->slots.end(), s));
  delete s;
  return DPGICP_OK;
}

int dpgicp_slot_set_pairs(dpgicp_slot *slot, const int32_t *src, const int32_t *tgt, const float *guess, int64_t n) {
  dpgicp_slot *s = live(slot);
  return s ? set_pairs_slot(s, src, tgt, guess, n) : DPGICP_E_INVALID;
}

int dpgicp_slot_set_pair_cost_hints(dpgicp_slot *slot, const float *hints, int64_t n) {
  dpgicp_slot *s = live(slot);
  return s ? set_pair_cost_hints_slot(s, hints, n) : DPGICP_E_INVALID;
}

int dpgicp_slot_run(dpgicp_slot *slot, const dpgicp_params *params) {
  dpgicp_slot *s = live(slot);
  return s ? run_slot(s, params, true, 0, 0) : DPGICP_E_INVALID;
}

int dpgicp_slot_run_range(dpgicp_slot *slot, const dpgicp_params *params, int64_t first, int64_t count) {
  dpgicp_slot *s = live(slot);
  return s ? run_slot(s, params, false, first, count) : DPGICP_E_INVALID;
}

int dpgicp_slot_fetch_results(dpgicp_slot *slot, dpgicp_result *out, int64_t n) {
  dpgicp_slot *s = live(slot);
  return s ? fetch_results_slot(s, out, 0, n) : DPGICP_E_INVALID;
}

int dpgicp_slot_fetch_results_range(dpgicp_slot *slot, dpgicp_result *out, int64_t first, int64_t count) {
  dpgicp_slot *s = live(slot);
  return s ? fetch_results_slot(s, out, first, count) : DPGICP_E_INVALID;
}

int dpgicp_slot_fetch_factors(dpgicp_slot *slot, dpgicp_factor *out, int64_t n) {
  dpgicp_slot *s = live(slot);
  return s ? fetch_factors_slot(s, out, n) : DPGICP_E_INVALID;
}

int dpgicp_slot_fetch_pairs(dpgicp_slot *slot, int32_t *src, int32_t *tgt, float *T, int64_t n) {
  dpgicp_slot *s = live(slot);
  if (!s) return DPGICP_E_INVALID;
  CU_TRY(s->ctx, cudaSetDevice(s->ctx->device));
  return fetch_pairs_from(s->ctx, stream_of(s), s->batch, src, tgt, T, n);
}

int dpgicp_slot_last_run_counters(dpgicp_slot *slot, uint64_t counters[8]) {
  dpgicp_slot *s = live(slot);
  return s && counters ? last_run_counters_slot(s, counters) : DPGICP_E_INVALID;
}

int dpgicp_slot_synchronize(dpgicp_slot *slot) {
  dpgicp_slot *s = live(slot);
  if (!s) return DPGICP_E_INVALID;
  CU_TRY(s->ctx, cudaSetDevice(s->ctx->device));
  CU_TRY(s->ctx, cudaStreamSynchronize(s->own));
  return DPGICP_OK;
}

int dpgicp_slot_query(dpgicp_slot *slot) {
  dpgicp_slot *s = live(slot);
  if (!s) return DPGICP_E_INVALID;
  CU_TRY(s->ctx, cudaSetDevice(s->ctx->device));
  const cudaError_t e = cudaStreamQuery(s->own);
  if (e == cudaErrorNotReady) { cudaGetLastError(); return 0; }
  CU_TRY(s->ctx, e);
  return 1;
}

int dpgicp_slot_enumerate_pairs_device(dpgicp_slot *slot, int32_t mode, float r_same, float r_other, int32_t rank,
                                       int32_t world, int64_t *n_total, int64_t *n_local) {
  dpgicp_slot *s = live(slot);
  return s ? enumerate_slot(s, mode, r_same, r_other, rank, world, n_total, n_local) : DPGICP_E_INVALID;
}

}  /* extern "C" */
