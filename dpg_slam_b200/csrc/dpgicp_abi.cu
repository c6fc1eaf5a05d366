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
#include <string>
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

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct Store {                 /* padded rows + counts on the device, counts mirrored on the host */
  DevBuf rows, count;
  int32_t pitch = 0, n_scans = 0, max_count = 0;
  std::vector<int32_t> h_count;
};

struct Batch {
  DevBuf tasks, results, order;
  bool has_order = false;
  PairTask *h_tasks = nullptr;   /* pinned */
  size_t h_tasks_cap = 0;
  cudaEvent_t h_tasks_free = nullptr;   /* recorded after the H2D copy out of h_tasks: the buffer may be rewritten */
  int64_t n_pairs = 0;
  int32_t max_scan = -1;         /* device-enumerated lists: highest scan (= node) index used; -1 = validated on the host */
};

struct Nodes {                   /* pose-graph node estimates on the device (dpgicp_set_nodes) */
  DevBuf xy, aux, pass;          /* float2 (x, y); float4 (theta, cosf(-theta), sinf(-theta), 0); int32 pass */
  DevBuf boxes;                  /* index-order box hierarchy, all levels back to back */
  int32_t n = 0;
  int levels = 0;
  int64_t level_off[8] = {0}, level_cnt[8] = {0};
};

}  // namespace

struct dpgicp_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  Store store, scratch_store;
  Batch batch, scratch_batch;
  Nodes nodes;                               /* dpgicp_set_nodes: the table of dpgicp_enumerate_pairs_device */
  Nodes list_nodes;                          /* dpgicp_enumerate_pairs: its own positions-only table */
  DevBuf enum_amb;                           /* enumeration: pairs whose guess the host re-derives */
  DevBuf stage, offsets, misc, corr, trig, enum_cnt;
  /* per (kernel, warps, shared memory): resident CTAs per SM or clusters per device — queried once, not on every run */
  std::map<std::tuple<const void *, int, size_t>, int> occupancy;
  cudaEvent_t stage_ev[9] = {nullptr};
  bool stage_timing = false;
  int last_stages = 0;
  void *h_pair = nullptr;                    /* pinned scratch of the single-pair call shapes */
  size_t h_pair_cap = 0;
  DevBuf d_pair;
  int gather_root_only = 0;
  bool gather_local = false;                 /* peers attached by dpgicp_gather_attach_local (no IPC mappings to close) */
  int trig_n = 0;
  float trig_min = 0.f, trig_inc = 0.f;
  DevBuf state[2], susp[2];                  /* suspended-pair state slots + pair lists, ping-pong between stages */
  unsigned long long *d_queue = nullptr;     /* [0..4] stage queue heads, [6],[7] suspended counts, [8..15] counters, [16..23] development phase timers, [24..28] pairs finished per stage */
  DevBuf gather;                             /* this rank's copy of the whole batch's records (fused gather)  */
  int64_t gather_n = 0;
  int gather_world = 0, gather_rank = 0;
  void *gather_peer[DPGICP_MAX_GATHER_RANKS] = {nullptr};
  int max_stages = 5;
  std::vector<int> chain, chain_cluster;     /* DPGICP_CHAIN: target warps (and "x<cluster size>") per stage (development knob) */
  int *d_bad = nullptr;
  void *h_stage = nullptr;                   /* pinned staging for subset uploads from pageable memory */
  size_t h_stage_cap = 0;
  double handover_factor = 2.0;              /* DPGICP_HANDOVER="f[,fc]": a stage hands over once at most f x (CTAs of the next stage) pairs are */
  double handover_cluster = 1.0;             /* left; fc x (clusters) when the next stage runs clusters (development knob; 0 = plain queue-dry rule) */
  int force_warps = 0;
  int force_ctas_per_sm = 0;
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

int reserve(dpgicp_ctx *ctx, DevBuf &b, size_t bytes) {
  if (bytes <= b.cap) return DPGICP_OK;
  if (b.p) { CU_TRY(ctx, cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
  size_t want = std::max(bytes, (size_t)256);
  CU_TRY(ctx, cudaMalloc(&b.p, want));
  b.cap = want;
  return DPGICP_OK;
}

void release(DevBuf &b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr; b.cap = 0;
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

template <int WARPS, int SEARCH, int CSIZE>
int launch_icp_t(dpgicp_ctx *ctx, const KernelParams &kp, size_t smem, int64_t max_items, int nw, int *grid_out) {
  auto kern = icp_pairs_kernel<WARPS, SEARCH, CSIZE>;
  const void *kfn = reinterpret_cast<const void *>(kern);
  /* the dynamic shared-memory opt-in and the occupancy of a shape do not change between runs: set / query once */
  {
    /* the attribute belongs to (device, function), not to a context: several contexts of one process share it, so it is
     * tracked process-wide and only ever raised */
    std::lock_guard<std::mutex> lock(g_optin_mutex);
    size_t &have = g_smem_optin[std::make_pair(ctx->device, kfn)];
    if (have < smem) {
      CU_TRY(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      have = smem;
    }
  }
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3((unsigned)nw * 32, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CSIZE; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CSIZE > 1 ? 1 : 0;
  int64_t units = 0;                        /* resident CTAs (CSIZE == 1) or clusters on the whole device */
  const auto key = std::make_tuple(kfn, nw, smem);
  auto occ = ctx->occupancy.find(key);
  if (occ != ctx->occupancy.end()) {
    units = occ->second;
  } else if (CSIZE > 1) {
    cfg.gridDim = dim3((unsigned)(ctx->sm_count / CSIZE) * CSIZE, 1, 1);
    int n_clusters = 0;
    CU_TRY(ctx, cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg));
    if (n_clusters < 1) return fail(ctx, DPGICP_E_TOOBIG, "no cluster of this shape fits the device");
    units = n_clusters;
    ctx->occupancy[key] = n_clusters;
  } else {
    int per_sm = 0;
    CU_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nw * 32, smem));
    if (per_sm < 1) return fail(ctx, DPGICP_E_TOOBIG, "scan too large for one CTA's shared memory");
    units = (int64_t)ctx->sm_count * per_sm;
    ctx->occupancy[key] = (int)units;
  }
  if (CSIZE == 1 && ctx->force_ctas_per_sm > 0) units = std::min<int64_t>(units, (int64_t)ctx->sm_count * ctx->force_ctas_per_sm);
  /* persistent grid: a whole number of resident CTAs per SM (or clusters), never more than work items */
  if (units > max_items) units = max_items;
  if (units < 1) units = 1;
  const int64_t grid = units * CSIZE;
  if (grid_out) {
    if (*grid_out < 0) { *grid_out = (int)units; return DPGICP_OK; }      /* query only */
    *grid_out = (int)units;
  }
  cfg.gridDim = dim3((unsigned)grid, 1, 1);
  CU_TRY(ctx, cudaLaunchKernelEx(&cfg, kern, kp));
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return DPGICP_OK;
}

/* nw warps per CTA run on the instantiation with the next power-of-two register budget; clusters (the last
 * stage only) use the 16-warp budget */
template <int SEARCH>
int launch_icp_w(dpgicp_ctx *ctx, int nw, int csize, const KernelParams &kp, size_t smem, int64_t n, int *grid_out) {
  nw = std::max(1, std::min(nw, 16));
  /* first stage of large scans: 12 warps with the 80-register budget so that two CTAs share an SM */
  if (csize == 1 && !kp.resume && nw > 8 && nw <= 12) return launch_icp_t<12, SEARCH, 1>(ctx, kp, smem, n, nw, grid_out);
  if (csize == 2) return launch_icp_t<16, SEARCH, 2>(ctx, kp, smem, n, nw, grid_out);
  if (csize == 4) return launch_icp_t<16, SEARCH, 4>(ctx, kp, smem, n, nw, grid_out);
  if (nw <= 1) return launch_icp_t<1, SEARCH, 1>(ctx, kp, smem, n, 1, grid_out);
  if (nw <= 2) return launch_icp_t<2, SEARCH, 1>(ctx, kp, smem, n, nw, grid_out);
  if (nw <= 4) return launch_icp_t<4, SEARCH, 1>(ctx, kp, smem, n, nw, grid_out);
  if (nw <= 8) return launch_icp_t<8, SEARCH, 1>(ctx, kp, smem, n, nw, grid_out);
  return launch_icp_t<16, SEARCH, 1>(ctx, kp, smem, n, nw, grid_out);
}

int launch_stage(dpgicp_ctx *ctx, int search, int nw, int csize, const KernelParams &kp, size_t smem, int64_t n, int *grid_out) {
  if (search == DPGICP_SEARCH_PROJECTIVE) return launch_icp_w<DPGICP_SEARCH_PROJECTIVE>(ctx, nw, csize, kp, smem, n, grid_out);
  if (search == DPGICP_SEARCH_PRUNED) return launch_icp_w<DPGICP_SEARCH_PRUNED>(ctx, nw, csize, kp, smem, n, grid_out);
  if (search == kSearchPrunedFlat) return launch_icp_w<kSearchPrunedFlat>(ctx, nw, csize, kp, smem, n, grid_out);
  if (search == kSearchPrunedStock) return launch_icp_w<kSearchPrunedStock>(ctx, nw, csize, kp, smem, n, grid_out);
  if (search == kSearchPrunedFlatStock) return launch_icp_w<kSearchPrunedFlatStock>(ctx, nw, csize, kp, smem, n, grid_out);
  return launch_icp_w<DPGICP_SEARCH_BRUTE>(ctx, nw, csize, kp, smem, n, grid_out);
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

int launch_icp(dpgicp_ctx *ctx, const Store &st, const Batch &b, const dpgicp_params *p, int32_t *corr_out,
               float *corr_d2, const int32_t *corr_seed = nullptr, int32_t *corr_nn_out = nullptr, int64_t first = 0,
               int64_t count = -1) {
  NvtxRange range("dpgicp: ICP + covariance stage chain");
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
  kp.counters = ctx->d_queue + 8;
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
  if (ctx->gather_world > 1 && corr_out == nullptr && &b == &ctx->batch) {
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
  /* shared memory of a stage: the reduction scratch grows with the CTA width */
  auto smem_of = [&](int warps) { return smem_bytes(n_cap, p->search == DPGICP_SEARCH_PROJECTIVE, trim, warps); };
  /* clouds of at most 32 groups: the pruned search's flat instantiation (one candidate round, no upper box level) */
  int search = p->search;
  if (search == DPGICP_SEARCH_PRUNED) {
    /* ... and the stock configuration's: point-to-point, no rejector, no parity hook */
    const bool stock = p->metric == DPGICP_METRIC_POINT_TO_POINT && !trim && corr_out == nullptr && corr_seed == nullptr;
    const bool flat = n_cap / kGroup <= kFlatMaxGroups;
    search = stock ? (flat ? kSearchPrunedFlatStock : kSearchPrunedStock) : (flat ? kSearchPrunedFlat : DPGICP_SEARCH_PRUNED);
  }

  /* stage widths (warps per pair): narrow CTAs for the bulk of the batch, wider ones for the pairs
   * still running when a stage's queue runs dry; each width is balanced against the tile count */
  const int tiles = n_cap / kTile;
  int w0 = ctx->force_warps;
  if (w0 <= 0) w0 = n_cap <= 512 ? 2 : (n_cap <= 2048 ? 4 : 12);
  struct StageShape { int warps, csize; };
  /* 34 tiles (1081 beams) -> 4, 7, 12 warps per CTA, then clusters of 4 CTAs x 9 warps (one tile per warp on four
   * SMs) for the last pairs: measured per-pass latency of one pair 28.7 / 17.9 / 11.4 / 6.3 us */
  StageShape targets[5] = {{w0, 1}, {std::min(16, 2 * w0), 1}, {16, 1}, {16, 4}, {16, 1}};
  int n_targets = (tiles >= 16 && !trim) ? 4 : 3;      /* the rejector's block-wide select does not span a cluster */
  if (!ctx->chain.empty()) {
    n_targets = 0;
    for (size_t k = 0; k < ctx->chain.size() && n_targets < 5; ++k)
      targets[n_targets++] = {ctx->chain[k], trim ? 1 : ctx->chain_cluster[k]};
  }
  StageShape shapes[5] = {{balanced_warps(tiles, targets[0].warps), 1}, {0, 1}, {0, 1}, {0, 1}, {0, 1}};
  int n_stages = 1;
  if (corr_out == nullptr) {
    for (int k = 1; k < n_targets && n_stages < ctx->max_stages; ++k) {
      /* a cluster of CTAs per pair is only used for the last stage (it never suspends) */
      const int cs = (k + 1 == n_targets || n_stages + 1 == ctx->max_stages) ? targets[k].csize : 1;
      const int w = balanced_warps(tiles, targets[k].warps, cs);
      if (w * cs <= shapes[n_stages - 1].warps * shapes[n_stages - 1].csize) continue;
      shapes[n_stages++] = {w, cs};
    }
  }
  /* Small batches (the online caller's handful of pairs, a single runIcp-shaped call): a stage whose WHOLE batch is within
   * the hand-over bound towards the next stage would see its queue dry at once and suspend every pair after its first
   * pass — a launch, a state round trip through HBM and a re-staging for nothing.  Start the chain at the first stage that
   * would keep its pairs (the last one at the latest). */
  while (n_stages > 1 && ctx->handover_factor > 0.0) {
    int next_units = -1;
    KernelParams kq = kp;
    kq.resume = 1;
    int rcq = launch_stage(ctx, search, shapes[1].warps, shapes[1].csize, kq, smem_of(shapes[1].warps), (int64_t)1 << 40, &next_units);
    if (rcq) return rcq;
    const long long bound = (long long)std::ceil((shapes[1].csize > 1 ? ctx->handover_cluster : ctx->handover_factor) * (double)next_units);
    if (count > bound) break;
    for (int k = 1; k < n_stages; ++k) shapes[k - 1] = shapes[k];
    --n_stages;
  }
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_queue, 0, 32 * sizeof(unsigned long long), ctx->stream));
  int grid_prev = 0;
  const bool timing = ctx->stage_timing && corr_out == nullptr;
  if (timing) { ctx->last_stages = n_stages; CU_TRY(ctx, cudaEventRecord(ctx->stage_ev[0], ctx->stream)); }
  if (n_stages > 1) {
    /* every stage can suspend at most one pair per CTA: size the state slots for stage 0's grid */
    int g0 = -1;
    int rc = launch_stage(ctx, search, shapes[0].warps, shapes[0].csize, kp, smem_of(shapes[0].warps), count, &g0);
    if (rc) return rc;
    for (int k = 0; k < 2; ++k) {
      if ((rc = reserve(ctx, ctx->state[k], (size_t)g0 * (size_t)kp.slot_bytes))) return rc;
      if ((rc = reserve(ctx, ctx->susp[k], (size_t)g0 * sizeof(long long)))) return rc;
    }
    kp.slot_cap = g0;
  }
  for (int sidx = 0; sidx < n_stages; ++sidx) {
    KernelParams ks = kp;
    ks.queue = ctx->d_queue + sidx;
    ks.resume = sidx > 0 ? 1 : 0;
    if (sidx > 0) {
      ks.in_count = reinterpret_cast<const unsigned int *>(ctx->d_queue + 6 + ((sidx - 1) & 1));
      ks.susp_in = (const long long *)ctx->susp[(sidx - 1) & 1].p;
      ks.state_in = (const unsigned char *)ctx->state[(sidx - 1) & 1].p;
    }
    ks.finished = ctx->d_queue + 24 + sidx;
    if (sidx + 1 < n_stages) {
      /* hand over once the next stage could run all that is left at once (clusters: exactly; CTAs: a third more,
       * the next stage's own queue-dry rule then takes over) */
      int next_units = -1;
      KernelParams kq = kp;
      kq.resume = 1;                        /* occupancy query for the shape the next stage will really use */
      int rcq = launch_stage(ctx, search, shapes[sidx + 1].warps, shapes[sidx + 1].csize, kq, smem_of(shapes[sidx + 1].warps), (int64_t)1 << 40, &next_units);
      if (rcq) return rcq;
      ks.handover = (long long)std::ceil((shapes[sidx + 1].csize > 1 ? ctx->handover_cluster : ctx->handover_factor) * (double)next_units);
      if (ctx->handover_factor <= 0.0) ks.handover = (long long)1 << 40;      /* development: the plain queue-dry rule */
      ks.out_count = reinterpret_cast<unsigned int *>(ctx->d_queue + 6 + (sidx & 1));
      ks.susp_out = (long long *)ctx->susp[sidx & 1].p;
      ks.state_out = (unsigned char *)ctx->state[sidx & 1].p;
      if (sidx >= 2)      /* the count cell is reused by stage sidx: clear it after stage sidx-1 consumed it */
        CU_TRY(ctx, cudaMemsetAsync(ctx->d_queue + 6 + (sidx & 1), 0, sizeof(unsigned long long), ctx->stream));
    }
    int grid = 0;
    const int64_t max_items = sidx == 0 ? count : (int64_t)grid_prev;
    int rc = launch_stage(ctx, search, shapes[sidx].warps, shapes[sidx].csize, ks, smem_of(shapes[sidx].warps), max_items, &grid);
    if (rc) return rc;
    grid_prev = grid;
    if (timing) CU_TRY(ctx, cudaEventRecord(ctx->stage_ev[sidx + 1], ctx->stream));
  }
  return DPGICP_OK;
}

int finish_store(dpgicp_ctx *ctx, Store &st, int n_scans) {
  /* counts back to the host (sizing of shared memory, argument validation) + range flag */
  st.h_count.resize((size_t)n_scans);
  int bad = 0;
  CU_TRY(ctx, cudaMemcpyAsync(st.h_count.data(), st.count.p, sizeof(int32_t) * (size_t)n_scans,
                              cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(&bad, ctx->d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  st.n_scans = n_scans;
  st.max_count = 0;
  for (int32_t c : st.h_count) st.max_count = std::max(st.max_count, c);
  if (bad) {
    st.n_scans = 0;
    return fail(ctx, DPGICP_E_RANGE, "scan store holds a non-finite point or |coordinate| > DPGICP_MAX_ABS_COORD");
  }
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

int upload_scans_into(dpgicp_ctx *ctx, Store &st, const void *points, size_t stride, const int64_t *offsets,
                      int32_t n_scans) {
  int64_t maxc = 0, total = 0;
  int rc = check_clouds(ctx, points, stride, offsets, n_scans, &maxc, &total);
  if (rc) return rc;
  const int pitch = (int)std::max<int64_t>(2, (maxc + 1) & ~(int64_t)1);
  if ((rc = reserve(ctx, st.rows, sizeof(float2) * (size_t)pitch * (size_t)std::max(n_scans, 1)))) return rc;
  if ((rc = reserve(ctx, st.count, sizeof(int32_t) * (size_t)std::max(n_scans, 1)))) return rc;
  if ((rc = reserve(ctx, ctx->stage, (size_t)total * stride + 16))) return rc;
  if ((rc = reserve(ctx, ctx->offsets, sizeof(int64_t) * ((size_t)n_scans + 1)))) return rc;
  st.pitch = pitch;
  st.n_scans = 0;
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_bad, 0, sizeof(int), ctx->stream));
  if (n_scans == 0) { st.max_count = 0; st.h_count.clear(); return DPGICP_OK; }
  if (total > 0)
    CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, points, (size_t)total * stride, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(ctx->offsets.p, offsets, sizeof(int64_t) * ((size_t)n_scans + 1),
                              cudaMemcpyHostToDevice, ctx->stream));
  pack_rows_kernel<<<n_scans, 256, 0, ctx->stream>>>((const unsigned char *)ctx->stage.p, stride,
                                                     (const long long *)ctx->offsets.p, n_scans, pitch,
                                                     (float2 *)st.rows.p, (int32_t *)st.count.p, ctx->d_bad);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return finish_store(ctx, st, n_scans);
}

int set_pairs_into(dpgicp_ctx *ctx, const Store &st, Batch &b, const int32_t *src, const int32_t *tgt,
                   const float *guess, const float *T_direct, int64_t n) {
  if (n < 0 || (n > 0 && (!src || !tgt || (!guess && !T_direct))))
    return fail(ctx, DPGICP_E_INVALID, "bad pair arguments");
  if (st.n_scans <= 0 && n > 0) return fail(ctx, DPGICP_E_STATE, "no scans uploaded");
  /* dpgicp_run is asynchronous: the previous list's H2D copy out of the pinned staging buffer may still be queued
   * behind a running kernel; wait for it before the buffer is rewritten (or freed) */
  if (b.h_tasks_free) CU_TRY(ctx, cudaEventSynchronize(b.h_tasks_free));
  else CU_TRY(ctx, cudaEventCreateWithFlags(&b.h_tasks_free, cudaEventDisableTiming));
  if ((size_t)n > b.h_tasks_cap) {
    if (b.h_tasks) cudaFreeHost(b.h_tasks);
    b.h_tasks = nullptr; b.h_tasks_cap = 0;
    CU_TRY(ctx, cudaMallocHost((void **)&b.h_tasks, sizeof(PairTask) * (size_t)n));
    b.h_tasks_cap = (size_t)n;
  }
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
    b.h_tasks[k] = t;
  }
  if (bad_index < n && bad_index <= bad_guess)
    return fail(ctx, DPGICP_E_INVALID, "pair index out of range at pair " + std::to_string(bad_index));
  if (bad_guess < n) return fail(ctx, DPGICP_E_RANGE, "non-finite guess at pair " + std::to_string(bad_guess));
  int rc;
  if ((rc = reserve(ctx, b.tasks, sizeof(PairTask) * (size_t)std::max<int64_t>(n, 1)))) return rc;
  if ((rc = reserve(ctx, b.results, sizeof(dpgicp_result) * (size_t)std::max<int64_t>(n, 1)))) return rc;
  if (n > 0)
    CU_TRY(ctx, cudaMemcpyAsync(b.tasks.p, b.h_tasks, sizeof(PairTask) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaEventRecord(b.h_tasks_free, ctx->stream));
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
  if (blob > ctx->h_pair_cap) {
    if (ctx->h_pair) { CU_TRY(ctx, cudaStreamSynchronize(ctx->stream)); cudaFreeHost(ctx->h_pair); }
    ctx->h_pair = nullptr; ctx->h_pair_cap = 0;
    CU_TRY(ctx, cudaMallocHost(&ctx->h_pair, blob));
    ctx->h_pair_cap = blob;
  } else {
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));       /* a previous call's copy out of the buffer (already done: every
                                                            * single-pair call ends with a synchronisation) */
  }
  float *rows = (float *)ctx->h_pair;
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
  int32_t *h_cnt = (int32_t *)((char *)ctx->h_pair + 2 * row_bytes);
  h_cnt[0] = na; h_cnt[1] = nb;
  int rc;
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

/* node estimates -> node table N on the device, plus the index-order box hierarchy the enumeration walks */
int set_nodes_impl(dpgicp_ctx *ctx, Nodes &N, const float *pose, const int32_t *pass, int32_t n, bool pose_is_xy) {
  N.n = 0;
  if (n == 0) return DPGICP_OK;
  std::vector<float> xy((size_t)n * 2), aux((size_t)n * 4);
  const int stride = pose_is_xy ? 2 : 3;
  for (int32_t k = 0; k < n; ++k) {
    const float x = pose[(size_t)stride * k], y = pose[(size_t)stride * k + 1], th = pose_is_xy ? 0.0f : pose[(size_t)stride * k + 2];
    if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(th))
      return fail(ctx, DPGICP_E_RANGE, "non-finite node estimate at node " + std::to_string(k));
    xy[2 * (size_t)k] = x; xy[2 * (size_t)k + 1] = y;
    const float ang = -th;                            /* Eigen::Rotation2Df(-theta_1), math_utils.cc:28 */
    aux[4 * (size_t)k] = th; aux[4 * (size_t)k + 1] = cosf(ang); aux[4 * (size_t)k + 2] = sinf(ang); aux[4 * (size_t)k + 3] = 0.f;
  }
  int rc;
  if ((rc = reserve(ctx, N.xy, sizeof(float) * 2 * (size_t)n))) return rc;
  if ((rc = reserve(ctx, N.aux, sizeof(float) * 4 * (size_t)n))) return rc;
  if ((rc = reserve(ctx, N.pass, sizeof(int32_t) * (size_t)n))) return rc;
  /* levels: L = 1 boxes of 32 nodes, L + 1 boxes of 32 level-L boxes, until one warp can test the top level at once */
  N.levels = 0;
  int64_t total = 0, cnt = n;
  do {
    cnt = (cnt + kEnumFan - 1) / kEnumFan;
    if (N.levels >= kEnumMaxLevels) return fail(ctx, DPGICP_E_TOOBIG, "too many nodes");
    N.level_off[N.levels] = total; N.level_cnt[N.levels] = cnt;
    total += cnt; ++N.levels;
  } while (cnt > kEnumFan);
  if ((rc = reserve(ctx, N.boxes, sizeof(NodeBox) * (size_t)total))) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(N.xy.p, xy.data(), sizeof(float) * 2 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(N.aux.p, aux.data(), sizeof(float) * 4 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(N.pass.p, pass, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  NodeBox *bx = (NodeBox *)N.boxes.p;
  {
    const int nb = (int)N.level_cnt[0], blocks = (nb + 3) / 4;
    node_boxes_leaf_kernel<<<blocks, 128, 0, ctx->stream>>>((const float2 *)N.xy.p, (const int32_t *)N.pass.p, n, bx, nb);
    ctx->launches++;
  }
  for (int L = 1; L < N.levels; ++L) {
    const int nb = (int)N.level_cnt[L], blocks = (nb + 3) / 4;
    node_boxes_up_kernel<<<blocks, 128, 0, ctx->stream>>>(bx + N.level_off[L - 1], (int)N.level_cnt[L - 1], bx + N.level_off[L], nb);
    ctx->launches++;
  }
  CU_TRY(ctx, cudaGetLastError());
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));         /* the host staging vectors go out of scope */
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
int fetch_pairs_from(dpgicp_ctx *ctx, const Batch &b, int32_t *src, int32_t *tgt, float *T, int64_t n) {
  if (n < 0 || n > b.n_pairs) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (n == 0) return DPGICP_OK;
  int rc;
  if ((rc = reserve(ctx, ctx->stage, (size_t)n * 24 + 64))) return rc;
  int32_t *d_src = (int32_t *)ctx->stage.p, *d_tgt = d_src + n;
  float4 *d_T = (float4 *)((char *)ctx->stage.p + (((size_t)n * 8 + 15) & ~(size_t)15));
  const int threads = 256;
  const long long blocks = (n + threads - 1) / threads;
  unpack_tasks_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>((const PairTask *)b.tasks.p, (long long)n, src ? d_src : nullptr,
                                                                   tgt ? d_tgt : nullptr, T ? d_T : nullptr);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  if (src) CU_TRY(ctx, cudaMemcpyAsync(src, d_src, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (tgt) CU_TRY(ctx, cudaMemcpyAsync(tgt, d_tgt, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (T) CU_TRY(ctx, cudaMemcpyAsync(T, d_T, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

/* Room for n_new more rows of at least need_pitch (even) points behind the rows of the store, every existing row kept
 * (the append path).  Rows and counts grow by doubling, so n one-scan appends copy O(n) rows in total; a scan longer
 * than the pitch re-pitches the kept rows on the device.  A buffer that moves is freed only after the stream has
 * drained: the copy out of it, and any dpgicp_run enqueued before the append, read it.  On failure the store is as
 * it was. */
int grow_store(dpgicp_ctx *ctx, Store &st, int n_new, int need_pitch) {
  const int n_old = st.n_scans;
  const int64_t rows = (int64_t)n_old + n_new;
  const int pitch = n_old > 0 ? std::max(st.pitch, need_pitch) : need_pitch;
  const size_t row_bytes = sizeof(float2) * (size_t)pitch;
  const bool move_rows = (n_old > 0 && pitch != st.pitch) || (size_t)rows * row_bytes > st.rows.cap;
  const bool move_count = (size_t)rows * sizeof(int32_t) > st.count.cap;
  DevBuf nr, nc;
  auto alloc = [&](DevBuf &b, size_t bytes) {
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e != cudaSuccess) {
      b.p = nullptr;
      return fail(ctx, e == cudaErrorMemoryAllocation ? DPGICP_E_NOMEM : DPGICP_E_CUDA,
                  std::string("cudaMalloc (scan store growth): ") + cudaGetErrorString(e));
    }
    b.cap = bytes;
    return (int)DPGICP_OK;
  };
  auto cuda = [&](cudaError_t e, const char *what) {
    return e == cudaSuccess ? (int)DPGICP_OK : fail(ctx, DPGICP_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  };
  int rc = DPGICP_OK;
  if (move_rows) {
    int64_t cap = st.pitch > 0 ? (int64_t)(st.rows.cap / (sizeof(float2) * (size_t)st.pitch)) : 0;
    if (rows > cap) cap = std::max(rows, 2 * cap);
    rc = alloc(nr, (size_t)cap * row_bytes);
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
    rc = alloc(nc, (size_t)cap * sizeof(int32_t));
    if (!rc && n_old > 0)
      rc = cuda(cudaMemcpyAsync(nc.p, st.count.p, (size_t)n_old * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream),
                "cudaMemcpyAsync (scan counts)");
  }
  if (!rc && (move_rows || move_count)) rc = cuda(cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize");
  if (rc) {
    cudaStreamSynchronize(ctx->stream);
    release(nr); release(nc);
    return rc;
  }
  if (move_rows) { release(st.rows); st.rows = nr; }
  if (move_count) { release(st.count); st.count = nc; }
  st.pitch = pitch;
  return DPGICP_OK;
}

/* the counts of the n_new rows just converted behind the store back to the host (only those) + the range flag; the
 * store takes them only when every point is in range */
int finish_append(dpgicp_ctx *ctx, Store &st, int n_new) {
  const size_t first = (size_t)st.n_scans;
  st.h_count.resize(first + (size_t)n_new);
  int bad = 0;
  CU_TRY(ctx, cudaMemcpyAsync(st.h_count.data() + first, (const int32_t *)st.count.p + first, sizeof(int32_t) * (size_t)n_new,
                              cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(&bad, ctx->d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (bad) {
    st.h_count.resize(first);
    return fail(ctx, DPGICP_E_RANGE, "appended scans hold a non-finite point or |coordinate| > DPGICP_MAX_ABS_COORD; "
                                     "the store is unchanged");
  }
  if (first == 0) st.max_count = 0;
  for (size_t k = first; k < st.h_count.size(); ++k) st.max_count = std::max(st.max_count, st.h_count[k]);
  st.n_scans = (int32_t)st.h_count.size();
  return DPGICP_OK;
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
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaMalloc((void **)&ctx->d_queue, 32 * sizeof(unsigned long long))) != cudaSuccess ||
      (e = cudaMalloc((void **)&ctx->d_bad, sizeof(int))) != cudaSuccess) {
    delete ctx;
    return fail(nullptr, DPGICP_E_CUDA, cudaGetErrorString(e));
  }
  for (cudaEvent_t &ev : ctx->stage_ev)
    if ((e = cudaEventCreate(&ev)) != cudaSuccess) { delete ctx; return fail(nullptr, DPGICP_E_CUDA, cudaGetErrorString(e)); }
  if (const char *w = std::getenv("DPGICP_WARPS")) ctx->force_warps = std::atoi(w);
  if (const char *c = std::getenv("DPGICP_CTAS_PER_SM")) ctx->force_ctas_per_sm = std::atoi(c);
  if (const char *c = std::getenv("DPGICP_HANDOVER")) {
    ctx->handover_factor = std::max(0.0, std::atof(c));
    if (const char *q = std::strchr(c, ',')) ctx->handover_cluster = std::max(0.0, std::atof(q + 1));
  }
  if (const char *c = std::getenv("DPGICP_STAGES")) ctx->max_stages = std::max(1, std::min(5, std::atoi(c)));
  if (const char *c = std::getenv("DPGICP_CHAIN")) {
    for (const char *q = c; *q;) {            /* e.g. "4,8,16,9x2": the last stage as clusters of 2 CTAs x 9 warps */
      ctx->chain.push_back(std::max(1, std::atoi(q)));
      int cs = 1;
      while (*q && *q != ',') { if (*q == 'x') cs = std::atoi(q + 1); ++q; }
      ctx->chain_cluster.push_back(cs == 2 || cs == 4 ? cs : 1);
      if (*q == ',') ++q;
    }
  }
  *out = ctx;
  return DPGICP_OK;
}

void dpgicp_destroy(dpgicp_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (Store *s : {&ctx->store, &ctx->scratch_store}) { release(s->rows); release(s->count); }
  for (Batch *b : {&ctx->batch, &ctx->scratch_batch}) {
    release(b->tasks); release(b->results); release(b->order);
    if (b->h_tasks) cudaFreeHost(b->h_tasks);
    if (b->h_tasks_free) cudaEventDestroy(b->h_tasks_free);
  }
  for (cudaEvent_t e : ctx->stage_ev) if (e) cudaEventDestroy(e);
  release(ctx->nodes.xy); release(ctx->nodes.aux); release(ctx->nodes.pass); release(ctx->nodes.boxes);
  release(ctx->list_nodes.xy); release(ctx->list_nodes.aux); release(ctx->list_nodes.pass); release(ctx->list_nodes.boxes);
  release(ctx->enum_cnt); release(ctx->enum_amb); release(ctx->d_pair);
  if (ctx->h_pair) cudaFreeHost(ctx->h_pair);
  gather_close(ctx);
  release(ctx->gather);
  release(ctx->stage); release(ctx->offsets); release(ctx->misc); release(ctx->corr); release(ctx->trig);
  for (int k = 0; k < 2; ++k) { release(ctx->state[k]); release(ctx->susp[k]); }
  if (ctx->d_queue) cudaFree(ctx->d_queue);
  if (ctx->d_bad) cudaFree(ctx->d_bad);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *dpgicp_last_error(const dpgicp_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int dpgicp_set_stream(dpgicp_ctx *ctx, void *stream) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (stream) {
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)stream;
    ctx->own_stream = false;
  } else if (!ctx->own_stream) {
    CU_TRY(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
  }
  return DPGICP_OK;
}

int dpgicp_synchronize(dpgicp_ctx *ctx) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

int dpgicp_upload_scans(dpgicp_ctx *ctx, const void *points, size_t stride, const int64_t *offsets, int32_t n_scans) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ctx->batch.n_pairs = 0;
  return upload_scans_into(ctx, ctx->store, points, stride, offsets, n_scans);
}

int dpgicp_upload_ranges(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans, int32_t n_beams, float angle_min,
                         float angle_max, float range_max, float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: upload ranges + scan->cloud");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_scans < 0 || n_beams < 2 || (n_scans > 0 && !ranges)) return fail(ctx, DPGICP_E_INVALID, "bad range-scan arguments");
  if (n_beams > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "n_beams exceeds DPGICP_MAX_POINTS");
  Store &st = ctx->store;
  ctx->batch.n_pairs = 0;
  const int pitch = (n_beams + 1) & ~1;
  int rc;
  if ((rc = reserve(ctx, st.rows, sizeof(float2) * (size_t)pitch * (size_t)std::max(n_scans, 1)))) return rc;
  if ((rc = reserve(ctx, st.count, sizeof(int32_t) * (size_t)std::max(n_scans, 1)))) return rc;
  if ((rc = reserve(ctx, ctx->stage, sizeof(float) * (size_t)n_scans * (size_t)n_beams + 16))) return rc;
  st.pitch = pitch;
  st.n_scans = 0;
  if (n_scans == 0) { st.max_count = 0; st.h_count.clear(); return DPGICP_OK; }
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_bad, 0, sizeof(int), ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, ranges, sizeof(float) * (size_t)n_scans * (size_t)n_beams,
                              cudaMemcpyHostToDevice, ctx->stream));
  /* createNode dpg_slam.cc:497: angle_inc = (max - min) / (n - 1.0), stored as float */
  const float angle_inc = (float)(((double)(float)(angle_max - angle_min)) / ((double)n_beams - 1.0));
  const float lc = cosf(ltheta), ls = sinf(ltheta);       /* Eigen::Rotation2Df(ltheta), host libm */
  const int threads = 128, warps_per_block = threads / 32;
  const int blocks = (n_scans + warps_per_block - 1) / warps_per_block;
  if ((rc = ensure_trig(ctx, n_beams, angle_min, angle_inc))) return rc;
  ranges_to_rows_kernel<<<blocks, threads, 0, ctx->stream>>>((const float *)ctx->stage.p, nullptr, n_scans, n_beams,
                                                            (const double2 *)ctx->trig.p, range_max, lx, ly, lc, ls, pitch,
                                                            (float2 *)st.rows.p, (int32_t *)st.count.p, ctx->d_bad);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return finish_store(ctx, st, n_scans);
}

int dpgicp_upload_ranges_subset(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans_total, int32_t n_beams,
                                const int32_t *scan_ids, int32_t n_ids, float angle_min, float angle_max, float range_max,
                                float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_scans_total < 0 || n_ids < 0 || n_beams < 2 || (n_ids > 0 && (!ranges || !scan_ids)))
    return fail(ctx, DPGICP_E_INVALID, "bad range-scan arguments");
  if (n_beams > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "n_beams exceeds DPGICP_MAX_POINTS");
  for (int32_t k = 0; k < n_ids; ++k)
    if (scan_ids[k] < 0 || scan_ids[k] >= n_scans_total)
      return fail(ctx, DPGICP_E_INVALID, "scan id out of range at position " + std::to_string(k));
  Store &st = ctx->store;
  ctx->batch.n_pairs = 0;
  const int pitch = (n_beams + 1) & ~1;
  int rc;
  if ((rc = reserve(ctx, st.rows, sizeof(float2) * (size_t)pitch * (size_t)std::max(n_ids, 1)))) return rc;
  if ((rc = reserve(ctx, st.count, sizeof(int32_t) * (size_t)std::max(n_ids, 1)))) return rc;
  st.pitch = pitch;
  st.n_scans = 0;
  if (n_ids == 0) { st.max_count = 0; st.h_count.clear(); return DPGICP_OK; }
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_bad, 0, sizeof(int), ctx->stream));
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
    if (bytes > ctx->h_stage_cap) {
      if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
      ctx->h_stage = nullptr; ctx->h_stage_cap = 0;
      CU_TRY(ctx, cudaMallocHost(&ctx->h_stage, bytes));
      ctx->h_stage_cap = bytes;
    }
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));       /* the buffer may still feed a previous copy */
    for (int32_t k = 0; k < n_ids; ++k)
      std::memcpy((float *)ctx->h_stage + (size_t)k * n_beams, ranges + (size_t)scan_ids[k] * n_beams, sizeof(float) * (size_t)n_beams);
    if ((rc = reserve(ctx, ctx->stage, bytes + 16))) return rc;
    CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, ctx->h_stage, bytes, cudaMemcpyHostToDevice, ctx->stream));
    d_in = (const float *)ctx->stage.p;
  }
  const float angle_inc = (float)(((double)(float)(angle_max - angle_min)) / ((double)n_beams - 1.0));
  const float lc = cosf(ltheta), ls = sinf(ltheta);
  const int threads = 128, warps_per_block = threads / 32;
  const int blocks = (n_ids + warps_per_block - 1) / warps_per_block;
  if ((rc = ensure_trig(ctx, n_beams, angle_min, angle_inc))) return rc;
  ranges_to_rows_kernel<<<blocks, threads, 0, ctx->stream>>>(d_in, d_ids, n_ids, n_beams, (const double2 *)ctx->trig.p, range_max,
                                                            lx, ly, lc, ls, pitch, (float2 *)st.rows.p, (int32_t *)st.count.p, ctx->d_bad);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return finish_store(ctx, st, n_ids);
}

int dpgicp_append_ranges(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans, int32_t n_beams, float angle_min,
                         float angle_max, float range_max, float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: append ranges + scan->cloud");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_scans < 0 || n_beams < 2 || (n_scans > 0 && !ranges)) return fail(ctx, DPGICP_E_INVALID, "bad range-scan arguments");
  if (n_beams > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "n_beams exceeds DPGICP_MAX_POINTS");
  Store &st = ctx->store;
  if ((int64_t)st.n_scans + n_scans > INT32_MAX) return fail(ctx, DPGICP_E_INVALID, "the store would hold more than 2^31 - 1 scans");
  if (n_scans == 0) return DPGICP_OK;
  const int first = st.n_scans;
  int rc;
  if ((rc = grow_store(ctx, st, n_scans, (n_beams + 1) & ~1))) return rc;
  if ((rc = reserve(ctx, ctx->stage, sizeof(float) * (size_t)n_scans * (size_t)n_beams + 16))) return rc;
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_bad, 0, sizeof(int), ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, ranges, sizeof(float) * (size_t)n_scans * (size_t)n_beams,
                              cudaMemcpyHostToDevice, ctx->stream));
  /* the conversion of dpgicp_upload_ranges, writing rows first .. first + n_scans - 1 */
  const float angle_inc = (float)(((double)(float)(angle_max - angle_min)) / ((double)n_beams - 1.0));
  const float lc = cosf(ltheta), ls = sinf(ltheta);
  const int threads = 128, warps_per_block = threads / 32;
  const int blocks = (n_scans + warps_per_block - 1) / warps_per_block;
  if ((rc = ensure_trig(ctx, n_beams, angle_min, angle_inc))) return rc;
  ranges_to_rows_kernel<<<blocks, threads, 0, ctx->stream>>>((const float *)ctx->stage.p, nullptr, n_scans, n_beams,
                                                            (const double2 *)ctx->trig.p, range_max, lx, ly, lc, ls, st.pitch,
                                                            (float2 *)st.rows.p + (size_t)first * st.pitch,
                                                            (int32_t *)st.count.p + first, ctx->d_bad);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return finish_append(ctx, st, n_scans);
}

int dpgicp_append_scans(dpgicp_ctx *ctx, const void *points, size_t stride, const int64_t *offsets, int32_t n_scans) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: append clouds");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int64_t maxc = 0, total = 0;
  int rc = check_clouds(ctx, points, stride, offsets, n_scans, &maxc, &total);
  if (rc) return rc;
  Store &st = ctx->store;
  if ((int64_t)st.n_scans + n_scans > INT32_MAX) return fail(ctx, DPGICP_E_INVALID, "the store would hold more than 2^31 - 1 scans");
  if (n_scans == 0) return DPGICP_OK;
  const int first = st.n_scans;
  if ((rc = grow_store(ctx, st, n_scans, (int)std::max<int64_t>(2, (maxc + 1) & ~(int64_t)1)))) return rc;
  if ((rc = reserve(ctx, ctx->stage, (size_t)total * stride + 16))) return rc;
  if ((rc = reserve(ctx, ctx->offsets, sizeof(int64_t) * ((size_t)n_scans + 1)))) return rc;
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_bad, 0, sizeof(int), ctx->stream));
  if (total > 0)
    CU_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, points, (size_t)total * stride, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(ctx->offsets.p, offsets, sizeof(int64_t) * ((size_t)n_scans + 1), cudaMemcpyHostToDevice,
                              ctx->stream));
  pack_rows_kernel<<<n_scans, 256, 0, ctx->stream>>>((const unsigned char *)ctx->stage.p, stride, (const long long *)ctx->offsets.p,
                                                     n_scans, st.pitch, (float2 *)st.rows.p + (size_t)first * st.pitch,
                                                     (int32_t *)st.count.p + first, ctx->d_bad);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return finish_append(ctx, st, n_scans);
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

int dpgicp_set_pairs(dpgicp_ctx *ctx, const int32_t *src, const int32_t *tgt, const float *guess, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: pair list");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  return set_pairs_into(ctx, ctx->store, ctx->batch, src, tgt, guess, nullptr, n);
}

int dpgicp_set_pair_cost_hints(dpgicp_ctx *ctx, const float *hints, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  Batch &b = ctx->batch;
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
  CU_TRY(ctx, cudaMemcpyAsync(b.order.p, order.data(), sizeof(long long) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));        /* `order` goes out of scope */
  b.has_order = true;
  return DPGICP_OK;
}

int dpgicp_run(dpgicp_ctx *ctx, const dpgicp_params *params) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_params(ctx, params);
  if (rc) return rc;
  if (ctx->batch.n_pairs == 0) return DPGICP_OK;               /* an empty batch is valid and does nothing */
  if (ctx->batch.n_pairs < 0) return fail(ctx, DPGICP_E_STATE, "no pair list set");
  if (ctx->store.n_scans <= 0) return fail(ctx, DPGICP_E_STATE, "no scans uploaded");
  if (ctx->batch.max_scan >= ctx->store.n_scans)
    return fail(ctx, DPGICP_E_STATE, "the enumerated pair list refers to nodes without a scan in the store (node k owns scan k)");
  return launch_icp(ctx, ctx->store, ctx->batch, params, nullptr, nullptr);
}

int dpgicp_run_range(dpgicp_ctx *ctx, const dpgicp_params *params, int64_t first, int64_t count) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = check_params(ctx, params);
  if (rc) return rc;
  if (first < 0 || count < 0 || first + count > ctx->batch.n_pairs) return fail(ctx, DPGICP_E_INVALID, "pair range outside the batch");
  if (count == 0) return DPGICP_OK;
  if (ctx->store.n_scans <= 0) return fail(ctx, DPGICP_E_STATE, "no scans uploaded");
  if (ctx->batch.max_scan >= ctx->store.n_scans)
    return fail(ctx, DPGICP_E_STATE, "the enumerated pair list refers to nodes without a scan in the store (node k owns scan k)");
  return launch_icp(ctx, ctx->store, ctx->batch, params, nullptr, nullptr, nullptr, nullptr, first, count);
}

int dpgicp_fetch_results_range(dpgicp_ctx *ctx, dpgicp_result *out, int64_t first, int64_t count) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (first < 0 || count < 0 || first + count > ctx->batch.n_pairs || (count > 0 && !out)) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (count > 0)
    CU_TRY(ctx, cudaMemcpyAsync(out, (const dpgicp_result *)ctx->batch.results.p + first, sizeof(dpgicp_result) * (size_t)count,
                                cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
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
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n < 0 || n > ctx->batch.n_pairs || (n > 0 && !out)) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (n > 0)
    CU_TRY(ctx, cudaMemcpyAsync(out, ctx->batch.results.p, sizeof(dpgicp_result) * (size_t)n, cudaMemcpyDeviceToHost,
                                ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

int dpgicp_fetch_factors(dpgicp_ctx *ctx, dpgicp_factor *out, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n < 0 || n > ctx->batch.n_pairs || (n > 0 && !out)) return fail(ctx, DPGICP_E_INVALID, "bad fetch arguments");
  if (n == 0) { CU_TRY(ctx, cudaStreamSynchronize(ctx->stream)); return DPGICP_OK; }
  int rc;
  if ((rc = reserve(ctx, ctx->stage, sizeof(dpgicp_factor) * (size_t)n))) return rc;
  const int threads = 128;
  const long long blocks = (n + threads - 1) / threads;
  factors_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>((const dpgicp_result *)ctx->batch.results.p,
                                                              (const PairTask *)ctx->batch.tasks.p, (long long)n,
                                                              (dpgicp_factor *)ctx->stage.p);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  CU_TRY(ctx, cudaMemcpyAsync(out, ctx->stage.p, sizeof(dpgicp_factor) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return DPGICP_OK;
}

static int gather_export_impl(dpgicp_ctx *ctx, int64_t n_global, int64_t n_alloc, unsigned char *handle_out) {
  static_assert(sizeof(cudaIpcMemHandle_t) == DPGICP_IPC_HANDLE_BYTES, "IPC handle size");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->gather_world > 0)
    return fail(ctx, DPGICP_E_STATE, "gather buffers are attached (peers may still store into this one): dpgicp_gather_detach on every rank first");
  /* a dedicated cudaMalloc allocation (IPC handles cover whole allocations) */
  release(ctx->gather);
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
    release(ctx->gather);
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
  *out_ptr = ctx->batch.results.p;
  *out_n = ctx->batch.n_pairs;
  return DPGICP_OK;
}

int dpgicp_last_run_counters(dpgicp_ctx *ctx, uint64_t counters[8]) {
  if (!ctx || !counters) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  unsigned long long h[8];
  CU_TRY(ctx, cudaMemcpyAsync(h, ctx->d_queue + 8, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 8; ++k) counters[k] = h[k];
  counters[4] = ctx->launches;
  return DPGICP_OK;
}

#ifdef DPGICP_PHASE_TIMING
/* development builds only: cycles thread 0 spent in each phase of the pass loop, summed over pairs */
int dpgicp_debug_phase_counters(dpgicp_ctx *ctx, uint64_t out[8]) {
  unsigned long long h[8];
  CU_TRY(ctx, cudaMemcpyAsync(h, ctx->d_queue + 16, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
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
  if ((rc = set_pairs_into(ctx, ctx->scratch_store, ctx->scratch_batch, &s, &t, guess, nullptr, 1))) return rc;
  if ((rc = launch_icp(ctx, ctx->scratch_store, ctx->scratch_batch, params, nullptr, nullptr))) return rc;
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
  if ((rc = set_pairs_into(ctx, ctx->scratch_store, ctx->scratch_batch, &s, &t, nullptr, T, 1))) return rc;
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
  if ((rc = launch_icp(ctx, ctx->scratch_store, ctx->scratch_batch, &p, d_corr, d_d2, prev_nn ? d_seed : nullptr, nn_out ? d_nn : nullptr))) return rc;
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
  cudaEvent_t e0, e1;
  CU_TRY(ctx, cudaEventCreate(&e0));
  CU_TRY(ctx, cudaEventCreate(&e1));
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
  cudaEventDestroy(e0); cudaEventDestroy(e1);
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
  rc = fetch_pairs_from(ctx, ctx->scratch_batch, src, tgt, nullptr, total);
  ctx->scratch_batch.n_pairs = 0;
  return rc;
}

int dpgicp_set_nodes(dpgicp_ctx *ctx, const float *pose, const int32_t *pass, int32_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n < 0 || (n > 0 && (!pose || !pass))) return fail(ctx, DPGICP_E_INVALID, "bad node arguments");
  return set_nodes_impl(ctx, ctx->nodes, pose, pass, n, false);
}

int dpgicp_enumerate_pairs_device(dpgicp_ctx *ctx, int32_t mode, float r_same, float r_other, int32_t rank, int32_t world,
                                  int64_t *n_total, int64_t *n_local) {
  if (!ctx) return DPGICP_E_INVALID;
  NvtxRange range("dpgicp: enumerate pairs (device)");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (mode != DPGICP_ENUM_REOPTIMIZE && mode != DPGICP_ENUM_ONLINE) return fail(ctx, DPGICP_E_INVALID, "mode must be DPGICP_ENUM_REOPTIMIZE or DPGICP_ENUM_ONLINE");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, DPGICP_E_INVALID, "bad shard arguments");
  if (!(r_same >= 0.0f) || !(r_other >= 0.0f)) return fail(ctx, DPGICP_E_INVALID, "radii must be >= 0");
  if (ctx->nodes.n <= 0) {
    if (n_total) *n_total = 0;
    if (n_local) *n_local = 0;
    ctx->batch.n_pairs = 0;
    return DPGICP_OK;
  }
  return enumerate_into(ctx, ctx->nodes, ctx->batch, mode, r_same, r_other, rank, world, n_total, n_local);
}

int dpgicp_fetch_pairs(dpgicp_ctx *ctx, int32_t *src, int32_t *tgt, float *T, int64_t n) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  return fetch_pairs_from(ctx, ctx->batch, src, tgt, T, n);
}

int dpgicp_convert_ranges_device(dpgicp_ctx *ctx, const float *d_ranges, int32_t n_scans, int32_t n_beams, float angle_min,
                                 float angle_max, float range_max, float lx, float ly, float ltheta) {
  if (!ctx) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n_scans < 0 || n_beams < 2 || (n_scans > 0 && !d_ranges)) return fail(ctx, DPGICP_E_INVALID, "bad range-scan arguments");
  if (n_beams > DPGICP_MAX_POINTS) return fail(ctx, DPGICP_E_TOOBIG, "n_beams exceeds DPGICP_MAX_POINTS");
  Store &st = ctx->store;
  ctx->batch.n_pairs = 0;
  const int pitch = (n_beams + 1) & ~1;
  int rc;
  if ((rc = reserve(ctx, st.rows, sizeof(float2) * (size_t)pitch * (size_t)std::max(n_scans, 1)))) return rc;
  if ((rc = reserve(ctx, st.count, sizeof(int32_t) * (size_t)std::max(n_scans, 1)))) return rc;
  st.pitch = pitch;
  st.n_scans = 0;
  if (n_scans == 0) { st.max_count = 0; st.h_count.clear(); return DPGICP_OK; }
  CU_TRY(ctx, cudaMemsetAsync(ctx->d_bad, 0, sizeof(int), ctx->stream));
  const float angle_inc = (float)(((double)(float)(angle_max - angle_min)) / ((double)n_beams - 1.0));
  const float lc = cosf(ltheta), ls = sinf(ltheta);
  const int threads = 128, warps_per_block = threads / 32;
  const int blocks = (n_scans + warps_per_block - 1) / warps_per_block;
  if ((rc = ensure_trig(ctx, n_beams, angle_min, angle_inc))) return rc;
  ranges_to_rows_kernel<<<blocks, threads, 0, ctx->stream>>>(d_ranges, nullptr, n_scans, n_beams, (const double2 *)ctx->trig.p,
                                                            range_max, lx, ly, lc, ls, pitch, (float2 *)st.rows.p,
                                                            (int32_t *)st.count.p, ctx->d_bad);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return finish_store(ctx, st, n_scans);
}

int dpgicp_enable_stage_timing(dpgicp_ctx *ctx, int32_t on) {
  if (!ctx) return DPGICP_E_INVALID;
  ctx->stage_timing = on != 0;
  ctx->last_stages = 0;
  return DPGICP_OK;
}

int dpgicp_last_run_stage_ms(dpgicp_ctx *ctx, float stage_ms[8], int32_t *n_stages) {
  if (!ctx || !stage_ms || !n_stages) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  *n_stages = 0;
  for (int k = 0; k < 8; ++k) stage_ms[k] = 0.f;
  if (!ctx->stage_timing || ctx->last_stages <= 0) return fail(ctx, DPGICP_E_STATE, "stage timing is off (dpgicp_enable_stage_timing) or nothing has run");
  CU_TRY(ctx, cudaEventSynchronize(ctx->stage_ev[ctx->last_stages]));
  for (int k = 0; k < ctx->last_stages; ++k) CU_TRY(ctx, cudaEventElapsedTime(&stage_ms[k], ctx->stage_ev[k], ctx->stage_ev[k + 1]));
  *n_stages = ctx->last_stages;
  return DPGICP_OK;
}

int dpgicp_fp32_probe(dpgicp_ctx *ctx, double *mul_add, double *fma) {
  if (!ctx || !mul_add || !fma) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc;
  if ((rc = reserve(ctx, ctx->misc, 256))) return rc;
  cudaEvent_t e0, e1;
  CU_TRY(ctx, cudaEventCreate(&e0));
  CU_TRY(ctx, cudaEventCreate(&e1));
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
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *mul_add = best[0]; *fma = best[1];
  return DPGICP_OK;
}

int dpgicp_fp32x2_probe(dpgicp_ctx *ctx, double *mul_add_packed) {
  if (!ctx || !mul_add_packed) return DPGICP_E_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc;
  if ((rc = reserve(ctx, ctx->misc, 256))) return rc;
  cudaEvent_t e0, e1;
  CU_TRY(ctx, cudaEventCreate(&e0));
  CU_TRY(ctx, cudaEventCreate(&e1));
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
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *mul_add_packed = best;
  return DPGICP_OK;
}

}  /* extern "C" */
