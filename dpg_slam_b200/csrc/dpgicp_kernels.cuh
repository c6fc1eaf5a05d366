/*
 * dpgicp_kernels.cuh — sm_100a device code of the scan-matching back end.
 *
 * One persistent CTA aligns one scan pair at a time, pulled from an atomic work queue (ICP
 * iteration counts vary 5..500 per pair, so static assignment would idle SMs).  Both clouds of
 * the pair are staged once in shared memory (1-D TMA bulk copies when rows are contiguous) and
 * every ICP iteration — correspondence search, reciprocity check, moment reduction, rigid solve,
 * convergence test, source update — runs on-chip; only the 112-byte result record goes back to
 * HBM.  Replaces the inside of DpgSLAM::runIcp (reference src/dpg_slam/dpg_slam.cc:362-446):
 * PCL's kd-tree correspondence estimation + SVD step + convergence criteria (SURVEY.md App. A)
 * and calculate_ICP_COV (src/icp_cov/cov_func_point_to_point.h:24-585, planar closed form
 * SURVEY.md App. B).
 *
 * Arithmetic contract (identical to oracle/dpg_oracle.c, see DESIGN.md): binary32 transform and
 * distances in individually rounded operations (no FMA: __f*_rn intrinsics and --fmad=false),
 * (d2, index)-lexicographic nearest neighbour, exact int64 fixed-point moment sums (order
 * independent, so any thread layout gives the same bits), binary64 closed-form planar step.
 *
 * Exact pruned search: points of a scan are in beam order, so kGroup (16) consecutive points form a
 * spatially compact group with an axis-aligned bounding box, and kSuper (16) consecutive groups an
 * upper-level box.  A warp handles a tile of 32 consecutive queries (one per lane); box-to-box
 * lower bounds, evaluated lane-parallel first over the upper boxes and then over the groups of the
 * surviving ones, select the groups that can still beat the tile's current bound, which is seeded
 * with the previous iteration's neighbour.  Lower bounds use the same rounding sequence as the
 * distance itself, so by monotonicity of rounding they never exceed a computed distance: pruning
 * is exact, no epsilons.  SEARCH_BRUTE scans every group through the same code.  In shared memory a
 * cloud is pair-interleaved — (x0, x1, y0, y1) per 16-byte word — so that the two distances of one
 * LDS.128 are five packed instructions (FADD2 FADD2 FMUL2 FMUL2 + the individually rounded packed
 * sum), their minimum a tree of three-input minima; the index of the minimum is looked up only when
 * a lane can strictly improve on its seed (sticky tie rule, include/dpgicp.h).
 * SEARCH_PROJECTIVE (north-star extension, approximate): every lane locates its query in the other
 * scan's beam order by bisection over bearing keys and scans a window around it; defined by the oracle.
 *
 * Execution shapes (DESIGN.md section 5.1): the host launches the kernel as a chain of stages with
 * growing warps per pair; a stage suspends the pairs still running once its queue is dry and few enough
 * are left for the next stage to run at once (state to HBM, restored bit for bit) and the last stage gives each remaining pair a thread-block cluster of
 * 4 CTAs that exchange exact partial sums through distributed shared memory.  With a multi-GPU
 * gather attached, the epilogue stores each record into every rank's buffer over NVLink.
 */
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dpgicp.h"

#include <cstdio>

/* -DDPGICP_CHECK: device-side assertions on everything the kernels index with computed values (work items, suspended-
 * state slots, neighbour seeds and matches, shared-memory capacities, gather slots, enumeration output positions) and on
 * the agreement of the CTAs of a cluster.  A failed check prints its text and traps, so the launch — and the test that
 * made it — fails loudly.  Compiled out of the product build; tools/build_variants.sh check=-DDPGICP_CHECK builds the
 * checked library and the GPU suite runs against it with DPGICP_LIBRARY. */
#ifdef DPGICP_CHECK
#define DPG_CHECK(cond)                                                                                    \
  do {                                                                                                     \
    if (!(cond)) {                                                                                         \
      printf("DPGICP_CHECK failed: %s (dpgicp_kernels.cuh:%d, block %d thread %d)\n", #cond, __LINE__,    \
             (int)blockIdx.x, (int)threadIdx.x);                                                           \
      __trap();                                                                                            \
    }                                                                                                      \
  } while (0)
#else
#define DPG_CHECK(cond) do { } while (0)
#endif

namespace dpg {

#ifndef DPGICP_GROUP
#define DPGICP_GROUP 16
#endif
constexpr int   kTile  = 32;            /* queries per warp (one per lane)                            */
constexpr int   kGroup = DPGICP_GROUP;  /* points per bounding-box group of a searched cloud          */
static_assert(kGroup == 8 || kGroup == 16 || kGroup == 32, "kGroup must be 8, 16 or 32");
/* internal instantiation of DPGICP_SEARCH_PRUNED for clouds of at most 32 groups (512 points — the reference's
 * down-sampled scans): all groups fit ONE lane-parallel round, so no upper box level is built or tested.  A compile-time
 * variant because a run-time branch in the candidate rounds cost the 1081-point batches 1.4 % (measured). */
constexpr int   kSearchPrunedFlat = 3;
constexpr int   kFlatMaxGroups = 32;
/* ... and of the stock configuration — point-to-point metric, no outlier rejector, no parity hook — with those run-time
 * branches compiled out of the pass loop (+1 % on the 1081-point batches, measured): the pruned search, plain and flat */
constexpr int   kSearchPrunedStock = 4;
constexpr int   kSearchPrunedFlatStock = 5;
__host__ __device__ constexpr bool search_is_projective(int s) { return s == DPGICP_SEARCH_PROJECTIVE; }
__host__ __device__ constexpr bool search_is_flat(int s) { return s == kSearchPrunedFlat || s == kSearchPrunedFlatStock; }
__host__ __device__ constexpr bool search_is_pruned(int s) { return s == DPGICP_SEARCH_PRUNED || s >= kSearchPrunedFlat; }
__host__ __device__ constexpr bool search_is_stock(int s) { return s == kSearchPrunedStock || s == kSearchPrunedFlatStock; }
constexpr int   kSuper = 16;            /* groups per box of the upper level of the search hierarchy  */
static_assert(DPGICP_MAX_POINTS / (kGroup * kSuper) <= 32, "the upper level is tested in ONE lane-parallel round: at most 32 boxes");
constexpr float kPad   = 1.0e30f;   /* coordinate of padded slots: any d2 against it is +inf      */
constexpr double kScaleLin  = 4294967296.0;      /* 2^32 */
constexpr double kScaleProd = 268435456.0;       /* 2^28 */
constexpr double kScaleD2   = 1099511627776.0;   /* 2^40 */
constexpr int   kMaxWarps = 32;
constexpr int   kCovChunk = 16;  /* tile partials per covariance reduction round: FIXED, the summation order must not
                                  * depend on the CTA width                                                         */
constexpr int   kStateHeader = 64;  /* bytes of scalars in front of a suspended pair's arrays      */
/* L.nn[i] between two passes: -1 = no gated forward neighbour; otherwise the neighbour's index, with kNnRejected set
 * when the pair failed the reciprocal test (it still seeds the next pass, but does not enter the sums) */
constexpr int   kNnRejected = 0x40000000;
constexpr int   kNnIndexMask = 0x3fffffff;

struct PairTask {            /* 24 bytes: pair indices + the guess as matrix entries (host libm) */
  int32_t src, tgt;
  float c, s, tx, ty;
};

struct StoreView {           /* scan store: padded rows of float2, beam order, MAX_RANGE dropped  */
  const float2 *pts;
  const int32_t *count;
  int32_t pitch;             /* points per row, even (rows are 16-byte aligned for TMA)           */
  int32_t n_scans;
};

/* scalars of a suspended pair (first kStateHeader bytes of its state slot) */
struct SuspHeader {
  float fc, fs, ftx, fty;
  double mse, mse_prev;
  int32_t iterations, last_k;
  uint32_t status;
  int32_t pad;
};
static_assert(sizeof(SuspHeader) <= kStateHeader, "state header too small");

struct KernelParams {
  StoreView store;
  const PairTask *tasks;
  dpgicp_result *results;
  unsigned long long *queue;      /* work-queue head of THIS stage                                */
  unsigned long long *counters;   /* [0] iterations [1] correspondences [2] distance evals [3] box tests */
  long long n_pairs;
  int32_t n_cap;                  /* smem capacity per cloud in points, multiple of 32            */
  int32_t max_iterations, use_reciprocal, divisor, metric, cov_mode, cov_cap;
  int32_t proj_window;            /* DPGICP_SEARCH_PROJECTIVE: candidates on each side of the projected index */
  float sensor_x, sensor_y;       /* ... and the laser origin the beam order turns around                      */
  float gate;                     /* binary32 floor of max_correspondence_distance^2              */
  float one;                      /* 1.0f, opaque to the compiler (see add2)                      */
  double eps, rot_thr, sensor_var;
  float live[3];
  /* dpgicp_correspondences hook: when corr_out != nullptr the kernel runs ONE pass for pair 0    */
  int32_t *corr_out;
  float *corr_d2_out;
  const int32_t *corr_seed;       /* ... seeded with these forward neighbours (nullptr: none)    */
  int32_t *corr_nn_out;           /* ... and reports this pass's gated forward neighbours (may be nullptr) */
  /* outlier rejection (DPGICP_OUTLIER_*; never combined with a cluster stage by the host) */
  int32_t outlier_mode;
  double outlier_param;
  /* staged execution (see icp_pairs_kernel): work items of stage > 0 are the pairs the previous
   * stage suspended when its queue ran dry; they are resumed by wider CTAs                        */
  const long long *order;             /* fresh stage only: item k is pair order[k] (nullptr = identity): callers that
                                       * know which pairs tend to run long put them first                         */
  int32_t resume;                     /* 0: items are fresh tasks; 1: items are susp_in[0..*in_count) */
  const unsigned int *in_count;
  const long long *susp_in;           /* pair index per suspended item; item k's state is slot k   */
  const unsigned char *state_in;
  unsigned int *out_count;            /* nullptr: final stage, never suspends                      */
  long long *susp_out;
  unsigned char *state_out;
  long long slot_bytes;               /* kStateHeader + 12 * n_cap                                 */
  /* hand-over rule of a stage that may suspend: once its queue is dry AND at most `handover` of its pairs are still
   * running, every CTA suspends its pair at the next pass boundary.  `handover` is what the next stage can run at
   * once: handing it more would only make pairs wait in its queue that could keep running here.            */
  unsigned long long *finished;       /* pairs of THIS stage that ran to completion                */
  long long handover;
  /* multi-GPU gather fused into the epilogue: with gather_world > 1 the record of local pair k also goes to
   * slot (gather_rank + k * gather_world) of EVERY rank's gather buffer — peer-mapped device memory, written
   * with plain stores over NVLink; no collective is launched                                              */
  dpgicp_result *gather_peer[DPGICP_MAX_GATHER_RANKS];
  int32_t gather_world, gather_rank;
  int32_t gather_fanout;              /* buffers written: gather_world (every rank's) or 1 (rank 0's only)        */
  long long pair_base;                /* dpgicp_run_range: tasks / results point at local pair pair_base of the batch */
  long long gather_slots;             /* records every attached gather buffer can hold                               */
  long long slot_cap;                 /* suspended-state slots available to a stage that may suspend                 */
};

/* ------------------------------------------------------------------------------------------------
 * small device helpers
 * ---------------------------------------------------------------------------------------------- */
__device__ __forceinline__ float dist2(float ax, float ay, float bx, float by) {
  const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by);
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}

__device__ __forceinline__ float2 xform(float c, float s, float tx, float ty, float2 p) {
  float2 r;
  r.x = __fadd_rn(__fadd_rn(__fmul_rn(c, p.x), __fmul_rn(-s, p.y)), tx);
  r.y = __fadd_rn(__fadd_rn(__fmul_rn(s, p.x), __fmul_rn(c, p.y)), ty);
  return r;
}

/* ---- packed binary32 pairs (sm_100 FADD2 / FMUL2): one issue slot for two individually rounded
 * operations; each half is the IEEE round-to-nearest result of the scalar instruction, so the bits are
 * those of __fsub_rn / __fmul_rn.  A float2 / half of a float4 loaded by LDS.64/.128 already sits in an
 * aligned register pair, so packing is free. ------------------------------------------------------ */
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float &lo, float &hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
/* a + b per half, individually rounded.  ptxas contracts a packed mul.rn feeding a packed add.rn into ONE FFMA2 (single
 * rounding!) whatever --fmad says — the scalar forms are left alone — and it also folds fma(a, 1.0f, b) back into that
 * add when it can see the constant.  So the sum is issued as fma(a, one, b) with `one` = (1.0f, 1.0f) read from the
 * kernel parameters: a * 1 is exact, the result is the correctly rounded a + b, and nothing can be fused into it. */
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b, f32x2 one) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(one), "l"(b));
  return r;
}
/* ---- pair-interleaved clouds in shared memory: points 2p and 2p+1 share one 16-byte word (x0, x1, y0, y1), so that one
 * LDS.128 of the scan loop delivers (x0, x1) and (y0, y1) as aligned register pairs and BOTH distances come out of five
 * packed instructions (two differences, two squares, one sum: 2.5 issue slots per distance instead of 3).  HBM rows and
 * TMA-staged rows are plain (x, y) pairs; the staging loops re-arrange each 32-point tile in place. ---- */
/* IL = true: pair-interleaved (the exact searches); IL = false: plain (x, y) pairs — the projective search reads single
 * points at per-lane indices, where one LDS.64 beats two LDS.32 plus the index arithmetic (measured: 442 k vs 530 k
 * pairs/s when it shared the interleaved layout) */
template <bool IL>
__device__ __forceinline__ float2 ld_pt(const float2 *cloud, int k) {
  if constexpr (!IL) return cloud[k];
  const float *f = reinterpret_cast<const float *>(cloud) + ((k >> 1) << 2) + (k & 1);
  return make_float2(f[0], f[2]);
}
template <bool IL>
__device__ __forceinline__ void st_pt(float2 *cloud, int k, float2 p) {
  if constexpr (!IL) { cloud[k] = p; return; }
  float *f = reinterpret_cast<float *>(cloud) + ((k >> 1) << 2) + (k & 1);
  f[0] = p.x; f[2] = p.y;
}
/* dist2(q, p) with q = (qx, qy), p = (px, py) packed: (qx - px)^2 + (qy - py)^2, same roundings as dist2() */
__device__ __forceinline__ float dist2_packed(f32x2 q, f32x2 p) {
  const f32x2 d = sub2(q, p);
  float sx, sy;
  unpack2(mul2(d, d), sx, sy);
  return __fadd_rn(sx, sy);
}

/* Blackwell warp-wide float min/max in one instruction (SASS CREDUX.MIN/MAX.F32) */
__device__ __forceinline__ float warp_min(float v) {
  float r;
  asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ float warp_max(float v) {
  float r;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}

__device__ __forceinline__ long long warp_sum_i64(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

/* lower bound of dist2(q, p) over all p in box b = (lox, loy, hix, hiy); same rounding sequence */
__device__ __forceinline__ float lb_point_box(f32x2 q, float4 b) {
  float lx, ly, hx, hy;
  unpack2(sub2(pack2(b.x, b.y), q), lx, ly);
  unpack2(sub2(q, pack2(b.z, b.w)), hx, hy);
  const f32x2 e = pack2(fmaxf(fmaxf(lx, hx), 0.0f), fmaxf(fmaxf(ly, hy), 0.0f));
  float sx, sy;
  unpack2(mul2(e, e), sx, sy);
  return __fadd_rn(sx, sy);
}
/* lower bound over all q in box a, p in box b */
__device__ __forceinline__ float lb_box_box(float4 a, float4 b) {
  float lx, ly, hx, hy;
  unpack2(sub2(pack2(b.x, b.y), pack2(a.z, a.w)), lx, ly);
  unpack2(sub2(pack2(a.x, a.y), pack2(b.z, b.w)), hx, hy);
  const f32x2 e = pack2(fmaxf(fmaxf(lx, hx), 0.0f), fmaxf(fmaxf(ly, hy), 0.0f));
  float sx, sy;
  unpack2(mul2(e, e), sx, sy);
  return __fadd_rn(sx, sy);
}

/* ---- mbarrier + 1-D TMA bulk copy (SASS UBLKCP) ------------------------------------------------ */
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
/* shared-memory loads from 32-bit shared-window addresses held in registers: the hot loops index the clouds and
 * boxes from bases computed once per search instead of re-deriving the window base in every iteration */
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
template <int OFF>
__device__ __forceinline__ float4 lds128_off(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr), "n"(OFF) : "memory");
  return v;
}
/* The shared-window address of an array is "window base + offset", and left to itself the compiler re-derives the window
 * base (S2UR SR_CgaCtaId, ULEA, ...: six dependent instructions, one of them with long latency) in front of every group
 * scan instead of keeping the sum in a register.  An empty asm that claims to modify the value makes it opaque: it can
 * no longer be rematerialised, only kept. */
#ifndef DPGICP_NO_KEEP
#define DPG_KEEP_IN_REGISTER(v) asm volatile("" : "+r"(v))
#else
#define DPG_KEEP_IN_REGISTER(v) do { } while (0)
#endif
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

/* ------------------------------------------------------------------------------------------------
 * shared-memory layout of one CTA
 * ---------------------------------------------------------------------------------------------- */
struct SmemLayout {
  float2 *tgt;      /* n_cap */
  float2 *src;      /* n_cap, current (incrementally transformed) source                           */
  int32_t *nn;      /* n_cap, forward neighbour of the previous pass (seed) / final correspondences */
  float4 *tbox;     /* n_cap/kGroup group boxes of the target                                        */
  float4 *sbox;     /* n_cap/kGroup group boxes of the current source                                */
  float4 *stile;    /* n_cap/32 boxes of the source tiles (query boxes of the forward search)        */
  float4 *tsup;     /* upper level: boxes of kSuper consecutive groups of the target ...             */
  float4 *ssup;     /* ... and of the current source                                                 */
  int32_t *tcnt;    /* n_cap/32 accepted per source tile (rank for the covariance cap)              */
  long long *red;   /* 48 int64: [0..15] totals of the pass, [16..47] this CTA's totals by pass parity (clusters) */
  double *dpart;    /* dpart_bytes(warps): per-warp int64 partials of the pass (two parities) / 16 tile partials of
                     * the covariance (deterministic order) / the rejector's histogram                            */
  float *step;      /* 4 */
  int32_t *ctl;     /* [0] item lo [1] item hi [2] stop [3] K [4] slot                               */
  uint64_t *mbar;
  float *fin;       /* 4: accumulated transform (c, s, tx, ty), read by the projective reciprocal test   */
  float *tkey;      /* projective search only: n_cap beam-order keys of the target ...                    */
  float *skey;      /* ... and of the untransformed source                                                */
  float *ad2;       /* outlier rejection only: n_cap squared distances of the accepted pairs (+inf: none)  */
  int lane;         /* this thread's lane, read from the special register ONCE (an S2R is long-latency; inlined helpers
                     * that each ask for threadIdx.x again get it re-read inside the hot loops)            */
};

/* scratch for the reductions, sized by the CTA width: 2 parities x warps x 12 int64 partials of a pass, and at least
 * kCovChunk x 12 doubles for the covariance (1536 bytes, which also holds the rejector's 256-bin histogram).  Narrow
 * CTAs are the ones that share an SM eight at a time, so every kilobyte counts there. */
__host__ __device__ inline size_t dpart_bytes(int warps) {
  const size_t pass = (size_t)2 * warps * 12 * 8, cov = (size_t)kCovChunk * 12 * 8;
  return pass > cov ? pass : cov;
}

__host__ __device__ inline int n_super_boxes(int n_groups) { return (n_groups + kSuper - 1) / kSuper; }

__host__ __device__ inline size_t smem_bytes(int n_cap, bool projective, bool trim, int warps) {
  const int g = n_cap / kGroup, t = n_cap / kTile;
  return (size_t)n_cap * (8 + 8 + 4) + (size_t)g * (16 + 16) + (size_t)t * (16 + 4) + (size_t)n_super_boxes(g) * (16 + 16) + 48 * 8 +
         dpart_bytes(warps) + 16 + 32 +
         16 + 64 + 16 + (projective ? (size_t)n_cap * 8 : 0) + (trim ? (size_t)n_cap * 4 : 0);
}

__device__ __forceinline__ SmemLayout carve(unsigned char *base, int n_cap, bool projective, int warps) {
  const int g = n_cap / kGroup, t = n_cap / kTile;
  SmemLayout L;
  size_t o = 0;
  L.tgt = (float2 *)(base + o);  o += (size_t)n_cap * 8;
  L.src = (float2 *)(base + o);  o += (size_t)n_cap * 8;
  L.nn = (int32_t *)(base + o);  o += (size_t)n_cap * 4;      /* n_cap % 32 == 0: stays 16-byte aligned */
  L.tbox = (float4 *)(base + o); o += (size_t)g * 16;
  L.sbox = (float4 *)(base + o); o += (size_t)g * 16;
  L.stile = (float4 *)(base + o); o += (size_t)t * 16;
  L.tsup = (float4 *)(base + o); o += (size_t)n_super_boxes(g) * 16;
  L.ssup = (float4 *)(base + o); o += (size_t)n_super_boxes(g) * 16;
  L.red = (long long *)(base + o); o += 48 * 8;
  L.dpart = (double *)(base + o);  o += dpart_bytes(warps);
  L.mbar = (uint64_t *)(base + o); o += 16;
  L.tcnt = (int32_t *)(base + o); o += (size_t)t * 4;
  L.step = (float *)(base + o);   o += 16;
  L.ctl = (int32_t *)(base + o);  o += 32;
  L.fin = (float *)(base + o);    o += 16;
  L.tkey = (float *)(base + o);                               /* present only when launched for the projective search */
  L.skey = L.tkey + n_cap;
  if (projective) o += (size_t)n_cap * 8;
  L.ad2 = (float *)(base + o);                                /* present only when launched with outlier rejection    */
  return L;
}

/* bounding box of the 32 points held one per lane (invalid lanes contribute nothing) */
__device__ __forceinline__ float4 warp_box(float2 p, bool valid) {
  const float inf = __int_as_float(0x7f800000);
  float4 b;
  b.x = warp_min(valid ? p.x : inf);
  b.y = warp_min(valid ? p.y : inf);
  b.z = warp_max(valid ? p.x : -inf);
  b.w = warp_max(valid ? p.y : -inf);
  return b;
}

/* Boxes of one tile (32 points, one per lane): the kGroup-point group boxes (every lane of a group
 * gets its group's box) and the whole tile's box. */
__device__ __forceinline__ void tile_boxes(float2 p, bool valid, float4 &gbox, float4 &tbox) {
  if (kGroup == kTile) {
    gbox = tbox = warp_box(p, valid);
    return;
  }
  const float inf = __int_as_float(0x7f800000);
  float4 b = make_float4(valid ? p.x : inf, valid ? p.y : inf, valid ? p.x : -inf, valid ? p.y : -inf);
#pragma unroll
  for (int o = 1; o < kGroup; o <<= 1) {
    b.x = fminf(b.x, __shfl_xor_sync(0xffffffffu, b.x, o));
    b.y = fminf(b.y, __shfl_xor_sync(0xffffffffu, b.y, o));
    b.z = fmaxf(b.z, __shfl_xor_sync(0xffffffffu, b.z, o));
    b.w = fmaxf(b.w, __shfl_xor_sync(0xffffffffu, b.w, o));
  }
  gbox = b;
  tbox.x = warp_min(b.x); tbox.y = warp_min(b.y); tbox.z = warp_max(b.z); tbox.w = warp_max(b.w);
}

/* store the boxes of tile `tile` of a cloud: group boxes into gb[], tile box into tb[] (may be null) */
__device__ __forceinline__ void store_tile_boxes(float2 p, bool valid, int tile, float4 *gb, float4 *tb, int lane) {
  float4 g, t;
  tile_boxes(p, valid, g, t);
  if ((lane & (kGroup - 1)) == 0) gb[tile * (kTile / kGroup) + lane / kGroup] = g;
  if (tb != nullptr && lane == 0) tb[tile] = t;
}

/* upper level of the hierarchy: box s covers groups [s * kSuper, (s + 1) * kSuper) — 256 consecutive points.  One warp
 * per box: sixteen lanes hold a group box each, four warp-wide minima / maxima.  Called by all warps between two
 * __syncthreads (group boxes complete -> upper boxes complete). */
__device__ __forceinline__ void build_super_boxes(const float4 *gb, int n_groups, float4 *sup, int warp, int nw, int lane) {
  const float inf = __int_as_float(0x7f800000);
  const int n_sup = n_super_boxes(n_groups);
  for (int sb = warp; sb < n_sup; sb += nw) {
    const int g = sb * kSuper + lane;
    float4 b = make_float4(inf, inf, -inf, -inf);
    if (lane < kSuper && g < n_groups) b = gb[g];
    b.x = warp_min(b.x); b.y = warp_min(b.y); b.z = warp_max(b.z); b.w = warp_max(b.w);
    if (lane == 0) sup[sb] = b;
  }
}

/* executed-work counters kept in registers by every warp, flushed once per CTA */
struct SearchStats {
  unsigned scans = 0, tests = 0, window_evals = 0;   /* window_evals: per lane (projective search) */
#ifdef DPGICP_STATS
  unsigned cands = 0, loose = 0, searches = 0, updates = 0;
#endif
};

/* largest binary32 strictly below a squared distance (d2 >= +0): "gd <= below(bd)" is "gd < bd" in one compare */
__device__ __forceinline__ float below(float d2) {
  return d2 > 0.0f ? __int_as_float(__float_as_int(d2) - 1) : -1.0f;
}

/* Candidate rounds of the pruned searches, two levels: ONE lane-parallel round over the upper boxes (256 points each, at
 * most 32 of them for DPGICP_MAX_POINTS), then per round the 2 x 16 groups of the next two surviving upper boxes — 2 to 3
 * rounds for a 1081-point scan where a flat pass over the groups takes 3, 3 to 4 instead of 8 for 4096 points.  An upper
 * box contains its groups' boxes and every operation of the lower bound is monotone, so its bound never exceeds
 * theirs: nothing a flat pass would have kept is dropped.  Groups still come in ascending order.  The brute-force
 * variant walks all groups, 32 per round.  FLAT (kSearchPrunedFlat): a cloud of at most 32 groups is tested in one flat
 * round and needs no upper level.  There is no branch around a test: a lane past the last box reads whatever follows the
 * array in this CTA's shared memory (at most 31 slots of 16 bytes further — the next box array, the reduction scratch —
 * always inside the allocation) and is masked out of the ballot.  Defines mask (bit b = group (b < 16 ? g0 : g1) + (b & 15)). */
#define DPG_ROUNDS_BEGIN(QBOX, BMAX)                                                                                     \
  int base__ = 0;                                                                                                        \
  unsigned up__ = 0u;                                                                                                    \
  if (PRUNED && !FLAT) {                                                                                                 \
    const bool c__ = (lb_box_box(QBOX, lds128(a_sup + lane * 16)) <= (BMAX)) & (lane < n_super_boxes(n_groups));         \
    up__ = __ballot_sync(0xffffffffu, c__);                                                                              \
    ++st.tests;                                                                                                          \
  }                                                                                                                      \
  for (;;) {                                                                                                             \
    unsigned mask;                                                                                                       \
    int g0, g1;                                                                                                          \
    if (PRUNED && FLAT) {                                                                                                \
      if (base__) break;                                                                                                 \
      base__ = 1;                                                                                                        \
      g0 = 0; g1 = kSuper;                                                                                               \
      const bool c__ = (lb_box_box(QBOX, lds128(a_boxes + lane * 16)) <= (BMAX)) & (lane < n_groups);                    \
      mask = __ballot_sync(0xffffffffu, c__);                                                                            \
      ++st.tests;                                                                                                        \
    } else if (PRUNED) {                                                                                                 \
      if (!up__) break;                                                                                                  \
      const int s0__ = __ffs(up__) - 1;                                                                                  \
      up__ &= up__ - 1;                                                                                                  \
      const bool two__ = up__ != 0u;                                                                                     \
      const int s1__ = two__ ? __ffs(up__) - 1 : s0__;                                                                   \
      up__ &= up__ - 1;                 /* 0 & anything = 0: harmless when there was no second box */                    \
      g0 = s0__ * kSuper; g1 = s1__ * kSuper;                                                                            \
      const int gl__ = (lane < kSuper ? g0 : g1) + (lane & (kSuper - 1));                                                \
      const bool c__ = (lb_box_box(QBOX, lds128(a_boxes + gl__ * 16)) <= (BMAX)) & (gl__ < n_groups) &                   \
                       ((lane < kSuper) | two__);                                                                        \
      mask = __ballot_sync(0xffffffffu, c__);                                                                            \
      ++st.tests;                                                                                                        \
    } else {                                                                                                             \
      if (base__ >= n_groups) break;                                                                                     \
      const int rem__ = n_groups - base__;                                                                               \
      mask = rem__ >= 32 ? 0xffffffffu : ((1u << rem__) - 1u);                                                           \
      g0 = base__; g1 = base__ + kSuper;                                                                                 \
      base__ += 32;                                                                                                      \
    }
#define DPG_ROUNDS_END }
#define DPG_NEXT_GROUP(G)                                                                                                \
      const int bit__ = __ffs(mask) - 1;                                                                                 \
      mask &= mask - 1;                                                                                                  \
      const int G = ((bit__ & kSuper) ? g1 : g0) + (bit__ & (kSuper - 1));

/* ------------------------------------------------------------------------------------------------
 * Exact forward nearest neighbour of one query per lane over a grouped cloud in shared memory.
 *   (bd, bj) in: the gate with bj = INT_MAX, or — seeded = true — the neighbour of the previous pass and its distance;
 *   out: the minimum squared distance and its index under the tie rule of include/dpgicp.h: a seeded lane keeps its
 *   seed unless a point is STRICTLY closer; otherwise the lowest index among the minimisers wins.
 *   Each lane carries thr = the largest group minimum that still changes its answer (bd, or the float just below bd
 *   for a lane still on its seed), so one compare decides whether the (d2, index) bookkeeping — first index attaining
 *   the group minimum, 2 instructions per point — has to run at all; with seeds that are still the nearest neighbours
 *   (the steady state of ICP) it never does.
 *   `qbox` is the bounding box of the active lanes' queries.  PRUNED = false scans every group.
 * ---------------------------------------------------------------------------------------------- */
template <bool PRUNED, bool FLAT>
__device__ __forceinline__ void nn_forward(const float2 *__restrict__ cloud, const float4 *__restrict__ boxes,
                                           const float4 *__restrict__ sup, int n_groups, float qx, float qy, bool active, float4 qbox,
                                           float &bd, int &bj, bool seeded, SearchStats &st, float gate, int lane,
                                           float one) {
  const f32x2 one2 = pack2(one, one);
  uint32_t a_cloud = smem_u32(cloud), a_boxes = smem_u32(boxes), a_sup = smem_u32(sup);
  DPG_KEEP_IN_REGISTER(a_cloud); DPG_KEEP_IN_REGISTER(a_boxes); DPG_KEEP_IN_REGISTER(a_sup);
  const f32x2 qx2 = pack2(qx, qx), qy2 = pack2(qy, qy);
  float thr = active ? (seeded ? below(bd) : bd) : -1.0f;
  float bmax = 0.0f;
  if (PRUNED) bmax = warp_max(thr);
#ifdef DPGICP_STATS
  st.searches++;
  if (bmax >= gate) st.loose++;
#endif
  DPG_ROUNDS_BEGIN(qbox, bmax)
#ifdef DPGICP_STATS
    if (PRUNED) st.cands += __popc(mask);
#endif
    while (mask) {
      DPG_NEXT_GROUP(g)
      ++st.scans;
      const uint32_t a_grp = a_cloud + g * (kGroup * 8);
      float dd[kGroup];
      float gd = __int_as_float(0x7f800000);
#define DPG_SCAN2(T)                                                                                  \
      if (2 * (T) < kGroup) {                                                                         \
        const float4 p = lds128_off<16 * (T)>(a_grp);     /* (x0, x1, y0, y1) of two points, broadcast */ \
        const f32x2 ex = sub2(qx2, pack2(p.x, p.y)), ey = sub2(qy2, pack2(p.z, p.w));                  \
        unpack2(add2(mul2(ex, ex), mul2(ey, ey), one2), dd[(2 * (T)) % kGroup], dd[(2 * (T) + 1) % kGroup]); \
        gd = fminf(fminf(gd, dd[(2 * (T)) % kGroup]), dd[(2 * (T) + 1) % kGroup]);                     \
      }
      DPG_SCAN2(0) DPG_SCAN2(1) DPG_SCAN2(2) DPG_SCAN2(3) DPG_SCAN2(4) DPG_SCAN2(5) DPG_SCAN2(6) DPG_SCAN2(7)
      DPG_SCAN2(8) DPG_SCAN2(9) DPG_SCAN2(10) DPG_SCAN2(11) DPG_SCAN2(12) DPG_SCAN2(13) DPG_SCAN2(14) DPG_SCAN2(15)
#undef DPG_SCAN2
      if (!__any_sync(0xffffffffu, gd <= thr)) continue;
#ifdef DPGICP_STATS
      st.updates++;
#endif
      int gj = kGroup - 1;                              /* first index attaining the minimum       */
#pragma unroll
      for (int t = kGroup - 2; t >= 0; --t)
        if (dd[t] == gd) gj = t;
      const int j = g * kGroup + gj;
      /* groups come in ascending order: a tie with an earlier group's point (j > bj) never wins */
      if (gd <= thr && (gd < bd || j < bj)) { bd = gd; bj = j; thr = gd; }
    }
  DPG_ROUNDS_END
}

/* ------------------------------------------------------------------------------------------------
 * Reciprocal test as an emptiness query: is any point of the cloud STRICTLY closer to this lane's query than bd?
 * (the asker wins exact ties, include/dpgicp.h).  No indices are tracked; a lane that has found a closer point stops
 * asking for scans.  A per-lane point-to-box test and a warp vote in front of every candidate group's scan skip the
 * groups no lane can use (21 % of the candidates, measured).
 * ---------------------------------------------------------------------------------------------- */
template <bool PRUNED, bool FLAT>
__device__ __forceinline__ bool nn_closer_exists(const float2 *__restrict__ cloud, const float4 *__restrict__ boxes,
                                                 const float4 *__restrict__ sup, int n_groups, float qx, float qy, bool active,
                                                 float4 qbox, float bd,
                                                 SearchStats &st, int lane, float one) {
  const f32x2 one2 = pack2(one, one);
  uint32_t a_cloud = smem_u32(cloud), a_boxes = smem_u32(boxes), a_sup = smem_u32(sup);
  DPG_KEEP_IN_REGISTER(a_cloud); DPG_KEEP_IN_REGISTER(a_boxes); DPG_KEEP_IN_REGISTER(a_sup);
  const f32x2 q2 = pack2(qx, qy), qx2 = pack2(qx, qx), qy2 = pack2(qy, qy);
  float thr = active ? below(bd) : -1.0f;               /* -1: this lane needs nothing (any more; or bd = 0: nothing can be closer) */
  bool closer = false;
  float bmax = 0.0f;
  if (PRUNED) bmax = warp_max(thr);
#ifdef DPGICP_STATS
  st.searches++;
#endif
  DPG_ROUNDS_BEGIN(qbox, bmax)
#ifdef DPGICP_STATS
    if (PRUNED) st.cands += __popc(mask);
#endif
    while (mask) {
      DPG_NEXT_GROUP(g)
      if (PRUNED) {
        const bool need = lb_point_box(q2, lds128(a_boxes + g * 16)) <= thr;
        if (!__any_sync(0xffffffffu, need)) continue;
      }
      ++st.scans;
      const uint32_t a_grp = a_cloud + g * (kGroup * 8);
      float gd = __int_as_float(0x7f800000);
#define DPG_SCAN2(T)                                                                                  \
      if (2 * (T) < kGroup) {                                                                         \
        const float4 p = lds128_off<16 * (T)>(a_grp);                                                 \
        const f32x2 ex = sub2(qx2, pack2(p.x, p.y)), ey = sub2(qy2, pack2(p.z, p.w));                  \
        float d0, d1;                                                                                 \
        unpack2(add2(mul2(ex, ex), mul2(ey, ey), one2), d0, d1);                                      \
        gd = fminf(fminf(gd, d0), d1);                                                                \
      }
      DPG_SCAN2(0) DPG_SCAN2(1) DPG_SCAN2(2) DPG_SCAN2(3) DPG_SCAN2(4) DPG_SCAN2(5) DPG_SCAN2(6) DPG_SCAN2(7)
      DPG_SCAN2(8) DPG_SCAN2(9) DPG_SCAN2(10) DPG_SCAN2(11) DPG_SCAN2(12) DPG_SCAN2(13) DPG_SCAN2(14) DPG_SCAN2(15)
#undef DPG_SCAN2
      if (gd <= thr) { closer = true; thr = -1.0f; }    /* a strictly closer point: this lane is done */
    }
  DPG_ROUNDS_END
  return closer;
}

/* ------------------------------------------------------------------------------------------------
 * One correspondence pass for one source tile (32 consecutive source points, one per lane).
 * Returns accept flag; j = matched target index, d = its squared distance.
 * PCL determineReciprocalCorrespondences (App. A.3-2): forward NN within the gate, then the target
 * point's own nearest source point must be the query ((d2, index)-lexicographic, like the forward).
 * ---------------------------------------------------------------------------------------------- */
/* ---- DPGICP_SEARCH_PROJECTIVE (include/dpgicp.h; defined by oracle/dpg_oracle.c correspondences_projective) ---- */
/* bearing key of a point seen from the laser origin: monotone in atan2 on (-pi, pi], no libm, IEEE division */
__device__ __forceinline__ float beam_key(float px, float py, float ox, float oy) {
  const float vx = __fsub_rn(px, ox), vy = __fsub_rn(py, oy);
  const float a = __fadd_rn(fabsf(vx), fabsf(vy));
  const float t = a > 0.0f ? __fdiv_rn(vy, a) : 0.0f;
  if (vx >= 0.0f) return t;
  return vy >= 0.0f ? __fsub_rn(2.0f, t) : __fsub_rn(-2.0f, t);
}
/* plain bisection over the stored order */
__device__ __forceinline__ int key_lower_bound(const float *keys, int n, float k) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (keys[mid] < k) lo = mid + 1; else hi = mid;
  }
  return lo;
}
/* (d2, index) argmin of (qx, qy) over cloud[c - W, c + W) clipped to [0, n): ascending scan, strict improvement */
__device__ __forceinline__ void nn_window(const float2 *cloud, int n, int c, int W, float qx, float qy, float &bd, int &bj,
                                          SearchStats &st) {
  const int j0 = c - W < 0 ? 0 : c - W, j1 = c + W > n ? n : c + W;
  const f32x2 q2 = pack2(qx, qy);
  bd = __int_as_float(0x7f800000);
  bj = -1;
  for (int j = j0; j < j1; ++j) {
    const float2 p = ld_pt<false>(cloud, j);
    const float d = dist2_packed(q2, pack2(p.x, p.y));
    if (d < bd) { bd = d; bj = j; }
  }
  st.window_evals += (unsigned)(j1 > j0 ? j1 - j0 : 0);
}

/* one correspondence pass of one source tile, projective search: every lane works alone */
__device__ __forceinline__ bool match_tile_projective(const SmemLayout &L, int tile, int ns, int nt, float gate,
                                                      bool reciprocal, int W, float ox, float oy, float2 &q, int &j_out,
                                                      float &d_out, bool &fwd_ok, SearchStats &st) {
  const int lane = L.lane;
  const int i = tile * kTile + lane;
  const bool valid = i < ns;
  q = ld_pt<false>(L.src, i);
  float bd = __int_as_float(0x7f800000);
  int bj = -1;
  if (valid) nn_window(L.tgt, nt, key_lower_bound(L.tkey, nt, beam_key(q.x, q.y, ox, oy)), W, q.x, q.y, bd, bj, st);
  fwd_ok = valid && bj >= 0 && bd <= gate;
  j_out = bj;
  d_out = bd;
  bool accept = fwd_ok;
  if (reciprocal && fwd_ok) {
    /* the matched target point in the source scan's own frame: R^T (r - t) */
    const float2 r = ld_pt<false>(L.tgt, bj);
    const float fc = L.fin[0], fs = L.fin[1];
    const float ex = __fsub_rn(r.x, L.fin[2]), ey = __fsub_rn(r.y, L.fin[3]);
    const float bx = __fadd_rn(__fmul_rn(fc, ex), __fmul_rn(fs, ey));
    const float by = __fsub_rn(__fmul_rn(fc, ey), __fmul_rn(fs, ex));
    float rd;
    int ri;
    nn_window(L.src, ns, key_lower_bound(L.skey, ns, beam_key(bx, by, ox, oy)), W, r.x, r.y, rd, ri, st);
    accept = (ri == i) && (rd <= gate);
  }
  return accept;
}

template <bool PRUNED, bool FLAT>
__device__ __forceinline__ bool match_tile(const SmemLayout &L, int tile, int ns, int n_groups_s,
                                           int n_groups_t, float gate, bool reciprocal, float one, float2 &q,
                                           int &j_out, float &d_out, bool &fwd_ok, SearchStats &st) {
  const int lane = L.lane;
  const int i = tile * kTile + lane;
  const bool valid = i < ns;
  q = ld_pt<true>(L.src, i);
  float bd = gate;
  int bj = 0x7fffffff;
  /* the previous pass's neighbour seeds the bound and is the tie preference (brute force and pruned search alike) */
  bool seeded = false;
  int seed = valid ? L.nn[i] : -1;
  if (seed >= 0) seed &= kNnIndexMask;
  DPG_CHECK(seed >= -1 && seed < n_groups_t * kGroup);
  if (seed >= 0) {
    const float2 p = ld_pt<true>(L.tgt, seed);
    const float d0 = dist2(q.x, q.y, p.x, p.y);
    if (d0 <= gate) { bd = d0; bj = seed; seeded = true; }
  }
  nn_forward<PRUNED, FLAT>(L.tgt, L.tbox, L.tsup, n_groups_t, q.x, q.y, valid, L.stile[tile], bd, bj, seeded, st, gate, lane, one);
  fwd_ok = valid && (bj != 0x7fffffff);
  DPG_CHECK(!fwd_ok || (bj >= 0 && bj < n_groups_t * kGroup && bd <= gate));
  j_out = bj;
  d_out = bd;
  bool accept = fwd_ok;
  if (reciprocal && __any_sync(0xffffffffu, fwd_ok)) {
    float2 r = make_float2(0.f, 0.f);
    if (fwd_ok) r = ld_pt<true>(L.tgt, bj);
    const float4 rbox = warp_box(r, fwd_ok);
    /* dist2(r, p) == dist2(p, r) bit for bit: fl(a-b) = -fl(b-a) and the square drops the sign, so source point i
     * itself is at exactly bd from r and "strictly closer than bd" is well defined */
    const bool closer = nn_closer_exists<PRUNED, FLAT>(L.src, L.sbox, L.ssup, n_groups_s, r.x, r.y, fwd_ok, rbox, bd, st, lane, one);
    accept = fwd_ok && !closer;
  }
  return accept;
}

struct KernelParams;
/* one correspondence pass of one source tile with the search strategy the kernel was instantiated for */
template <int SEARCH, typename KP>
__device__ __forceinline__ bool match_any(const SmemLayout &L, const KP &P, int tile, int ns, int nt, int gs, int gt,
                                          float2 &q, int &j, float &d, bool &fwd, SearchStats &st) {
  if constexpr (search_is_projective(SEARCH))
    return match_tile_projective(L, tile, ns, nt, P.gate, P.use_reciprocal != 0, P.proj_window, P.sensor_x, P.sensor_y, q, j,
                                 d, fwd, st);
  else
    return match_tile<search_is_pruned(SEARCH), search_is_flat(SEARCH)>(L, tile, ns, gs, gt, P.gate, P.use_reciprocal != 0, P.one, q, j, d, fwd, st);
}

/* ------------------------------------------------------------------------------------------------
 * covariance finishing (3x3 algebra), mirrors oracle/dpg_oracle.c orc_cov_censi
 * sums: [0] n_h [1] SA [2] SB [3] SE   (Hessian, all pairs)
 *       [4] n_d [5] Sdx [6] Sdy [7] SA_d [8] SB_d [9] S(dx^2+dy^2) [10] S(A^2+B^2)  (capped set)
 * ---------------------------------------------------------------------------------------------- */
__device__ inline uint32_t finish_cov(const double *S, double sensor_var, const float *live, double *cov) {
  double H[9], M[9], Hi[9];
  H[0] = 2.0 * S[0]; H[1] = 0.0;        H[2] = -2.0 * S[2];
  H[3] = 0.0;        H[4] = 2.0 * S[0]; H[5] = 2.0 * S[1];
  H[6] = H[2];       H[7] = H[5];       H[8] = -2.0 * S[3];
  M[0] = 8.0 * S[4]; M[1] = 0.0;        M[2] = 4.0 * (S[6] - S[8]);
  M[3] = 0.0;        M[4] = 8.0 * S[4]; M[5] = 4.0 * (S[7] - S[5]);
  M[6] = M[2];       M[7] = M[5];       M[8] = 4.0 * S[9] + 4.0 * S[10];
  bool ok = S[0] > 0.0;
  const double a = H[0], b = H[1], c = H[2], d = H[4], e = H[5], f = H[8];
  const double c00 = d * f - e * e, c01 = c * e - b * f, c02 = b * e - c * d;
  const double det = a * c00 + b * c01 + c * c02;
  if (!(fabs(det) > 0.0) || !isfinite(det)) ok = false;
  if (ok) {
    const double id = 1.0 / det;
    Hi[0] = c00 * id; Hi[1] = c01 * id; Hi[2] = c02 * id;
    Hi[3] = Hi[1];    Hi[4] = (a * f - c * c) * id; Hi[5] = (b * c - a * e) * id;
    Hi[6] = Hi[2];    Hi[7] = Hi[5];    Hi[8] = (a * d - b * b) * id;
    double Tm[9];
    for (int r = 0; r < 3; ++r)
      for (int q = 0; q < 3; ++q)
        Tm[3 * r + q] = Hi[3 * r] * M[q] + Hi[3 * r + 1] * M[3 + q] + Hi[3 * r + 2] * M[6 + q];
    for (int r = 0; r < 3; ++r)
      for (int q = 0; q < 3; ++q)
        cov[3 * r + q] =
            sensor_var * (Tm[3 * r] * Hi[q] + Tm[3 * r + 1] * Hi[3 + q] + Tm[3 * r + 2] * Hi[6 + q]);
    for (int k = 0; k < 9; ++k)
      if (!isfinite(cov[k])) ok = false;
  }
  if (!ok) {
    for (int k = 0; k < 9; ++k) cov[k] = 0.0;
    cov[0] = live[0]; cov[4] = live[1]; cov[8] = live[2];
    return DPGICP_FLAG_COV_SINGULAR;
  }
  return 0u;
}

/* per-pair terms of the covariance sums for source point p (untransformed) and target q */
__device__ __forceinline__ void cov_terms(double px, double py, double qx, double qy, double c, double s,
                                          double x, double y, bool in_h, bool in_d, double *acc) {
  const double A = px * c - py * s, B = px * s + py * c;
  const double dx = x - qx, dy = y - qy;
  if (in_h) {
    acc[0] += 1.0; acc[1] += A; acc[2] += B; acc[3] += A * dx + B * dy;
  }
  if (in_d) {
    acc[4] += 1.0; acc[5] += dx; acc[6] += dy; acc[7] += A; acc[8] += B;
    acc[9] += dx * dx + dy * dy; acc[10] += A * A + B * B;
  }
}

/* deterministic block reduction of 11 doubles: lanes by xor-shuffle, warps summed in order */
template <int WARPS>
__device__ __forceinline__ void block_sum11(double *acc, double *dpart, double *out /* thread 0 */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 11; ++k) acc[k] = warp_sum_f64(acc[k]);
  if (lane == 0)
    for (int k = 0; k < 11; ++k) dpart[warp * 12 + k] = acc[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < 11; ++k) {
      double v = 0.0;
      for (int w = 0; w < WARPS; ++w) v = __dadd_rn(v, dpart[w * 12 + k]);
      out[k] = v;
    }
  }
  __syncthreads();
}

/* ------------------------------------------------------------------------------------------------
 * Rigid steps (thread 0 of the CTA), mirroring oracle/dpg_oracle.c operation for operation.
 * red[0..8] = nine exact fixed-point sums (meaning depends on the metric), red[9] = sum d2, red[10] = K
 * ---------------------------------------------------------------------------------------------- */
/* point-to-point: planar Procrustes in binary64 (PCL TransformationEstimationSVD on z = 0 data).
 * Division by K and by the norm are multiplications by one reciprocal each, so the dependent chain is
 * reciprocal(K) || sums -> sqrt -> reciprocal -> products (this runs on one thread per pass). */
__device__ __forceinline__ void solve_p2p(const long long *red, double invK, float st[4]) {
  const double spx = __dmul_rn((double)red[0], 1.0 / kScaleLin);
  const double spy = __dmul_rn((double)red[1], 1.0 / kScaleLin);
  const double sqx = __dmul_rn((double)red[2], 1.0 / kScaleLin);
  const double sqy = __dmul_rn((double)red[3], 1.0 / kScaleLin);
  const double dot = __dmul_rn((double)(red[4] + red[7]), 1.0 / kScaleProd);
  const double crs = __dmul_rn((double)(red[5] - red[6]), 1.0 / kScaleProd);
  const double a = __dsub_rn(dot, __dmul_rn(__dadd_rn(__dmul_rn(spx, sqx), __dmul_rn(spy, sqy)), invK));
  const double b = __dsub_rn(crs, __dmul_rn(__dsub_rn(__dmul_rn(spx, sqy), __dmul_rn(spy, sqx)), invK));
  const double h = __dsqrt_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)));
  double c = 1.0, s = 0.0;
  if (h > 0.0) { const double rh = __ddiv_rn(1.0, h); c = __dmul_rn(a, rh); s = __dmul_rn(b, rh); }
  const double mpx = __dmul_rn(spx, invK), mpy = __dmul_rn(spy, invK);
  const double mqx = __dmul_rn(sqx, invK), mqy = __dmul_rn(sqy, invK);
  const double tx = __dsub_rn(mqx, __dsub_rn(__dmul_rn(c, mpx), __dmul_rn(s, mpy)));
  const double ty = __dsub_rn(mqy, __dadd_rn(__dmul_rn(s, mpx), __dmul_rn(c, mpy)));
  st[0] = (float)c; st[1] = (float)s; st[2] = (float)tx; st[3] = (float)ty;
}

/* point-to-line: one Gauss-Newton step from the 3x3 normal equations, Cholesky; the rotation is the
 * Cayley map of dtheta/2 (rational, no libm).  Returns false when A is not positive definite. */
__device__ __forceinline__ bool solve_p2l(const long long *red, float st[4]) {
  const double inv = 1.0 / kScaleProd;
  const double a11 = __dmul_rn((double)red[0], inv), a12 = __dmul_rn((double)red[1], inv);
  const double a13 = __dmul_rn((double)red[2], inv), a22 = __dmul_rn((double)red[3], inv);
  const double a23 = __dmul_rn((double)red[4], inv), a33 = __dmul_rn((double)red[5], inv);
  const double b1 = -__dmul_rn((double)red[6], inv), b2 = -__dmul_rn((double)red[7], inv);
  const double b3 = -__dmul_rn((double)red[8], inv);
  if (!(a11 > 0.0)) return false;
  const double l11 = __dsqrt_rn(a11);
  const double l21 = __ddiv_rn(a12, l11), l31 = __ddiv_rn(a13, l11);
  const double d22 = __dsub_rn(a22, __dmul_rn(l21, l21));
  if (!(d22 > 0.0)) return false;
  const double l22 = __dsqrt_rn(d22);
  const double l32 = __ddiv_rn(__dsub_rn(a23, __dmul_rn(l31, l21)), l22);
  const double d33 = __dsub_rn(__dsub_rn(a33, __dmul_rn(l31, l31)), __dmul_rn(l32, l32));
  if (!(d33 > 0.0)) return false;
  const double l33 = __dsqrt_rn(d33);
  const double y1 = __ddiv_rn(b1, l11);
  const double y2 = __ddiv_rn(__dsub_rn(b2, __dmul_rn(l21, y1)), l22);
  const double y3 = __ddiv_rn(__dsub_rn(__dsub_rn(b3, __dmul_rn(l31, y1)), __dmul_rn(l32, y2)), l33);
  const double x3 = __ddiv_rn(y3, l33);
  const double x2 = __ddiv_rn(__dsub_rn(y2, __dmul_rn(l32, x3)), l22);
  const double x1 = __ddiv_rn(__dsub_rn(__dsub_rn(y1, __dmul_rn(l21, x2)), __dmul_rn(l31, x3)), l11);
  if (!isfinite(x1) || !isfinite(x2) || !isfinite(x3)) return false;
  const double u = __dmul_rn(0.5, x3);
  const double uu = __dmul_rn(u, u);
  const double den = __dadd_rn(1.0, uu);
  st[0] = (float)__ddiv_rn(__dsub_rn(1.0, uu), den);
  st[1] = (float)__ddiv_rn(__dadd_rn(u, u), den);
  st[2] = (float)x1;
  st[3] = (float)x2;
  return true;
}

/* fixed-point term: round-to-nearest-even of v * 2^28 */
__device__ __forceinline__ long long fxp(double v) { return __double2ll_rn(__dmul_rn(v, kScaleProd)); }

/* ------------------------------------------------------------------------------------------------
 * Moment sums of one accepted pair (q = current source point, target j, d = squared distance): m[0..8] are the
 * nine exact fixed-point sums of the metric, m[9] = sum d2 (2^40).  Mirrors oracle/dpg_oracle.c accumulate_moments /
 * accumulate_normal_eq term for term.
 * ---------------------------------------------------------------------------------------------- */
template <bool IL, typename KP>
__device__ __forceinline__ void accumulate_pair(const SmemLayout &L, const KP &P, bool p2l, float2 q, int j, float d, int nt,
                                                long long (&m)[10], int &m_k) {
  const float2 t = ld_pt<IL>(L.tgt, j);
  const double px = q.x, py = q.y, qx = t.x, qy = t.y;
  if (p2l) {
    /* line through the matched target point and its closer beam neighbour (oracle:
     * accumulate_normal_eq); m0..m5 = A (11,12,13,22,23,33), m6..m8 = sum J^T r */
    int j2 = -1;
    float best = __int_as_float(0x7f800000);
    if (j - 1 >= 0) { const float2 a = ld_pt<IL>(L.tgt, j - 1); best = dist2(q.x, q.y, a.x, a.y); j2 = j - 1; }
    if (j + 1 < nt) {
      const float2 a = ld_pt<IL>(L.tgt, j + 1);
      const float dn = dist2(q.x, q.y, a.x, a.y);
      if (dn < best) { best = dn; j2 = j + 1; }
    }
    bool line = false;
    double nx = 0.0, ny = 0.0;
    if (j2 >= 0) {
      const float2 a = ld_pt<IL>(L.tgt, j2);
      const float seg = dist2(a.x, a.y, t.x, t.y);
      if (seg > 0.0f && seg <= P.gate) {
        const double tx = __dsub_rn((double)a.x, qx), ty = __dsub_rn((double)a.y, qy);
        const double len = __dsqrt_rn(__dadd_rn(__dmul_rn(tx, tx), __dmul_rn(ty, ty)));
        nx = __ddiv_rn(-ty, len);
        ny = __ddiv_rn(tx, len);
        line = true;
      }
    }
    const double ex = __dsub_rn(px, qx), ey = __dsub_rn(py, qy);
    if (line) {
      const double r = __dadd_rn(__dmul_rn(nx, ex), __dmul_rn(ny, ey));
      const double j3 = __dsub_rn(__dmul_rn(ny, px), __dmul_rn(nx, py));
      m[0] += fxp(__dmul_rn(nx, nx)); m[1] += fxp(__dmul_rn(nx, ny)); m[2] += fxp(__dmul_rn(nx, j3));
      m[3] += fxp(__dmul_rn(ny, ny)); m[4] += fxp(__dmul_rn(ny, j3)); m[5] += fxp(__dmul_rn(j3, j3));
      m[6] += fxp(__dmul_rn(nx, r)); m[7] += fxp(__dmul_rn(ny, r)); m[8] += fxp(__dmul_rn(j3, r));
    } else {
      m[0] += fxp(1.0); m[2] += fxp(-py);
      m[3] += fxp(1.0); m[4] += fxp(px);
      m[5] += fxp(__dadd_rn(__dmul_rn(px, px), __dmul_rn(py, py)));
      m[6] += fxp(ex); m[7] += fxp(ey);
      m[8] += fxp(__dsub_rn(__dmul_rn(px, ey), __dmul_rn(py, ex)));
    }
  } else {
    /* point-to-point moments: sums of p, q (2^32) and of the four products (2^28) */
    m[0] += __double2ll_rn(__dmul_rn(px, kScaleLin));
    m[1] += __double2ll_rn(__dmul_rn(py, kScaleLin));
    m[2] += __double2ll_rn(__dmul_rn(qx, kScaleLin));
    m[3] += __double2ll_rn(__dmul_rn(qy, kScaleLin));
    m[4] += fxp(__dmul_rn(px, qx));
    m[5] += fxp(__dmul_rn(px, qy));
    m[6] += fxp(__dmul_rn(py, qx));
    m[7] += fxp(__dmul_rn(py, qy));
  }
  m[9] += __double2ll_rn(__dmul_rn((double)d, kScaleD2));
  m_k += 1;
}

/* ------------------------------------------------------------------------------------------------
 * Outlier rejection threshold tau (include/dpgicp.h DPGICP_OUTLIER_*; oracle: orc_outlier_threshold) over the accepted
 * squared distances L.ad2[0 .. n_pad) (+inf = not accepted).  Exact block-wide radix select: four rounds of 8 bits over
 * the binary32 patterns (d2 >= +0, so the patterns order like the values), a 256-bin histogram in shared memory per
 * round.  Every thread of the CTA calls it between two __syncthreads-separated phases; all get the same tau
 * (+inf only when no pair was accepted).  With 1 or 2 accepted pairs the rule still applies, as in the oracle and
 * DESIGN §5.8: the pass then stops on K < 3 either way, but the kept set is what the parity hook returns and the
 * record's n_correspondences counts.  Scratch: L.dpart (free between the passes' reductions) and L.ctl[5..7].
 * ---------------------------------------------------------------------------------------------- */
__device__ __forceinline__ float select_tau(const SmemLayout &L, int n_pad, int mode, double param) {
  const float inf = __int_as_float(0x7f800000);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthreads = blockDim.x;
  int *hist = reinterpret_cast<int *>(L.dpart);
  int *sel = L.ctl + 5;
  if (tid == 0) sel[0] = 0;
  __syncthreads();
  int c = 0;
  for (int k = tid; k < n_pad; k += nthreads) c += (L.ad2[k] < inf) ? 1 : 0;
  c = __reduce_add_sync(0xffffffffu, c);
  if (lane == 0 && c) atomicAdd(&sel[0], c);
  __syncthreads();
  const int K = sel[0];
  if (K < 1) return inf;
  int r;
  if (mode == DPGICP_OUTLIER_TRIMMED) {
    int keep = (int)floor(__dmul_rn(param, (double)K));
    keep = keep < 3 ? 3 : keep;
    keep = keep > K ? K : keep;
    r = keep - 1;
  } else {
    r = K / 2;
  }
  uint32_t prefix = 0;
  for (int round = 0; round < 4; ++round) {
    const int shift = 24 - 8 * round;
    for (int k = tid; k < 256; k += nthreads) hist[k] = 0;
    __syncthreads();
    const uint32_t himask = round == 0 ? 0u : (0xffffffffu << (shift + 8));
    for (int k = tid; k < n_pad; k += nthreads) {
      const uint32_t key = __float_as_uint(L.ad2[k]);
      if (key < 0x7f800000u && (key & himask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1);
    }
    __syncthreads();
    if (warp == 0) {
      int h[8], tot = 0;
#pragma unroll
      for (int u = 0; u < 8; ++u) { h[u] = hist[lane * 8 + u]; tot += h[u]; }
      int incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      const int excl = incl - tot;
      const bool mine = r >= excl && r < incl;         /* exactly one lane: the bins hold K > r keys in all */
      int bin = 0, before = 0;
      if (mine) {
        int acc = excl;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (r >= acc && r < acc + h[u]) { bin = lane * 8 + u; before = acc; }
          acc += h[u];
        }
      }
      DPG_CHECK(__popc(__ballot_sync(0xffffffffu, mine)) == 1);
      const int src = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
      bin = __shfl_sync(0xffffffffu, bin, src);
      before = __shfl_sync(0xffffffffu, before, src);
      if (lane == 0) { sel[1] = bin; sel[2] = before; }
    }
    __syncthreads();
    prefix |= (uint32_t)sel[1] << shift;
    r -= sel[2];
  }
  const float stat = __uint_as_float(prefix);
  if (mode == DPGICP_OUTLIER_TRIMMED) return stat;
  const double lim = __dmul_rn((double)stat, param);
  float tau = __double2float_rn(lim);
  if ((double)tau > lim) tau = __uint_as_float(__float_as_uint(tau) - 1u);   /* nextafterf(tau, -inf), tau > 0 here */
  return tau;
}

/* ------------------------------------------------------------------------------------------------
 * The persistent ICP + covariance kernel.
 *
 * Staged execution.  ICP iteration counts are heavy-tailed (corridor workload: median 37, p99 174,
 * max 305 passes), so a fixed CTA shape either wastes the machine on the last long pairs (narrow
 * CTAs: few warps left running) or wastes issue slots on the bulk (wide CTAs).  The host therefore
 * launches the same kernel as a chain of stages with growing WARPS.  A stage works through its queue;
 * once the queue is EMPTY, every CTA suspends the pair it is on at the next pass boundary (current
 * source cloud, neighbour seeds and a few scalars go to a state slot in HBM) and the stage ends with
 * all SMs still busy.  The next, wider stage resumes the suspended pairs — at most one per CTA of the
 * previous stage — with more warps per pair.  The last stage runs to completion.  State is restored
 * bit for bit, so staging cannot change results (tested: any chain == single stage).
 * ---------------------------------------------------------------------------------------------- */
/* resident CTAs per SM the register allocation is held to (DPGICP_TARGET_WARPS resident warps per SM) */
#ifndef DPGICP_TARGET_WARPS
#define DPGICP_TARGET_WARPS 28
#endif
/* CTAs of up to 4 warps: 28 resident warps per SM (7 x 4 warps, 72 registers) for the general instantiations, 32 (8 x 4
 * warps, 64 registers; fits since the reduction scratch is sized by the CTA width) for the stock-configuration ones.
 * Measured: with the general kernel the 64-register build spills in the pass loop and 8 CTAs equal 7 (471.6 k vs 474.4 k
 * pairs/s); the stock kernel, with the point-to-line / rejector / hook code compiled out, spills less and gains
 * (486 k -> 497 k pairs/s corridor, 692 k -> 711 k loop closure). */
#ifndef DPGICP_TARGET_WARPS_NARROW
#define DPGICP_TARGET_WARPS_NARROW 28
#endif
#ifndef DPGICP_TARGET_WARPS_NARROW_STOCK
#define DPGICP_TARGET_WARPS_NARROW_STOCK 32
#endif
__host__ __device__ constexpr int min_ctas(int warps, int search) {
  const int target = warps <= 4 ? (search_is_stock(search) ? DPGICP_TARGET_WARPS_NARROW_STOCK : DPGICP_TARGET_WARPS_NARROW)
                                : DPGICP_TARGET_WARPS;
  return (target / warps) < 1 ? 1 : (target / warps) > 16 ? 16 : (target / warps);   /* 16, 17, 32 -> 1 */
}

/* CSIZE > 1: a thread-block CLUSTER of CSIZE CTAs (one per SM) works on one pair — used by the host for the
 * last stage of the chain, where a few long pairs are all that is left and one SM cannot run a pass faster
 * (it is bound by its issue rate).  Every CTA of the cluster stages both clouds in its own shared memory and
 * keeps them identical (each applies every step to all source points — redundant but exact); the search
 * tiles are split over the CTAs; the per-warp partial sums of all CTAs are read through distributed shared
 * memory after one cluster barrier per pass, so every CTA forms the same exact integer totals and takes the
 * same step and the same stop decision without any broadcast.  CTA 0 writes the record. */
template <int CSIZE>
__device__ __forceinline__ void pair_sync() {
  if constexpr (CSIZE > 1) cooperative_groups::this_cluster().sync();
  else __syncthreads();
}
template <int CSIZE, typename T>
__device__ __forceinline__ T *peer_smem(T *p, int rank) {
  if constexpr (CSIZE > 1) return cooperative_groups::this_cluster().map_shared_rank(p, rank);
  else return p;
}

template <int WARPS, int SEARCH, int CSIZE>
__global__ void __launch_bounds__(WARPS * 32, min_ctas(WARPS, SEARCH)) icp_pairs_kernel(const KernelParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  SmemLayout L = carve(smem_raw, P.n_cap, search_is_projective(SEARCH), (int)(blockDim.x >> 5));
  int tid = threadIdx.x;
  DPG_KEEP_IN_REGISTER(tid);
  int lane = tid & 31;
  DPG_KEEP_IN_REGISTER(lane);
  L.lane = lane;
  const int warp = tid >> 5;
  const int nw = blockDim.x >> 5;            /* warps of this CTA: <= WARPS (and <= 16), chosen by the host so
                                              * that the pair's tiles divide evenly among them                 */
  const int nthreads = blockDim.x;
  int crank = 0;                             /* rank of this CTA in its cluster                                */
  if constexpr (CSIZE > 1) crank = (int)cooperative_groups::this_cluster().block_rank();
  const int tile0 = crank * nw + warp, tile_stride = nw * CSIZE;     /* search tiles of this warp             */
  const int div = P.divisor;
  constexpr int GPT = kTile / kGroup;        /* groups per tile */
  uint32_t mbar_phase = 0;
  constexpr bool IL = !search_is_projective(SEARCH);   /* cloud layout in shared memory: pair-interleaved or plain */
  constexpr bool STOCK = search_is_stock(SEARCH);      /* point-to-point, no rejector, no parity hook: the host's promise */
  const bool trim = !STOCK && (CSIZE == 1) && P.outlier_mode != DPGICP_OUTLIER_NONE;   /* the host never combines it with clusters */
  const bool p2l = !STOCK && P.metric == DPGICP_METRIC_POINT_TO_LINE;

  if (tid == 0) mbar_init(L.mbar, 1);
  __syncthreads();
  /* a CTA may address a peer's shared memory only once every CTA of the cluster has started: one cluster barrier
   * before the first work fetch (which stores the item into the peers' control words) */
  if constexpr (CSIZE > 1) cooperative_groups::this_cluster().sync();

  SearchStats stats;
  unsigned long long c_iters = 0, c_corr = 0;
  const unsigned long long n_items =
      P.resume ? (unsigned long long)(*P.in_count) : (unsigned long long)P.n_pairs;

  for (;;) {
    /* ---- fetch the next work item ----------------------------------------------------------- */
    if (tid == 0 && crank == 0) {
      const unsigned long long k = atomicAdd(P.queue, 1ull);
      for (int r = 0; r < CSIZE; ++r) {               /* every CTA of the cluster works on the same item */
        int32_t *c = peer_smem<CSIZE>(L.ctl, r);
        c[0] = (int32_t)(k & 0xffffffffu);
        c[1] = (int32_t)(k >> 32);
      }
    }
    pair_sync<CSIZE>();
    const unsigned long long item = ((unsigned long long)(uint32_t)L.ctl[1] << 32) | (uint32_t)L.ctl[0];
    if (item >= n_items) break;
    const long long pair = P.resume ? P.susp_in[item] : (P.order ? P.order[item] : (long long)item);
    const unsigned char *slot_in = P.resume ? P.state_in + (size_t)item * (size_t)P.slot_bytes : nullptr;
    DPG_CHECK(pair >= 0 && pair < P.n_pairs);
    const PairTask task = P.tasks[pair];
    DPG_CHECK(task.src >= 0 && task.src < P.store.n_scans && task.tgt >= 0 && task.tgt < P.store.n_scans);
    const float2 *srow = P.store.pts + (size_t)task.src * P.store.pitch;
    const float2 *trow = P.store.pts + (size_t)task.tgt * P.store.pitch;
    const int ns_full = P.store.count[task.src], nt_full = P.store.count[task.tgt];
    const int ns = (ns_full + div - 1) / div, nt = (nt_full + div - 1) / div;
    const int ts = (ns + kTile - 1) / kTile, tt = (nt + kTile - 1) / kTile;   /* tiles           */
    const int gs = ts * GPT, gt = tt * GPT;                                    /* box groups      */
    DPG_CHECK(ns >= 0 && nt >= 0 && ts * kTile <= P.n_cap && tt * kTile <= P.n_cap);

    /* ---- stage both clouds in shared memory ------------------------------------------------- */
    {
      /* contiguous rows: 1-D TMA bulk copies completing on one mbarrier; a resumed pair takes its
       * current source cloud and neighbour seeds from its state slot */
      const bool tma_t = (div == 1), tma_s = (div == 1) || P.resume;
      fence_proxy_async();
      __syncthreads();
      if (tid == 0) {
        const uint32_t bt = tma_t ? (uint32_t)((nt * 8 + 15) & ~15) : 0u;
        const uint32_t bs = tma_s ? (uint32_t)((ns * 8 + 15) & ~15) : 0u;
        const uint32_t bn = P.resume ? (uint32_t)((ns * 4 + 15) & ~15) : 0u;
        mbar_expect_tx(L.mbar, bt + bs + bn);
        if (bt) bulk_g2s(L.tgt, trow, bt, L.mbar);
        if (bs) bulk_g2s(L.src, P.resume ? (const void *)(slot_in + kStateHeader) : (const void *)srow, bs, L.mbar);
        if (bn) bulk_g2s(L.nn, slot_in + kStateHeader + (size_t)P.n_cap * 8, bn, L.mbar);
      }
      if (!tma_t) for (int k = tid; k < nt; k += nthreads) L.tgt[k] = __ldg(trow + (size_t)k * div);
      if (!tma_s) for (int k = tid; k < ns; k += nthreads) L.src[k] = __ldg(srow + (size_t)k * div);
      mbar_wait(L.mbar, mbar_phase);
      mbar_phase ^= 1u;
    }
    __syncthreads();
    /* every warp re-arranges its tiles in place from the staged (x, y) rows to pair-interleaved words (all 32 lanes
     * read their point before any lane writes), pads to whole tiles, applies the guess to the source (PCL
     * transformCloud(input, guess), App. A.2) and forms the boxes.  A resumed source already is pair-interleaved. */
    for (int t = warp; t < tt; t += nw) {
      const int k = t * kTile + lane;
      const float2 p = k < nt ? L.tgt[k] : make_float2(kPad, kPad);
      __syncwarp();
      st_pt<IL>(L.tgt, k, p);
      if constexpr (search_is_projective(SEARCH)) L.tkey[k] = beam_key(p.x, p.y, P.sensor_x, P.sensor_y);
      else store_tile_boxes(p, k < nt, t, L.tbox, nullptr, lane);
    }
    for (int t = warp; t < ts; t += nw) {
      const int k = t * kTile + lane;
      float2 p = make_float2(kPad, kPad);
      if (k < ns) p = P.resume ? ld_pt<IL>(L.src, k) : L.src[k];
      __syncwarp();
      if constexpr (search_is_projective(SEARCH)) {
        /* keys of the UNTRANSFORMED source (a resumed pair holds the current one: take the original from the store) */
        float2 o = p;
        if (P.resume && k < ns) o = __ldg(srow + (size_t)k * div);
        L.skey[k] = beam_key(o.x, o.y, P.sensor_x, P.sensor_y);
      }
      if (!P.resume) {
        if (k < ns) p = xform(task.c, task.s, task.tx, task.ty, p);
        L.nn[k] = (!STOCK && P.corr_seed != nullptr && k < ns) ? P.corr_seed[k] : -1;
      }
      if (!P.resume || k >= ns) st_pt<IL>(L.src, k, p);
      if constexpr (!search_is_projective(SEARCH)) store_tile_boxes(p, k < ns, t, L.sbox, L.stile, lane);
    }
    if (search_is_projective(SEARCH) && tid == 0) {
      /* accumulated transform the source in shared memory has been moved by so far */
      if (P.resume) {
        const SuspHeader h = *reinterpret_cast<const SuspHeader *>(slot_in);
        L.fin[0] = h.fc; L.fin[1] = h.fs; L.fin[2] = h.ftx; L.fin[3] = h.fty;
      } else {
        L.fin[0] = task.c; L.fin[1] = task.s; L.fin[2] = task.tx; L.fin[3] = task.ty;
      }
    }
    __syncthreads();
    if constexpr (search_is_pruned(SEARCH) && !search_is_flat(SEARCH)) {      /* upper level of the box hierarchy, from the complete group boxes */
      build_super_boxes(L.tbox, gt, L.tsup, warp, nw, lane);
      build_super_boxes(L.sbox, gs, L.ssup, warp, nw, lane);
      __syncthreads();
    }

    /* ---- parity hook: a single correspondence pass ------------------------------------------ */
    if (!STOCK && P.corr_out != nullptr) {
      for (int tile = warp; tile < ts; tile += nw) {
        float2 q; int j; float d; bool fwd;
        const bool acc = match_any<SEARCH>(L, P, tile, ns, nt, gs, gt, q, j, d, fwd, stats);
        const int i = tile * kTile + lane;
        if (trim) L.ad2[i] = acc ? d : __int_as_float(0x7f800000);
        if (i < ns) {
          P.corr_out[i] = acc ? j : -1;
          P.corr_d2_out[i] = fwd ? d : __int_as_float(0x7f800000);
          if (P.corr_nn_out != nullptr) P.corr_nn_out[i] = fwd ? j : -1;
        }
      }
      if (trim) {
        __syncthreads();
        const float tau = select_tau(L, ts * kTile, P.outlier_mode, P.outlier_param);
        for (int i = tid; i < ns; i += nthreads)
          if (!(L.ad2[i] <= tau)) P.corr_out[i] = -1;
      }
      continue;
    }

    /* ---- ICP iterations (PCL IterativeClosestPoint::computeTransformation, App. A.3) -------- */
    float fc = task.c, fs = task.s, ftx = task.tx, fty = task.ty;   /* thread 0: final transform  */
    int iterations = 0, last_k = 0;
    uint32_t status = 0;
    double mse = 0.0, mse_prev = 1.7976931348623157e308;
    if (ns <= 0 || nt <= 0) status |= DPGICP_FLAG_EMPTY_INPUT;
    if (P.resume && tid == 0) {
      const SuspHeader h = *reinterpret_cast<const SuspHeader *>(slot_in);
      fc = h.fc; fs = h.fs; ftx = h.ftx; fty = h.fty;
      mse = h.mse; mse_prev = h.mse_prev; iterations = h.iterations; last_k = h.last_k; status = h.status;
    }

    int stop = 0;
    int parity = 0;                       /* the partial-sum slots are double-buffered by pass parity: peers may
                                           * still be reading the previous pass's slots                         */
#ifdef DPGICP_PHASE_TIMING
    long long ph[6] = {0, 0, 0, 0, 0, 0};
#define PH_MARK(k) do { if (tid == 0) { const long long now__ = clock64(); ph[k] += now__ - ph_t; ph_t = now__; } } while (0)
    long long ph_t = clock64();
#else
#define PH_MARK(k) do { } while (0)
#endif
    for (;;) {
      /* phase 1: the searches.  Their result goes to L.nn (neighbour + rejected bit), so that the twenty registers of
       * moment accumulators are not live across the search loops */
      for (int tile = tile0; tile < ts; tile += tile_stride) {
        float2 q; int j; float d; bool fwd;
        const bool acc = match_any<SEARCH>(L, P, tile, ns, nt, gs, gt, q, j, d, fwd, stats);
        const int i = tile * kTile + lane;
        if (i < ns) L.nn[i] = fwd ? (acc ? j : (j | kNnRejected)) : -1;   /* seed (and tie preference) of the next pass */
        if (trim) L.ad2[i] = acc ? d : __int_as_float(0x7f800000);
      }
      /* outlier rejection: threshold from the accepted distances of the whole pair */
      float tau = __int_as_float(0x7f800000);
      if (trim) {
        __syncthreads();
        tau = select_tau(L, ts * kTile, P.outlier_mode, P.outlier_param);
      }
      /* phase 2: the sums over the accepted (and kept) pairs of this warp's tiles */
      long long m[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
      int m_k = 0;
      for (int tile = tile0; tile < ts; tile += tile_stride) {
        const int i = tile * kTile + lane;
        const int v = (i < ns) ? L.nn[i] : -1;
        if (v >= 0 && !(v & kNnRejected)) {
          const float2 q = ld_pt<IL>(L.src, i);
          const float2 t = ld_pt<IL>(L.tgt, v);
          const float d = dist2(q.x, q.y, t.x, t.y);          /* the search's own value: same operands, same roundings */
          if (!trim || d <= tau) accumulate_pair<IL>(L, P, p2l, q, v, d, nt, m, m_k);
        }
      }
      PH_MARK(0);                                     /* own tiles */
      /* exact integer reduction: warp shuffles, then one shared atomic per warp and value */
#pragma unroll
      for (int k = 0; k < 10; ++k) m[k] = warp_sum_i64(m[k]);
      m_k = __reduce_add_sync(0xffffffffu, m_k);
      if (lane == 0) {
        /* per-warp partials in shared memory (plain stores; a 64-bit shared atomicAdd is a CAS spin loop);
         * the slots alias L.dpart, which is only used by the covariance after the pass loop */
        long long *w = reinterpret_cast<long long *>(L.dpart) + (parity * nw + warp) * 12;
#pragma unroll
        for (int k = 0; k < 10; ++k) w[k] = m[k];
        w[10] = (long long)m_k;
      }
      PH_MARK(1);                                     /* warp reduction + partial slots */
      __syncthreads();                                /* all warps of this CTA have stored */
      PH_MARK(2);                                     /* wait for the other warps */

      if constexpr (CSIZE > 1) {
        /* cluster: each CTA first folds its own warps into one set of 11 totals, so that a peer reads
         * 11 values per CTA through distributed shared memory (latency ~200 cycles each), not 11 per warp */
        if (warp == 0 && lane < 11) {
          const long long *w = reinterpret_cast<const long long *>(L.dpart) + parity * nw * 12 + lane;
          long long tot = 0;
          for (int q = 0; q < nw; ++q) tot += w[q * 12];
          L.red[16 + parity * 16 + lane] = tot;
        }
        pair_sync<CSIZE>();                           /* every CTA of the pair has published its totals */
        if (warp == 0) {
          if (lane < 11) {
            long long v[CSIZE];
#pragma unroll
            for (int r = 0; r < CSIZE; ++r) v[r] = peer_smem<CSIZE>(L.red, r)[16 + parity * 16 + lane];
            long long tot = 0;
#pragma unroll
            for (int r = 0; r < CSIZE; ++r) tot += v[r];
            L.red[lane] = tot;
          }
          __syncwarp();
        }
      } else if (warp == 0) {
        /* exact integer totals: lane k adds value k over the warps (any order gives the same bits) */
        if (lane < 11) {
          const long long *w = reinterpret_cast<const long long *>(L.dpart) + parity * nw * 12 + lane;
          long long tot = 0;
          for (int q = 0; q < nw; ++q) tot += w[q * 12];
          L.red[lane] = tot;
        }
        __syncwarp();
      }
      parity ^= 1;
      if (tid == 0) {
        /* has this stage's queue run dry?  (read early, the L2 round trip overlaps the solve) */
        unsigned long long qhead = 0, done = 0;
        if (P.out_count != nullptr) {
          qhead = *reinterpret_cast<volatile unsigned long long *>(P.queue);
          done = *reinterpret_cast<volatile unsigned long long *>(P.finished);
        }
        const int K = (int)L.red[10];
        last_k = K;
        int st = 0;
        float stp[4];
        if (K < 3) {                                   /* App. A.3-4 */
          status |= DPGICP_STOP_NO_CORRESPONDENCES;
          st = 2;
        } else if (p2l && !solve_p2l(L.red, stp)) {
          status |= DPGICP_STOP_DEGENERATE;            /* geometry does not constrain the pose */
          st = 2;
        } else {
          const double invK = __ddiv_rn(1.0, (double)K);
          if (!p2l) solve_p2p(L.red, invK, stp);
          const float sc = stp[0], ss = stp[1], stx = stp[2], sty = stp[3];
          L.step[0] = sc; L.step[1] = ss; L.step[2] = stx; L.step[3] = sty;
          /* final = step * final (App. A.3-6) */
          const float nc = __fadd_rn(__fmul_rn(sc, fc), __fmul_rn(-ss, fs));
          const float nsn = __fadd_rn(__fmul_rn(ss, fc), __fmul_rn(sc, fs));
          const float ntx = __fadd_rn(__fadd_rn(__fmul_rn(sc, ftx), __fmul_rn(-ss, fty)), stx);
          const float nty = __fadd_rn(__fadd_rn(__fmul_rn(ss, ftx), __fmul_rn(sc, fty)), sty);
          fc = nc; fs = nsn; ftx = ntx; fty = nty;
          if constexpr (search_is_projective(SEARCH)) { L.fin[0] = fc; L.fin[1] = fs; L.fin[2] = ftx; L.fin[3] = fty; }
          ++iterations;
          mse = __dmul_rn(__dmul_rn((double)L.red[9], 1.0 / kScaleD2), invK);
          /* DefaultConvergenceCriteria (App. A.5), in PCL's order */
          const float tr = __fsub_rn(__fadd_rn(__fadd_rn(sc, sc), 1.0f), 1.0f);
          const double cos_angle = __dmul_rn(0.5, (double)tr);
          const float tsq = __fadd_rn(__fmul_rn(stx, stx), __fmul_rn(sty, sty));
          if (iterations >= P.max_iterations) {
            status |= DPGICP_STOP_ITERATIONS | DPGICP_FLAG_CONVERGED; st = 1;
          } else if (cos_angle >= P.rot_thr && (double)tsq <= P.eps) {
            status |= DPGICP_STOP_TRANSFORM | DPGICP_FLAG_CONVERGED; st = 1;
          } else if (fabs(__dsub_rn(mse, mse_prev)) < 1e-12) {
            status |= DPGICP_STOP_ABS_MSE | DPGICP_FLAG_CONVERGED; st = 1;
          } else {
            mse_prev = mse;
            if (P.out_count != nullptr && qhead >= n_items && (long long)(n_items - done) <= P.handover) {
              /* queue dry and few enough pairs left: hand this pair to the next (wider) stage */
              st = 3;
              L.ctl[4] = (int32_t)atomicAdd(P.out_count, 1u);
            }
          }
        }
        L.ctl[2] = st;
        L.ctl[3] = K;
      }
      PH_MARK(3);                                     /* solve + convergence */
      __syncthreads();
      stop = L.ctl[2];
#ifdef DPGICP_CHECK
      if constexpr (CSIZE > 1) {                      /* every CTA of the cluster took the same decision from the same totals */
        pair_sync<CSIZE>();
        if (tid == 0)
          for (int r = 0; r < CSIZE; ++r) {
            const int32_t *c = peer_smem<CSIZE>(L.ctl, r);
            DPG_CHECK(c[2] == L.ctl[2] && c[3] == L.ctl[3]);
          }
        pair_sync<CSIZE>();
      }
#endif
      c_corr += (tid == 0 && crank == 0) ? (unsigned long long)L.ctl[3] : 0ull;
      if (stop == 2) break;
      /* src' = step * src' in place (App. A.3-6) and refresh the source boxes */
      {
        const float sc = L.step[0], ss = L.step[1], stx = L.step[2], sty = L.step[3];
        for (int t = warp; t < ts; t += nw) {
          const int k = t * kTile + lane;
          float2 p = ld_pt<IL>(L.src, k);
          if (k < ns) { p = xform(sc, ss, stx, sty, p); st_pt<IL>(L.src, k, p); }
          if constexpr (!search_is_projective(SEARCH)) store_tile_boxes(p, k < ns, t, L.sbox, L.stile, lane);
        }
      }
      if (tid == 0 && crank == 0) ++c_iters;
      PH_MARK(4);                                     /* transform + boxes (own tiles) */
      __syncthreads();
      PH_MARK(5);                                     /* wait */
      if (stop) break;
      if constexpr (search_is_pruned(SEARCH) && !search_is_flat(SEARCH)) {
        build_super_boxes(L.sbox, gs, L.ssup, warp, nw, lane);
        __syncthreads();
      }
    }
#ifdef DPGICP_PHASE_TIMING
    if (tid == 0)
      for (int k = 0; k < 6; ++k) atomicAdd(P.counters + 8 + k, (unsigned long long)ph[k]);   /* d_queue[16..21] */
#endif

    if (stop == 3) {
      /* ---- suspend: current source cloud + seeds + scalars -> state slot, pair -> next queue --- */
      DPG_CHECK(L.ctl[4] >= 0 && (long long)L.ctl[4] < P.slot_cap);
      unsigned char *slot = P.state_out + (size_t)(uint32_t)L.ctl[4] * (size_t)P.slot_bytes;
      float2 *s_src = reinterpret_cast<float2 *>(slot + kStateHeader);
      int32_t *s_nn = reinterpret_cast<int32_t *>(slot + kStateHeader + (size_t)P.n_cap * 8);
      /* the cloud goes out as it lies in shared memory (pair-interleaved words): whole pairs, so ns rounded up to even */
      for (int k = tid; k < ((ns + 1) & ~1); k += nthreads) s_src[k] = L.src[k];
      for (int k = tid; k < ns; k += nthreads) s_nn[k] = L.nn[k];
      if (tid == 0) {
        SuspHeader h;
        h.fc = fc; h.fs = fs; h.ftx = ftx; h.fty = fty; h.mse = mse; h.mse_prev = mse_prev;
        h.iterations = iterations; h.last_k = last_k; h.status = status; h.pad = 0;
        *reinterpret_cast<SuspHeader *>(slot) = h;
        P.susp_out[(uint32_t)L.ctl[4]] = pair;
      }
      continue;            /* the queue is dry: the next fetch ends this CTA */
    }

    /* ---- covariance (calculate_ICP_COV) + result record --------------------------------------
     * The 11 binary64 sums are formed in an order that does not depend on WARPS (a pair may finish in
     * any stage): per 32-element tile by a fixed xor-shuffle tree, tiles added in ascending order by
     * thread 0, 16 tile partials at a time through L.dpart. */
    double S[11];
#pragma unroll
    for (int k = 0; k < 11; ++k) S[k] = 0.0;
    uint32_t cov_flag = 0;
    const int cov_mode = P.cov_mode;
    if constexpr (CSIZE > 1) pair_sync<CSIZE>();     /* peers have finished reading this CTA's partial-sum slots */
    if (cov_mode != DPGICP_COV_REFERENCE_LIVE) {
      /* pose as cov.h:26-35: x,y float entries widened, a = (double)atan2f(T10, T00); all threads */
      if (tid == 0) { L.step[0] = fc; L.step[1] = fs; L.step[2] = ftx; L.step[3] = fty; }
      __syncthreads();
      const float Tc = L.step[0], Ts = L.step[1], Ttx = L.step[2], Tty = L.step[3];
      const double x = (double)Ttx, y = (double)Tty;
      const double a = (double)atan2f(Ts, Tc);
      const double ca = cos(a), sa = sin(a);
      int n_cov = 0, nd = 0;
      if (cov_mode == DPGICP_COV_CENSI_INDEXPAIR) {
        /* full clouds paired by index (dpg_slam.cc:430), Hessian over all, D-term over the cap */
        n_cov = ns_full < nt_full ? ns_full : nt_full;
        nd = (P.cov_cap > 0 && n_cov > P.cov_cap) ? P.cov_cap : n_cov;
      } else {
        /* CENSI_CORR: correspondences at the final pose: src'' = final * src (original points) */
        __syncthreads();
        for (int t = warp; t < ts; t += nw) {
          const int k = t * kTile + lane;
          float2 p = make_float2(kPad, kPad);
          if (k < ns) { p = xform(Tc, Ts, Ttx, Tty, __ldg(srow + (size_t)k * div)); }
          st_pt<IL>(L.src, k, p);
          if constexpr (!search_is_projective(SEARCH)) store_tile_boxes(p, k < ns, t, L.sbox, L.stile, lane);
        }
        __syncthreads();
        if constexpr (search_is_pruned(SEARCH) && !search_is_flat(SEARCH)) {
          build_super_boxes(L.sbox, gs, L.ssup, warp, nw, lane);
          __syncthreads();
        }
        for (int tile = tile0; tile < ts; tile += tile_stride) {
          float2 q; int j; float d; bool fwd;
          const bool ok = match_any<SEARCH>(L, P, tile, ns, nt, gs, gt, q, j, d, fwd, stats);
          const unsigned bal = __ballot_sync(0xffffffffu, ok);
          const int i = tile * kTile + lane;
          if (i < ns) L.nn[i] = ok ? j : -1;
          if (trim) L.ad2[i] = ok ? d : __int_as_float(0x7f800000);
          if (lane == 0) L.tcnt[tile] = __popc(bal);
        }
        if (trim) {
          /* the same rejector as in the iterations, on the correspondences at the final pose */
          __syncthreads();
          const float tau = select_tau(L, ts * kTile, P.outlier_mode, P.outlier_param);
          for (int tile = tile0; tile < ts; tile += tile_stride) {
            const int i = tile * kTile + lane;
            const bool keep = L.ad2[i] <= tau && L.ad2[i] < __int_as_float(0x7f800000);
            const unsigned bal = __ballot_sync(0xffffffffu, keep);
            if (i < ns && !keep) L.nn[i] = -1;
            if (lane == 0) L.tcnt[tile] = __popc(bal);
          }
        }
        pair_sync<CSIZE>();
        n_cov = ns;
      }
      const int cov_tiles = (n_cov + kTile - 1) / kTile;
      for (int chunk = 0; chunk < cov_tiles; chunk += kCovChunk) {
        const int chunk_end = chunk + kCovChunk < cov_tiles ? chunk + kCovChunk : cov_tiles;
        /* tile t belongs to CTA (t / nw) % CSIZE, warp t % nw — the same split as the search tiles */
        int tile_first = tile0;
        if (tile_first < chunk) tile_first += ((chunk - tile_first + tile_stride - 1) / tile_stride) * tile_stride;
        for (int tile = tile_first; tile < chunk_end; tile += tile_stride) {
          double acc[11];
#pragma unroll
          for (int k = 0; k < 11; ++k) acc[k] = 0.0;
          const int i = tile * kTile + lane;
          if (cov_mode == DPGICP_COV_CENSI_INDEXPAIR) {
            if (i < n_cov) {
              const float2 p = __ldg(srow + i), q = __ldg(trow + i);
              cov_terms(p.x, p.y, q.x, q.y, ca, sa, x, y, true, i < nd, acc);
            }
          } else {
            int prefix = 0;
            for (int t = lane; t < tile; t += 32) prefix += peer_smem<CSIZE>(L.tcnt, (t / nw) % CSIZE)[t];
            prefix = __reduce_add_sync(0xffffffffu, prefix);
            const int j = (i < ns) ? L.nn[i] : -1;
            const unsigned bal = __ballot_sync(0xffffffffu, j >= 0);
            const int rank = prefix + __popc(bal & ((1u << lane) - 1u));
            if (j >= 0) {
              const float2 p = __ldg(srow + (size_t)i * div);
              const float2 q = ld_pt<IL>(L.tgt, j);
              const bool in_d = (P.cov_cap <= 0) || (rank < P.cov_cap);
              cov_terms(p.x, p.y, q.x, q.y, ca, sa, x, y, true, in_d, acc);
            }
          }
#pragma unroll
          for (int k = 0; k < 11; ++k) acc[k] = warp_sum_f64(acc[k]);
          if (lane == 0)
            for (int k = 0; k < 11; ++k) L.dpart[(tile - chunk) * 12 + k] = acc[k];
        }
        pair_sync<CSIZE>();
        if (tid == 0 && crank == 0)
          for (int t = 0; t < chunk_end - chunk; ++t) {
            const double *dp = peer_smem<CSIZE>(L.dpart, ((chunk + t) / nw) % CSIZE) + t * 12;
            for (int k = 0; k < 11; ++k) S[k] = __dadd_rn(S[k], dp[k]);
          }
        pair_sync<CSIZE>();
      }
    }

    if (tid == 0 && crank == 0) {
      static_assert(sizeof(dpgicp_result) % 16 == 0, "the fused gather copies records in 16-byte words");
      alignas(16) dpgicp_result r;
      r.tx = ftx; r.ty = fty;
      r.theta = atan2f(fs, fc);                      /* Rotation2Df::fromRotationMatrix().angle() */
      r.rot_c = fc; r.rot_s = fs;
      r.iterations = iterations;
      r.n_correspondences = last_k;
      r.mse = mse;
#pragma unroll
      for (int k = 0; k < 9; ++k) r.cov[k] = 0.0;
      if (cov_mode == DPGICP_COV_REFERENCE_LIVE) {   /* cov.h:572-575 */
        r.cov[0] = P.live[0]; r.cov[4] = P.live[1]; r.cov[8] = P.live[2];
      } else {
        cov_flag = finish_cov(S, P.sensor_var, P.live, r.cov);
      }
      r.status = status | cov_flag;
      P.results[pair] = r;
      if (P.out_count != nullptr) atomicAdd(P.finished, 1ull);
      if (P.gather_world > 1) {
        /* fused gather: seven 16-byte stores per peer, straight into every rank's buffer at the global slot */
        const long long slot = (long long)P.gather_rank + (P.pair_base + pair) * (long long)P.gather_world;
        DPG_CHECK(slot >= 0 && slot < P.gather_slots);
        const int4 *src = reinterpret_cast<const int4 *>(&r);
        for (int g = 0; g < P.gather_fanout; ++g) {
          int4 *dst = reinterpret_cast<int4 *>(P.gather_peer[g] + slot);
#pragma unroll
          for (int q = 0; q < (int)(sizeof(dpgicp_result) / 16); ++q) dst[q] = src[q];
        }
      }
    }
  }

  if constexpr (CSIZE > 1) pair_sync<CSIZE>();       /* no CTA leaves while a peer may still address its shared memory */

  /* executed-work counters (one set of atomics per CTA) */
  if (lane == 0) {
    atomicAdd(P.counters + 2, (unsigned long long)stats.scans * (kGroup * 32ull));
  }
  if constexpr (search_is_projective(SEARCH)) {
    const unsigned we = __reduce_add_sync(0xffffffffu, stats.window_evals);   /* per-lane counts, may wrap past 2^32 per warp: an executed-work statistic only */
    if (lane == 0) atomicAdd(P.counters + 2, (unsigned long long)we);
  }
  if (lane == 0) {
    atomicAdd(P.counters + 3, (unsigned long long)stats.tests * 32ull);
#ifdef DPGICP_STATS
    atomicAdd(P.counters + 5, (unsigned long long)stats.cands);
    atomicAdd(P.counters + 6, (unsigned long long)stats.loose);
    atomicAdd(P.counters + 7, (unsigned long long)stats.searches);
#endif
  }
  if (tid == 0) {
    atomicAdd(P.counters + 0, c_iters);
    atomicAdd(P.counters + 1, c_corr);
  }
}

/* ------------------------------------------------------------------------------------------------
 * Standalone covariance kernel (calculate_ICP_COV call shape): one CTA per item, clouds paired by
 * index.  HBM-bound: 16 bytes read per index pair.
 * ---------------------------------------------------------------------------------------------- */
struct CovItem {
  const float2 *p, *q;      /* data_pi, model_qi (packed float2) */
  int32_t n_p, n_q;
  float c, s, tx, ty;       /* T(0,0), T(1,0), T(0,3), T(1,3)    */
};

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) cov_indexpair_kernel(const CovItem *items, int n_items, int cov_mode,
                                                                  int cov_cap, double sensor_var, float lx,
                                                                  float ly, float lt, double *cov_out,
                                                                  uint32_t *status_out) {
  __shared__ double dpart[kMaxWarps * 12];
  const int item = blockIdx.x;
  if (item >= n_items) return;
  const CovItem it = items[item];
  const float live[3] = {lx, ly, lt};
  double S[11];
  double acc[11];
#pragma unroll
  for (int k = 0; k < 11; ++k) acc[k] = 0.0;
  if (cov_mode != DPGICP_COV_REFERENCE_LIVE) {
    /* pose as cov.h:26-35; the trigonometry once per CTA, broadcast through shared memory */
    if (threadIdx.x == 0) {
      const double a = (double)atan2f(it.s, it.c);
      dpart[0] = cos(a); dpart[1] = sin(a);
    }
    __syncthreads();
    const double x = (double)it.tx, y = (double)it.ty;
    const double ca = dpart[0], sa = dpart[1];
    __syncthreads();                                   /* dpart is reused by the reduction below */
    const int nh = it.n_p < it.n_q ? it.n_p : it.n_q;
    const int nd = (cov_cap > 0 && nh > cov_cap) ? cov_cap : nh;
    /* two index pairs per 16-byte load (rows are 16-byte aligned): 32 bytes in flight per thread and trip */
    const float4 *p4 = reinterpret_cast<const float4 *>(it.p), *q4 = reinterpret_cast<const float4 *>(it.q);
    for (int k2 = threadIdx.x; 2 * k2 < nh; k2 += WARPS * 32) {
      const float4 p = __ldg(p4 + k2), q = __ldg(q4 + k2);
      const int k = 2 * k2;
      cov_terms(p.x, p.y, q.x, q.y, ca, sa, x, y, true, k < nd, acc);
      if (k + 1 < nh) cov_terms(p.z, p.w, q.z, q.w, ca, sa, x, y, true, k + 1 < nd, acc);
    }
  }
  block_sum11<WARPS>(acc, dpart, S);
  if (threadIdx.x == 0) {
    double cov[9];
    uint32_t flag = 0;
    if (cov_mode == DPGICP_COV_REFERENCE_LIVE) {
      for (int k = 0; k < 9; ++k) cov[k] = 0.0;
      cov[0] = lx; cov[4] = ly; cov[8] = lt;
    } else {
      flag = finish_cov(S, sensor_var, live, cov);
    }
    for (int k = 0; k < 9; ++k) cov_out[(size_t)item * 9 + k] = cov[k];
    status_out[item] = flag;
  }
}

/* ------------------------------------------------------------------------------------------------
 * Scan-store builders
 * ---------------------------------------------------------------------------------------------- */
/* CSR points (arbitrary stride) -> padded rows; flags non-finite / out-of-range coordinates */
__global__ void pack_rows_kernel(const unsigned char *__restrict__ pts, size_t stride, const long long *offsets,
                                 int n_scans, int pitch, float2 *rows, int32_t *count, int *bad) {
  const int scan = blockIdx.x;
  if (scan >= n_scans) return;
  const long long o0 = offsets[scan], o1 = offsets[scan + 1];
  const int n = (int)(o1 - o0);
  if (threadIdx.x == 0) count[scan] = n;
  for (int k = threadIdx.x; k < pitch; k += blockDim.x) {
    float2 v = make_float2(0.f, 0.f);
    if (k < n) {
      const float *f = reinterpret_cast<const float *>(pts + (size_t)(o0 + k) * stride);
      v = make_float2(f[0], f[1]);
      if (!(fabsf(v.x) <= DPGICP_MAX_ABS_COORD) || !(fabsf(v.y) <= DPGICP_MAX_ABS_COORD)) atomicExch(bad, 1);
    }
    rows[(size_t)scan * pitch + k] = v;
  }
}

/* raw ranges -> base_link points, MAX_RANGE dropped, beam order kept (createNode
 * dpg_slam.cc:497-506, dpg_measurement.h:41-46,102-104, dpg_node.cc:13-22).  One warp per scan,
 * ballot-prefix compaction.  The beam directions are the same for every scan, so cos/sin of
 * angle_i = angle_inc * i + angle_min come from a table the host computed once with its own libm in
 * binary64 — bit for bit what the oracle (and the reference's double overloads) use, and the kernel
 * is left with a multiply per coordinate: HBM-bound, 4 B in + 8 B out per beam. */
__global__ void ranges_to_rows_kernel(const float *__restrict__ ranges, const int32_t *__restrict__ scan_ids, int n_scans,
                                      int n_beams, const double2 *__restrict__ trig, float range_max, float lx, float ly,
                                      float lc, float ls, int pitch, float2 *rows, int32_t *count, int *bad) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_scans) return;
  /* store row `warp` is scan scan_ids[warp] of the input (identity when null); `ranges` may be pinned host
   * memory, read directly over PCIe in coalesced 128-byte requests */
  const float *r = ranges + (size_t)(scan_ids ? scan_ids[warp] : warp) * n_beams;
  float2 *row = rows + (size_t)warp * pitch;
  int n = 0;
  for (int base = 0; base < n_beams; base += 128) {
    /* four coalesced loads (and their table entries) in flight before the first dependent compaction step */
    float rg[4];
    double2 cs[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = base + 32 * u + lane;
      rg[u] = range_max;
      cs[u] = make_double2(0.0, 0.0);
      if (i < n_beams) { rg[u] = __ldg(r + i); cs[u] = __ldg(trig + i); }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const bool keep = !(rg[u] >= range_max);          /* out-of-range lanes hold range_max */
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (keep) {
        const float px = (float)__dmul_rn((double)rg[u], cs[u].x);
        const float py = (float)__dmul_rn((double)rg[u], cs[u].y);
        const float rx = __fadd_rn(__fmul_rn(lc, px), __fmul_rn(-ls, py));
        const float ry = __fadd_rn(__fmul_rn(ls, px), __fmul_rn(lc, py));
        const float2 v = make_float2(__fadd_rn(lx, rx), __fadd_rn(ly, ry));
        if (!(fabsf(v.x) <= DPGICP_MAX_ABS_COORD) || !(fabsf(v.y) <= DPGICP_MAX_ABS_COORD)) atomicExch(bad, 1);
        row[n + __popc(bal & ((1u << lane) - 1u))] = v;
      }
      n += __popc(bal);
    }
  }
  for (int k = n + lane; k < pitch; k += 32) row[k] = make_float2(0.f, 0.f);
  if (lane == 0) count[warp] = n;
}

/* rows of pitch `old_pitch` -> rows of the larger pitch `new_pitch` (both even, so every row starts on a 16-byte
 * boundary and is a whole number of float4 = two points).  One warp per row, 16-byte loads and stores; the old
 * row's padding is already zero, the new tail is zero-filled: every row keeps its contents and stays zero-padded. */
__global__ void repitch_rows_kernel(const float4 *__restrict__ src, int n_rows, int old_pitch, int new_pitch,
                                    float4 *__restrict__ dst) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_rows) return;
  const int old_q = old_pitch >> 1, new_q = new_pitch >> 1;
  const float4 *in = src + (size_t)warp * old_q;
  float4 *out = dst + (size_t)warp * new_q;
  for (int k = lane; k < new_q; k += 32) out[k] = k < old_q ? __ldg(in + k) : make_float4(0.f, 0.f, 0.f, 0.f);
}

/* ------------------------------------------------------------------------------------------------
 * Candidate-pair enumeration on the device (the callers of runIcp: reoptimize dpg_slam.cc:79-107 and
 * updatePoseGraphObsConstraints dpg_slam.cc:255-300), output left in device memory as the pair batch.
 *
 * Pose-graph nodes are created along the trajectory (1 m / 30 deg apart, parameters.h:242,254), so consecutive node
 * indices are spatially compact — the same property the ICP kernel uses for beam-ordered points.  A hierarchy of
 * bounding boxes over INDEX ranges (32 nodes per leaf box, 32 boxes per parent, ...) is therefore tight, and
 * traversing it in index order visits the candidates j of a node i in ascending j: the reference's loop order falls
 * out without any sort.  One warp per node i walks the hierarchy top-down (32 children tested per step, one per
 * lane, a ballot per step); the leaf step applies the reference's float gate to 32 nodes at once.  Box lower bounds
 * use the gate's own rounding sequence, so by monotonicity of rounding the pruning is exact.  A count pass, a device
 * exclusive scan and a fill pass keep the global order: pair position = start[i] + rank of j among node i's hits.
 * The fill pass also derives every pair's guess from the node estimates (dpg_slam.cc:364-378).
 * Worst case (node indices in no spatial order) degrades to all-pairs tests; pose-graph nodes are never like that.
 * ---------------------------------------------------------------------------------------------- */
struct NodeBox {               /* 32 bytes: bounding box + pass range of an index range of nodes */
  float lox, loy, hix, hiy;
  int32_t pass_lo, pass_hi, pad0, pad1;
};
constexpr int kEnumFan = 32;   /* children per box = lanes of the warp testing them */
constexpr int kEnumMaxLevels = 7;

/* a pair listed for the host: its slot in the shard's list and its guess angle; the host replaces (a, b) = (g2, 0)
 * with its libm's (cos g2, sin g2) and amb_scatter_kernel writes them into the pair */
struct AmbPair {
  long long slot;
  float a, b;
};

struct EnumParams {
  const float2 *xy;            /* node positions                                          */
  const int32_t *pass;         /* node pass numbers                                       */
  const float4 *aux;           /* (theta, cosf(-theta), sinf(-theta), 0) per node          */
  const NodeBox *boxes;        /* level L (1-based) starts at level_off[L - 1]            */
  long long level_off[kEnumMaxLevels];
  int32_t level_cnt[kEnumMaxLevels];
  int32_t levels;
  int32_t n;
  float r_same, r_other;
  unsigned long long *cnt;     /* count pass: pairs per node out; fill pass: start offsets in */
  PairTask *tasks;             /* fill pass: this shard's pair list                         */
  int32_t rank, world;
  long long n_local;           /* capacity of tasks: this shard's pair count                 */
  unsigned long long *amb_count; /* pairs whose cos/sin sit too close to a binary32 rounding boundary for two */
  AmbPair *amb_list;           /* libm implementations to be guaranteed to agree: the host re-derives these */
  long long amb_cap;           /* entries of amb_list; the count goes on past it (the host then grows the list) */
};

/* the reference's gate: float distance between two node estimates against the same-pass / other-pass radius */
__device__ __forceinline__ bool node_gate(float2 a, int pa, float2 b, int pb, float r_same, float r_other) {
  const float dx = __fsub_rn(a.x, b.x), dy = __fsub_rn(a.y, b.y);
  const float dist = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
  return dist <= ((pa == pb) ? r_same : r_other);
}

/* can any node inside `bx` pass the gate against query (q, pq)?  Lower bound of the gate's distance, same roundings */
__device__ __forceinline__ bool box_may_pass(const NodeBox bx, float2 q, int pq, float r_same, float r_other) {
  const float ex = fmaxf(fmaxf(__fsub_rn(bx.lox, q.x), __fsub_rn(q.x, bx.hix)), 0.0f);
  const float ey = fmaxf(fmaxf(__fsub_rn(bx.loy, q.y), __fsub_rn(q.y, bx.hiy)), 0.0f);
  const float lb = __fsqrt_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)));
  float r;
  if (pq < bx.pass_lo || pq > bx.pass_hi) r = r_other;            /* no node of the query's pass inside */
  else if (bx.pass_lo == bx.pass_hi) r = r_same;                  /* only nodes of the query's pass     */
  else r = fmaxf(r_same, r_other);
  return lb <= r;                                                 /* empty boxes have lb = +inf / NaN   */
}

/* leaf boxes: one warp per box of kEnumFan consecutive nodes */
__global__ void node_boxes_leaf_kernel(const float2 *__restrict__ xy, const int32_t *__restrict__ pass, int n,
                                       NodeBox *__restrict__ out, int n_boxes) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= n_boxes) return;
  const int k = b * kEnumFan + lane;
  const float inf = __int_as_float(0x7f800000);
  float lox = inf, loy = inf, hix = -inf, hiy = -inf;
  int plo = 0x7fffffff, phi = -0x7fffffff - 1;
  if (k < n) { const float2 p = xy[k]; lox = hix = p.x; loy = hiy = p.y; plo = phi = pass[k]; }
  lox = warp_min(lox); loy = warp_min(loy); hix = warp_max(hix); hiy = warp_max(hiy);
  plo = __reduce_min_sync(0xffffffffu, plo); phi = __reduce_max_sync(0xffffffffu, phi);
  if (lane == 0) { NodeBox o = {lox, loy, hix, hiy, plo, phi, 0, 0}; out[b] = o; }
}

/* parent boxes: one warp per box of kEnumFan consecutive child boxes */
__global__ void node_boxes_up_kernel(const NodeBox *__restrict__ in, int n_in, NodeBox *__restrict__ out, int n_out) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= n_out) return;
  const int k = b * kEnumFan + lane;
  const float inf = __int_as_float(0x7f800000);
  float lox = inf, loy = inf, hix = -inf, hiy = -inf;
  int plo = 0x7fffffff, phi = -0x7fffffff - 1;
  if (k < n_in) { const NodeBox c = in[k]; lox = c.lox; loy = c.loy; hix = c.hix; hiy = c.hiy; plo = c.pass_lo; phi = c.pass_hi; }
  lox = warp_min(lox); loy = warp_min(loy); hix = warp_max(hix); hiy = warp_max(hiy);
  plo = __reduce_min_sync(0xffffffffu, plo); phi = __reduce_max_sync(0xffffffffu, phi);
  if (lane == 0) { NodeBox o = {lox, loy, hix, hiy, plo, phi, 0, 0}; out[b] = o; }
}

/* is the double v so close to the midpoint of two adjacent binary32 values that a libm with a different (sub-ulp)
 * error could round it the other way?  (29 mantissa bits are dropped: the midpoint pattern is 1 followed by zeros) */
__device__ __forceinline__ bool near_f32_rounding_boundary(double v) {
  const unsigned low = (unsigned)(__double_as_longlong(v) & 0x1fffffffll);
  const int d = (int)low - 0x10000000;
  return (d < 0 ? -d : d) <= 32;
}

/* the pair task of (source node src, target node tgt): indices + the guess of runIcp (dpg_slam.cc:364-378) in the
 * arithmetic of dpgicp_relative_guess (math_utils.cc:20-34, math_utils.h:13-16) and of the Matrix4f initialiser */
__device__ __forceinline__ PairTask make_pair_task(const EnumParams &E, int src, int tgt, long long slot) {
  const float2 p1 = E.xy[tgt], p2 = E.xy[src];
  const float4 a1 = E.aux[tgt];
  const float th2 = E.aux[src].x;
  const float tx = __fsub_rn(p2.x, p1.x), ty = __fsub_rn(p2.y, p1.y);
  const float c = a1.y, sn = a1.z;                                   /* Rotation2Df(-theta_1), host libm */
  PairTask t;
  t.src = src; t.tgt = tgt;
  t.tx = __fadd_rn(__fmul_rn(c, tx), __fmul_rn(-sn, ty));
  t.ty = __fadd_rn(__fmul_rn(sn, tx), __fmul_rn(c, ty));
  double d = (double)__fsub_rn(th2, a1.x);                           /* AngleMod, evaluated in binary64 */
  d = __dsub_rn(d, __dmul_rn(6.283185307179586, rint(__ddiv_rn(d, 6.283185307179586))));
  const double g2 = (double)(float)d;
  double sd, cd;
  sincos(g2, &sd, &cd);
  t.c = (float)cd; t.s = (float)sd;
  if (near_f32_rounding_boundary(cd) || near_f32_rounding_boundary(sd)) {
    const unsigned long long k = atomicAdd(E.amb_count, 1ull);
    if (k < (unsigned long long)E.amb_cap) { AmbPair p; p.slot = slot; p.a = (float)g2; p.b = 0.f; E.amb_list[k] = p; }
  }
  return t;
}

/* the host's cos / sin of the listed pairs' guess angles into their pair tasks */
__global__ void amb_scatter_kernel(const AmbPair *__restrict__ list, long long n, PairTask *__restrict__ tasks) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const AmbPair p = list[k];
  tasks[p.slot].c = p.a;
  tasks[p.slot].s = p.b;
}

/* DPGICP_ENUM_REOPTIMIZE: one warp per node i.  FILL = false counts node i's pairs into cnt[i]; FILL = true writes
 * them (E.cnt then holds the exclusive scan of the counts). */
template <bool FILL>
__global__ void __launch_bounds__(128) enumerate_reopt_kernel(const EnumParams E) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= E.n) return;
  unsigned long long count = 0, pos = 0;
  if (FILL) pos = E.cnt[i];
  auto emit = [&](unsigned long long at, int src, int tgt) {
    if ((long long)(at % (unsigned long long)E.world) == (long long)E.rank) {
      const long long slot = (long long)(at / (unsigned long long)E.world);
      DPG_CHECK(slot >= 0 && slot < E.n_local && src >= 0 && src < E.n && tgt >= 0 && tgt < E.n);
      E.tasks[slot] = make_pair_task(E, src, tgt, slot);
    }
  };
  if (i >= 1) {                                   /* the successive pair comes first (dpg_slam.cc:83-89) */
    if (FILL && lane == 0) emit(pos, i, i - 1);
    ++pos; ++count;
  }
  const int jmax = i - 1;                          /* gated candidates: j < i - 1 (dpg_slam.cc:91) */
  if (jmax > 0) {
    const float2 q = E.xy[i];
    const int pq = E.pass[i];
    unsigned mask[kEnumMaxLevels + 1];
    int base[kEnumMaxLevels + 1];
    const int top = E.levels;
    /* span[L] = nodes covered by one box of level L */
    auto test_boxes = [&](int L, int first) -> unsigned {
      const int c = first + lane;
      long long span = kEnumFan;
      for (int k = 1; k < L; ++k) span *= kEnumFan;
      bool ok = c < E.level_cnt[L - 1] && (long long)c * span < (long long)jmax;
      if (ok) ok = box_may_pass(E.boxes[E.level_off[L - 1] + c], q, pq, E.r_same, E.r_other);
      return __ballot_sync(0xffffffffu, ok);
    };
    int level = top;
    base[top] = 0;
    mask[top] = test_boxes(top, 0);
    for (;;) {
      while (level <= top && mask[level] == 0u) ++level;
      if (level > top) break;
      const int b = __ffs(mask[level]) - 1;
      mask[level] &= mask[level] - 1u;
      const int idx = base[level] + b;
      if (level == 1) {
        const int j = idx * kEnumFan + lane;
        bool ok = j < jmax;
        if (ok) ok = node_gate(E.xy[j], E.pass[j], q, pq, E.r_same, E.r_other);
        const unsigned bal = __ballot_sync(0xffffffffu, ok);
        if (FILL && ok) emit(pos + (unsigned long long)__popc(bal & ((1u << lane) - 1u)), i, j);
        pos += (unsigned long long)__popc(bal);
        count += (unsigned long long)__popc(bal);
      } else {
        --level;
        base[level] = idx * kEnumFan;
        mask[level] = test_boxes(level, base[level]);
      }
    }
  }
  if (!FILL && lane == 0) E.cnt[i] = count;
}

/* DPGICP_ENUM_ONLINE: the newest node is n-1, the preceding node pre = n-2; candidates i < n-3 are gated against the
 * PRECEDING node and attach to it.  One warp per chunk of 32 candidates; cnt[chunk] as above.  Pair 0 is the
 * successive pair (src n-1, tgt n-2), counted with chunk 0. */
template <bool FILL>
__global__ void __launch_bounds__(128) enumerate_online_kernel(const EnumParams E, int n_chunks) {
  const int chunk = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (chunk >= n_chunks) return;
  const int pre = E.n - 2, jmax = E.n - 3;
  unsigned long long pos = 0;
  if (FILL) pos = E.cnt[chunk];
  auto emit = [&](unsigned long long at, int src, int tgt) {
    if ((long long)(at % (unsigned long long)E.world) == (long long)E.rank) {
      const long long slot = (long long)(at / (unsigned long long)E.world);
      DPG_CHECK(slot >= 0 && slot < E.n_local && src >= 0 && src < E.n && tgt >= 0 && tgt < E.n);
      E.tasks[slot] = make_pair_task(E, src, tgt, slot);
    }
  };
  unsigned long long count = 0;
  if (chunk == 0) {
    if (FILL && lane == 0) emit(pos, E.n - 1, pre);
    ++pos; ++count;
  }
  const int j = chunk * 32 + lane;
  bool ok = j < jmax;
  if (ok) ok = node_gate(E.xy[j], E.pass[j], E.xy[pre], E.pass[pre], E.r_same, E.r_other);
  const unsigned bal = __ballot_sync(0xffffffffu, ok);
  if (FILL && ok) emit(pos + (unsigned long long)__popc(bal & ((1u << lane) - 1u)), pre, j);
  count += (unsigned long long)__popc(bal);
  if (!FILL && lane == 0) E.cnt[chunk] = count;
}

/* exclusive scan of n 64-bit counts in place, v[n] = total: one CTA (the arrays are a few MB at most and sit in L2) */
__global__ void __launch_bounds__(1024) scan_u64_kernel(unsigned long long *v, int n) {
  __shared__ unsigned long long wsum[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (n + 1023) / 1024;
  const int lo = tid * per < n ? tid * per : n, hi = lo + per < n ? lo + per : n;
  unsigned long long sum = 0;
  for (int k = lo; k < hi; ++k) sum += v[k];
  unsigned long long incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    unsigned long long w = wsum[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    wsum[lane] = wi - w;                       /* exclusive prefix of the warp totals */
    if (lane == 31) v[n] = wi;                 /* grand total */
  }
  __syncthreads();
  unsigned long long run = wsum[warp] + (incl - sum);
  for (int k = lo; k < hi; ++k) { const unsigned long long t = v[k]; v[k] = run; run += t; }
}

/* unpack a pair list for the host: indices and the guess entries */
__global__ void unpack_tasks_kernel(const PairTask *__restrict__ tasks, long long n, int32_t *src, int32_t *tgt, float4 *T) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const PairTask t = tasks[k];
  if (src) src[k] = t.src;
  if (tgt) tgt[k] = t.tgt;
  if (T) T[k] = make_float4(t.c, t.s, t.tx, t.ty);
}

/* ------------------------------------------------------------------------------------------------
 * Records -> pose-graph factors (addObservationConstraint, dpg_slam.cc:331-338): information = cov^-1
 * by cofactors, R = its upper Cholesky factor.  One thread per pair; HBM-bound (136 B in, 96 B out).
 * Individually rounded binary64 operations, mirrored by oracle/dpg_oracle.c orc_factor.
 * ---------------------------------------------------------------------------------------------- */
__global__ void factors_kernel(const dpgicp_result *__restrict__ rec, const PairTask *__restrict__ tasks, long long n,
                               dpgicp_factor *__restrict__ out) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const dpgicp_result r = rec[k];
  dpgicp_factor f;
  f.from_node = tasks[k].tgt; f.to_node = tasks[k].src;
  f.tx = r.tx; f.ty = r.ty; f.theta = r.theta;
  const double a = r.cov[0], b = r.cov[1], c = r.cov[2], d = r.cov[4], e = r.cov[5], g = r.cov[8];
  /* information matrix by cofactors of the symmetric covariance */
  const double c00 = __dsub_rn(__dmul_rn(d, g), __dmul_rn(e, e));
  const double c01 = __dsub_rn(__dmul_rn(c, e), __dmul_rn(b, g));
  const double c02 = __dsub_rn(__dmul_rn(b, e), __dmul_rn(c, d));
  const double det = __dadd_rn(__dadd_rn(__dmul_rn(a, c00), __dmul_rn(b, c01)), __dmul_rn(c, c02));
  bool ok = (det > 0.0) && isfinite(det);
  double R[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  if (ok) {
    const double id = __ddiv_rn(1.0, det);
    const double i00 = __dmul_rn(c00, id), i01 = __dmul_rn(c01, id), i02 = __dmul_rn(c02, id);
    const double i11 = __dmul_rn(__dsub_rn(__dmul_rn(a, g), __dmul_rn(c, c)), id);
    const double i12 = __dmul_rn(__dsub_rn(__dmul_rn(b, c), __dmul_rn(a, e)), id);
    const double i22 = __dmul_rn(__dsub_rn(__dmul_rn(a, d), __dmul_rn(b, b)), id);
    /* upper Cholesky: info = R^T R */
    ok = i00 > 0.0;
    if (ok) {
      const double r00 = __dsqrt_rn(i00);
      const double r01 = __ddiv_rn(i01, r00), r02 = __ddiv_rn(i02, r00);
      const double p11 = __dsub_rn(i11, __dmul_rn(r01, r01));
      ok = p11 > 0.0;
      if (ok) {
        const double r11 = __dsqrt_rn(p11);
        const double r12 = __ddiv_rn(__dsub_rn(i12, __dmul_rn(r01, r02)), r11);
        const double p22 = __dsub_rn(__dsub_rn(i22, __dmul_rn(r02, r02)), __dmul_rn(r12, r12));
        ok = p22 > 0.0;
        if (ok) {
          const double r22 = __dsqrt_rn(p22);
          R[0] = r00; R[1] = r01; R[2] = r02; R[4] = r11; R[5] = r12; R[8] = r22;
          for (int q = 0; q < 9; ++q) ok = ok && isfinite(R[q]);
        }
      }
    }
  }
  if (!ok)
    for (int q = 0; q < 9; ++q) R[q] = 0.0;
  for (int q = 0; q < 9; ++q) f.sqrt_info[q] = R[q];
  f.status = r.status | (ok ? 0u : DPGICP_FLAG_FACTOR_INVALID);
  out[k] = f;
}

/* ------------------------------------------------------------------------------------------------
 * FP32-pipe probe: the roofline denominator of the distance loop, measured on the device in use.
 * 8 independent dependent-chains per thread of separately rounded FMUL + FADD (the instruction mix
 * the bit-exact distance loop is allowed to use; FMA = false) or of FFMA (FMA = true, for context).
 * ---------------------------------------------------------------------------------------------- */
template <bool FMA>
__global__ void __launch_bounds__(256) fp32_probe_kernel(float *out, int iters, float a, float b) {
  float x[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) x[k] = (float)(threadIdx.x + k) * 1e-3f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      if (FMA) x[k] = __fmaf_rn(x[k], a, b);
      else x[k] = __fadd_rn(__fmul_rn(x[k], a), b);
    }
  }
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) s += x[k];
  if (s == 123.456f) out[0] = s;       /* keeps the chains alive; practically never true */
}

/* the same chains with packed pairs, two individually rounded results per instruction: FMUL2 then the packed sum in
 * the form the distance loop issues it (add2: an FFMA2 by an opaque 1.0f, because ptxas would contract a packed
 * mul.rn + add.rn pair into ONE fused FFMA2 — which is what this probe measured, unnoticed, until round 2: half the
 * instructions it was credited with) */
__global__ void __launch_bounds__(256) fp32x2_probe_kernel(float *out, int iters, float a, float b, float one) {
  f32x2 x[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) x[k] = pack2((float)(threadIdx.x + k) * 1e-3f, (float)(threadIdx.x + k) * 2e-3f);
  const f32x2 a2 = pack2(a, a), b2 = pack2(b, b), one2 = pack2(one, one);
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = add2(mul2(x[k], a2), b2, one2);
  }
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) { float lo, hi; unpack2(x[k], lo, hi); s += lo + hi; }
  if (s == 123.456f) out[0] = s;
}

}  // namespace dpg
