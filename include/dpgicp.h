/*
 * dpgicp.h — C ABI of the B200 scan-matching back end (batched 2D ICP + Censi covariance).
 *
 * This is the drop-in boundary for ONE path of DPG-SLAM: the inside of
 *   bool DpgSLAM::runIcp(DpgNode&, DpgNode&, pair<pair<Vector2f,float>,MatrixXd>&)
 *        (reference: src/dpg_slam/dpg_slam.cc:362-446, decl src/dpg_slam/dpg_slam.h:630)
 *   void calculate_ICP_COV(Ptr data_pi, Ptr model_qi, Matrix4f&, MatrixXd&, float, float, float)
 *        (reference: src/icp_cov/cov_func_point_to_point.h:24-585)
 * plus the batch form the two callers need (dpg_slam.cc:85,101,263,295).
 *
 * Plain C, plain-old-data only; no C++/torch/CUDA types cross this boundary.  All functions
 * return 0 on success and a negative DPGICP_E_* code on failure (never throw); the message of
 * the last failure on a context is available from dpgicp_last_error().  There is no CPU
 * fallback: without a CUDA device dpgicp_create() fails with DPGICP_E_NODEVICE.
 *
 * Ownership: the caller owns every host buffer; the library owns device buffers inside the
 * opaque context.  A context is single-owner (one host thread at a time), as the reference's
 * callers are single-threaded (src/dpg_slam/dpg_slam_main.cc:328).
 */
#ifndef DPGICP_H
#define DPGICP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPGICP_ABI_VERSION 5

/* ---- error codes ------------------------------------------------------------------------- */
#define DPGICP_OK            0
#define DPGICP_E_INVALID    -1   /* bad argument (NULL, negative size, index out of range, ...)  */
#define DPGICP_E_NODEVICE   -2   /* no CUDA device / device ordinal not present                   */
#define DPGICP_E_CUDA       -3   /* a CUDA runtime call failed (see dpgicp_last_error)            */
#define DPGICP_E_NOMEM      -4   /* host or device allocation failed                              */
#define DPGICP_E_RANGE      -5   /* non-finite point or |coordinate| > DPGICP_MAX_ABS_COORD       */
#define DPGICP_E_STATE      -6   /* call order violated (e.g. run before pairs were set)          */
#define DPGICP_E_TOOBIG     -7   /* a scan has more points than DPGICP_MAX_POINTS                 */

/* Arithmetic-contract limits (DESIGN.md "arithmetic contract"): coordinates are binary32 metres,
 * moment sums are exact 64-bit fixed point, which needs these bounds.                           */
#define DPGICP_MAX_ABS_COORD 1000.0f
#define DPGICP_MAX_POINTS    8192

/* ---- enumerations ------------------------------------------------------------------------ */
/* error metric minimised by each ICP step */
#define DPGICP_METRIC_POINT_TO_POINT 0   /* what the reference runs (PCL ICP, dpg_slam.cc:387)   */
#define DPGICP_METRIC_POINT_TO_LINE  1   /* north-star extension; no reference counterpart: each matched
                                          * target point contributes the line through it and its closer beam
                                          * neighbour; one Gauss-Newton step per iteration from the 3x3 normal
                                          * equations (Cholesky); DESIGN.md "point-to-line"               */

/* Tie rule of the exact searches (BRUTE, PRUNED).  FLANN's order among points at EXACTLY the same binary32 distance
 * is unspecified (SURVEY.md App. A.3-2), so the library fixes one that is cheap on the GPU:
 *   forward     the neighbour is the point matched in the previous iteration of the same pair when it is among the
 *               minimisers ("sticky"), else the lowest index among them;
 *   reciprocal  (i, j) is kept iff no source point is STRICTLY closer to target j than source i (the asker wins ties).
 * For inputs without exact distance ties this is plain nearest-neighbour search.                                  */
/* nearest-neighbour search strategy; BRUTE and PRUNED are exact and give identical correspondences */
#define DPGICP_SEARCH_BRUTE   0
#define DPGICP_SEARCH_PRUNED  1          /* beam-order block bounding boxes + seeded bound       */
#define DPGICP_SEARCH_PROJECTIVE 2       /* north-star extension; no reference counterpart (PCL searches exactly).
                                          * APPROXIMATE neighbour by projection onto the other scan's beam order:
                                          *   key(v), v = point - (sensor_x, sensor_y): a = |vx| + |vy|, t = a > 0 ? vy / a : 0,
                                          *   key = vx >= 0 ? t : (vy >= 0 ? 2 - t : -2 - t)     (binary32, monotone in the bearing)
                                          *   c = lower_bound of key(query) in the searched scan's keys (plain bisection over the
                                          *   stored order, whether or not the keys are sorted); candidates = indices
                                          *   [c - W, c + W) inside the scan, W = projective_window; the (d2, index)-
                                          *   lexicographic minimum among them is the neighbour.
                                          * Forward: query = current source point, searched = target.  Reciprocal: query = the
                                          * matched target point taken back to the source frame by the inverse of the current
                                          * transform, searched keys = the untransformed source scan, distances to the current
                                          * source points.  Defined by oracle/dpg_oracle.c (orc_correspondences_ex).      */

/* outlier rejection after the reciprocal test (north-star "outlier-trim logic").  The reference registers no
 * correspondence rejector (dpg_slam.cc:408-412; setRANSACIterations is inert in stock PCL ICP), so the default is
 * NONE; the other modes are defined by oracle/dpg_oracle.c (orc_outlier_threshold).  K = accepted correspondences of
 * the pass, d2 their squared distances (binary32):
 *   TRIMMED  keep_n = max(3, floor(outlier_param * K)); tau = keep_n-th smallest d2; keep d2 <= tau
 *            (PCL CorrespondenceRejectorTrimmed with overlap ratio outlier_param in (0, 1]);
 *   MEDIAN   med = d2 of rank K / 2; tau = largest binary32 <= (double)med * outlier_param; keep d2 <= tau
 *            (PCL CorrespondenceRejectorMedianDistance with factor outlier_param > 0).
 * Ties at tau are all kept, so the kept set does not depend on any ordering of equal values.  The same rejector is
 * applied to the correspondences the CENSI_CORR covariance is formed on.                                          */
#define DPGICP_OUTLIER_NONE    0
#define DPGICP_OUTLIER_TRIMMED 1
#define DPGICP_OUTLIER_MEDIAN  2

/* what is written to result.cov (SURVEY.md §8a "covariance modes") */
#define DPGICP_COV_REFERENCE_LIVE  0     /* diag(sx2, sy2, st2): cov_func_point_to_point.h:572-575 */
#define DPGICP_COV_CENSI_INDEXPAIR 1     /* intended formula, clouds paired by index as dpg_slam.cc:430 */
#define DPGICP_COV_CENSI_CORR      2     /* intended formula on the final ICP correspondences    */
/* CENSI_CORR pair set: one correspondence pass at the FINAL pose (down-sampled source moved by the final transform),
 * seeded with the last ICP pass's forward neighbours, then the reciprocal test and the outlier rejector (if any).  The
 * kept pairs in source-index order, p = the untransformed down-sampled source point: the Hessian runs over all of them,
 * the D-term over the first cov_cap (all when cov_cap = 0).  CENSI_INDEXPAIR: the full clouds paired by index,
 * n_h = min(n_source, n_target), the D-term over the first min(n_h, cov_cap). */

/* result.status: low byte = stop reason, higher bits = flags */
#define DPGICP_STOP_MASK              0xffu
#define DPGICP_STOP_NONE              0u   /* never ran                                          */
#define DPGICP_STOP_ITERATIONS        1u   /* max_iterations reached (PCL reports converged)     */
#define DPGICP_STOP_TRANSFORM         2u   /* step below transformation_epsilon                  */
#define DPGICP_STOP_ABS_MSE           3u   /* |mse - mse_prev| < 1e-12                           */
#define DPGICP_STOP_NO_CORRESPONDENCES 4u  /* fewer than 3 pairs: converged == false                 */
#define DPGICP_STOP_DEGENERATE        5u   /* point-to-line only: normal equations not positive definite
                                            * (geometry does not constrain the pose); converged == false */
#define DPGICP_FLAG_CONVERGED         0x100u  /* == what icp.hasConverged() returns, dpg_slam.cc:445 */
#define DPGICP_FLAG_COV_SINGULAR      0x200u  /* Hessian not invertible; cov fell back to the LIVE diagonal */
#define DPGICP_FLAG_EMPTY_INPUT       0x400u  /* a cloud of the pair had no points                */
#define DPGICP_FLAG_FACTOR_INVALID    0x800u  /* dpgicp_factor only: cov is not positive definite  */

/* ---- parameter block (defaults = src/dpg_slam/parameters.h, see dpgicp_default_params) ---- */
typedef struct dpgicp_params {
  int32_t max_iterations;              /* 500    parameters.h:146 */
  int32_t use_reciprocal;              /* 1      parameters.h:201 */
  int32_t ransac_iterations;           /* 50     parameters.h:191 — stored, inert (as in stock PCL ICP) */
  int32_t downsample_divisor;          /* 5      parameters.h:402 — 1 = "1081-beam" benchmark setting */
  int32_t metric;                      /* DPGICP_METRIC_*  (default point-to-point)              */
  int32_t search;                      /* DPGICP_SEARCH_*  (default pruned)                      */
  int32_t cov_mode;                    /* DPGICP_COV_*     (default REFERENCE_LIVE = drop-in)    */
  int32_t cov_cap;                     /* 200    cov_func_point_to_point.h:307; 0 = no cap       */
  double  transformation_epsilon;      /* 5e-9   parameters.h:159 */
  double  max_correspondence_distance; /* 0.6    parameters.h:173; must be <= 30 m (fixed-point sums) */
  double  cov_sensor_variance;         /* 0.01   cov_func_point_to_point.h:554 (cov_z = 0.01 I)  */
  float   laser_x_variance;            /* 0.5    parameters.h:374 */
  float   laser_y_variance;            /* 0.5    parameters.h:385 */
  float   laser_theta_variance;        /* 0.3    parameters.h:396 */
  int32_t projective_window;           /* 8      DPGICP_SEARCH_PROJECTIVE only: W, candidates on each side (1..1024)   */
  float   sensor_x, sensor_y;          /* 0.2, 0 DPGICP_SEARCH_PROJECTIVE only: laser origin in the cloud (base_link)
                                        *        frame, parameters.h:319-339 — the centre the beam order turns around  */
  int32_t outlier_mode;                /* DPGICP_OUTLIER_* (default NONE = stock PCL ICP, dpg_slam.cc:408-412)        */
  int32_t reserved0;                   /* 0                                                                           */
  double  outlier_param;               /* TRIMMED: overlap ratio in (0, 1]; MEDIAN: factor > 0                         */
} dpgicp_params;

/* ---- fixed-size result record (112 bytes) ------------------------------------------------- */
typedef struct dpgicp_result {
  float    tx, ty;        /* T(0,3), T(1,3) of the final transform: pose of source in target frame */
  float    theta;         /* atan2f(T(1,0), T(0,0))                       dpg_slam.cc:434-439       */
  float    rot_c, rot_s;  /* T(0,0), T(1,0) — the raw rotation entries theta was taken from         */
  int32_t  iterations;    /* ICP iterations executed                                               */
  uint32_t status;        /* DPGICP_STOP_* | DPGICP_FLAG_*                                          */
  int32_t  n_correspondences; /* of the last executed iteration                                    */
  double   mse;           /* mean squared correspondence distance of the last executed iteration   */
  double   cov[9];        /* 3x3, axes (x, y, theta), row-major (symmetric)  cov.h:564-566,573-575  */
} dpgicp_result;

/* ---- pose-graph factor (the hand-off of addObservationConstraint, dpg_slam.cc:331-338) -------- */
/* BetweenFactor<Pose2>(from, to, Pose2(tx, ty, theta), noiseModel::Gaussian::Covariance(cov)): GTSAM
 * turns the covariance into the upper-triangular square-root information R (R^T R = cov^-1); it is
 * computed here on the device so the host does no per-factor linear algebra
 * (noiseModel::Gaussian::SqrtInformation(R)).                                                     */
typedef struct dpgicp_factor {          /* 96 bytes */
  int32_t  from_node, to_node;          /* target scan (node_1), source scan (node_2)                 */
  float    tx, ty, theta;               /* pose of to_node in from_node's frame                        */
  uint32_t status;                      /* the record's status | DPGICP_FLAG_FACTOR_INVALID           */
  double   sqrt_info[9];                /* R, row-major, upper triangular; zeros when invalid          */
} dpgicp_factor;

typedef struct dpgicp_ctx dpgicp_ctx;
typedef struct dpgicp_slot dpgicp_slot;

/* ---- lifetime ------------------------------------------------------------------------------ */
int  dpgicp_abi_version(void);
int  dpgicp_default_params(dpgicp_params *p);
int  dpgicp_create(int device_ordinal, dpgicp_ctx **out_ctx);
void dpgicp_destroy(dpgicp_ctx *ctx);
const char *dpgicp_last_error(const dpgicp_ctx *ctx);   /* ctx may be NULL: last create() error */

/* Launch work of this context on an existing CUDA stream (a cudaStream_t passed as void*), e.g.
 * the caller's framework stream so that its events bracket our kernels.  NULL = own stream.   */
int  dpgicp_set_stream(dpgicp_ctx *ctx, void *cuda_stream);
int  dpgicp_synchronize(dpgicp_ctx *ctx);

/* ---- scan store (replaces the per-node cached clouds, dpg_node.cc:8-26) --------------------- */
/* Upload n_scans ragged clouds.  Scan k owns points [offsets[k], offsets[k+1]) of `points`;
 * a point is two consecutive floats (x, y) at byte stride `stride_bytes` (8 = packed float2,
 * 16 = pcl::PointXYZ layout {x,y,z,pad}; z is ignored, the reference sets it to 0).
 * Replaces any previous store.                                                                 */
int  dpgicp_upload_scans(dpgicp_ctx *ctx, const void *points, size_t stride_bytes,
                         const int64_t *offsets, int32_t n_scans);

/* Upload raw range scans and convert on the device (createNode dpg_slam.cc:488-513 +
 * getCachedPointCloudFromNode dpg_node.cc:8-26): angle_i = angle_inc*i + angle_min (float),
 * p = (r cos a, r sin a), drop r >= range_max, then laser->base_link pose (lx, ly, ltheta).    */
int  dpgicp_upload_ranges(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans, int32_t n_beams,
                          float angle_min, float angle_max, float range_max,
                          float laser_x, float laser_y, float laser_theta);

/* The same conversion for a SUBSET of the scans of a host array: store row k = scan scan_ids[k].  A GPU that
 * holds a shard of the pairs needs only the scans its pairs touch.  When `ranges` is page-locked host memory the
 * kernel reads the selected rows directly over PCIe (no staging, only those rows cross the bus); pageable
 * memory is gathered through an internal pinned buffer.                                                      */
int  dpgicp_upload_ranges_subset(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans_total, int32_t n_beams,
                                 const int32_t *scan_ids, int32_t n_ids, float angle_min, float angle_max,
                                 float range_max, float laser_x, float laser_y, float laser_theta);

/* Append n_scans range scans to the store: they become rows scan_count() .. scan_count() + n_scans - 1, so node k of
 * an online caller can own row k without the earlier scans being sent again (createNode, dpg_slam.cc:462-513, one
 * call per new node).  Same conversion and arguments as dpgicp_upload_ranges: every appended row and its count are bit
 * for bit what one dpgicp_upload_ranges of all the scans would hold.  Existing rows, the current pair batch and the
 * node table stay valid (indices only grow).  After dpgicp_upload_ranges_subset the appended scans take the next row
 * numbers, whatever scans the subset's rows came from.  An empty (or never uploaded) store is started.
 * Storage grows by doubling; a scan longer than the store's row pitch re-pitches the store on the device.
 * Failure leaves the store as it was: a non-finite or out-of-range point gives DPGICP_E_RANGE with scan_count()
 * unchanged and every earlier row intact (unlike a full upload, which empties the store); bad arguments give
 * DPGICP_E_INVALID and n_beams > DPGICP_MAX_POINTS gives DPGICP_E_TOOBIG, both before any device work.  Stream-ordered
 * with a dpgicp_run enqueued before it: the run reads the store as it was.                                        */
int  dpgicp_append_ranges(dpgicp_ctx *ctx, const float *ranges, int32_t n_scans, int32_t n_beams,
                          float angle_min, float angle_max, float range_max,
                          float laser_x, float laser_y, float laser_theta);
/* The same for point clouds, with the layout and offsets of dpgicp_upload_scans (a scan over DPGICP_MAX_POINTS points
 * gives DPGICP_E_TOOBIG).                                                                                        */
int  dpgicp_append_scans(dpgicp_ctx *ctx, const void *points, size_t stride_bytes,
                         const int64_t *offsets, int32_t n_scans);

int  dpgicp_scan_count(const dpgicp_ctx *ctx);
/* copy scan k of the store back to the host (packed float2); *n_points in = capacity, out = count */
int  dpgicp_download_scan(dpgicp_ctx *ctx, int32_t scan, float *xy, int32_t *n_points);

/* ---- batched alignment ---------------------------------------------------------------------- */
/* The runIcp batch: pair k aligns source scan src_idx[k] (node_2) onto target scan tgt_idx[k]
 * (node_1) starting from guess[3k..3k+2] = (dx, dy, dtheta), the pose of node_2 in node_1's frame
 * (dpg_slam.cc:364-378).  Synchronous; writes n_pairs records to out (host memory).            */
int  dpgicp_submit_pairs(dpgicp_ctx *ctx, const int32_t *src_idx, const int32_t *tgt_idx,
                         const float *guess, int64_t n_pairs, const dpgicp_params *params,
                         dpgicp_result *out);

/* Same work split into resident steps (what the benchmark's device-resident figure times):      */
int  dpgicp_set_pairs(dpgicp_ctx *ctx, const int32_t *src_idx, const int32_t *tgt_idx,
                      const float *guess, int64_t n_pairs);            /* H2D of the pair list   */
int  dpgicp_run(dpgicp_ctx *ctx, const dpgicp_params *params);         /* async on ctx stream    */
/* Optional scheduling hint for the pair list set last: expected relative cost per pair (e.g. the iteration counts of
 * the previous alignment of the same pairs — reoptimize(), dpg_slam.cc:35-120, re-aligns every pair after each pass).
 * Pairs are then started in descending hint order, so long alignments do not start last.  Results do not depend on
 * it (tested).  NULL clears the hint; set_pairs clears it too.                                                  */
int  dpgicp_set_pair_cost_hints(dpgicp_ctx *ctx, const float *hints, int64_t n_pairs);
int  dpgicp_fetch_results(dpgicp_ctx *ctx, dpgicp_result *out, int64_t n_pairs); /* D2H + sync   */
/* Part of the resident pair list: pairs [first, first + count) (asynchronous like dpgicp_run; records, fused-gather
 * slots and factors keep the indices of the whole list).  Lets a caller stream a very large enumerated list through
 * the device in slices, or warm up on a prefix.  The *_range fetches copy the matching records.                 */
int  dpgicp_run_range(dpgicp_ctx *ctx, const dpgicp_params *params, int64_t first, int64_t count);
int  dpgicp_fetch_results_range(dpgicp_ctx *ctx, dpgicp_result *out, int64_t first, int64_t count);
/* Records of the last dpgicp_run turned into pose-graph factors on the device (one per pair, pair order). */
int  dpgicp_fetch_factors(dpgicp_ctx *ctx, dpgicp_factor *out, int64_t n_pairs);
/* device address of the record array written by dpgicp_run (n_pairs * sizeof(dpgicp_result));
 * lets a multi-GPU host gather records device-to-device (NCCL) without a host bounce.          */
int  dpgicp_results_device_ptr(dpgicp_ctx *ctx, void **out_ptr, int64_t *out_n_pairs);
/* ---- multi-GPU gather fused into the kernel (one context per GPU, one process per GPU or not) --------------
 * Scan pairs are independent, so pair k of a global batch runs on rank k % world (round-robin) and the ONLY
 * exchange is the gather of the records.  Instead of a collective after the kernel, every rank exports a buffer
 * sized for the whole batch (CUDA IPC handle, 64 bytes), attaches all ranks' buffers, and from then on dpgicp_run
 * stores each finished record straight into slot (rank + k * world) of every rank's buffer (peer stores over
 * NVLink from the kernel's epilogue).  After all ranks have synchronised, every buffer holds the whole batch in
 * global pair order.                                                                                       */
#define DPGICP_IPC_HANDLE_BYTES   64
#define DPGICP_MAX_GATHER_RANKS   16
int  dpgicp_gather_export(dpgicp_ctx *ctx, int64_t n_global_pairs, unsigned char handle_out[DPGICP_IPC_HANDLE_BYTES]);
/* root-only gathers (dpgicp_gather_set_root_only): ranks other than 0 receive nothing, so they only declare the size of
 * the global batch (a one-record placeholder allocation backs the handle)                                   */
int  dpgicp_gather_declare(dpgicp_ctx *ctx, int64_t n_global_pairs, unsigned char handle_out[DPGICP_IPC_HANDLE_BYTES]);
/* handles = world * 64 bytes in rank order (this rank's own entry is ignored and may be anything) */
int  dpgicp_gather_attach(dpgicp_ctx *ctx, const unsigned char *handles, int32_t world, int32_t rank);
int  dpgicp_gather_detach(dpgicp_ctx *ctx);
/* copy the first n records of this rank's gather buffer to the host (caller has synchronised all ranks) */
int  dpgicp_gather_fetch(dpgicp_ctx *ctx, dpgicp_result *out, int64_t n_global_pairs);
int  dpgicp_gather_fetch_range(dpgicp_ctx *ctx, dpgicp_result *out, int64_t first, int64_t count);
int  dpgicp_gather_device_ptr(dpgicp_ctx *ctx, void **out_ptr, int64_t *out_n_global_pairs);

/* executed-work counters of the last dpgicp_run, summed over pairs (after synchronisation):
 * [0] iterations, [1] correspondences, [2] distance evaluations, [3] block tests, [4] kernel launches */
int  dpgicp_last_run_counters(dpgicp_ctx *ctx, uint64_t counters[8]);

/* ---- single-call shapes of the two reference functions -------------------------------------- */
/* runIcp shape: two clouds + guess -> record.  source = node_2 cloud, target = node_1 cloud,
 * both NOT yet down-sampled (params->downsample_divisor is applied inside, dpg_slam.cc:397-402). */
int  dpgicp_single_pair(dpgicp_ctx *ctx,
                        const void *source_points, int32_t n_source,
                        const void *target_points, int32_t n_target, size_t stride_bytes,
                        const float guess[3], const dpgicp_params *params, dpgicp_result *out);

/* calculate_ICP_COV shape: data_pi, model_qi, Matrix4f (column-major 16 floats), three variances
 * -> 3x3 double.  cov_mode LIVE reproduces the reference's live output; CENSI_INDEXPAIR its
 * intended one (the clouds are paired by index, as the reference passes them).                  */
int  dpgicp_cov(dpgicp_ctx *ctx,
                const void *data_pi, int32_t n_data, const void *model_qi, int32_t n_model,
                size_t stride_bytes, const float transform_colmajor[16],
                const dpgicp_params *params, double cov_out[9], uint32_t *status_out);

/* Batched form over the scan store: item k is calculate_ICP_COV(data_pi = scan data_idx[k], model_qi = scan
 * model_idx[k], T[k]) with T[k] = (T(0,0), T(1,0), T(0,3), T(1,3)) of the 4x4 transform; cov_out = 9 doubles and
 * status_out = one word per item.  One CTA per item; HBM-bound (16 bytes read per index pair).  kernel_ms (may be
 * NULL) receives the device time of the kernel alone (CUDA events on the context's stream).                 */
int  dpgicp_cov_pairs(dpgicp_ctx *ctx, const int32_t *data_idx, const int32_t *model_idx, const float *T,
                      int64_t n_items, const dpgicp_params *params, double *cov_out, uint32_t *status_out,
                      float *kernel_ms);

/* Host helper, no device work: the guess runIcp derives from two node pose estimates
 * (dpg_slam.cc:364-370 = math_utils::inverseTransformPoint, math_utils.cc:20-34, and AngleMod,
 * math_utils.h:13-16), in the reference's float arithmetic.  pose = (x, y, theta).             */
int  dpgicp_relative_guess(const float node_1_pose[3], const float node_2_pose[3], float guess[3]);

/* ---- parity / inspection hook ---------------------------------------------------------------- */
/* One correspondence pass at a given iterate: the source cloud (already down-sampled) is
 * transformed by T = [c -s tx; s c ty] exactly as one ICP iteration would, then matched.
 * corr_tgt[i] = matched target index or -1; corr_d2[i] = squared distance (binary32).
 * This is what the "correspondence sets bit-exact at equal iterate" tests call.                 */
int  dpgicp_correspondences(dpgicp_ctx *ctx,
                            const void *source_points, int32_t n_source,
                            const void *target_points, int32_t n_target, size_t stride_bytes,
                            const float T[4] /* c, s, tx, ty */, const dpgicp_params *params,
                            int32_t *corr_tgt, float *corr_d2);

/* The same pass with the tie preference of an ICP run in progress: prev_nn[i] = forward neighbour of source point i
 * in the previous pass (-1 = none; NULL = all none, i.e. dpgicp_correspondences), nn_out[i] (may be NULL) = this
 * pass's gated forward neighbour — what the next pass would be seeded with.                                      */
int  dpgicp_correspondences_seeded(dpgicp_ctx *ctx,
                                   const void *source_points, int32_t n_source,
                                   const void *target_points, int32_t n_target, size_t stride_bytes,
                                   const float T[4], const dpgicp_params *params, const int32_t *prev_nn,
                                   int32_t *corr_tgt, float *corr_d2, int32_t *nn_out);

/* ---- candidate-pair enumeration (callers' distance gate, dpg_slam.cc:91-98,275-282) ---------- */
/* For node i (ascending) and every j < i-1 ... emits (src=i, tgt=j) when the node positions are
 * within same_pass_radius (same pass) or other_pass_radius (different pass), plus every
 * successive pair (src=i, tgt=i-1) — the pair set of one DpgSLAM::reoptimize().  Output order is
 * the reference's loop order.  *n_pairs in = capacity, out = count (DPGICP_E_TOOBIG if short).
 * Radii must be >= 0 (NaN: DPGICP_E_INVALID).  This form is independent of the device-resident one below: it uses a
 * node table of its own and leaves the table of dpgicp_set_nodes and the current batch as they were.            */
int  dpgicp_enumerate_pairs(dpgicp_ctx *ctx, const float *node_xy, const int32_t *node_pass,
                            int32_t n_nodes, float same_pass_radius, float other_pass_radius,
                            int32_t *src_idx, int32_t *tgt_idx, int64_t *n_pairs);

/* ---- device-resident form of the callers (pose-graph nodes in, pair batch left on the device) --------------
 * Node k of the pose graph owns scan k of the store.  dpgicp_set_nodes uploads the node estimates
 * (x, y, theta per node, DpgNode::getEstimatedPosition) and pass numbers.  dpgicp_enumerate_pairs_device then builds
 * the pair list of one caller ON THE DEVICE, in the reference's loop order, together with every pair's guess
 * (dpg_slam.cc:364-378, the arithmetic of dpgicp_relative_guess + the Matrix4f cos/sin), and leaves it as the
 * context's current batch: dpgicp_run / fetch_results / fetch_factors follow with no host round trip of the list.
 *   DPGICP_ENUM_REOPTIMIZE  DpgSLAM::reoptimize (dpg_slam.cc:79-107): for i = 1..n-1: (src i, tgt i-1), then every
 *                           j < i-1 within same_pass_radius / other_pass_radius of node i -> (src i, tgt j).
 *   DPGICP_ENUM_ONLINE      DpgSLAM::updatePoseGraphObsConstraints (dpg_slam.cc:255-300) for new node n-1 with
 *                           preceding node n-2: (src n-1, tgt n-2), then every i <= n-4 within the radius of the
 *                           PRECEDING node -> (src n-2, tgt i)   [loop closures attach to the preceding node and the
 *                           loop runs to dpg_nodes_.size() - 2 exclusive, dpg_slam.cc:275-299].
 * Sharding: of the global list only the pairs with (global index % shard_world) == shard_rank become this context's
 * batch (round-robin, as the multi-GPU path shards); local pair k is global pair shard_rank + k * shard_world.
 * n_pairs_total / n_pairs_local (may be NULL) receive the global and the local count.  Radii must be >= 0
 * (NaN: DPGICP_E_INVALID).  Any legal node table enumerates: guesses whose cos / sin lie next to a binary32 rounding
 * boundary are re-derived with the host's libm, however many pairs share one (e.g. a recurring heading difference). */
#define DPGICP_ENUM_REOPTIMIZE 0
#define DPGICP_ENUM_ONLINE     1
int  dpgicp_set_nodes(dpgicp_ctx *ctx, const float *node_pose_xytheta, const int32_t *node_pass, int32_t n_nodes);
/* Change part of the node table of dpgicp_set_nodes and/or grow it.  After the call the table holds n_nodes nodes;
 * node ids[k] takes the estimate pose_xytheta[3k..3k+2] and pass[k]; every other node keeps what it had.
 *   Result: the table is bit for bit what one dpgicp_set_nodes of the equivalent full arrays holds (positions, theta
 *     and its host-libm cosf / sinf, pass numbers, every box level), so enumerated lists, guesses, records and factors
 *     are identical too, whatever changed (a node that moves away and shrinks its box, a change of pass range).
 *   Size: n_nodes >= the current count (a table never set counts as 0, so this call may start one); every id in
 *     [current count, n_nodes) is listed; ids are distinct and in [0, n_nodes).  n_ids = 0 with an unchanged n_nodes
 *     does nothing.
 *   Errors leave the table as it was: DPGICP_E_INVALID for a shrinking n_nodes, a new id not listed, a duplicate or
 *     out-of-range id, or NULL arrays with n_ids > 0; DPGICP_E_RANGE for a non-finite estimate.  Both are found on the
 *     host before any device write.  DPGICP_E_NOMEM from the capacity growth also leaves the table as it was; a CUDA
 *     error (DPGICP_E_CUDA) once the device work has been enqueued empties the table, as a failed dpgicp_set_nodes
 *     does.
 *   Cost: host work and the host-to-device copy scale with n_ids, not n_nodes: the listed rows are scattered and only
 *     the leaf boxes (32 nodes each) that hold a listed node are refit, then the upper levels (at most n_nodes / 1024
 *     boxes).  Capacity grows by doubling, so appending one node per call is amortised O(1).
 *   Ordering: as dpgicp_set_nodes.  The table is per context and the enumeration reads it synchronously; a run
 *     already enqueued in any slot keeps the guesses its batch was enumerated with.  The call returns once its work is
 *     enqueued on the context's stream.  dpgicp_set_nodes still replaces the whole table and may be mixed with this
 *     call in any order; dpgicp_enumerate_pairs (host list) uses a table of its own and is unaffected.             */
int  dpgicp_update_nodes(dpgicp_ctx *ctx, int32_t n_nodes, const int32_t *ids, const float *pose_xytheta,
                         const int32_t *pass, int32_t n_ids);
int  dpgicp_enumerate_pairs_device(dpgicp_ctx *ctx, int32_t mode, float same_pass_radius, float other_pass_radius,
                                   int32_t shard_rank, int32_t shard_world, int64_t *n_pairs_total,
                                   int64_t *n_pairs_local);
/* the current batch's pair list back on the host (any of the outputs may be NULL): indices and the guess as the
 * Matrix4f entries T = (T(0,0), T(1,0), T(0,3), T(1,3)) per pair                                                */
int  dpgicp_fetch_pairs(dpgicp_ctx *ctx, int32_t *src_idx, int32_t *tgt_idx, float *T, int64_t n_pairs);
/* scan store from raw ranges that are ALREADY in device memory (e.g. all-gathered there over NCCL); same conversion
 * as dpgicp_upload_ranges                                                                                       */
int  dpgicp_convert_ranges_device(dpgicp_ctx *ctx, const float *d_ranges, int32_t n_scans, int32_t n_beams,
                                  float angle_min, float angle_max, float range_max,
                                  float laser_x, float laser_y, float laser_theta);

/* ---- single-process multi-GPU (host code in C/C++: one context per GPU driven by one thread) ----------------
 * The fused gather for contexts that live in ONE process: instead of CUDA IPC handles the contexts are given each
 * other's gather buffers directly (peer access is enabled between their devices).  ctxs[r] becomes rank r of
 * `world`; every context allocates a buffer for n_global_pairs records.  root_only != 0: records are stored only
 * into rank 0's buffer (what a single host-side pose-graph update needs) instead of into every rank's.          */
int  dpgicp_gather_attach_local(dpgicp_ctx **ctxs, int32_t world, int64_t n_global_pairs, int32_t root_only);
/* the cross-process form (dpgicp_gather_export / _attach) with root_only != 0 stores into rank 0's buffer only; set
 * before dpgicp_run, on every rank alike                                                                        */
int  dpgicp_gather_set_root_only(dpgicp_ctx *ctx, int32_t root_only);
/* device time of every stage launch of dpgicp_run (CUDA events between the launches of the stage chain): switch it
 * on, run, then read the last run's per-stage times in ms (synchronises on the last stage); *n_stages <= 8       */
int  dpgicp_enable_stage_timing(dpgicp_ctx *ctx, int32_t on);
int  dpgicp_last_run_stage_ms(dpgicp_ctx *ctx, float stage_ms[8], int32_t *n_stages);

/* ---- measurement aid ------------------------------------------------------------------------- */
/* Measures this device's FP32 CUDA-core throughput with the two instruction mixes that matter for
 * the roofline of the distance loop: separately rounded FMUL+FADD (what the bit-exact loop may use)
 * and FFMA (for context).  Results in operations per second (one FMUL, FADD or FFMA = 1 op).     */
int  dpgicp_fp32_probe(dpgicp_ctx *ctx, double *ops_per_s_mul_add, double *ops_per_s_fma);
/* The same chains issued as packed pairs (sm_100 FMUL2 + the packed sum the distance loop uses): operations per
 * second, one packed instruction = 2 operations.  Measured equal to the scalar rate: a packed instruction takes two
 * pipe cycles, so packing saves issue slots, not FP32 time.                                         */
int  dpgicp_fp32x2_probe(dpgicp_ctx *ctx, double *ops_per_s_mul_add_packed);

/* ---- batch slots: several pair batches in flight on one context ------------------------------------------------
 * The batch calls above (dpgicp_set_pairs, _run, _fetch_*, dpgicp_enumerate_pairs_device, stage timing, the fused
 * gather) act on the context's DEFAULT slot, which runs on the context's stream (dpgicp_set_stream).  A slot created
 * here holds a batch of its own (pair list, cost hints, records, counters) and runs it on a CUDA stream of its own on
 * the context's device, so a caller can prepare and launch batch k+1 while batch k still runs.  Every slot shares the
 * context's scan store and node table: one copy of the store serves every batch in flight.
 *   for (k = 0; k < n_batches; ++k) {
 *     dpgicp_slot *s = slot[k % K];
 *     if (k >= K) dpgicp_slot_fetch_results(s, out[k - K], n[k - K]);     // waits for that batch only
 *     dpgicp_slot_set_pairs(s, src[k], tgt[k], guess[k], n[k]);
 *     dpgicp_slot_run(s, &params);                                        // returns at once
 *   }
 * Ordering rules (enforced by the library with stream events and synchronisations):
 *   - a slot's run reads the store as it was when the run was enqueued, and waits for the store writes (upload, append,
 *     convert) and the enumeration into that slot enqueued before it;
 *   - dpgicp_upload_scans / _upload_ranges / _upload_ranges_subset / _convert_ranges_device replace the store: they wait
 *     for every slot's enqueued work and empty every slot's batch.  dpgicp_append_* writes only rows no enqueued run
 *     reads and does not wait, unless the store has to move (growth, re-pitch): the old buffers are then freed only
 *     after every slot's stream has drained;
 *   - dpgicp_set_nodes and dpgicp_update_nodes do not wait: no run reads the node table (the enumeration does, and it
 *     is synchronous);
 *   - dpgicp_slot_enumerate_pairs_device runs on the context's stream and returns when the list is on the device, as
 *     dpgicp_enumerate_pairs_device does; it first waits for the slot's own enqueued work;
 *   - the fused multi-GPU gather (dpgicp_gather_attach*) applies to the default slot only: a slot's run writes its
 *     local records only, whether or not a gather is attached;
 *   - records do not depend on what runs concurrently (bit-equal to the same batch run alone).
 * Returns: DPGICP_E_INVALID for a NULL or destroyed slot (as for bad arguments), DPGICP_E_STATE for a run before the
 * slot's first pair list.  Errors are reported through dpgicp_last_error of the slot's context.  A slot belongs to the
 * thread that owns its context.                                                                                  */
int  dpgicp_slot_create(dpgicp_ctx *ctx, dpgicp_slot **out_slot);
/* waits for the slot's work, then frees it; dpgicp_destroy destroys the slots of the context still alive */
int  dpgicp_slot_destroy(dpgicp_slot *slot);
/* the slot forms of dpgicp_set_pairs, _set_pair_cost_hints, _run, _run_range, _fetch_results, _fetch_results_range,
 * _fetch_factors, _fetch_pairs, _last_run_counters ([4] counts the launches of the whole context) and _synchronize */
int  dpgicp_slot_set_pairs(dpgicp_slot *slot, const int32_t *src_idx, const int32_t *tgt_idx, const float *guess,
                           int64_t n_pairs);
int  dpgicp_slot_set_pair_cost_hints(dpgicp_slot *slot, const float *hints, int64_t n_pairs);
int  dpgicp_slot_run(dpgicp_slot *slot, const dpgicp_params *params);
int  dpgicp_slot_run_range(dpgicp_slot *slot, const dpgicp_params *params, int64_t first, int64_t count);
int  dpgicp_slot_fetch_results(dpgicp_slot *slot, dpgicp_result *out, int64_t n_pairs);
int  dpgicp_slot_fetch_results_range(dpgicp_slot *slot, dpgicp_result *out, int64_t first, int64_t count);
int  dpgicp_slot_fetch_factors(dpgicp_slot *slot, dpgicp_factor *out, int64_t n_pairs);
int  dpgicp_slot_fetch_pairs(dpgicp_slot *slot, int32_t *src_idx, int32_t *tgt_idx, float *T, int64_t n_pairs);
int  dpgicp_slot_last_run_counters(dpgicp_slot *slot, uint64_t counters[8]);
int  dpgicp_slot_synchronize(dpgicp_slot *slot);
/* non-blocking: 1 when the slot's enqueued work is done, 0 while it runs, < 0 on error */
int  dpgicp_slot_query(dpgicp_slot *slot);
/* dpgicp_enumerate_pairs_device with the list and guesses left as the slot's batch */
int  dpgicp_slot_enumerate_pairs_device(dpgicp_slot *slot, int32_t mode, float same_pass_radius, float other_pass_radius,
                                        int32_t shard_rank, int32_t shard_world, int64_t *n_pairs_total,
                                        int64_t *n_pairs_local);

#ifdef __cplusplus
}
#endif
#endif /* DPGICP_H */
