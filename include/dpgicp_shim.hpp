/*
 * dpgicp_shim.hpp — header-only C++ shim that re-exposes the reference's two call shapes on top
 * of the C ABI (dpgicp.h), on plain arrays laid out like the reference's PCL/Eigen types:
 *
 *   bool DpgSLAM::runIcp(DpgNode &node_1, DpgNode &node_2,
 *                        std::pair<std::pair<Eigen::Vector2f,float>, Eigen::MatrixXd> &icp_results)
 *                                             (reference src/dpg_slam/dpg_slam.h:630, dpg_slam.cc:362-446)
 *   void calculate_ICP_COV(cloud data_pi, cloud model_qi, Eigen::Matrix4f &transform,
 *                          Eigen::MatrixXd &ICP_COV, float sx2, float sy2, float st2)
 *                                             (reference src/icp_cov/cov_func_point_to_point.h:24)
 *
 * PCL/Eigen are not needed to compile this header: PointXYZ below has pcl::PointXYZ's 16-byte
 * layout {x, y, z, pad}, Matrix4f is 16 column-major floats, the covariance is 9 doubles
 * (row-major == column-major by symmetry).  INTEGRATION.md shows the three-line adapter from the
 * real PCL/Eigen types.
 */
#ifndef DPGICP_SHIM_HPP
#define DPGICP_SHIM_HPP

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <functional>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "dpgicp.h"

namespace dpgicp_shim {

struct alignas(16) PointXYZ {   /* == pcl::PointXYZ memory layout */
  float x, y, z, pad;
};
using Cloud = std::vector<PointXYZ>;

struct Pose2f {                 /* node estimate: DpgNode::getEstimatedPosition() */
  float x, y, theta;
};

struct IcpResults {             /* the reference's pair<pair<Vector2f,float>, MatrixXd> flattened */
  float tx = 0, ty = 0, theta = 0;
  double cov[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  dpgicp_result record{};
};

/* The node table a context was last sent by syncNodes.  diff() lists the rows of a new estimate vector whose bits
 * differ from it, then the new rows; it asks for the whole table instead (returns true) when there is no table yet,
 * the vector is shorter, or more than kFullShare of its rows would go. */
class NodeMirror {
 public:
  /* update_nodes costs host work per listed row, set_nodes per node; at 50 000 nodes on an NVIDIA B200 (1000 W,
   * 1965 MHz) update_nodes takes 0.37 ms for 25 % of the rows and 0.65 ms for 50 % against 0.47-0.49 ms for set_nodes
   * (profiles/online_nodes.json, "share": measured through the Python wrapper, which has the same threshold) */
  static constexpr double kFullShare = 0.3;
  bool diff(const Pose2f *poses, const int32_t *pass, int32_t n, std::vector<int32_t> &ids, std::vector<float> &flat,
            std::vector<int32_t> &ids_pass) const {
    ids.clear(); flat.clear(); ids_pass.clear();
    if (!valid_ || (size_t)n < pose_.size()) return true;
    const int32_t m = (int32_t)pose_.size();
    auto same = [&](int32_t i, int32_t k) {      /* rows i .. i + k - 1, bit for bit */
      return i + k <= m && std::memcmp(&poses[i], &pose_[(size_t)i], sizeof(Pose2f) * (size_t)k) == 0 &&
             std::memcmp(&pass[i], &pass_[(size_t)i], sizeof(int32_t) * (size_t)k) == 0;
    };
    for (int32_t b = 0; b < n; b += 256) {      /* whole blocks first: an unchanged block costs two memcmp */
      const int32_t e = std::min(n, b + 256);
      if (same(b, e - b)) continue;
      for (int32_t i = b; i < e; ++i) {
        if (same(i, 1)) continue;
        ids.push_back(i);
        if ((double)ids.size() > kFullShare * n) return true;
        flat.insert(flat.end(), {poses[i].x, poses[i].y, poses[i].theta});
        ids_pass.push_back(pass[i]);
      }
    }
    return false;
  }
  /* after the table was sent: the whole vector (full) or the rows diff() listed */
  void commit(const Pose2f *poses, const int32_t *pass, int32_t n, bool full, const std::vector<int32_t> &ids) {
    if (full) {
      pose_.assign(poses, poses + n); pass_.assign(pass, pass + n);
    } else {
      pose_.resize((size_t)n); pass_.resize((size_t)n);
      for (int32_t i : ids) { pose_[(size_t)i] = poses[i]; pass_[(size_t)i] = pass[i]; }
    }
    valid_ = true;
  }
  void clear() { valid_ = false; pose_.clear(); pass_.clear(); }

 private:
  bool valid_ = false;
  std::vector<Pose2f> pose_;
  std::vector<int32_t> pass_;
};

inline std::vector<float> flatten(const Pose2f *poses, size_t n) {
  std::vector<float> flat(n * 3);
  for (size_t i = 0; i < n; ++i) { flat[3 * i] = poses[i].x; flat[3 * i + 1] = poses[i].y; flat[3 * i + 2] = poses[i].theta; }
  return flat;
}

class ScanMatcher {
 public:
  explicit ScanMatcher(int device = 0) {
    int rc = dpgicp_create(device, &ctx_);
    if (rc != DPGICP_OK) throw std::runtime_error(std::string("dpgicp_create: ") + dpgicp_last_error(nullptr));
    dpgicp_default_params(&params_);
  }
  ~ScanMatcher() { dpgicp_destroy(ctx_); }
  ScanMatcher(const ScanMatcher &) = delete;
  ScanMatcher &operator=(const ScanMatcher &) = delete;

  dpgicp_params &params() { return params_; }   /* PoseGraphParameters' ICP fields, parameters.h */
  dpgicp_ctx *ctx() { return ctx_; }
  const char *last_error() const { return dpgicp_last_error(ctx_); }

  /* runIcp: source = node_2, target = node_1, guess from the two pose estimates
   * (dpg_slam.cc:364-378).  Returns icp.hasConverged() (dpg_slam.cc:445).  Unlike the reference's
   * early `return false` (dpg_slam.cc:422-426) the result is always written.  A library/CUDA
   * failure is reported like a non-converged alignment (false) with last_error() set. */
  bool runIcp(const Cloud &node_1_cloud, const Pose2f &node_1_pose, const Cloud &node_2_cloud,
              const Pose2f &node_2_pose, IcpResults &icp_results) {
    const float p1[3] = {node_1_pose.x, node_1_pose.y, node_1_pose.theta};
    const float p2[3] = {node_2_pose.x, node_2_pose.y, node_2_pose.theta};
    float guess[3];
    dpgicp_relative_guess(p1, p2, guess);
    dpgicp_result r{};
    int rc = dpgicp_single_pair(ctx_, node_2_cloud.data(), (int32_t)node_2_cloud.size(), node_1_cloud.data(),
                                (int32_t)node_1_cloud.size(), sizeof(PointXYZ), guess, &params_, &r);
    if (rc != DPGICP_OK) return false;
    icp_results.tx = r.tx; icp_results.ty = r.ty; icp_results.theta = r.theta;
    for (int k = 0; k < 9; ++k) icp_results.cov[k] = r.cov[k];
    icp_results.record = r;
    return (r.status & DPGICP_FLAG_CONVERGED) != 0;
  }

  /* calculate_ICP_COV with the reference's argument order.  transform = Matrix4f column-major. */
  void calculate_ICP_COV(const Cloud &data_pi, const Cloud &model_qi, const float transform[16], double ICP_COV[9],
                         float laser_x_variance, float laser_y_variance, float laser_theta_variance) {
    dpgicp_params p = params_;
    p.laser_x_variance = laser_x_variance;
    p.laser_y_variance = laser_y_variance;
    p.laser_theta_variance = laser_theta_variance;
    if (p.cov_mode == DPGICP_COV_CENSI_CORR) p.cov_mode = DPGICP_COV_CENSI_INDEXPAIR;
    uint32_t status = 0;
    int rc = dpgicp_cov(ctx_, data_pi.data(), (int32_t)data_pi.size(), model_qi.data(), (int32_t)model_qi.size(),
                        sizeof(PointXYZ), transform, &p, ICP_COV, &status);
    if (rc != DPGICP_OK) throw std::runtime_error(std::string("dpgicp_cov: ") + last_error());
  }

  /* Batch form of the callers' loops (dpg_slam.cc:79-107, 255-300): pairs are independent until
   * optimizeGraph (dpg_slam.cc:119,313), so enumerate -> one submit -> addObservationConstraint. */
  void uploadRanges(const std::vector<float> &ranges, int n_scans, int n_beams, float angle_min, float angle_max,
                    float range_max, float lx = 0.2f, float ly = 0.0f, float ltheta = 0.0f) {
    check(dpgicp_upload_ranges(ctx_, ranges.data(), n_scans, n_beams, angle_min, angle_max, range_max, lx, ly, ltheta),
          "dpgicp_upload_ranges");
  }
  void uploadClouds(const std::vector<Cloud> &clouds) {
    std::vector<PointXYZ> all;
    std::vector<int64_t> off(1, 0);
    for (const Cloud &c : clouds) { all.insert(all.end(), c.begin(), c.end()); off.push_back((int64_t)all.size()); }
    check(dpgicp_upload_scans(ctx_, all.data(), sizeof(PointXYZ), off.data(), (int32_t)clouds.size()),
          "dpgicp_upload_scans");
  }
  /* online form (createNode, dpg_slam.cc:462-513): the new node's scan(s) become the next rows of the store, earlier
   * rows stay on the device; n_scans * n_beams floats at `ranges` */
  void appendRanges(const float *ranges, int n_scans, int n_beams, float angle_min, float angle_max, float range_max,
                    float lx = 0.2f, float ly = 0.0f, float ltheta = 0.0f) {
    check(dpgicp_append_ranges(ctx_, ranges, n_scans, n_beams, angle_min, angle_max, range_max, lx, ly, ltheta),
          "dpgicp_append_ranges");
  }
  void appendClouds(const std::vector<Cloud> &clouds) {
    std::vector<PointXYZ> all;
    std::vector<int64_t> off(1, 0);
    for (const Cloud &c : clouds) { all.insert(all.end(), c.begin(), c.end()); off.push_back((int64_t)all.size()); }
    check(dpgicp_append_scans(ctx_, all.data(), sizeof(PointXYZ), off.data(), (int32_t)clouds.size()),
          "dpgicp_append_scans");
  }
  /* node ids[k] takes poses[k] and pass[k]; the table then holds n_nodes nodes (dpgicp_update_nodes) */
  void updateNodes(int32_t n_nodes, const std::vector<int32_t> &ids, const std::vector<Pose2f> &poses,
                   const std::vector<int32_t> &pass) {
    if (poses.size() != ids.size() || pass.size() != ids.size()) throw std::runtime_error("updateNodes: length mismatch");
    mirror_.clear();
    const std::vector<float> flat = flatten(poses.data(), poses.size());
    check(dpgicp_update_nodes(ctx_, n_nodes, ids.data(), flat.data(), pass.data(), (int32_t)ids.size()), "dpgicp_update_nodes");
  }
  /* the whole estimate vector after calculateEstimate(): only the rows that changed since the last syncNodes, and the
   * new ones, go to the device; the first call, or one where most rows changed, sends the whole table.  The diff is
   * taken against what the last syncNodes sent, so syncNodes (or updateNodes, after which the next syncNodes sends
   * everything) must be the only writer of the table: dpgicp_set_nodes / dpgicp_update_nodes called on ctx()
   * directly are not seen, and the next syncNodes would diff against a stale table. */
  void syncNodes(const Pose2f *poses, const int32_t *pass, int32_t n_nodes) {
    std::vector<int32_t> ids, ids_pass;
    std::vector<float> flat;
    const bool full = mirror_.diff(poses, pass, n_nodes, ids, flat, ids_pass);
    mirror_.clear();
    if (full) {
      const std::vector<float> all = flatten(poses, (size_t)n_nodes);
      check(dpgicp_set_nodes(ctx_, all.data(), pass, n_nodes), "dpgicp_set_nodes");
    } else {
      check(dpgicp_update_nodes(ctx_, n_nodes, ids.data(), flat.data(), ids_pass.data(), (int32_t)ids.size()),
            "dpgicp_update_nodes");
    }
    mirror_.commit(poses, pass, n_nodes, full, ids);
  }
  void syncNodes(const std::vector<Pose2f> &poses, const std::vector<int32_t> &pass) {
    if (pass.size() != poses.size()) throw std::runtime_error("syncNodes: length mismatch");
    syncNodes(poses.data(), pass.data(), (int32_t)poses.size());
  }
  /* node poses -> (source, target) list of one reoptimize() */
  void enumeratePairs(const std::vector<Pose2f> &poses, const std::vector<int32_t> &pass, float same_pass_radius,
                      float other_pass_radius, std::vector<int32_t> &src, std::vector<int32_t> &tgt) {
    std::vector<float> xy(poses.size() * 2);
    for (size_t i = 0; i < poses.size(); ++i) { xy[2 * i] = poses[i].x; xy[2 * i + 1] = poses[i].y; }
    int64_t n = 0;
    int rc = dpgicp_enumerate_pairs(ctx_, xy.data(), pass.data(), (int32_t)poses.size(), same_pass_radius,
                                    other_pass_radius, nullptr, nullptr, &n);
    if (rc != DPGICP_OK && rc != DPGICP_E_TOOBIG) check(rc, "dpgicp_enumerate_pairs");
    src.assign((size_t)n, 0); tgt.assign((size_t)n, 0);
    if (n > 0)
      check(dpgicp_enumerate_pairs(ctx_, xy.data(), pass.data(), (int32_t)poses.size(), same_pass_radius,
                                   other_pass_radius, src.data(), tgt.data(), &n), "dpgicp_enumerate_pairs");
  }
  /* guesses from node estimates, then one batched submit */
  std::vector<dpgicp_result> runIcpBatch(const std::vector<Pose2f> &poses, const std::vector<int32_t> &src,
                                         const std::vector<int32_t> &tgt) {
    std::vector<float> guess(src.size() * 3);
    for (size_t k = 0; k < src.size(); ++k) {
      const Pose2f &a = poses[(size_t)tgt[k]], &b = poses[(size_t)src[k]];
      const float p1[3] = {a.x, a.y, a.theta}, p2[3] = {b.x, b.y, b.theta};
      dpgicp_relative_guess(p1, p2, &guess[3 * k]);
    }
    std::vector<dpgicp_result> out(src.size());
    check(dpgicp_submit_pairs(ctx_, src.data(), tgt.data(), guess.data(), (int64_t)src.size(), &params_, out.data()),
          "dpgicp_submit_pairs");
    return out;
  }
  /* the batch just run as pose-graph factors: BetweenFactor<Pose2>(from, to, Pose2(tx, ty, theta),
   * noiseModel::Gaussian::SqrtInformation(R)) — addObservationConstraint, dpg_slam.cc:331-338 */
  std::vector<dpgicp_factor> factors(size_t n) {
    std::vector<dpgicp_factor> out(n);
    check(dpgicp_fetch_factors(ctx_, out.data(), (int64_t)n), "dpgicp_fetch_factors");
    return out;
  }

  /* One more batch in flight over this matcher's scan store (dpgicp_slot_*): run() returns at once, the fetches wait
   * for this slot's batch only.  Must not outlive its ScanMatcher. */
  class Slot {
   public:
    explicit Slot(ScanMatcher &sm) : sm_(sm) { sm_.check(dpgicp_slot_create(sm_.ctx_, &slot_), "dpgicp_slot_create"); }
    ~Slot() { dpgicp_slot_destroy(slot_); }
    Slot(const Slot &) = delete;
    Slot &operator=(const Slot &) = delete;

    dpgicp_slot *get() { return slot_; }
    void setPairs(const std::vector<int32_t> &src, const std::vector<int32_t> &tgt, const std::vector<float> &guess) {
      if (tgt.size() != src.size() || guess.size() != 3 * src.size()) throw std::runtime_error("Slot::setPairs: length mismatch");
      sm_.check(dpgicp_slot_set_pairs(slot_, src.data(), tgt.data(), guess.data(), (int64_t)src.size()), "dpgicp_slot_set_pairs");
    }
    /* the caller's pair list built on the device into this slot; returns the local pair count */
    int64_t enumeratePairs(int32_t mode, float same_pass_radius, float other_pass_radius) {
      int64_t n = 0;
      sm_.check(dpgicp_slot_enumerate_pairs_device(slot_, mode, same_pass_radius, other_pass_radius, 0, 1, nullptr, &n),
                "dpgicp_slot_enumerate_pairs_device");
      return n;
    }
    void run() { sm_.check(dpgicp_slot_run(slot_, &sm_.params_), "dpgicp_slot_run"); }
    void runRange(int64_t first, int64_t count) {
      sm_.check(dpgicp_slot_run_range(slot_, &sm_.params_, first, count), "dpgicp_slot_run_range");
    }
    void fetchResults(dpgicp_result *out, int64_t first, int64_t count) {
      sm_.check(dpgicp_slot_fetch_results_range(slot_, out, first, count), "dpgicp_slot_fetch_results_range");
    }
    std::vector<dpgicp_factor> factors(size_t n) {
      std::vector<dpgicp_factor> out(n);
      sm_.check(dpgicp_slot_fetch_factors(slot_, out.data(), (int64_t)n), "dpgicp_slot_fetch_factors");
      return out;
    }
    void pairs(std::vector<int32_t> &src, std::vector<int32_t> &tgt, int64_t n) {
      src.assign((size_t)n, 0); tgt.assign((size_t)n, 0);
      sm_.check(dpgicp_slot_fetch_pairs(slot_, src.data(), tgt.data(), nullptr, n), "dpgicp_slot_fetch_pairs");
    }
    bool done() {
      const int rc = dpgicp_slot_query(slot_);
      if (rc < 0) sm_.check(rc, "dpgicp_slot_query");
      return rc == 1;
    }
    void synchronize() { sm_.check(dpgicp_slot_synchronize(slot_), "dpgicp_slot_synchronize"); }

   private:
    ScanMatcher &sm_;
    dpgicp_slot *slot_ = nullptr;
  };

 private:
  void check(int rc, const char *what) {
    if (rc != DPGICP_OK) throw std::runtime_error(std::string(what) + ": " + last_error());
  }
  dpgicp_ctx *ctx_ = nullptr;
  dpgicp_params params_{};
  NodeMirror mirror_;
};

/* ------------------------------------------------------------------------------------------------
 * The batch form of the two callers on G GPUs of one box, driven from ONE host process in C++ (the role of the
 * reference's data runner, src/runner/dpg_data_runner_main.cc:95-128, and of DpgSLAM::reoptimize /
 * updatePoseGraphObsConstraints, dpg_slam.cc:35-120, 255-314).  One dpgicp context per device; the scan store and
 * the node table are replicated; the pair list is enumerated ON every device, each keeping its round-robin shard
 * (global pair k -> context k % G); the records are gathered by peer stores from the kernels' epilogues into
 * context 0's buffer (dpgicp_gather_attach_local, no collective, no host interleave).  The same device may be listed
 * more than once (two contexts on one GPU), which is how a single-GPU box exercises this path.
 * ---------------------------------------------------------------------------------------------- */
class MultiGpuScanMatcher {
 public:
  explicit MultiGpuScanMatcher(const std::vector<int> &devices) {
    if (devices.empty() || devices.size() > DPGICP_MAX_GATHER_RANKS) throw std::runtime_error("MultiGpuScanMatcher: 1..16 devices");
    for (int d : devices) {
      dpgicp_ctx *c = nullptr;
      if (dpgicp_create(d, &c) != DPGICP_OK) {
        const std::string msg = dpgicp_last_error(nullptr);
        for (dpgicp_ctx *q : ctx_) dpgicp_destroy(q);
        throw std::runtime_error("dpgicp_create(device " + std::to_string(d) + "): " + msg);
      }
      ctx_.push_back(c);
    }
    dpgicp_default_params(&params_);
  }
  ~MultiGpuScanMatcher() {
    for (dpgicp_ctx *c : ctx_) dpgicp_gather_detach(c);
    for (dpgicp_ctx *c : ctx_) dpgicp_destroy(c);
  }
  MultiGpuScanMatcher(const MultiGpuScanMatcher &) = delete;
  MultiGpuScanMatcher &operator=(const MultiGpuScanMatcher &) = delete;

  dpgicp_params &params() { return params_; }
  int world() const { return (int)ctx_.size(); }
  dpgicp_ctx *ctx(int r) { return ctx_[(size_t)r]; }

  /* replicate the scan store (raw ranges, converted on each device) */
  void uploadRanges(const std::vector<float> &ranges, int n_scans, int n_beams, float angle_min, float angle_max,
                    float range_max, float lx = 0.2f, float ly = 0.0f, float ltheta = 0.0f) {
    each([&](int r) {
      return dpgicp_upload_ranges(ctx_[(size_t)r], ranges.data(), n_scans, n_beams, angle_min, angle_max, range_max, lx, ly, ltheta);
    }, "dpgicp_upload_ranges");
  }
  /* node estimates (DpgNode::getEstimatedPosition) and pass numbers; node k owns scan k */
  void setNodes(const std::vector<Pose2f> &poses, const std::vector<int32_t> &pass) {
    mirror_.clear();
    const std::vector<float> flat = flatten(poses.data(), poses.size());
    each([&](int r) { return dpgicp_set_nodes(ctx_[(size_t)r], flat.data(), pass.data(), (int32_t)poses.size()); }, "dpgicp_set_nodes");
  }
  /* ScanMatcher::updateNodes / syncNodes on every context (syncNodes: the same only-writer rule, for every ctx(r)) */
  void updateNodes(int32_t n_nodes, const std::vector<int32_t> &ids, const std::vector<Pose2f> &poses,
                   const std::vector<int32_t> &pass) {
    if (poses.size() != ids.size() || pass.size() != ids.size()) throw std::runtime_error("updateNodes: length mismatch");
    mirror_.clear();
    const std::vector<float> flat = flatten(poses.data(), poses.size());
    each([&](int r) { return dpgicp_update_nodes(ctx_[(size_t)r], n_nodes, ids.data(), flat.data(), pass.data(), (int32_t)ids.size()); },
         "dpgicp_update_nodes");
  }
  void syncNodes(const std::vector<Pose2f> &poses, const std::vector<int32_t> &pass) {
    if (pass.size() != poses.size()) throw std::runtime_error("syncNodes: length mismatch");
    const int32_t n = (int32_t)poses.size();
    std::vector<int32_t> ids, ids_pass;
    std::vector<float> flat;
    const bool full = mirror_.diff(poses.data(), pass.data(), n, ids, flat, ids_pass);
    mirror_.clear();
    if (full) {
      flat = flatten(poses.data(), poses.size());
      each([&](int r) { return dpgicp_set_nodes(ctx_[(size_t)r], flat.data(), pass.data(), n); }, "dpgicp_set_nodes");
    } else {
      each([&](int r) { return dpgicp_update_nodes(ctx_[(size_t)r], n, ids.data(), flat.data(), ids_pass.data(), (int32_t)ids.size()); },
           "dpgicp_update_nodes");
    }
    mirror_.commit(poses.data(), pass.data(), n, full, ids);
  }
  /* the caller's pair list (DPGICP_ENUM_REOPTIMIZE / _ONLINE) built on every device; returns the global pair count */
  int64_t enumeratePairs(int32_t mode, float same_pass_radius, float other_pass_radius) {
    std::vector<int64_t> total(ctx_.size(), 0);
    local_.assign(ctx_.size(), 0);
    each([&](int r) {
      return dpgicp_enumerate_pairs_device(ctx_[(size_t)r], mode, same_pass_radius, other_pass_radius, r, world(),
                                           &total[(size_t)r], &local_[(size_t)r]);
    }, "dpgicp_enumerate_pairs_device");
    n_total_ = total[0];
    return n_total_;
  }
  /* align every pair: all devices run concurrently; records land in context 0's gather buffer in global order */
  std::vector<dpgicp_result> runIcpBatch() {
    std::vector<dpgicp_result> out((size_t)n_total_);
    if (n_total_ == 0) return out;
    if (world() > 1 && dpgicp_gather_attach_local(ctx_.data(), world(), n_total_, /*root_only=*/1) != DPGICP_OK)
      throw std::runtime_error(std::string("dpgicp_gather_attach_local: ") + first_error());
    for (int r = 0; r < world(); ++r)                      /* dpgicp_run only launches: one thread starts them all */
      if (dpgicp_run(ctx_[(size_t)r], &params_) != DPGICP_OK) throw std::runtime_error(std::string("dpgicp_run: ") + dpgicp_last_error(ctx_[(size_t)r]));
    for (int r = 0; r < world(); ++r)
      if (dpgicp_synchronize(ctx_[(size_t)r]) != DPGICP_OK) throw std::runtime_error(std::string("dpgicp_synchronize: ") + dpgicp_last_error(ctx_[(size_t)r]));
    const int rc = world() > 1 ? dpgicp_gather_fetch(ctx_[0], out.data(), n_total_) : dpgicp_fetch_results(ctx_[0], out.data(), n_total_);
    if (rc != DPGICP_OK) throw std::runtime_error(std::string("fetch records: ") + dpgicp_last_error(ctx_[0]));
    return out;
  }
  /* the global pair list (source, target node per pair) in the reference's loop order */
  void pairs(std::vector<int32_t> &src, std::vector<int32_t> &tgt) {
    src.assign((size_t)n_total_, 0); tgt.assign((size_t)n_total_, 0);
    for (int r = 0; r < world(); ++r) {
      const int64_t n = local_[(size_t)r];
      std::vector<int32_t> s((size_t)n), t((size_t)n);
      if (dpgicp_fetch_pairs(ctx_[(size_t)r], s.data(), t.data(), nullptr, n) != DPGICP_OK)
        throw std::runtime_error(std::string("dpgicp_fetch_pairs: ") + dpgicp_last_error(ctx_[(size_t)r]));
      for (int64_t k = 0; k < n; ++k) { src[(size_t)(r + k * world())] = s[(size_t)k]; tgt[(size_t)(r + k * world())] = t[(size_t)k]; }
    }
  }

 private:
  /* the same host-side call on every context, one thread per context (a context is single-owner, contexts are independent) */
  void each(const std::function<int(int)> &fn, const char *what) {
    std::vector<int> rc(ctx_.size(), 0);
    if (ctx_.size() == 1) {
      rc[0] = fn(0);
    } else {
      std::vector<std::thread> th;
      for (int r = 0; r < world(); ++r) th.emplace_back([&, r] { rc[(size_t)r] = fn(r); });
      for (std::thread &t : th) t.join();
    }
    for (int r = 0; r < world(); ++r)
      if (rc[(size_t)r] != DPGICP_OK) throw std::runtime_error(std::string(what) + " (context " + std::to_string(r) + "): " + dpgicp_last_error(ctx_[(size_t)r]));
  }
  const char *first_error() {
    for (dpgicp_ctx *c : ctx_) if (dpgicp_last_error(c)[0]) return dpgicp_last_error(c);
    return "";
  }
  std::vector<dpgicp_ctx *> ctx_;
  std::vector<int64_t> local_;
  int64_t n_total_ = 0;
  dpgicp_params params_{};
  NodeMirror mirror_;
};

}  // namespace dpgicp_shim
#endif
