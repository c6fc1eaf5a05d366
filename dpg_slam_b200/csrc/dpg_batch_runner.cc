/*
 * dpg_batch_runner.cc — batch runner: drives the scan-matching path over a whole trajectory in one
 * submission.  It takes the role of the reference's data runner (src/runner/dpg_data_runner_main.cc:
 * 38-53,95-128, which replays rosbags into the SLAM node one scan at a time) for offline data, and
 * of the two caller loops of runIcp (src/dpg_slam/dpg_slam.cc:79-107 reoptimize, 255-300
 * updatePoseGraphObsConstraints): enumerate the distance-gated pairs, submit them as ONE batch,
 * hand the records to the pose-graph update.  Host C++ only; all arithmetic of the path runs
 * behind the C ABI (include/dpgicp.h) on the GPU.
 *
 * Input is either a synthetic trajectory (--synthetic corridor|office) or a scan log (--log FILE):
 *   header  : char magic[8] = "DPGSCAN1"; int32 n_scans, n_beams; float angle_min, angle_max,
 *             range_max, laser_x, laser_y, laser_theta
 *   per scan: float pose_est[3] (x, y, theta of base_link); int32 pass; float ranges[n_beams]
 * Output: one JSON line with counts, timings and result statistics; --out FILE writes the records
 * (src, tgt, tx, ty, theta, cov[9], status) as CSV for the pose-graph side.
 *
 * --gpus N (devices 0..N-1) or --devices a,b,... runs the batch on several GPUs from this one process
 * (dpgicp_shim::MultiGpuScanMatcher): store and node table replicated, the pair list enumerated on every device with
 * its round-robin shard kept, records gathered into device a's buffer by peer stores.  The CSV is identical for any N.
 * --caller online enumerates the pairs of one updatePoseGraphObsConstraints call for the newest node instead of a
 * whole reoptimize().
 * --replay runs the reference's online loop instead of one batch (replay() below): every log scan becomes a node, is
 * appended to the scan store and aligned with its predecessor and its loop-closure candidates; a reoptimize() runs at
 * every pass boundary.  The CSV gains a leading column `update` (k, or reopt@k); the JSON line reports per-update times.
 * --inflight K (K >= 2) enumerates the pair list into K batch slots of one context and runs it in batches of
 * --batch-pairs pairs with K batches in flight (batch b on slot b % K, launched once that slot's previous batch is
 * fetched).  The CSV is identical to --inflight 1.
 * --nodes full|sync (with --replay) chooses how each alignment batch brings the node table up to date: full sends the
 * whole table (dpgicp_set_nodes), sync sends the estimates that changed since the last batch and the new node
 * (ScanMatcher::syncNodes -> dpgicp_update_nodes).  The CSV is identical for both.
 */
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "dpgicp.h"
#include "dpgicp_shim.hpp"

extern "C" {
double dpgsynth_uniform(uint64_t seed, uint64_t a, uint64_t b);
int dpgsynth_world_corridor(double x_from, double x_to, double width, double period, uint64_t seed, float *segs, int cap);
int dpgsynth_world_office(double size, int n_boxes, uint64_t seed, int variant, double moved_fraction, float *segs, int cap);
int dpgsynth_is_free(const float *segs, int nseg, double x, double y, double margin);
int dpgsynth_inside_box(const float *segs, int nseg, double x, double y);
void dpgsynth_cast_scans(const float *segs, int nseg, const double *poses, int n_scans, int n_beams, float angle_min,
                         float angle_max, float range_min, float range_max, double noise_sigma, uint64_t seed,
                         double laser_x, double laser_y, int threads, float *ranges_out);
}

namespace {

struct ScanLog {
  int32_t n_scans = 0, n_beams = 0;
  float angle_min = -2.35619449f, angle_max = 2.35619449f, range_max = 30.f, lx = 0.2f, ly = 0.f, lt = 0.f;
  std::vector<dpgicp_shim::Pose2f> est;
  std::vector<int32_t> pass;
  std::vector<float> ranges;
};

double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

bool read_log(const char *path, ScanLog &L) {
  FILE *f = std::fopen(path, "rb");
  if (!f) return false;
  char magic[8];
  bool ok = std::fread(magic, 1, 8, f) == 8 && std::memcmp(magic, "DPGSCAN1", 8) == 0;
  ok = ok && std::fread(&L.n_scans, 4, 1, f) == 1 && std::fread(&L.n_beams, 4, 1, f) == 1;
  float hdr[6];
  ok = ok && std::fread(hdr, 4, 6, f) == 6;
  if (ok) {
    L.angle_min = hdr[0]; L.angle_max = hdr[1]; L.range_max = hdr[2]; L.lx = hdr[3]; L.ly = hdr[4]; L.lt = hdr[5];
    ok = L.n_scans >= 0 && L.n_beams >= 2 && L.n_beams <= DPGICP_MAX_POINTS;
  }
  if (ok) {
    L.est.resize((size_t)L.n_scans); L.pass.resize((size_t)L.n_scans);
    L.ranges.resize((size_t)L.n_scans * (size_t)L.n_beams);
    for (int s = 0; ok && s < L.n_scans; ++s) {
      float p[3];
      ok = std::fread(p, 4, 3, f) == 3 && std::fread(&L.pass[(size_t)s], 4, 1, f) == 1 &&
           std::fread(&L.ranges[(size_t)s * (size_t)L.n_beams], 4, (size_t)L.n_beams, f) == (size_t)L.n_beams;
      L.est[(size_t)s] = {p[0], p[1], p[2]};
    }
  }
  std::fclose(f);
  return ok;
}

bool write_log(const char *path, const ScanLog &L) {
  FILE *f = std::fopen(path, "wb");
  if (!f) return false;
  std::fwrite("DPGSCAN1", 1, 8, f);
  std::fwrite(&L.n_scans, 4, 1, f); std::fwrite(&L.n_beams, 4, 1, f);
  const float hdr[6] = {L.angle_min, L.angle_max, L.range_max, L.lx, L.ly, L.lt};
  std::fwrite(hdr, 4, 6, f);
  for (int s = 0; s < L.n_scans; ++s) {
    const float p[3] = {L.est[(size_t)s].x, L.est[(size_t)s].y, L.est[(size_t)s].theta};
    std::fwrite(p, 4, 3, f); std::fwrite(&L.pass[(size_t)s], 4, 1, f);
    std::fwrite(&L.ranges[(size_t)s * (size_t)L.n_beams], 4, (size_t)L.n_beams, f);
  }
  return std::fclose(f) == 0;
}

/* hashed Gaussian (Box-Muller over dpgsynth_uniform) for odometry drift on the estimates */
double gauss(uint64_t seed, uint64_t a, uint64_t b) {
  const double u1 = dpgsynth_uniform(seed, a, 2 * b) + 1e-18, u2 = dpgsynth_uniform(seed, a, 2 * b + 1);
  return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2);
}

/* corridor trajectory in `passes` passes (BASELINE config 2 is one pass): poses 1 m apart, the
 * node gate of the reference (parameters.h:242) */
void make_synthetic(const std::string &kind, int n_scans, int n_beams, int passes, uint64_t seed, ScanLog &L) {
  L.n_scans = n_scans; L.n_beams = n_beams;
  std::vector<double> poses((size_t)n_scans * 3);
  std::vector<float> segs((size_t)4 << 16);
  int nseg;
  const int per_pass = (n_scans + passes - 1) / passes;
  if (kind == "office") {
    const double size = 40.0;
    nseg = dpgsynth_world_office(size, 60, seed, 0, 0.05, segs.data(), 1 << 16);
    double x = 0.5 * size, y = 0.5 * size, th = 0.0;
    uint64_t tries = 0;
    while (!dpgsynth_is_free(segs.data(), nseg, x, y, 0.4) || dpgsynth_inside_box(segs.data(), nseg, x, y)) {
      x = 1.0 + (size - 2.0) * dpgsynth_uniform(seed, 900, tries); y = 1.0 + (size - 2.0) * dpgsynth_uniform(seed, 901, tries); ++tries;
    }
    for (int s = 0; s < n_scans; ++s) {
      poses[3 * s] = x; poses[3 * s + 1] = y; poses[3 * s + 2] = th;
      for (int k = 0; k < 64; ++k) {
        const double nt = th + (dpgsynth_uniform(seed, (uint64_t)s, 10 + (uint64_t)k) - 0.5);
        const double nx = x + std::cos(nt), ny = y + std::sin(nt);
        if (nx > 0.5 && nx < size - 0.5 && ny > 0.5 && ny < size - 0.5 && dpgsynth_is_free(segs.data(), nseg, nx, ny, 0.35) &&
            !dpgsynth_inside_box(segs.data(), nseg, nx, ny)) { x = nx; y = ny; th = nt; break; }
        th += 1.0 + 1.5 * dpgsynth_uniform(seed, (uint64_t)s, 200 + (uint64_t)k);
      }
    }
  } else {
    nseg = dpgsynth_world_corridor(0.0, per_pass + 10.0, 2.5, 4.0, seed, segs.data(), 1 << 16);
    for (int s = 0; s < n_scans; ++s) {
      const int k = s % per_pass, pass = s / per_pass;
      const bool back = (pass & 1) != 0;                         /* odd passes drive back */
      poses[3 * s] = back ? 5.0 + (per_pass - 1 - k) : 5.0 + k;
      poses[3 * s + 1] = 0.6 * (dpgsynth_uniform(seed, (uint64_t)s, 1) - 0.5);
      poses[3 * s + 2] = (back ? M_PI : 0.0) + 0.1 * (dpgsynth_uniform(seed, (uint64_t)s, 2) - 0.5);
    }
  }
  L.ranges.resize((size_t)n_scans * (size_t)n_beams);
  dpgsynth_cast_scans(segs.data(), nseg, poses.data(), n_scans, n_beams, L.angle_min, L.angle_max, 0.02f, L.range_max,
                      0.01, seed, L.lx, L.ly, 0, L.ranges.data());
  L.est.resize((size_t)n_scans); L.pass.resize((size_t)n_scans);
  for (int s = 0; s < n_scans; ++s) {
    L.est[(size_t)s] = {(float)(poses[3 * s] + 0.05 * gauss(seed, (uint64_t)s, 5)),
                        (float)(poses[3 * s + 1] + 0.05 * gauss(seed, (uint64_t)s, 6)),
                        (float)(poses[3 * s + 2] + 0.02 * gauss(seed, (uint64_t)s, 7))};
    L.pass[(size_t)s] = s / per_pass;
  }
}

double percentile(std::vector<double> v, double q) {      /* nearest rank */
  if (v.empty()) return 0.0;
  std::sort(v.begin(), v.end());
  return v[(size_t)std::lround(q * (double)(v.size() - 1))];
}

/* The reference's runtime shape, node by node (the data runner feeds scans one at a time, runner.cc:95-128):
 *   for k = 0 .. n-1:
 *     if k > 0 and pass[k] != pass[k-1]:   reoptimize() over nodes 0..k-1   (incrementPassNumber, slam.cc:25-33)
 *     append scan k                        (createNode, dpg_slam.cc:462-513)
 *     if k >= 1: pairs of node k           (updatePoseGraphObsConstraints, dpg_slam.cc:255-314)
 * Each alignment batch is node table -> enumerate on the device -> run -> records + factors back (the hand-off to
 * addObservationConstraint).  Node estimates are the log's; a pose-graph optimiser would update them in between.  The
 * node table goes whole (set_nodes) or as the rows that changed (sync_nodes). */
int replay(const ScanLog &L, const dpgicp_params &params, float r_same, float r_other, int device, bool sync_nodes,
           const std::string &csv_out) {
  dpgicp_shim::ScanMatcher sm(device);
  dpgicp_ctx *ctx = sm.ctx();
  auto check = [&](int rc, const char *what) {
    if (rc != DPGICP_OK) throw std::runtime_error(std::string(what) + ": " + dpgicp_last_error(ctx));
  };
  std::vector<float> pose((size_t)L.n_scans * 3);
  for (int s = 0; s < L.n_scans; ++s) {
    pose[3 * (size_t)s] = L.est[(size_t)s].x; pose[3 * (size_t)s + 1] = L.est[(size_t)s].y; pose[3 * (size_t)s + 2] = L.est[(size_t)s].theta;
  }
  struct Row { int update; bool reopt; dpgicp_factor fac; dpgicp_result rec; };
  std::vector<Row> rows;
  std::vector<dpgicp_result> rec;
  std::vector<dpgicp_factor> fac;
  std::vector<double> t_append, t_nodes, t_erf, t_total;
  int n_online = 0, n_reopt = 0;
  size_t online_pairs = 0;
  /* one alignment batch over nodes 0..n_nodes-1; returns the set_nodes and the enumerate + run + fetch times */
  auto align = [&](int n_nodes, int mode, int update, double *dt_nodes, double *dt_erf) {
    const double t0 = now_s();
    if (sync_nodes) sm.syncNodes(L.est.data(), L.pass.data(), n_nodes);
    else check(dpgicp_set_nodes(ctx, pose.data(), L.pass.data(), n_nodes), "dpgicp_set_nodes");
    const double t1 = now_s();
    int64_t n = 0;
    check(dpgicp_enumerate_pairs_device(ctx, mode, r_same, r_other, 0, 1, &n, nullptr), "dpgicp_enumerate_pairs_device");
    check(dpgicp_run(ctx, &params), "dpgicp_run");
    rec.resize((size_t)n); fac.resize((size_t)n);
    check(dpgicp_fetch_results(ctx, rec.data(), n), "dpgicp_fetch_results");
    check(dpgicp_fetch_factors(ctx, fac.data(), n), "dpgicp_fetch_factors");
    const double t2 = now_s();
    *dt_nodes = t1 - t0; *dt_erf = t2 - t1;
    for (int64_t k = 0; k < n; ++k) rows.push_back({update, mode == DPGICP_ENUM_REOPTIMIZE, fac[(size_t)k], rec[(size_t)k]});
    return (size_t)n;
  };
  const double t_start = now_s();
  for (int k = 0; k < L.n_scans; ++k) {
    double dn, de;
    if (k > 0 && L.pass[(size_t)k] != L.pass[(size_t)k - 1]) { align(k, DPGICP_ENUM_REOPTIMIZE, k, &dn, &de); ++n_reopt; }
    const double a0 = now_s();
    sm.appendRanges(&L.ranges[(size_t)k * (size_t)L.n_beams], 1, L.n_beams, L.angle_min, L.angle_max, L.range_max, L.lx, L.ly, L.lt);
    const double a1 = now_s();
    if (k >= 1) {
      online_pairs += align(k + 1, DPGICP_ENUM_ONLINE, k, &dn, &de);
      t_append.push_back(a1 - a0); t_nodes.push_back(dn); t_erf.push_back(de); t_total.push_back(a1 - a0 + dn + de);
      ++n_online;
    }
  }
  const double replay_s = now_s() - t_start;
  if (!csv_out.empty()) {
    FILE *f = std::fopen(csv_out.c_str(), "w");
    if (!f) { std::fprintf(stderr, "cannot write %s\n", csv_out.c_str()); return 1; }
    std::fprintf(f, "update,src,tgt,tx,ty,theta,c00,c01,c02,c10,c11,c12,c20,c21,c22,iterations,status\n");
    for (const Row &w : rows) {
      const dpgicp_result &r = w.rec;
      std::fprintf(f, w.reopt ? "reopt@%d," : "%d,", w.update);
      std::fprintf(f, "%d,%d,%.9g,%.9g,%.9g", w.fac.to_node, w.fac.from_node, r.tx, r.ty, r.theta);
      for (int c = 0; c < 9; ++c) std::fprintf(f, ",%.17g", r.cov[c]);
      std::fprintf(f, ",%d,%u\n", r.iterations, r.status);
    }
    std::fclose(f);
  }
  auto ms = [](const std::vector<double> &v, double q) { return 1e3 * percentile(v, q); };
  std::printf("{\"mode\": \"replay\", \"nodes\": \"%s\", \"scans\": %d, \"beams\": %d, \"online_updates\": %d, \"reoptimize_batches\": %d, "
              "\"pairs\": %zu, \"online_pairs\": %zu, "
              "\"update_ms_median\": {\"append\": %.4f, \"set_nodes\": %.4f, \"enumerate_run_fetch\": %.4f, \"total\": %.4f}, "
              "\"update_ms_p90\": {\"append\": %.4f, \"set_nodes\": %.4f, \"enumerate_run_fetch\": %.4f, \"total\": %.4f}, "
              "\"replay_s\": %.6f}\n",
              sync_nodes ? "sync" : "full", L.n_scans, L.n_beams, n_online, n_reopt, rows.size(), online_pairs,
              ms(t_append, 0.5), ms(t_nodes, 0.5), ms(t_erf, 0.5), ms(t_total, 0.5),
              ms(t_append, 0.9), ms(t_nodes, 0.9), ms(t_erf, 0.9), ms(t_total, 0.9), replay_s);
  return 0;
}

}  // namespace

int main(int argc, char **argv) {
  std::string synthetic = "corridor", log_in, log_out, csv_out;
  int n_scans = 501, n_beams = 1081, passes = 1, device = 0;
  std::vector<int> devices;
  int32_t caller = DPGICP_ENUM_REOPTIMIZE;
  bool successive_only = false, replay_log = false;
  std::string nodes = "full";
  int inflight = 1;
  int64_t batch_pairs = 5000;
  uint64_t seed = 2;
  dpgicp_params params;
  dpgicp_default_params(&params);
  float r_same = 5.0f, r_other = 2.0f;                       /* parameters.h:212,224 */
  for (int i = 1; i < argc; ++i) {
    const std::string a = argv[i];
    auto next = [&](const char *what) -> const char * {
      if (i + 1 >= argc) { std::fprintf(stderr, "%s needs a value\n", what); std::exit(2); }
      return argv[++i];
    };
    if (a == "--synthetic") synthetic = next("--synthetic");
    else if (a == "--log") log_in = next("--log");
    else if (a == "--write-log") log_out = next("--write-log");
    else if (a == "--out") csv_out = next("--out");
    else if (a == "--scans") n_scans = std::atoi(next("--scans"));
    else if (a == "--beams") n_beams = std::atoi(next("--beams"));
    else if (a == "--passes") passes = std::atoi(next("--passes"));
    else if (a == "--seed") seed = (uint64_t)std::atoll(next("--seed"));
    else if (a == "--device") device = std::atoi(next("--device"));
    else if (a == "--gpus") { const int g = std::atoi(next("--gpus")); devices.clear(); for (int d = 0; d < g; ++d) devices.push_back(d); }
    else if (a == "--devices") {
      devices.clear();
      for (const char *q = next("--devices"); *q;) { devices.push_back(std::atoi(q)); while (*q && *q != ',') ++q; if (*q == ',') ++q; }
    }
    else if (a == "--caller") { const std::string c = next("--caller"); caller = c == "online" ? DPGICP_ENUM_ONLINE : DPGICP_ENUM_REOPTIMIZE; }
    else if (a == "--outlier-mode") params.outlier_mode = std::atoi(next("--outlier-mode"));
    else if (a == "--outlier-param") params.outlier_param = std::atof(next("--outlier-param"));
    else if (a == "--divisor") params.downsample_divisor = std::atoi(next("--divisor"));
    else if (a == "--cov-mode") params.cov_mode = std::atoi(next("--cov-mode"));
    else if (a == "--metric") params.metric = std::atoi(next("--metric"));
    else if (a == "--search") params.search = std::atoi(next("--search"));
    else if (a == "--window") params.projective_window = std::atoi(next("--window"));
    else if (a == "--same-pass-radius") r_same = (float)std::atof(next("--same-pass-radius"));
    else if (a == "--other-pass-radius") r_other = (float)std::atof(next("--other-pass-radius"));
    else if (a == "--successive-only") successive_only = true;
    else if (a == "--replay") replay_log = true;
    else if (a == "--nodes") nodes = next("--nodes");
    else if (a == "--inflight") inflight = std::atoi(next("--inflight"));
    else if (a == "--batch-pairs") batch_pairs = std::atoll(next("--batch-pairs"));
    else {
      std::fprintf(stderr,
                   "usage: dpg_batch_runner [--synthetic corridor|office | --log FILE] [--scans N] [--beams N] [--passes N]\n"
                   "         [--seed S] [--divisor D] [--cov-mode 0|1|2] [--metric 0|1] [--search 0|1|2] [--window W] [--successive-only]\n"
                   "         [--same-pass-radius R] [--other-pass-radius R] [--write-log FILE] [--out FILE.csv] [--device K]\n"
                   "         [--gpus N | --devices a,b,...] [--caller reoptimize|online] [--outlier-mode 0|1|2 --outlier-param X]\n"
                   "         [--replay [--nodes full|sync]] [--inflight K [--batch-pairs N]]\n");
      return a == "--help" ? 0 : 2;
    }
  }
  ScanLog L;
  if (!log_in.empty()) {
    if (!read_log(log_in.c_str(), L)) { std::fprintf(stderr, "cannot read scan log %s\n", log_in.c_str()); return 1; }
  } else {
    if (n_scans < 2 || n_beams < 2 || passes < 1) { std::fprintf(stderr, "bad sizes\n"); return 2; }
    make_synthetic(synthetic, n_scans, n_beams, passes, seed, L);
  }
  if (!log_out.empty() && !write_log(log_out.c_str(), L)) { std::fprintf(stderr, "cannot write %s\n", log_out.c_str()); return 1; }

  if (inflight < 1 || batch_pairs < 1) { std::fprintf(stderr, "dpg_batch_runner: --inflight and --batch-pairs must be >= 1\n"); return 2; }
  if (inflight > 1 && (replay_log || successive_only || !devices.empty())) {
    std::fprintf(stderr, "dpg_batch_runner: --inflight K > 1 runs the enumerated batch of one context (--device K); it is not "
                         "supported with --replay, --successive-only, --gpus or --devices\n");
    return 2;
  }
  if (nodes != "full" && (nodes != "sync" || !replay_log)) {
    std::fprintf(stderr, "dpg_batch_runner: --nodes is full or sync, and sync applies to --replay only\n");
    return 2;
  }
  if (replay_log && !devices.empty()) {
    std::fprintf(stderr, "dpg_batch_runner: --replay runs on one device (--device K); --gpus / --devices are not supported "
                         "with it (online batches are tens of pairs)\n");
    return 2;
  }

  try {
    if (replay_log) return replay(L, params, r_same, r_other, device, nodes == "sync", csv_out);
    std::vector<int32_t> src, tgt;
    std::vector<dpgicp_result> res;
    double t0, t1, t2, t3;
    if (devices.empty()) devices.push_back(device);
    if (successive_only) {
      dpgicp_shim::ScanMatcher sm(devices[0]);
      sm.params() = params;
      t0 = now_s();
      sm.uploadRanges(L.ranges, L.n_scans, L.n_beams, L.angle_min, L.angle_max, L.range_max, L.lx, L.ly, L.lt);
      t1 = now_s();
      for (int i = 1; i < L.n_scans; ++i) { src.push_back(i); tgt.push_back(i - 1); }
      t2 = now_s();
      res = sm.runIcpBatch(L.est, src, tgt);
      t3 = now_s();
    } else if (inflight > 1) {
      dpgicp_shim::ScanMatcher sm(devices[0]);
      sm.params() = params;
      t0 = now_s();
      sm.uploadRanges(L.ranges, L.n_scans, L.n_beams, L.angle_min, L.angle_max, L.range_max, L.lx, L.ly, L.lt);
      t1 = now_s();
      std::vector<float> flat((size_t)L.n_scans * 3);
      for (int i = 0; i < L.n_scans; ++i) { flat[3 * (size_t)i] = L.est[(size_t)i].x; flat[3 * (size_t)i + 1] = L.est[(size_t)i].y; flat[3 * (size_t)i + 2] = L.est[(size_t)i].theta; }
      if (dpgicp_set_nodes(sm.ctx(), flat.data(), L.pass.data(), L.n_scans) != DPGICP_OK)
        throw std::runtime_error(std::string("dpgicp_set_nodes: ") + sm.last_error());
      std::vector<std::unique_ptr<dpgicp_shim::ScanMatcher::Slot>> slots;
      int64_t n = 0;
      for (int k = 0; k < inflight; ++k) {
        slots.emplace_back(new dpgicp_shim::ScanMatcher::Slot(sm));
        n = slots.back()->enumeratePairs(caller, r_same, r_other);
      }
      t2 = now_s();
      res.resize((size_t)n);
      std::vector<int64_t> pending((size_t)inflight, -1);         /* first pair of the batch each slot has in flight */
      auto fetch = [&](int k) {
        const int64_t f = pending[(size_t)k];
        if (f >= 0) slots[(size_t)k]->fetchResults(&res[(size_t)f], f, std::min(batch_pairs, n - f));
        pending[(size_t)k] = -1;
      };
      for (int64_t first = 0, b = 0; first < n; first += batch_pairs, ++b) {
        const int k = (int)(b % inflight);
        fetch(k);
        slots[(size_t)k]->runRange(first, std::min(batch_pairs, n - first));
        pending[(size_t)k] = first;
      }
      for (int k = 0; k < inflight; ++k) fetch(k);
      t3 = now_s();
      slots[0]->pairs(src, tgt, n);
    } else {
      /* the callers' form: nodes in, pair list enumerated and kept on the device(s), records gathered back */
      dpgicp_shim::MultiGpuScanMatcher sm(devices);
      sm.params() = params;
      t0 = now_s();
      sm.uploadRanges(L.ranges, L.n_scans, L.n_beams, L.angle_min, L.angle_max, L.range_max, L.lx, L.ly, L.lt);
      t1 = now_s();
      sm.setNodes(L.est, L.pass);
      sm.enumeratePairs(caller, r_same, r_other);
      t2 = now_s();
      res = sm.runIcpBatch();
      t3 = now_s();
      sm.pairs(src, tgt);
    }
    size_t converged = 0, singular = 0;
    double it_sum = 0;
    for (const dpgicp_result &r : res) {
      converged += (r.status & DPGICP_FLAG_CONVERGED) ? 1 : 0;
      singular += (r.status & DPGICP_FLAG_COV_SINGULAR) ? 1 : 0;
      it_sum += r.iterations;
    }
    if (!csv_out.empty()) {
      FILE *f = std::fopen(csv_out.c_str(), "w");
      if (!f) { std::fprintf(stderr, "cannot write %s\n", csv_out.c_str()); return 1; }
      std::fprintf(f, "src,tgt,tx,ty,theta,c00,c01,c02,c10,c11,c12,c20,c21,c22,iterations,status\n");
      for (size_t k = 0; k < res.size(); ++k) {
        const dpgicp_result &r = res[k];
        std::fprintf(f, "%d,%d,%.9g,%.9g,%.9g", src[k], tgt[k], r.tx, r.ty, r.theta);
        for (int c = 0; c < 9; ++c) std::fprintf(f, ",%.17g", r.cov[c]);
        std::fprintf(f, ",%d,%u\n", r.iterations, r.status);
      }
      std::fclose(f);
    }
    std::printf("{\"scans\": %d, \"beams\": %d, \"gpus\": %zu, \"inflight\": %d, \"pairs\": %zu, \"converged\": %zu, \"cov_singular\": %zu, "
                "\"mean_iterations\": %.2f, \"upload_s\": %.6f, \"enumerate_s\": %.6f, \"icp_cov_s\": %.6f, "
                "\"pairs_per_s\": %.1f}\n",
                L.n_scans, L.n_beams, devices.size(), inflight, res.size(), converged, singular, res.empty() ? 0.0 : it_sum / (double)res.size(),
                t1 - t0, t2 - t1, t3 - t2, res.empty() ? 0.0 : (double)res.size() / (t3 - t2));
  } catch (const std::exception &e) {
    std::fprintf(stderr, "dpg_batch_runner: %s\n", e.what());
    return 1;
  }
  return 0;
}
