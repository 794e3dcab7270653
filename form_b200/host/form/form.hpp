// form::Estimator - the FORM front end, B200 build.
//
// Same public surface as the reference's form.hpp
// (/root/reference/form/form.hpp:40-84): struct Estimator with nested Params
// {extraction, matcher, constraints, scans, map, num_threads}, public members
// m_params / m_extractor / m_constraints / m_matcher / m_keyscanner /
// m_keypoint_map, current_lidar_estimate() and
//   std::tuple<std::vector<PlanarFeat>, std::vector<PointFeat>>
//   register_scan(const std::vector<PointXYZf>&) noexcept
// with the stage order of /root/reference/form/form.cpp:40-114.  Everything
// data-parallel (extraction, map rebuild, matching, linearisation, map insert)
// is executed by the HotPath (the CUDA library); the dense fixed-lag smoother
// and the key-scan bookkeeping stay on the host.
//
// Differences a maintainer should know (see INTEGRATION.md):
//   * poses are form::Pose3 (pose3.hpp) instead of gtsam::Pose3;
//   * m_matcher / m_keypoint_map are thin handles: the matches and the keypoint
//     maps live in device memory and are reached through them;
//   * a failure inside the hot path (bad scan size, CUDA error) is recorded in
//     last_error() and register_scan returns empty keypoints instead of
//     std::terminate (the reference throws through a noexcept function).
#pragma once

#include "form/constraints.hpp"
// FORM_HOTPATH_INJECTED_ONLY (test infrastructure: the oracle library): the estimator only ever
// runs over an injected HotPath and the translation unit must not reference the CUDA library.
#ifndef FORM_HOTPATH_INJECTED_ONLY
#include "form/gpu_hotpath.hpp"
#endif
#include "form/hotpath.hpp"
#include "form/keyscanner.hpp"
#include "form/pose3.hpp"
#include "form/types.hpp"

#include <memory>
#include <string>
#include <tuple>
#include <vector>

namespace form {

/// form::MatcherParams, matcher.hpp:32-41
struct MatcherParams {
  double max_dist_matching = 0.8;
  double new_pose_threshold = 1e-4;
  size_t max_num_rematches = 30;
};

/// form::KeypointMapParams, map.hpp:97-100
struct KeypointMapParams {
  double min_dist_map = 0.1;
};

/// form::FeatureExtractor, extraction.hpp:57-101: same Params, same extract().
class FeatureExtractor {
public:
  struct Params {
    size_t neighbor_points = 5;
    size_t num_sectors = 6;
    double planar_threshold = 1.0;
    size_t planar_feats_per_sector = 50;
    size_t point_feats_per_sector = 3;
    double radius = 1.0;
    size_t min_points = 5;
    double min_norm_squared = 1.0;
    double max_norm_squared = 100.0 * 100.0;
    int num_columns = 1024;
    int num_rows = 64;
  };

  Params params;

  explicit FeatureExtractor(const Params &params_, size_t num_threads = 0)
      : params(params_), m_num_threads(num_threads) {}

  /// Shares the Estimator's hot path; a stand-alone extractor creates its own
  /// CUDA context on first use.
  void set_hotpath(std::shared_ptr<HotPath> hp) { m_hotpath = std::move(hp); }

  template <typename Point>
  [[nodiscard]] std::tuple<std::vector<PlanarFeat>, std::vector<PointFeat>>
  extract(const std::vector<Point> &scan, size_t scan_idx) const {
    static_assert(sizeof(Point) == sizeof(PointXYZf), "scan points must be 16-byte x,y,z,_ floats");
    if (!m_hotpath) {
#ifndef FORM_HOTPATH_INJECTED_ONLY
      HotPathParams hp;
      fill(hp);
      m_hotpath = std::make_shared<GpuHotPath>(hp, 0, nullptr, 2);
#else
      throw HotPathError("FeatureExtractor: no hot path injected");
#endif
    }
    std::vector<PlanarFeat> planar;
    std::vector<PointFeat> point;
    m_hotpath->extract(reinterpret_cast<const PointXYZf *>(scan.data()), scan.size(), scan_idx, planar,
                       point);
    return std::make_tuple(std::move(planar), std::move(point));
  }

  void fill(HotPathParams &hp) const {
    hp.neighbor_points = params.neighbor_points;
    hp.num_sectors = params.num_sectors;
    hp.planar_threshold = params.planar_threshold;
    hp.planar_feats_per_sector = params.planar_feats_per_sector;
    hp.point_feats_per_sector = params.point_feats_per_sector;
    hp.radius = params.radius;
    hp.min_points = params.min_points;
    hp.min_norm_squared = params.min_norm_squared;
    hp.max_norm_squared = params.max_norm_squared;
    hp.num_columns = params.num_columns;
    hp.num_rows = params.num_rows;
    hp.num_threads = m_num_threads;
  }

private:
  size_t m_num_threads;
  mutable std::shared_ptr<HotPath> m_hotpath;
};

/// Handle standing in for form::Matcher<Point> (matcher.hpp:44-115): parameters
/// on the host, matches in device memory.
struct MatcherHandle {
  MatcherParams m_params;
};

/// Handle standing in for the tuple of form::KeypointMap (map.hpp:108-143).
struct KeypointMapHandle {
  KeypointMapParams m_params;
  std::shared_ptr<HotPath> hotpath;
  /// to_voxel_map(values, .) flattened: every stored keypoint in the world frame
  /// (what FORM::map() iterates, bindings.cpp:96-119).
  void world_keypoints(const Values &values, std::vector<PlanarFeat> &planar,
                       std::vector<PointFeat> &point) const {
    std::vector<ScanPose> poses;
    for (const auto &kv : values) poses.push_back({kv.first, kv.second});
    hotpath->world_keypoints(poses.data(), poses.size(), planar, point);
  }
};

struct Estimator {
  struct Params {
    FeatureExtractor::Params extraction;
    MatcherParams matcher;
    ConstraintManager::Params constraints;
    KeyScanner::Params scans;
    KeypointMapParams map;
    size_t num_threads = 0;
    int device = 0; // CUDA device of this estimator (one sequence per context)
  };

  Params m_params;
  FeatureExtractor m_extractor;
  ConstraintManager m_constraints;
  MatcherHandle m_matcher;
  KeyScanner m_keyscanner;
  KeypointMapHandle m_keypoint_map;
  std::shared_ptr<HotPath> m_hotpath;

  Estimator() : Estimator(Params()) {}

  /// form.cpp:31-38.  Creates the CUDA context; throws HotPathError when no
  /// usable B200 is present (there is no CPU fallback).
  explicit Estimator(const Params &params) : Estimator(params, nullptr) {}

  /// Injection point for tests / tracing: run the same host logic over another
  /// HotPath implementation.
  Estimator(const Params &params, std::shared_ptr<HotPath> hotpath)
      : m_params(params), m_extractor(params.extraction, params.num_threads),
        m_constraints(params.constraints), m_matcher{params.matcher}, m_keyscanner(params.scans),
        m_keypoint_map{params.map, nullptr}, m_hotpath(std::move(hotpath)) {
    if (!m_hotpath) {
#ifndef FORM_HOTPATH_INJECTED_ONLY
      const size_t window = 1 + params.scans.max_num_recent_scans +
                            (params.scans.max_num_keyscans > 0 ? (size_t)params.scans.max_num_keyscans + 1 : 64) + 2;
      m_hotpath = std::make_shared<GpuHotPath>(hotpath_params(params), params.device, nullptr,
                                               (int)std::min<size_t>(window, 128));
#else
      throw HotPathError("Estimator: no hot path injected");
#endif
    }
    m_extractor.set_hotpath(m_hotpath);
    m_constraints.set_hotpath(m_hotpath.get());
    m_keypoint_map.hotpath = m_hotpath;
  }

  static HotPathParams hotpath_params(const Params &p) {
    HotPathParams hp;
    FeatureExtractor(p.extraction, p.num_threads).fill(hp);
    hp.max_dist_matching = p.matcher.max_dist_matching;
    hp.min_dist_map = p.map.min_dist_map;
    hp.sigma = p.constraints.planar_constraint_sigma;
    return hp;
  }

  Pose3 current_lidar_estimate() { return m_constraints.get_current_pose(); }
  const std::string &last_error() const { return m_last_error; }

  /// form.cpp:40-114
  std::tuple<std::vector<PlanarFeat>, std::vector<PointFeat>>
  register_scan(const std::vector<PointXYZf> &scan) noexcept {
    return register_scan(scan.data(), scan.size());
  }

  std::tuple<std::vector<PlanarFeat>, std::vector<PointFeat>>
  register_scan(const PointXYZf *scan, size_t n) noexcept {
    return register_impl([&](size_t scan_idx, std::vector<PlanarFeat> &planar, std::vector<PointFeat> &point) {
      m_hotpath->extract(scan, n, scan_idx, planar, point);
    });
  }

  /// register_scan on a raw sensor cloud: n records in the layout given to set_cloud_format (a
  /// driver's unordered points, missing returns absent).  They are organised into the scan on the
  /// device (rule R8, DESIGN.md §4); every later stage is register_scan's.  Errors (no format, more
  /// records than the format's max_records, ...) are reported through last_error().
  std::tuple<std::vector<PlanarFeat>, std::vector<PointFeat>> register_cloud(const void *records,
                                                                              size_t n) noexcept {
    return register_impl([&](size_t scan_idx, std::vector<PlanarFeat> &planar, std::vector<PointFeat> &point) {
      m_hotpath->extract_cloud(records, n, scan_idx, planar, point);
    });
  }

  /// Record layout and organisation rule of the clouds register_cloud receives (throws HotPathError).
  void set_cloud_format(const formgpu_cloud_format &fmt) { m_hotpath->set_cloud_format(fmt); }

  size_t icp_iterations() const { return m_icp_iterations; }

private:
  /// form.cpp:40-114; `extract` is the feature extraction step (form.cpp:53-55) of the input at hand
  template <typename Extract>
  std::tuple<std::vector<PlanarFeat>, std::vector<PointFeat>> register_impl(Extract &&extract) noexcept {
    std::tuple<std::vector<PlanarFeat>, std::vector<PointFeat>> keypoints;
    struct ScanBracket { // tells a pooled hot path that this sequence is inside register_scan
      HotPath &hp;
      explicit ScanBracket(HotPath &h) : hp(h) { hp.begin_scan(); }
      ~ScanBracket() { hp.end_scan(); }
    } bracket(*m_hotpath);
    try {
      // ---- initialisation (form.cpp:49-50) ----
      const Pose3 prediction = m_constraints.predict_next();
      const size_t scan_idx = m_constraints.step(prediction);

      // ---- feature extraction (form.cpp:53-55) ----
      extract(scan_idx, std::get<0>(keypoints), std::get<1>(keypoints));
      const size_t num_keypoints = std::get<0>(keypoints).size() + std::get<1>(keypoints).size();

      // ---- world map at the latest smoothed poses (form.cpp:61-65) ----
      const std::vector<ScanPose> poses = m_constraints.scan_poses(m_constraints.get_values());
      m_hotpath->map_rebuild(poses.data(), poses.size());

      // ---- ICP loop (form.cpp:70-89) ----
      Values new_values;
      std::vector<PairCount> counts;
      for (size_t idx = 0; idx < m_params.matcher.max_num_rematches; ++idx) {
        const Pose3 before = m_constraints.get_current_pose();
        if (m_constraints.fused_schedule()) {
          // match (:75-79) and the first linearisation of optimize(true) (:82) in one
          // hot-path call; the LM then starts from those blocks
          const std::vector<ScanPose> now = m_constraints.scan_poses(m_constraints.get_values());
          m_hotpath->associate_linearize(scan_idx, now.data(), now.size(), counts, m_first_blocks);
          m_constraints.set_current_counts(counts);
          new_values = m_constraints.optimize(true, &m_first_blocks);
        } else {
          m_hotpath->associate(before, counts);            // :75-79
          m_constraints.set_current_counts(counts);
          new_values = m_constraints.optimize(true);        // :82
        }
        const Pose3 after = new_values.at(scan_idx);
        const double diff = norm6(before.localCoordinates(after));
        ++m_icp_iterations;
        if (diff < m_params.matcher.new_pose_threshold) break; // :85-87
        m_constraints.update_current_pose(after);          // :88
      }

      // ---- full nonlinear optimisation (form.cpp:92-93) ----
      new_values = m_constraints.optimize(false);
      m_constraints.update_values(new_values);

      // ---- map insertion (form.cpp:99-101) ----
      size_t np = 0, nq = 0;
      m_hotpath->commit_scan(np, nq);

      // ---- key-scan selection + marginalisation (form.cpp:104-111) ----
      const auto connections = [&](ScanIndex i) {
        return m_constraints.num_recent_connections(i, m_keyscanner.oldest_rf());
      };
      const std::vector<ScanIndex> marg = m_keyscanner.step(scan_idx, num_keypoints, connections);
      m_constraints.marginalize(marg);
    } catch (const std::exception &e) {
      m_last_error = e.what();
      std::get<0>(keypoints).clear();
      std::get<1>(keypoints).clear();
    }
    return keypoints;
  }

  std::string m_last_error;
  size_t m_icp_iterations = 0;
  std::vector<double> m_first_blocks;
};

} // namespace form
