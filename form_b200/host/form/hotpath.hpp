// The seam between FORM's host code and its per-scan data-parallel hot path.
//
// Each virtual below is one of the places where the reference's
// Estimator::register_scan (/root/reference/form/form.cpp:40-114) and
// ConstraintManager (/root/reference/form/optimization/constraints.cpp) call
// into feature extraction, the keypoint/voxel maps, the matcher and the
// factor linearisation.  The product implementation (GpuHotPath,
// gpu_hotpath.hpp) forwards 1:1 to the C-ABI in include/formgpu.h; tests plug
// the CPU oracle in behind the same interface so both pipelines share every
// line of host logic.
#pragma once

#include "form/pose3.hpp"
#include "form/types.hpp"
#include "formgpu.h"

#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

namespace form {

/// Parameters of the hot path (the reference spreads them over
/// FeatureExtractor::Params extraction.hpp:59-88, MatcherParams matcher.hpp:32-41,
/// KeypointMapParams map.hpp:97-100, ConstraintManager::Params constraints.hpp:60).
struct HotPathParams {
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
  double max_dist_matching = 0.8;
  double min_dist_map = 0.1;
  double sigma = 0.1;
  size_t num_threads = 0;
};

/// A (older scan i, newer scan j) pair, j > i: m_constraints[j][i] in
/// constraints.hpp:91-99.
struct PairKey {
  uint64_t i;
  uint64_t j;
};

/// Correspondence counts of pair (i, current scan) after an association.
struct PairCount {
  uint64_t i;
  uint32_t n_planar;
  uint32_t n_point;
};

struct ScanPose {
  uint64_t scan;
  Pose3 pose;
};

class HotPathError : public std::runtime_error {
public:
  using std::runtime_error::runtime_error;
  HotPathError(const std::string &msg, int code_) : std::runtime_error(msg), code(code_) {}
  int code = 0; // FORMGPU_* status of the failing call, 0 when not from the C-ABI
};

class HotPath {
public:
  virtual ~HotPath() = default;

  /// Brackets of one Estimator::register_scan.  A stand-alone context ignores them; the
  /// pooled implementation (batch_dispatch.hpp) uses them to know which sequences to wait
  /// for when it forms a batch.
  virtual void begin_scan() {}
  virtual void end_scan() {}

  /// FeatureExtractor::extract (extraction.hpp:99-101).  Also makes scan_idx the
  /// "current scan" whose keypoints later calls match and commit.
  virtual void extract(const PointXYZf *scan, size_t n, uint64_t scan_idx,
                       std::vector<PlanarFeat> &planar, std::vector<PointFeat> &point) = 0;

  /// Raw sensor clouds (formgpu_set_cloud_format / formgpu_extract_cloud): the record layout of the
  /// clouds extract_cloud() receives, then extract() of the organised cloud (rule R8).  Hot paths that
  /// do not organise clouds (the CPU oracle, trace recording) keep these defaults.
  virtual void set_cloud_format(const formgpu_cloud_format &) {
    throw HotPathError("this hot path does not organise raw clouds", FORMGPU_ERR_UNSUPPORTED);
  }
  virtual void extract_cloud(const void *, size_t, uint64_t, std::vector<PlanarFeat> &, std::vector<PointFeat> &) {
    throw HotPathError("this hot path does not organise raw clouds", FORMGPU_ERR_UNSUPPORTED);
  }
  /// Counters of the last organisation (formgpu_cloud_stats_last).
  virtual void cloud_stats(formgpu_cloud_stats &) {
    throw HotPathError("this hot path does not organise raw clouds", FORMGPU_ERR_UNSUPPORTED);
  }

  /// KeypointMap::to_voxel_map for both keypoint types (map.hpp:137,
  /// form.cpp:61-65): re-transform every stored keypoint with the given poses
  /// and rebuild the voxel hash (the reparative step).
  virtual void map_rebuild(const ScanPose *poses, size_t n_poses) = 0;

  /// Matcher::match<0> and match<1> (matcher.hpp:67-112, form.cpp:75-79) for the
  /// current scan at pose `pose_k`: replaces the current scan's correspondences
  /// and reports the per-pair counts.
  virtual void associate(const Pose3 &pose_k, std::vector<PairCount> &counts) = 0;

  /// associate() at the current scan's pose in `poses`, then linearize() of every non-empty
  /// pair (i, current scan) at `poses`: the start of one ICP iteration (form.cpp:75-82).
  /// blocks receives 91 doubles per entry of counts.  Implementations may fuse the two
  /// into one device round trip; the default simply calls them in turn.
  virtual void associate_linearize(uint64_t current_scan, const ScanPose *poses, size_t n_poses,
                                   std::vector<PairCount> &counts, std::vector<double> &blocks) {
    const Pose3 *pose_k = nullptr;
    for (size_t p = 0; p < n_poses; ++p)
      if (poses[p].scan == current_scan) pose_k = &poses[p].pose;
    if (!pose_k) throw HotPathError("associate_linearize: no pose for the current scan");
    associate(*pose_k, counts);
    std::vector<PairKey> pairs;
    for (const auto &c : counts) pairs.push_back({c.i, current_scan});
    blocks.assign(91 * pairs.size(), 0.0);
    if (!pairs.empty()) linearize(pairs.data(), pairs.size(), poses, n_poses, blocks.data());
  }

  /// DenseFactor::linearize of FeatureFactor(X(i), X(j)) for each pair
  /// (gtsam.hpp:67-86, factor.cpp:141-186): 91 doubles per pair, the packed
  /// upper triangle of the 13x13 augmented information matrix.
  virtual void linearize(const PairKey *pairs, size_t n_pairs, const ScanPose *poses,
                         size_t n_poses, double *out91) = 0;

  /// 0.5 * |r / sigma|^2 per pair (NoiseModelFactor::error), for LM trial steps.
  virtual void error(const PairKey *pairs, size_t n_pairs, const ScanPose *poses,
                     size_t n_poses, double *out) = 0;

  /// KeypointMap::insert_matches for both types (map.hpp:142, form.cpp:99-101).
  virtual void commit_scan(size_t &n_planar_added, size_t &n_point_added) = 0;

  /// KeypointMap::remove + ConstraintManager's erase of every pair touching the
  /// scans (map.hpp:130-133, constraints.cpp:186-194).
  virtual void remove_scans(const uint64_t *scans, size_t n) = 0;

  /// World-frame copy of the stored keypoints (FORM::map(), bindings.cpp:96-119).
  virtual void world_keypoints(const ScanPose *poses, size_t n_poses,
                               std::vector<PlanarFeat> &planar, std::vector<PointFeat> &point) = 0;
};

} // namespace form
