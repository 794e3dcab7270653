// HotPath implemented by the CUDA library through its C-ABI (include/formgpu.h).
// This is the only hot-path implementation the product links; a failing call
// throws HotPathError with the library's message - there is no CPU fallback.
#pragma once

#include "form/hotpath.hpp"
#include "formgpu.h"

#include <string>

namespace form {

static_assert(sizeof(ScanPose) == sizeof(formgpu_scan_pose), "ScanPose layout");
static_assert(sizeof(PairKey) == sizeof(formgpu_pair), "PairKey layout");
static_assert(sizeof(PairCount) == sizeof(formgpu_pair_count), "PairCount layout");
static_assert(sizeof(PlanarFeat) == sizeof(formgpu_planar_feat), "PlanarFeat layout");
static_assert(sizeof(PointFeat) == sizeof(formgpu_point_feat), "PointFeat layout");
static_assert(sizeof(PointXYZf) == sizeof(formgpu_point4f), "PointXYZf layout");

inline formgpu_params to_formgpu_params(const HotPathParams &p, int max_window_scans = 64) {
  formgpu_params g;
  formgpu_default_params(&g);
  g.neighbor_points = (int32_t)p.neighbor_points;
  g.num_sectors = (int32_t)p.num_sectors;
  g.planar_feats_per_sector = (int32_t)p.planar_feats_per_sector;
  g.point_feats_per_sector = (int32_t)p.point_feats_per_sector;
  g.min_points = (int32_t)p.min_points;
  g.num_columns = p.num_columns;
  g.num_rows = p.num_rows;
  g.planar_threshold = p.planar_threshold;
  g.radius = p.radius;
  g.min_norm_squared = p.min_norm_squared;
  g.max_norm_squared = p.max_norm_squared;
  g.max_dist_matching = p.max_dist_matching;
  g.min_dist_map = p.min_dist_map;
  g.sigma = p.sigma;
  g.max_window_scans = max_window_scans;
  return g;
}

/// Field-wise equality of two context configurations (every field a context reads).
inline bool same_formgpu_params(const formgpu_params &a, const formgpu_params &b) {
  return a.neighbor_points == b.neighbor_points && a.num_sectors == b.num_sectors &&
         a.planar_feats_per_sector == b.planar_feats_per_sector &&
         a.point_feats_per_sector == b.point_feats_per_sector && a.min_points == b.min_points &&
         a.num_columns == b.num_columns && a.num_rows == b.num_rows && a.max_window_scans == b.max_window_scans &&
         a.planar_threshold == b.planar_threshold && a.radius == b.radius &&
         a.min_norm_squared == b.min_norm_squared && a.max_norm_squared == b.max_norm_squared &&
         a.max_dist_matching == b.max_dist_matching && a.min_dist_map == b.min_dist_map && a.sigma == b.sigma &&
         a.max_batch_scans == b.max_batch_scans;
}

class GpuHotPath : public HotPath {
public:
  explicit GpuHotPath(const HotPathParams &p, int device = 0, void *stream = nullptr,
                      int max_window_scans = 64) {
    formgpu_params g = to_formgpu_params(p);
    g.max_window_scans = max_window_scans;
    const int rc = formgpu_create(&g, device, stream, &m_ctx);
    if (rc != FORMGPU_OK)
      throw HotPathError(std::string("formgpu_create: ") + formgpu_last_error(nullptr));
    // page-locked output buffers: the kernels write the keypoint structs straight into them
    m_planar_cap = formgpu_max_planar(m_ctx);
    m_point_cap = formgpu_max_point(m_ctx);
    m_planar = static_cast<PlanarFeat *>(formgpu_alloc_pinned(m_planar_cap * sizeof(PlanarFeat)));
    m_point = static_cast<PointFeat *>(formgpu_alloc_pinned(m_point_cap * sizeof(PointFeat)));
    if (!m_planar || !m_point) {
      formgpu_free_pinned(m_planar);
      formgpu_free_pinned(m_point);
      formgpu_destroy(m_ctx);
      throw HotPathError("formgpu_alloc_pinned failed");
    }
  }
  ~GpuHotPath() override {
    formgpu_destroy(m_ctx);
    formgpu_free_pinned(m_planar);
    formgpu_free_pinned(m_point);
  }
  GpuHotPath(const GpuHotPath &) = delete;
  GpuHotPath &operator=(const GpuHotPath &) = delete;

  formgpu_ctx *ctx() const { return m_ctx; }

  void extract(const PointXYZf *scan, size_t n, uint64_t scan_idx, std::vector<PlanarFeat> &planar,
               std::vector<PointFeat> &point) override {
    size_t np = 0, nq = 0;
    check(formgpu_extract(m_ctx, reinterpret_cast<const formgpu_point4f *>(scan), n, scan_idx,
                          reinterpret_cast<formgpu_planar_feat *>(m_planar), m_planar_cap, &np,
                          reinterpret_cast<formgpu_point_feat *>(m_point), m_point_cap, &nq));
    planar.assign(m_planar, m_planar + np);
    point.assign(m_point, m_point + nq);
  }

  /// formgpu_extract into the adapter's own buffers without building vectors (what a
  /// caller that owns its buffers pays): returns the counts, data stays in planar_buffer().
  void extract_raw(const PointXYZf *scan, size_t n, uint64_t scan_idx, size_t &n_planar,
                   size_t &n_point) {
    check(formgpu_extract(m_ctx, reinterpret_cast<const formgpu_point4f *>(scan), n, scan_idx,
                          reinterpret_cast<formgpu_planar_feat *>(m_planar), m_planar_cap, &n_planar,
                          reinterpret_cast<formgpu_point_feat *>(m_point), m_point_cap, &n_point));
  }
  const PlanarFeat *planar_buffer() const { return m_planar; }
  const PointFeat *point_buffer() const { return m_point; }

  void set_cloud_format(const formgpu_cloud_format &fmt) override { check(formgpu_set_cloud_format(m_ctx, &fmt)); }

  void extract_cloud(const void *records, size_t n, uint64_t scan_idx, std::vector<PlanarFeat> &planar,
                     std::vector<PointFeat> &point) override {
    size_t np = 0, nq = 0;
    check(formgpu_extract_cloud(m_ctx, records, n, scan_idx, reinterpret_cast<formgpu_planar_feat *>(m_planar),
                                m_planar_cap, &np, reinterpret_cast<formgpu_point_feat *>(m_point), m_point_cap, &nq));
    planar.assign(m_planar, m_planar + np);
    point.assign(m_point, m_point + nq);
  }

  void cloud_stats(formgpu_cloud_stats &s) override { check(formgpu_cloud_stats_last(m_ctx, &s)); }

  /// Scan already resident in device memory; nothing is copied back.
  void extract_device(const void *scan_dev, size_t n, uint64_t scan_idx, size_t &n_planar,
                      size_t &n_point) {
    check(formgpu_extract_device(m_ctx, static_cast<const formgpu_point4f *>(scan_dev), n, scan_idx,
                                 &n_planar, &n_point));
  }

  void map_rebuild(const ScanPose *poses, size_t n_poses) override {
    check(formgpu_map_rebuild(m_ctx, reinterpret_cast<const formgpu_scan_pose *>(poses), n_poses));
  }

  void associate(const Pose3 &pose_k, std::vector<PairCount> &counts) override {
    counts.resize(256);
    size_t n = 0;
    check(formgpu_associate(m_ctx, reinterpret_cast<const formgpu_pose *>(&pose_k),
                            reinterpret_cast<formgpu_pair_count *>(counts.data()), counts.size(), &n));
    counts.resize(n);
  }

  void associate_linearize(uint64_t, const ScanPose *poses, size_t n_poses,
                           std::vector<PairCount> &counts, std::vector<double> &blocks) override {
    counts.resize(256);
    blocks.resize(91 * 256);
    size_t n = 0;
    check(formgpu_associate_linearize(m_ctx, reinterpret_cast<const formgpu_scan_pose *>(poses), n_poses,
                                      reinterpret_cast<formgpu_pair_count *>(counts.data()), counts.size(),
                                      &n, blocks.data()));
    counts.resize(n);
    blocks.resize(91 * n);
  }

  void linearize(const PairKey *pairs, size_t n_pairs, const ScanPose *poses, size_t n_poses,
                 double *out91) override {
    check(formgpu_linearize(m_ctx, reinterpret_cast<const formgpu_pair *>(pairs), n_pairs,
                            reinterpret_cast<const formgpu_scan_pose *>(poses), n_poses, out91));
  }

  void error(const PairKey *pairs, size_t n_pairs, const ScanPose *poses, size_t n_poses,
             double *out) override {
    check(formgpu_error(m_ctx, reinterpret_cast<const formgpu_pair *>(pairs), n_pairs,
                        reinterpret_cast<const formgpu_scan_pose *>(poses), n_poses, out));
  }

  void commit_scan(size_t &n_planar_added, size_t &n_point_added) override {
    check(formgpu_commit_scan(m_ctx, &n_planar_added, &n_point_added));
  }

  void remove_scans(const uint64_t *scans, size_t n) override {
    check(formgpu_remove_scans(m_ctx, scans, n));
  }

  void world_keypoints(const ScanPose *poses, size_t n_poses, std::vector<PlanarFeat> &planar,
                       std::vector<PointFeat> &point) override {
    size_t np = 0, nq = 0;
    // query sizes first (capacity error reports the counts)
    int rc = formgpu_world_keypoints(m_ctx, reinterpret_cast<const formgpu_scan_pose *>(poses),
                                     n_poses, nullptr, 0, &np, nullptr, 0, &nq);
    if (rc != FORMGPU_OK && rc != FORMGPU_ERR_CAPACITY) check(rc);
    planar.resize(np);
    point.resize(nq);
    if (np + nq == 0) return;
    check(formgpu_world_keypoints(m_ctx, reinterpret_cast<const formgpu_scan_pose *>(poses), n_poses,
                                  reinterpret_cast<formgpu_planar_feat *>(planar.data()), np, &np,
                                  reinterpret_cast<formgpu_point_feat *>(point.data()), nq, &nq));
  }

private:
  void check(int rc) const {
    if (rc != FORMGPU_OK)
      throw HotPathError(std::string("formgpu error ") + std::to_string(rc) + ": " +
                             formgpu_last_error(m_ctx),
                         rc);
  }
  formgpu_ctx *m_ctx = nullptr;
  PlanarFeat *m_planar = nullptr; // page-locked, formgpu_max_planar entries
  PointFeat *m_point = nullptr;
  size_t m_planar_cap = 0, m_point_cap = 0;
};

} // namespace form
