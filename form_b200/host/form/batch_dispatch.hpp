// Many live form::Estimators on ONE GPU: a dispatcher that funnels their hot-path calls
// through formgpu_batch_submit (include/formgpu.h), so that calls of the same kind from
// different sequences share one launch per kernel.
//
// Each Estimator runs on its own host thread, exactly as a stand-alone one would, over a
// BatchedHotPath: every HotPath call (the seams of /root/reference/form/form.cpp:40-114)
// becomes a formgpu_request that is posted to the dispatcher and blocks until it has been
// executed.  The dispatcher thread submits as soon as every sequence that is currently
// inside register_scan has posted (or after a short linger, so one sequence busy in its
// smoother does not stall the others) - dynamic batching, as inference servers do it.
// Results are those of the single-sequence entry points (index work bit-identical, blocks
// to 1e-12), so an Estimator cannot tell whether it runs alone or in a pool.
#pragma once

#include "form/gpu_hotpath.hpp"
#include "form/hotpath.hpp"

#include <chrono>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace form {

class BatchDispatcher {
public:
  /// n_sequences sequences with the same hot-path parameters.
  BatchDispatcher(const HotPathParams &hp, int device, size_t n_sequences, int max_window_scans = 64,
                  std::chrono::microseconds linger = std::chrono::microseconds(200))
      : BatchDispatcher(std::vector<formgpu_params>(n_sequences, to_formgpu_params(hp, max_window_scans)), device,
                        linger) {}
  /// One sequence per entry of `params` (hot-path parameters and window of its context): sensors of
  /// different shapes and parameter variants in one batch (formgpu_batch_create_mixed).
  BatchDispatcher(const std::vector<formgpu_params> &params, int device,
                  std::chrono::microseconds linger = std::chrono::microseconds(200))
      : m_linger(linger), m_slots(params.size()), m_params(params) {
    const int rc = formgpu_batch_create_mixed(params.data(), device, nullptr, params.size(), &m_batch);
    if (rc != FORMGPU_OK)
      throw HotPathError(std::string("formgpu_batch_create: ") + formgpu_batch_last_error(nullptr));
    m_thread = std::thread([this] { run(); });
  }
  ~BatchDispatcher() {
    {
      std::lock_guard<std::mutex> lk(m_mu);
      m_stop = true;
    }
    m_cv_work.notify_all();
    if (m_thread.joinable()) m_thread.join();
    formgpu_batch_destroy(m_batch);
  }
  BatchDispatcher(const BatchDispatcher &) = delete;
  BatchDispatcher &operator=(const BatchDispatcher &) = delete;

  size_t size() const { return m_slots.size(); }
  formgpu_batch *batch() const { return m_batch; }
  formgpu_ctx *ctx(size_t i) const { return formgpu_batch_ctx(m_batch, i); }
  /// The parameters sequence i's context was created with.
  const formgpu_params &params(size_t i) const { return m_params[i]; }
  uint64_t submits() const { return m_submits; }
  uint64_t requests() const { return m_requests; }

  /// A sequence announces that it is (not) inside register_scan: only busy sequences are
  /// waited for when a batch is formed.
  void set_busy(size_t seq, bool busy) {
    std::lock_guard<std::mutex> lk(m_mu);
    if (m_slots[seq].busy != busy) {
      m_slots[seq].busy = busy;
      m_busy += busy ? 1 : -1;
    }
    m_cv_work.notify_all();
  }

  /// Message of the last submission that failed as a whole ("" if none).
  std::string batch_error() {
    std::lock_guard<std::mutex> lk(m_mu);
    return m_batch_error;
  }

  /// Execute one request of sequence `seq` (blocking).  Returns the request's status; the
  /// message of a failure is formgpu_last_error(ctx(seq)).
  int execute(size_t seq, formgpu_request &req) {
    std::unique_lock<std::mutex> lk(m_mu);
    Slot &s = m_slots[seq];
    req.sequence = (uint32_t)seq;
    s.req = &req;
    s.done = false;
    if (m_pending++ == 0) m_first_post = std::chrono::steady_clock::now();
    m_cv_work.notify_all();
    m_cv_done.wait(lk, [&] { return s.done; });
    return req.status;
  }

private:
  struct Slot {
    formgpu_request *req = nullptr;
    bool done = true;
    bool busy = false;
  };

  void run() {
    std::vector<formgpu_request> reqs;
    std::vector<size_t> owner;
    std::unique_lock<std::mutex> lk(m_mu);
    for (;;) {
      m_cv_work.wait(lk, [&] { return m_stop || m_pending > 0; });
      if (m_stop) return;
      // linger until every busy sequence has posted, but no longer than m_linger after the
      // first request of this batch
      const auto deadline = m_first_post + m_linger;
      while (!m_stop && m_pending < std::max<size_t>(m_busy, 1) &&
             m_cv_work.wait_until(lk, deadline) != std::cv_status::timeout) {
      }
      if (m_stop) return;
      reqs.clear();
      owner.clear();
      for (size_t i = 0; i < m_slots.size(); ++i)
        if (m_slots[i].req && !m_slots[i].done) {
          reqs.push_back(*m_slots[i].req);
          owner.push_back(i);
        }
      m_pending = 0;
      lk.unlock();
      // per-request status is in reqs[k]; a submission that aborts as a whole (bad request list,
      // CUDA error while queueing) stamps its code on every request it did not reject individually
      const int rc = formgpu_batch_submit(m_batch, reqs.data(), reqs.size());
      lk.lock();
      if (rc != FORMGPU_OK) {
        m_batch_error = formgpu_batch_last_error(m_batch);
        for (auto &q : reqs)
          if (q.status == FORMGPU_OK) q.status = rc; // belt and braces: never report an unprocessed request as done
      }
      for (size_t k = 0; k < reqs.size(); ++k) {
        Slot &s = m_slots[owner[k]];
        *s.req = reqs[k];
        s.req = nullptr;
        s.done = true;
      }
      m_submits += 1;
      m_requests += reqs.size();
      m_cv_done.notify_all();
    }
  }

  formgpu_batch *m_batch = nullptr;
  std::chrono::microseconds m_linger;
  std::mutex m_mu;
  std::condition_variable m_cv_work, m_cv_done;
  std::vector<Slot> m_slots;
  std::vector<formgpu_params> m_params;
  size_t m_pending = 0, m_busy = 0;
  std::chrono::steady_clock::time_point m_first_post;
  bool m_stop = false;
  uint64_t m_submits = 0, m_requests = 0;
  std::string m_batch_error; // message of the last submission that failed as a whole
  std::thread m_thread;
};

/// HotPath of ONE sequence of a BatchDispatcher: every call is posted as a formgpu_request.
class BatchedHotPath : public HotPath {
public:
  BatchedHotPath(std::shared_ptr<BatchDispatcher> pool, size_t seq) : m_pool(std::move(pool)), m_seq(seq) {
    formgpu_ctx *c = m_pool->ctx(seq);
    m_planar_cap = formgpu_max_planar(c);
    m_point_cap = formgpu_max_point(c);
    m_planar = static_cast<PlanarFeat *>(formgpu_alloc_pinned(m_planar_cap * sizeof(PlanarFeat)));
    m_point = static_cast<PointFeat *>(formgpu_alloc_pinned(m_point_cap * sizeof(PointFeat)));
    if (!m_planar || !m_point) {
      formgpu_free_pinned(m_planar);
      formgpu_free_pinned(m_point);
      throw HotPathError("formgpu_alloc_pinned failed");
    }
  }
  ~BatchedHotPath() override {
    formgpu_free_pinned(m_planar);
    formgpu_free_pinned(m_point);
  }

  /// Estimator::register_scan brackets itself with these so the dispatcher knows whom to wait for.
  void begin_scan() override { m_pool->set_busy(m_seq, true); }
  void end_scan() override { m_pool->set_busy(m_seq, false); }

  void extract(const PointXYZf *scan, size_t n, uint64_t scan_idx, std::vector<PlanarFeat> &planar,
               std::vector<PointFeat> &point) override {
    formgpu_request r{};
    r.op = FORMGPU_OP_EXTRACT;
    r.scan = reinterpret_cast<const formgpu_point4f *>(scan);
    r.n_points = n;
    r.scan_idx = scan_idx;
    r.planar_out = reinterpret_cast<formgpu_planar_feat *>(m_planar);
    r.planar_cap = m_planar_cap;
    r.point_out = reinterpret_cast<formgpu_point_feat *>(m_point);
    r.point_cap = m_point_cap;
    run(r);
    planar.assign(m_planar, m_planar + r.n_planar);
    point.assign(m_point, m_point + r.n_point);
  }

  /// Not batched: straight on the sequence's context.  Only call while no request of this sequence
  /// is in flight (before its first scan, or between scans).
  void set_cloud_format(const formgpu_cloud_format &fmt) override {
    const int rc = formgpu_set_cloud_format(m_pool->ctx(m_seq), &fmt);
    if (rc != FORMGPU_OK) fail(rc);
  }

  /// A FORMGPU_REQ_CLOUD extraction: the pool's clouds are organised by one launch per kernel.
  void extract_cloud(const void *records, size_t n, uint64_t scan_idx, std::vector<PlanarFeat> &planar,
                     std::vector<PointFeat> &point) override {
    formgpu_request r{};
    r.op = FORMGPU_OP_EXTRACT;
    r.flags = FORMGPU_REQ_CLOUD;
    r.scan = static_cast<const formgpu_point4f *>(records);
    r.n_points = n;
    r.scan_idx = scan_idx;
    r.planar_out = reinterpret_cast<formgpu_planar_feat *>(m_planar);
    r.planar_cap = m_planar_cap;
    r.point_out = reinterpret_cast<formgpu_point_feat *>(m_point);
    r.point_cap = m_point_cap;
    run(r);
    planar.assign(m_planar, m_planar + r.n_planar);
    point.assign(m_point, m_point + r.n_point);
  }

  void cloud_stats(formgpu_cloud_stats &s) override {
    const int rc = formgpu_cloud_stats_last(m_pool->ctx(m_seq), &s);
    if (rc != FORMGPU_OK) fail(rc);
  }

  void map_rebuild(const ScanPose *poses, size_t n_poses) override {
    formgpu_request r{};
    r.op = FORMGPU_OP_MAP_REBUILD;
    r.poses = reinterpret_cast<const formgpu_scan_pose *>(poses);
    r.n_poses = n_poses;
    run(r);
  }

  void associate(const Pose3 &pose_k, std::vector<PairCount> &counts) override {
    counts.resize(256);
    formgpu_request r{};
    r.op = FORMGPU_OP_ASSOCIATE;
    r.pose_k = reinterpret_cast<const formgpu_pose *>(&pose_k);
    r.counts_out = reinterpret_cast<formgpu_pair_count *>(counts.data());
    r.counts_cap = counts.size();
    run(r);
    counts.resize(r.n_counts);
  }

  void associate_linearize(uint64_t, const ScanPose *poses, size_t n_poses, std::vector<PairCount> &counts,
                           std::vector<double> &blocks) override {
    counts.resize(256);
    blocks.resize(91 * 256);
    formgpu_request r{};
    r.op = FORMGPU_OP_ASSOC_LIN;
    r.poses = reinterpret_cast<const formgpu_scan_pose *>(poses);
    r.n_poses = n_poses;
    r.counts_out = reinterpret_cast<formgpu_pair_count *>(counts.data());
    r.counts_cap = counts.size();
    r.out = blocks.data();
    run(r);
    counts.resize(r.n_counts);
    blocks.resize(91 * r.n_counts);
  }

  void linearize(const PairKey *pairs, size_t n_pairs, const ScanPose *poses, size_t n_poses,
                 double *out91) override {
    stage3(FORMGPU_OP_LINEARIZE, pairs, n_pairs, poses, n_poses, out91);
  }
  void error(const PairKey *pairs, size_t n_pairs, const ScanPose *poses, size_t n_poses, double *out) override {
    stage3(FORMGPU_OP_ERROR, pairs, n_pairs, poses, n_poses, out);
  }

  void commit_scan(size_t &n_planar_added, size_t &n_point_added) override {
    formgpu_request r{};
    r.op = FORMGPU_OP_COMMIT;
    run(r);
    n_planar_added = r.n_planar;
    n_point_added = r.n_point;
  }

  void remove_scans(const uint64_t *scans, size_t n) override {
    formgpu_request r{};
    r.op = FORMGPU_OP_REMOVE;
    r.scans = scans;
    r.n_scans = n;
    run(r);
  }

  /// Not batched (FORM::map(), once per query): straight on the sequence's context, which
  /// shares the batch's stream.  Only call while no request of this sequence is in flight.
  void world_keypoints(const ScanPose *poses, size_t n_poses, std::vector<PlanarFeat> &planar,
                       std::vector<PointFeat> &point) override {
    formgpu_ctx *c = m_pool->ctx(m_seq);
    size_t np = 0, nq = 0;
    int rc = formgpu_world_keypoints(c, reinterpret_cast<const formgpu_scan_pose *>(poses), n_poses, nullptr,
                                     0, &np, nullptr, 0, &nq);
    if (rc != FORMGPU_OK && rc != FORMGPU_ERR_CAPACITY) fail(rc);
    planar.resize(np);
    point.resize(nq);
    if (np + nq == 0) return;
    rc = formgpu_world_keypoints(c, reinterpret_cast<const formgpu_scan_pose *>(poses), n_poses,
                                 reinterpret_cast<formgpu_planar_feat *>(planar.data()), np, &np,
                                 reinterpret_cast<formgpu_point_feat *>(point.data()), nq, &nq);
    if (rc != FORMGPU_OK) fail(rc);
  }

private:
  void stage3(uint32_t op, const PairKey *pairs, size_t n_pairs, const ScanPose *poses, size_t n_poses,
              double *out) {
    formgpu_request r{};
    r.op = op;
    r.pairs = reinterpret_cast<const formgpu_pair *>(pairs);
    r.n_pairs = n_pairs;
    r.poses = reinterpret_cast<const formgpu_scan_pose *>(poses);
    r.n_poses = n_poses;
    r.out = out;
    run(r);
  }
  void run(formgpu_request &r) {
    const int rc = m_pool->execute(m_seq, r);
    if (rc != FORMGPU_OK) fail(rc);
  }
  [[noreturn]] void fail(int rc) const {
    std::string msg = formgpu_last_error(m_pool->ctx(m_seq));
    const std::string batch = m_pool->batch_error();
    if (!batch.empty()) msg += (msg.empty() ? "" : "; ") + std::string("batch: ") + batch;
    throw HotPathError(std::string("formgpu error ") + std::to_string(rc) + ": " + msg, rc);
  }

  std::shared_ptr<BatchDispatcher> m_pool;
  size_t m_seq;
  PlanarFeat *m_planar = nullptr;
  PointFeat *m_point = nullptr;
  size_t m_planar_cap = 0, m_point_cap = 0;
};

} // namespace form
