// Lock-step replay of the recorded hot-path traces of MANY independent sequences through
// formgpu_batch_submit (include/formgpu.h): every round takes the next pending call of each
// sequence and submits them together, so calls of the same kind share one launch per
// kernel.  The per-sequence call order - and therefore every result - is that of
// form::replay (trace.hpp) on a private context.
#pragma once

#include "form/gpu_hotpath.hpp"
#include "form/trace.hpp"

#include <chrono>
#include <cstdlib>
#include <memory>

namespace form {

class BatchReplay {
public:
  /// What the calls of one scan of one sequence handed back, in call order.
  struct Captured {
    std::vector<PairCount> counts;  // every ASSOCIATE / ASSOC_LIN
    std::vector<double> blocks;     // 91 per pair, every ASSOC_LIN / LINEARIZE
    std::vector<double> errors;     // one per pair, every ERROR
    std::vector<uint64_t> keypoint_counts; // EXTRACT: planar, point; COMMIT: novel planar, point
    std::vector<PlanarFeat> planar; // host-scan replays only
    std::vector<PointFeat> point;
  };

  /// traces[s] drives sequence s.  `stream` = cudaStream_t of the batch (nullptr: private).
  BatchReplay(const std::vector<const Trace *> &traces, const HotPathParams &hp, int device,
              void *stream, int max_window_scans)
      : BatchReplay(traces, std::vector<formgpu_params>(traces.size(), to_formgpu_params(hp, max_window_scans)),
                    device, stream) {}
  /// traces[s] drives sequence s, whose context is configured by params[s] (sensor shape and
  /// hot-path parameters may differ between sequences: formgpu_batch_create_mixed).
  BatchReplay(const std::vector<const Trace *> &traces, const std::vector<formgpu_params> &params, int device,
              void *stream)
      : m_traces(traces), m_stats(traces.size()), m_seq(traces.size()) {
    if (params.size() != traces.size()) throw HotPathError("BatchReplay: one params entry per trace");
    for (size_t s = 0; s < params.size(); ++s)
      m_seq[s].points = (size_t)params[s].num_rows * (size_t)params[s].num_columns;
    if (const char *env = std::getenv("FORM_REPLAY_PREFETCH")) m_prefetch = env[0] != '0';
    const int rc = formgpu_batch_create_mixed(params.data(), device, stream, traces.size(), &m_batch);
    if (rc != FORMGPU_OK)
      throw HotPathError(std::string("formgpu_batch_create: ") + formgpu_batch_last_error(nullptr));
    for (auto &s : m_seq) {
      s.counts.resize(256);
      s.out.resize(91 * 256);
    }
  }
  ~BatchReplay() { formgpu_batch_destroy(m_batch); }
  BatchReplay(const BatchReplay &) = delete;
  BatchReplay &operator=(const BatchReplay &) = delete;

  formgpu_batch *batch() const { return m_batch; }
  size_t size() const { return m_traces.size(); }
  ReplayStats &stats(size_t s) { return m_stats[s]; }
  /// on: every later run keeps what the calls of its last scan return for sequence s
  void capture_last_scan(size_t s, bool on) { m_seq[s].capture = on; }
  const Captured &captured(size_t s) const { return m_seq[s].last; }

  /// Replays scans [first, last) of every sequence.  scans[s][k] = scan k of sequence s
  /// (device pointers when on_device, host pointers otherwise; host scans come back as
  /// f64 keypoint structs in page-locked buffers, as formgpu_extract does).  Returns the
  /// wall time in seconds; `rounds` (optional) receives the number of submits.
  double run(size_t first, size_t last, const formgpu_point4f *const *const *scans, bool on_device,
             size_t *rounds = nullptr) {
    begin(first, last, on_device);
    const auto t0 = std::chrono::steady_clock::now();
    while (submit_next(scans)) finish_round();
    if (rounds) *rounds = m_rounds;
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }

  // ---- the same replay in three steps, for a host thread that drives several batches ----
  /// Positions every sequence at scan `first`.
  void begin(size_t first, size_t last, bool on_device) {
    const size_t S = m_traces.size();
    if (!on_device) ensure_host_buffers();
    for (size_t s = 0; s < S; ++s) {
      const Trace &t = *m_traces[s];
      const size_t lo = std::min(first, t.num_scans()), hi = std::min(last, t.num_scans());
      m_seq[s].op = lo < hi ? t.scan_begin[lo] : 0;
      m_seq[s].end = lo < hi ? t.op_end(hi - 1) : 0;
      m_seq[s].scan_hi = hi;
      m_seq[s].last_begin = lo < hi ? t.scan_begin[hi - 1] : 0;
      if (m_seq[s].capture) m_seq[s].last = Captured();
    }
    m_on_device = on_device;
    m_rounds = 0;
    m_reqs.reserve(S);
  }
  /// Queues the next pending call of every sequence (formgpu_batch_submit_async); false when
  /// every sequence has reached its end.
  bool submit_next(const formgpu_point4f *const *const *scans) {
    m_scans = scans;
    m_reqs.clear();
    m_owner.clear();
    for (size_t s = 0; s < m_traces.size(); ++s) {
      Seq &q = m_seq[s];
      if (q.op >= q.end) continue;
      m_reqs.push_back(make_request(s, (*m_traces[s]).ops[q.op], scans[s], m_on_device));
      m_owner.push_back(s);
    }
    if (m_reqs.empty()) return false;
    const int rc = formgpu_batch_submit_async(m_batch, m_reqs.data(), m_reqs.size());
    if (rc != FORMGPU_OK)
      throw HotPathError(std::string("formgpu_batch_submit: ") + formgpu_batch_last_error(m_batch));
    return true;
  }
  /// Waits for the round queued by submit_next and advances the sequences.
  void finish_round() {
    const int rc = formgpu_batch_wait(m_batch);
    if (rc != FORMGPU_OK)
      throw HotPathError(std::string("formgpu_batch_submit: ") + formgpu_batch_last_error(m_batch));
    for (size_t r = 0; r < m_reqs.size(); ++r) {
      const size_t s = m_owner[r];
      const TraceOp &op = (*m_traces[s]).ops[m_seq[s].op];
      account(s, op, m_reqs[r]);
      if (m_seq[s].capture && m_seq[s].op >= m_seq[s].last_begin) capture(s, op, m_reqs[r]);
      m_seq[s].op += 1;
      // a log is being reprocessed: the next scan of the sequence is known, so its upload starts
      // as soon as the extraction of this one has completed (the scan buffers alternate)
      if (m_prefetch && !m_on_device && op.kind == TraceOp::EXTRACT && m_scans && op.scan + 1 < m_seq[s].scan_hi)
        formgpu_batch_prefetch_scan(m_batch, s, m_scans[s][op.scan + 1], m_seq[s].points);
    }
    ++m_rounds;
  }
  size_t rounds() const { return m_rounds; }
  /// true when finish_round() would not block (the round in flight has completed)
  bool round_done() const {
    const int d = formgpu_batch_done(m_batch);
    if (d < 0) throw HotPathError(std::string("formgpu_batch_done: ") + formgpu_batch_last_error(m_batch));
    return d == 1;
  }

  /// One host thread, several batches (one stream each) on the same GPU: the thread queues a
  /// round on every batch before it waits for the first, so reps.size() rounds are in flight
  /// while it builds the next ones.  Returns the wall time in seconds.
  static double run_pipelined(const std::vector<BatchReplay *> &reps, size_t first, size_t last,
                              const formgpu_point4f *const *const *const *scans, bool on_device) {
    std::vector<uint8_t> flying(reps.size(), 0);
    for (BatchReplay *r : reps) r->begin(first, last, on_device);
    const auto t0 = std::chrono::steady_clock::now();
    size_t n_flying = 0;
    for (size_t i = 0; i < reps.size(); ++i) {
      flying[i] = reps[i]->submit_next(scans[i]);
      n_flying += flying[i];
    }
    while (n_flying) {
      for (size_t i = 0; i < reps.size(); ++i) {
        if (!flying[i]) continue;
        reps[i]->finish_round();
        flying[i] = reps[i]->submit_next(scans[i]);
        if (!flying[i]) --n_flying;
      }
    }
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }

private:
  struct Seq {
    size_t op = 0, end = 0;
    size_t points = 0;  // rows x cols of the sequence's sensor
    size_t scan_hi = 0; // scans [.., scan_hi) belong to the run in progress
    size_t last_begin = 0; // first op of scan scan_hi - 1
    uint64_t cur_scan = 0;
    size_t cur_np = 0, cur_nq = 0;
    std::vector<PairCount> counts;
    std::vector<double> out;
    PlanarFeat *planar = nullptr; // page-locked (host-scan replays only)
    PointFeat *point = nullptr;
    size_t planar_cap = 0, point_cap = 0;
    bool capture = false;
    Captured last;
  };

  void capture(size_t s, const TraceOp &op, const formgpu_request &r) {
    Seq &q = m_seq[s];
    Captured &c = q.last;
    switch (op.kind) {
    case TraceOp::EXTRACT:
    case TraceOp::COMMIT:
      c.keypoint_counts.push_back(r.n_planar);
      c.keypoint_counts.push_back(r.n_point);
      if (op.kind == TraceOp::EXTRACT && r.planar_out) {
        c.planar.assign(q.planar, q.planar + r.n_planar);
        c.point.assign(q.point, q.point + r.n_point);
      }
      break;
    case TraceOp::ASSOCIATE:
    case TraceOp::ASSOC_LIN:
      c.counts.insert(c.counts.end(), q.counts.begin(), q.counts.begin() + r.n_counts);
      if (op.kind == TraceOp::ASSOC_LIN) c.blocks.insert(c.blocks.end(), q.out.begin(), q.out.begin() + 91 * r.n_counts);
      break;
    case TraceOp::LINEARIZE:
      c.blocks.insert(c.blocks.end(), q.out.begin(), q.out.begin() + 91 * op.pairs.size());
      break;
    case TraceOp::ERROR:
      c.errors.insert(c.errors.end(), q.out.begin(), q.out.begin() + op.pairs.size());
      break;
    default:
      break;
    }
  }

  void ensure_host_buffers() {
    if (m_host_ready) return;
    for (size_t i = 0; i < m_seq.size(); ++i) {
      Seq &s = m_seq[i];
      formgpu_ctx *c = formgpu_batch_ctx(m_batch, i);
      s.planar_cap = formgpu_max_planar(c);
      s.point_cap = formgpu_max_point(c);
      s.planar = static_cast<PlanarFeat *>(formgpu_alloc_pinned(s.planar_cap * sizeof(PlanarFeat)));
      s.point = static_cast<PointFeat *>(formgpu_alloc_pinned(s.point_cap * sizeof(PointFeat)));
      if (!s.planar || !s.point) throw HotPathError("formgpu_alloc_pinned failed");
      m_pinned.emplace_back(s.planar, formgpu_free_pinned);
      m_pinned.emplace_back(s.point, formgpu_free_pinned);
    }
    m_host_ready = true;
  }

  formgpu_request make_request(size_t s, const TraceOp &op, const formgpu_point4f *const *scans,
                               bool on_device) {
    Seq &q = m_seq[s];
    formgpu_request r{};
    r.sequence = (uint32_t)s;
    switch (op.kind) {
    case TraceOp::EXTRACT:
      r.op = FORMGPU_OP_EXTRACT;
      r.flags = on_device ? FORMGPU_REQ_SCAN_ON_DEVICE : 0u;
      r.scan = scans[op.scan];
      r.n_points = q.points;
      r.scan_idx = op.scan;
      if (!on_device) {
        r.planar_out = reinterpret_cast<formgpu_planar_feat *>(q.planar);
        r.planar_cap = q.planar_cap;
        r.point_out = reinterpret_cast<formgpu_point_feat *>(q.point);
        r.point_cap = q.point_cap;
      }
      break;
    case TraceOp::MAP_REBUILD:
      r.op = FORMGPU_OP_MAP_REBUILD;
      r.poses = reinterpret_cast<const formgpu_scan_pose *>(op.poses.data());
      r.n_poses = op.poses.size();
      break;
    case TraceOp::ASSOCIATE:
      r.op = FORMGPU_OP_ASSOCIATE;
      r.pose_k = reinterpret_cast<const formgpu_pose *>(&op.pose);
      r.counts_out = reinterpret_cast<formgpu_pair_count *>(q.counts.data());
      r.counts_cap = q.counts.size();
      break;
    case TraceOp::ASSOC_LIN:
      r.op = FORMGPU_OP_ASSOC_LIN;
      r.poses = reinterpret_cast<const formgpu_scan_pose *>(op.poses.data());
      r.n_poses = op.poses.size();
      r.counts_out = reinterpret_cast<formgpu_pair_count *>(q.counts.data());
      r.counts_cap = q.counts.size();
      r.out = q.out.data();
      break;
    case TraceOp::LINEARIZE:
    case TraceOp::ERROR: {
      const bool err = op.kind == TraceOp::ERROR;
      r.op = err ? FORMGPU_OP_ERROR : FORMGPU_OP_LINEARIZE;
      const size_t need = (err ? 1 : 91) * op.pairs.size();
      if (q.out.size() < need) q.out.resize(need);
      r.pairs = reinterpret_cast<const formgpu_pair *>(op.pairs.data());
      r.n_pairs = op.pairs.size();
      r.poses = reinterpret_cast<const formgpu_scan_pose *>(op.poses.data());
      r.n_poses = op.poses.size();
      r.out = q.out.data();
      break;
    }
    case TraceOp::COMMIT:
      r.op = FORMGPU_OP_COMMIT;
      break;
    case TraceOp::REMOVE:
      r.op = FORMGPU_OP_REMOVE;
      r.scans = op.ids.data();
      r.n_scans = op.ids.size();
      break;
    }
    return r;
  }

  // same bookkeeping as form::replay (trace.hpp): work counters for the algorithmic bytes
  void account(size_t s, const TraceOp &op, const formgpu_request &r) {
    Seq &q = m_seq[s];
    ReplayStats &st = m_stats[s];
    auto &table = st.table;
    auto lookup = [&](const PairKey &p) -> std::pair<uint32_t, uint32_t> {
      for (const auto &e : table)
        if (e.first.i == p.i && e.first.j == p.j) return e.second;
      return {0, 0};
    };
    auto refresh_rows = [&]() {
      table.erase(std::remove_if(table.begin(), table.end(),
                                 [&](const auto &e) { return e.first.j == q.cur_scan; }),
                  table.end());
      for (size_t c = 0; c < r.n_counts; ++c) {
        table.push_back({{q.counts[c].i, q.cur_scan}, {q.counts[c].n_planar, q.counts[c].n_point}});
        st.assoc_planar += q.counts[c].n_planar;
        st.assoc_point += q.counts[c].n_point;
      }
    };
    switch (op.kind) {
    case TraceOp::EXTRACT:
      q.cur_scan = op.scan;
      q.cur_np = r.n_planar;
      q.cur_nq = r.n_point;
      st.scans += 1;
      st.points += q.points;
      st.planar_kp += r.n_planar;
      st.point_kp += r.n_point;
      break;
    case TraceOp::MAP_REBUILD:
      st.map_rebuilds += 1;
      break;
    case TraceOp::ASSOCIATE:
      st.assoc_calls += 1;
      st.assoc_queries += q.cur_np + q.cur_nq;
      refresh_rows();
      break;
    case TraceOp::ASSOC_LIN:
      st.assoc_calls += 1;
      st.assoc_queries += q.cur_np + q.cur_nq;
      refresh_rows();
      st.lin_calls += 1;
      st.lin_pairs += r.n_counts;
      for (size_t p = 0; p < r.n_counts; ++p) {
        st.lin_planar += q.counts[p].n_planar;
        st.lin_point += q.counts[p].n_point;
        st.checksum += q.out[91 * p + 90];
      }
      break;
    case TraceOp::LINEARIZE:
      st.lin_calls += 1;
      st.lin_pairs += op.pairs.size();
      for (size_t p = 0; p < op.pairs.size(); ++p) {
        const auto c = lookup(op.pairs[p]);
        st.lin_planar += c.first;
        st.lin_point += c.second;
        st.checksum += q.out[91 * p + 90];
      }
      break;
    case TraceOp::ERROR:
      st.err_calls += 1;
      st.err_pairs += op.pairs.size();
      for (size_t p = 0; p < op.pairs.size(); ++p) {
        const auto c = lookup(op.pairs[p]);
        st.err_planar += c.first;
        st.err_point += c.second;
        st.checksum += q.out[p];
      }
      break;
    case TraceOp::COMMIT:
      st.novel_planar += r.n_planar;
      st.novel_point += r.n_point;
      st.map_points += r.n_planar + r.n_point;
      break;
    case TraceOp::REMOVE:
      table.erase(std::remove_if(table.begin(), table.end(),
                                 [&](const auto &e) {
                                   for (uint64_t id : op.ids)
                                     if (e.first.i == id || e.first.j == id) return true;
                                   return false;
                                 }),
                  table.end());
      break;
    }
  }

  std::vector<const Trace *> m_traces;
  std::vector<ReplayStats> m_stats;
  std::vector<Seq> m_seq;
  formgpu_batch *m_batch = nullptr;
  bool m_host_ready = false;
  bool m_on_device = false;
  bool m_prefetch = true;        // FORM_REPLAY_PREFETCH=0: every scan is uploaded by its EXTRACT request
  const formgpu_point4f *const *const *m_scans = nullptr;
  size_t m_rounds = 0;
  std::vector<formgpu_request> m_reqs; // the round in flight (must outlive formgpu_batch_wait)
  std::vector<size_t> m_owner;
  std::vector<std::unique_ptr<void, void (*)(void *)>> m_pinned;
};

} // namespace form
