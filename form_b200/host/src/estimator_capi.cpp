// libformhost.so: form::Estimator and the trace replayer over the CUDA hot path.
#include "form/batch_dispatch.hpp"
#include "form/batch_replay.hpp"
#include "form/capi_impl.hpp"

#include <atomic>
#include <thread>

using namespace form;
using namespace form::capi;

namespace {
std::string g_error;
std::shared_ptr<HotPath> make_gpu(const HotPathParams &hp, const formhost_est_params &p) {
  const int window = p.hot.max_window_scans > 0 ? p.hot.max_window_scans : 64;
  return std::make_shared<GpuHotPath>(hp, p.device, nullptr, window);
}
} // namespace

extern "C" {

void formhost_default_est_params(formhost_est_params *p) {
  std::memset(p, 0, sizeof(*p));
  formgpu_default_params(&p->hot);
  p->new_pose_threshold = 1e-4;
  p->keyscan_match_ratio = 0.1;
  p->max_num_rematches = 30;
  p->disable_smoothing = 0;
  p->max_num_keyscans = 50;
  p->max_num_recent_scans = 10;
  p->max_steps_unused_keyscan = 10;
  p->num_threads = 0;
  p->device = 0;
  p->record_trace = 0;
}

const char *formhost_last_error(void) { return g_error.c_str(); }

void *formhost_est_create(const formhost_est_params *p) { return est_create(p, make_gpu, g_error); }
void formhost_est_destroy(void *h) { delete static_cast<EstimatorHandle *>(h); }
const char *formhost_est_error(void *h) { return static_cast<EstimatorHandle *>(h)->error.c_str(); }

int formhost_est_register_scan(void *h, const formgpu_point4f *scan, size_t n,
                               formgpu_planar_feat *planar, size_t planar_cap, size_t *n_planar,
                               formgpu_point_feat *point, size_t point_cap, size_t *n_point) {
  return est_register_scan(static_cast<EstimatorHandle *>(h), scan, n, planar, planar_cap, n_planar,
                           point, point_cap, n_point);
}
void formhost_est_pose(void *h, formgpu_pose *out) { est_pose(static_cast<EstimatorHandle *>(h), out); }
int formhost_est_window(void *h, formgpu_scan_pose *out, size_t cap, size_t *n) {
  return est_window(static_cast<EstimatorHandle *>(h), out, cap, n);
}
void formhost_est_stats(void *h, uint64_t out[8]) { est_stats(static_cast<EstimatorHandle *>(h), out); }
int formhost_est_map(void *h, formgpu_planar_feat *planar, size_t planar_cap, size_t *n_planar,
                     formgpu_point_feat *point, size_t point_cap, size_t *n_point) {
  return est_map(static_cast<EstimatorHandle *>(h), planar, planar_cap, n_planar, point, point_cap,
                 n_point);
}
/// The context behind the estimator (profiling, launch counts).
void *formhost_est_ctx(void *h) {
  auto *g = dynamic_cast<GpuHotPath *>(static_cast<EstimatorHandle *>(h)->backend.get());
  return g ? g->ctx() : nullptr;
}
/// Borrowed pointer to the recorded trace (valid while the estimator lives).
const void *formhost_est_trace(void *h) { return &static_cast<EstimatorHandle *>(h)->trace; }
size_t formhost_trace_num_scans(const void *t) { return static_cast<const Trace *>(t)->num_scans(); }
size_t formhost_trace_num_ops(const void *t) { return static_cast<const Trace *>(t)->ops.size(); }

/// A fresh CUDA context that replays a recorded trace.  `stream` may be a
/// cudaStream_t the caller times with its own events (NULL = private stream).
void *formhost_replay_create(const void *trace, const formhost_est_params *p, void *stream) {
  try {
    auto r = std::make_unique<ReplayHandle>();
    r->trace = static_cast<const Trace *>(trace);
    const Estimator::Params ep = to_estimator_params(*p);
    const int window = p->hot.max_window_scans > 0 ? p->hot.max_window_scans : 64;
    r->backend = std::make_shared<GpuHotPath>(Estimator::hotpath_params(ep), p->device, stream, window);
    r->points_per_scan = (size_t)p->hot.num_rows * p->hot.num_columns;
    return r.release();
  } catch (const std::exception &e) {
    g_error = e.what();
    return nullptr;
  }
}
void formhost_replay_destroy(void *r) { delete static_cast<ReplayHandle *>(r); }
void *formhost_replay_ctx(void *r) {
  return static_cast<GpuHotPath *>(static_cast<ReplayHandle *>(r)->backend.get())->ctx();
}

/// Replay with HOST scans: every EXTRACT copies the scan to the device and the
/// keypoints back, as Estimator::register_scan does.  Returns seconds, < 0 on error.
double formhost_replay_run_host(void *r, size_t first, size_t last,
                                const formgpu_point4f *const *scans) {
  auto *rh = static_cast<ReplayHandle *>(r);
  auto *gpu = static_cast<GpuHotPath *>(rh->backend.get());
  try {
    const auto t0 = std::chrono::steady_clock::now();
    replay(*rh->trace, *rh->backend, first, last,
           [&](uint64_t scan_idx, size_t &np, size_t &nq) {
             // straight through formgpu_extract: host scan in, f64 keypoint structs out
             gpu->extract_raw(reinterpret_cast<const PointXYZf *>(scans[scan_idx]),
                              rh->points_per_scan, scan_idx, np, nq);
           },
           rh->points_per_scan, rh->stats);
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  } catch (const std::exception &e) {
    g_error = e.what();
    return -1.0;
  }
}

/// Replay with scans already resident in DEVICE memory (scans_dev[s] = device
/// pointer); keypoints stay on the device.  Returns seconds, < 0 on error.
double formhost_replay_run_device(void *rv, size_t first, size_t last,
                                  const formgpu_point4f *const *scans_dev) {
  auto *r = static_cast<ReplayHandle *>(rv);
  auto *gpu = static_cast<GpuHotPath *>(r->backend.get());
  try {
    const auto t0 = std::chrono::steady_clock::now();
    replay(*r->trace, *r->backend, first, last,
           [&](uint64_t scan_idx, size_t &np, size_t &nq) {
             gpu->extract_device(scans_dev[scan_idx], r->points_per_scan, scan_idx, np, nq);
           },
           r->points_per_scan, r->stats);
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  } catch (const std::exception &e) {
    g_error = e.what();
    return -1.0;
  }
}

/// Several independent sequences on ONE GPU: replay[i] (its own context and stream) is
/// driven by its own host thread over scans_dev[i] (device pointers of its sequence).
/// Returns the wall time in seconds from a common start to the last thread finishing
/// (every replay call is synchronous, so all device work is done by then), < 0 on error.
double formhost_replay_run_device_multi(void *const *replays, size_t n_replays, size_t first, size_t last,
                                        const formgpu_point4f *const *const *scans_dev) {
  std::vector<std::thread> threads;
  std::vector<int> failed(n_replays, 0);
  std::atomic<size_t> ready{0};
  std::atomic<bool> go{false};
  for (size_t i = 0; i < n_replays; ++i) {
    threads.emplace_back([&, i] {
      auto *r = static_cast<ReplayHandle *>(replays[i]);
      auto *gpu = static_cast<GpuHotPath *>(r->backend.get());
      ready.fetch_add(1);
      while (!go.load(std::memory_order_acquire)) {
      }
      try {
        replay(*r->trace, *r->backend, first, last,
               [&](uint64_t scan_idx, size_t &np, size_t &nq) {
                 gpu->extract_device(scans_dev[i][scan_idx], r->points_per_scan, scan_idx, np, nq);
               },
               r->points_per_scan, r->stats);
      } catch (const std::exception &e) {
        failed[i] = 1;
      }
    });
  }
  while (ready.load() < n_replays) {
  }
  const auto t0 = std::chrono::steady_clock::now();
  go.store(true, std::memory_order_release);
  for (auto &t : threads) t.join();
  const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  for (int f : failed)
    if (f) return -1.0;
  return dt;
}

// ---- pool: many LIVE estimators on one GPU behind a batching dispatcher ----

/// A pool of n sequences sharing one formgpu_batch; formhost_pool_est_create(pool, i) gives
/// the form::Estimator of sequence i (same handle type as formhost_est_create: use the
/// formhost_est_* calls on it, each sequence from its own host thread).
void *formhost_pool_create(const formhost_est_params *p, size_t n_sequences, int linger_us) {
  try {
    const Estimator::Params ep = to_estimator_params(*p);
    const int window = p->hot.max_window_scans > 0 ? p->hot.max_window_scans : 64;
    auto *pool = new std::shared_ptr<BatchDispatcher>(std::make_shared<BatchDispatcher>(
        Estimator::hotpath_params(ep), p->device, n_sequences, window,
        std::chrono::microseconds(linger_us > 0 ? linger_us : 200)));
    return pool;
  } catch (const std::exception &e) {
    g_error = e.what();
    return nullptr;
  }
}
void formhost_pool_destroy(void *pool) { delete static_cast<std::shared_ptr<BatchDispatcher> *>(pool); }
void formhost_pool_stats(void *pool, uint64_t out[2]) {
  auto &d = *static_cast<std::shared_ptr<BatchDispatcher> *>(pool);
  out[0] = d->submits();
  out[1] = d->requests();
}
void *formhost_pool_est_create(void *pool, const formhost_est_params *p, size_t seq) {
  auto &d = *static_cast<std::shared_ptr<BatchDispatcher> *>(pool);
  if (seq >= d->size()) {
    g_error = "formhost_pool_est_create: sequence index outside the pool";
    return nullptr;
  }
  auto make = [&](const HotPathParams &, const formhost_est_params &) -> std::shared_ptr<HotPath> {
    return std::make_shared<BatchedHotPath>(d, seq);
  };
  return est_create(p, make, g_error);
}

// ---- batched replay: many sequences per launch (formgpu_batch_submit) ----

/// traces[s] (borrowed, from formhost_est_trace) drives sequence s of a fresh batch.
void *formhost_batch_replay_create(const void *const *traces, size_t n, const formhost_est_params *p,
                                   void *stream) {
  try {
    std::vector<const Trace *> tr;
    for (size_t i = 0; i < n; ++i) tr.push_back(static_cast<const Trace *>(traces[i]));
    const Estimator::Params ep = to_estimator_params(*p);
    const int window = p->hot.max_window_scans > 0 ? p->hot.max_window_scans : 64;
    return new BatchReplay(tr, Estimator::hotpath_params(ep), p->device, stream, window);
  } catch (const std::exception &e) {
    g_error = e.what();
    return nullptr;
  }
}
void formhost_batch_replay_destroy(void *r) { delete static_cast<BatchReplay *>(r); }
void *formhost_batch_replay_batch(void *r) { return static_cast<BatchReplay *>(r)->batch(); }

/// Replays scans [first, last) of every sequence in lock step; scans[s][k] = scan k of
/// sequence s (device pointers when on_device != 0).  Returns seconds, < 0 on error.
double formhost_batch_replay_run(void *r, size_t first, size_t last,
                                 const formgpu_point4f *const *const *scans, int on_device,
                                 size_t *rounds) {
  try {
    return static_cast<BatchReplay *>(r)->run(first, last, scans, on_device != 0, rounds);
  } catch (const std::exception &e) {
    g_error = e.what();
    return -1.0;
  }
}

/// Several batches on one GPU, one host thread (and stream) each: while one batch waits for
/// its round, the others prepare and queue theirs.  scans[b] as for formhost_batch_replay_run.
/// Returns the wall time from a common start to the last batch finishing, < 0 on error.
double formhost_batch_replay_run_multi(void *const *replays, size_t n, size_t first, size_t last,
                                       const formgpu_point4f *const *const *const *scans, int on_device) {
  std::vector<std::thread> threads;
  std::vector<int> failed(n, 0);
  std::atomic<size_t> ready{0};
  std::atomic<bool> go{false};
  for (size_t i = 0; i < n; ++i) {
    threads.emplace_back([&, i] {
      ready.fetch_add(1);
      while (!go.load(std::memory_order_acquire)) {
      }
      try {
        static_cast<BatchReplay *>(replays[i])->run(first, last, scans[i], on_device != 0);
      } catch (const std::exception &e) {
        g_error = e.what();
        failed[i] = 1;
      }
    });
  }
  while (ready.load() < n) {
  }
  const auto t0 = std::chrono::steady_clock::now();
  go.store(true, std::memory_order_release);
  for (auto &t : threads) t.join();
  const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  for (int f : failed)
    if (f) return -1.0;
  return dt;
}

/// The same job with `n_threads` host threads, each driving its share of the batches in a
/// software pipeline (BatchReplay::run_pipelined): a thread queues one round on each of its
/// batches before it waits for the first, so n / n_threads rounds per thread are in flight.
/// n_threads = 0 or >= n: one thread per batch.  Returns seconds, < 0 on error.
double formhost_batch_replay_run_pipelined(void *const *replays, size_t n, size_t n_threads, size_t first,
                                           size_t last, const formgpu_point4f *const *const *const *scans,
                                           int on_device) {
  if (n == 0) return 0.0;
  if (n_threads == 0 || n_threads > n) n_threads = n;
  // No batch belongs to a thread: every thread walks over ALL batches and serves whichever has its
  // round completed (formgpu_batch_done polls a word in host memory) - collect it, queue the next
  // round, move on.  With fixed ownership the timed region ended with the slowest thread's batches
  // (a thread that shares a core, or is descheduled, held its streams idle): 3.6-8.7 k scans/s from
  // run to run with 8 threads x 1 batch.
  struct Slot {
    std::atomic<bool> busy{false};
    bool flying = false, finished = false;
  };
  std::vector<Slot> slots(n);
  std::atomic<size_t> n_finished{0};
  std::atomic<bool> abort_all{false};
  std::vector<std::thread> threads;
  std::vector<int> failed(n_threads, 0);
  for (size_t i = 0; i < n; ++i) static_cast<BatchReplay *>(replays[i])->begin(first, last, on_device != 0);
  std::atomic<size_t> ready{0};
  std::atomic<bool> go{false};
  for (size_t t = 0; t < n_threads; ++t) {
    threads.emplace_back([&, t] {
      ready.fetch_add(1);
      while (!go.load(std::memory_order_acquire)) {
      }
      try {
        size_t i = t * n / n_threads; // start at different batches
        while (n_finished.load(std::memory_order_acquire) < n && !abort_all.load(std::memory_order_relaxed)) {
          i = i + 1 < n ? i + 1 : 0;
          Slot &sl = slots[i];
          if (sl.finished || sl.busy.exchange(true, std::memory_order_acquire)) continue;
          if (!sl.finished) {
            BatchReplay *r = static_cast<BatchReplay *>(replays[i]);
            bool submit = !sl.flying;
            if (sl.flying && r->round_done()) {
              r->finish_round();
              sl.flying = false;
              submit = true;
            }
            if (submit) {
              sl.flying = r->submit_next(scans[i]);
              if (!sl.flying) {
                sl.finished = true;
                n_finished.fetch_add(1, std::memory_order_release);
              }
            }
          }
          sl.busy.store(false, std::memory_order_release);
        }
      } catch (const std::exception &e) {
        g_error = e.what();
        failed[t] = 1;
        abort_all.store(true);
      }
    });
  }
  while (ready.load() < n_threads) {
  }
  const auto t0 = std::chrono::steady_clock::now();
  go.store(true, std::memory_order_release);
  for (auto &t : threads) t.join();
  const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  for (int f : failed)
    if (f) return -1.0;
  return dt;
}

/// Work counters of sequence `seq`, or summed over all sequences when seq < 0.
void formhost_batch_replay_stats(void *r, int seq, uint64_t out[20], double *checksum) {
  auto *b = static_cast<BatchReplay *>(r);
  std::memset(out, 0, 20 * sizeof(uint64_t));
  double cs = 0.0;
  for (size_t s = 0; s < b->size(); ++s) {
    if (seq >= 0 && (size_t)seq != s) continue;
    ReplayHandle tmp;
    tmp.stats = b->stats(s);
    uint64_t v[20];
    double c = 0.0;
    replay_stats(&tmp, v, &c);
    for (int k = 0; k < 20; ++k) out[k] += v[k];
    cs += c;
  }
  if (checksum) *checksum = cs;
}
/// on != 0: every later run keeps what the calls of its last scan returned for sequence `seq`.
void formhost_batch_replay_capture(void *r, size_t seq, int on) {
  auto *b = static_cast<BatchReplay *>(r);
  if (seq < b->size()) b->capture_last_scan(seq, on != 0);
}

/// What the calls of the last scan of sequence `seq` returned in the latest run with capture on.
/// what: 0 pair counts (16 B records), 1 blocks (91 doubles per pair), 2 errors (doubles),
/// 3 planar / 4 point keypoints (72 / 40 B records, host-scan runs only), 5 keypoint counts
/// (uint64: extracted planar, point, then committed novel planar, point).  Copies at most `cap`
/// elements to `out` (may be null) and returns how many there are.
size_t formhost_batch_replay_captured(void *r, size_t seq, int what, void *out, size_t cap) {
  auto *b = static_cast<BatchReplay *>(r);
  if (seq >= b->size()) return 0;
  const BatchReplay::Captured &c = b->captured(seq);
  auto copy = [&](const auto &v) {
    if (out) std::memcpy(out, v.data(), std::min(cap, v.size()) * sizeof(v[0]));
    return v.size();
  };
  switch (what) {
  case 0: return copy(c.counts);
  case 1: return copy(c.blocks);
  case 2: return copy(c.errors);
  case 3: return copy(c.planar);
  case 4: return copy(c.point);
  case 5: return copy(c.keypoint_counts);
  default: return 0;
  }
}

void formhost_batch_replay_reset_stats(void *r) {
  auto *b = static_cast<BatchReplay *>(r);
  for (size_t s = 0; s < b->size(); ++s) {
    auto table = std::move(b->stats(s).table);
    b->stats(s) = ReplayStats();
    b->stats(s).table = std::move(table);
  }
}

void formhost_replay_stats(void *r, uint64_t out[20], double *checksum) {
  replay_stats(static_cast<ReplayHandle *>(r), out, checksum);
}
void formhost_replay_reset_stats(void *r) {
  auto *h = static_cast<ReplayHandle *>(r);
  auto table = std::move(h->stats.table);
  h->stats = ReplayStats();
  h->stats.table = std::move(table);
}

} // extern "C"
