// C-ABI (include/formgpu.h): batched submit - the hot-path calls of MANY independent
// sequences in one launch per kernel.
//
// One sequence alone cannot fill a B200: a per-scan request is < 1 MB and every call is
// a dependent round trip (DESIGN.md 5).  A formgpu_batch owns S contexts (one per
// sequence) on one stream; formgpu_batch_submit takes at most one pending call per
// sequence, groups the calls by kind and issues ONE grid per kernel for each group -
// blockIdx.z (or blockIdx.y for stage 1) selects the sequence, whose argument block the
// CTA copies from a device array.  The kernel bodies are the single-sequence ones, so
// the results are bit-identical to S separate contexts; only the launch is shared.
// All groups are queued before the first wait, so the GPU runs them back to back while
// the host collects results through the same mapped-memory flags as the single calls.
#include "api_common.hpp"

#include <cuda.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <functional>
#include <new>
#include <tuple>

using namespace formgpu;

struct formgpu_batch {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::vector<formgpu_ctx *> ctx;
  mutable std::string err;
  // argument staging: pinned host ring + device mirror, bump-allocated per submit
  unsigned char *h_args = nullptr, *d_args = nullptr;
  size_t args_cap = 0, args_used = 0;
  Profiler prof;
  // scratch reused across submits
  std::vector<AssocPlan> assoc_plans;
  std::vector<ExtractArgs> extract_args;
  std::vector<CommitPlan> commit_plans;
  std::vector<std::vector<int>> lin_indices;
  std::vector<unsigned long long> lin_seqs;
  std::vector<LinTask> tasks_scratch;
  // extraction launches with at least this many rows use the many-row kernel variants
  // (kernels.hpp: kManyRowsMin; FORMGPU_MANY_ROWS_MIN overrides it, for tests and tuning)
  int many_rows_min = kManyRowsMin;
  // 13x13 blocks of a submission: the evaluation kernels write plain doubles into d_blocks and ONE
  // copy-engine transfer per submission takes them to h_blocks (page-locked).  SM stores of
  // sequence-tagged words into mapped host memory (the single-sequence protocol) move twice the
  // bytes in 8-byte PCIe writes and kept the evaluation CTAs resident until the writes drained:
  // 52 us per launch of ~1000 pairs, i.e. ~28 GB/s of PCIe stores.  Errors still come back as
  // tagged words.
  double *d_blocks = nullptr, *h_blocks = nullptr;
  size_t blocks_cap = 0, blocks_used = 0; // doubles
  std::vector<size_t> assoc_block_off, lin_block_off; // per sequence: offset into h_blocks, or kNoBlocks
  // Completion of a submission: ONE 32-bit stream write (cuStreamWriteValue32) into mapped host
  // memory behind the last operation of the submission; the host polls the word - no CUDA call
  // while it waits.  The process-wide rate of CUDA API calls is what bounds the batched engine
  // (~70 calls per scan from 15 threads, ~1.5 us each under the driver's lock), so a submission
  // makes as few as it can: no events, copies on the batch's own stream.
  volatile uint32_t *h_done = nullptr; // [0] submission counter reached, [1] keypoint copies of the collect phase
  CUdeviceptr d_done = 0;              // device address of h_done
  uint32_t done_seq = 0, kp_seq = 0;
  uint32_t done_polls = 0;
  // FORMGPU_BATCH_TRACE=1: host-side timing of the submissions, by kind of round (with / without
  // an extraction), printed when the batch is destroyed - a development probe
  struct Trace {
    bool on = false;
    double build_us[2] = {0, 0}, collect_us[2] = {0, 0}, flight_us[2] = {0, 0}, idle_us = 0;
    double extract_wait_us = 0, dma_us = 0, blocks_wait_us = 0;
    size_t rounds[2] = {0, 0};
    size_t build_outliers = 0;
    std::chrono::steady_clock::time_point t_submit, t_built, t_done;
    bool have_done = false;
    int kind = 0;
  } trace;
  // the submission in flight (formgpu_batch_submit_async ... formgpu_batch_wait)
  struct Pending {
    bool active = false;
    formgpu_request *reqs = nullptr;
    size_t n = 0;
    int first_error = FORMGPU_OK;
    std::vector<size_t> live_extract, live_assoc, live_lin[2], live_commit;
  } pend;
};

namespace {

std::string g_batch_error;

int bfail(formgpu_batch *b, int code, const std::string &msg) {
  if (b) b->err = msg;
  return code;
}

#define BATCH_CUDA(b, expr)                                                                  \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return bfail((b), FORMGPU_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); \
  } while (0)

size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

constexpr size_t kNoBlocks = ~(size_t)0;

// room for `doubles` block words of one submission (called before anything of it is staged)
int ensure_blocks(formgpu_batch *b, size_t doubles) {
  if (doubles <= b->blocks_cap) return FORMGPU_OK;
  BATCH_CUDA(b, cudaStreamSynchronize(b->stream));
  size_t cap = std::max<size_t>(b->blocks_cap * 2, 91 * 1024);
  while (cap < doubles) cap *= 2;
  if (b->d_blocks) cudaFree(b->d_blocks);
  if (b->h_blocks) cudaFreeHost(b->h_blocks);
  b->d_blocks = b->h_blocks = nullptr;
  b->blocks_cap = 0;
  BATCH_CUDA(b, cudaMalloc(reinterpret_cast<void **>(&b->d_blocks), cap * sizeof(double)));
  BATCH_CUDA(b, cudaHostAlloc(reinterpret_cast<void **>(&b->h_blocks), cap * sizeof(double), cudaHostAllocDefault));
  b->blocks_cap = cap;
  return FORMGPU_OK;
}

// cuStreamWriteValue32 through the runtime's driver-entry-point lookup (no link dependency on
// libcuda); nullptr when the driver does not offer it - a one-thread kernel writes the word then
typedef CUresult (*StreamWrite32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
StreamWrite32Fn stream_write32_fn() {
  static const StreamWrite32Fn fn = [] {
    void *p = nullptr;
    if (std::getenv("FORMGPU_NO_STREAM_MEMOPS")) return (StreamWrite32Fn) nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &p, cudaEnableDefault, &qr) != cudaSuccess ||
        qr != cudaDriverEntryPointSuccess)
      p = nullptr;
    cudaGetLastError();
    return reinterpret_cast<StreamWrite32Fn>(p);
  }();
  return fn;
}

__global__ void flag_write_kernel(volatile uint32_t *flag, uint32_t value) {
  __threadfence_system();
  *flag = value;
}

// queue "h_done[word] = value" behind everything already on the batch's stream
int queue_flag(formgpu_batch *b, int word, uint32_t value) {
  if (StreamWrite32Fn fn = stream_write32_fn()) {
    const CUresult r = fn(reinterpret_cast<CUstream>(b->stream), b->d_done + 4u * (unsigned)word, value, 0u);
    if (r == CUDA_SUCCESS) return FORMGPU_OK;
  }
  flag_write_kernel<<<1, 1, 0, b->stream>>>(reinterpret_cast<volatile uint32_t *>(b->d_done) + word, value);
  BATCH_CUDA(b, cudaGetLastError());
  return FORMGPU_OK;
}

// Spin (no CUDA call) until h_done[word] == value; the stream state is looked at every 4096 polls
// so that a faulted kernel cannot hang the caller.
int wait_done(formgpu_batch *b, int word, uint32_t value) {
  volatile uint32_t *f = b->h_done + word;
  for (unsigned spins = 0;; ++spins) {
    if (*f == value) {
      std::atomic_thread_fence(std::memory_order_acquire); // results are read after the word
      return FORMGPU_OK;
    }
    if ((spins & 0xfff) == 0xfff) {
      const cudaError_t e = cudaStreamQuery(b->stream);
      if (e == cudaSuccess) {
        if (*f == value) return FORMGPU_OK;
        return bfail(b, FORMGPU_ERR_STATE, "submission finished without raising its completion word");
      }
      if (e != cudaErrorNotReady)
        return bfail(b, FORMGPU_ERR_CUDA, std::string("submission failed: ") + cudaGetErrorString(e));
    }
    poll_relax(spins);
  }
}

// make room for `bytes` more staged argument bytes (contents staged so far are kept)
int ensure_args(formgpu_batch *b, size_t bytes) {
  if (b->args_used + bytes <= b->args_cap) return FORMGPU_OK;
  // no kernel of this submit has been queued yet (arguments are uploaded once, after the
  // last group is staged) and the previous submit's were waited for at submit start
  BATCH_CUDA(b, cudaStreamSynchronize(b->stream));
  size_t cap = std::max<size_t>(b->args_cap * 2, 1 << 20);
  while (cap < b->args_used + bytes) cap *= 2;
  unsigned char *h = nullptr, *d = nullptr;
  BATCH_CUDA(b, cudaHostAlloc(reinterpret_cast<void **>(&h), cap, cudaHostAllocDefault));
  BATCH_CUDA(b, cudaMalloc(reinterpret_cast<void **>(&d), cap));
  if (b->h_args) {
    std::memcpy(h, b->h_args, b->args_used);
    cudaFreeHost(b->h_args);
  }
  if (b->d_args) cudaFree(b->d_args);
  b->h_args = h;
  b->d_args = d;
  b->args_cap = cap;
  return FORMGPU_OK;
}

// stage `count` argument blocks; *offset = their position in the device mirror once the
// submit's single upload has run
template <typename T> int stage_args(formgpu_batch *b, const T *src, size_t count, size_t *offset) {
  const size_t bytes = round_up(count * sizeof(T), 256);
  const int rc = ensure_args(b, bytes);
  if (rc) return rc;
  std::memcpy(b->h_args + b->args_used, src, count * sizeof(T));
  *offset = b->args_used;
  b->args_used += bytes;
  return FORMGPU_OK;
}
template <typename T> const T *staged(const formgpu_batch *b, size_t offset) {
  return reinterpret_cast<const T *>(b->d_args + offset);
}

// Blocks / errors of the listed tasks of several contexts in ONE launch, evaluated from the
// contexts' pair-moment caches (moments.cu): one CTA per task, ctx_args[task.ctx_index] is the
// task's context.
int stage_lin_groups(formgpu_batch *b, const std::vector<LinArgs> &ctx_args, const std::vector<LinTask> &tasks,
                     bool error_only, std::vector<std::function<int()>> &launchers) {
  if (tasks.empty()) return FORMGPU_OK;
  size_t off_ctx = 0, off_tasks = 0;
  int rc = stage_args(b, ctx_args.data(), ctx_args.size(), &off_ctx);
  if (rc) return rc;
  rc = stage_args(b, tasks.data(), tasks.size(), &off_tasks);
  if (rc) return rc;
  const int n_tasks = (int)tasks.size();
  launchers.push_back([=]() -> int {
    BATCH_CUDA(b, eval_batch_launch(staged<LinArgs>(b, off_ctx), staged<LinTask>(b, off_tasks), n_tasks, error_only,
                                    b->stream, b->prof));
    return FORMGPU_OK;
  });
  return FORMGPU_OK;
}

} // namespace

extern "C" {

const char *formgpu_batch_last_error(const formgpu_batch *b) {
  return b ? b->err.c_str() : g_batch_error.c_str();
}

int formgpu_batch_create(const formgpu_params *p, int device, void *stream, size_t n_sequences,
                         formgpu_batch **out) {
  if (!p || !out || n_sequences == 0 || n_sequences > 4096) {
    g_batch_error = "formgpu_batch_create: bad argument";
    return FORMGPU_ERR_INVALID_ARG;
  }
  const std::vector<formgpu_params> params(n_sequences, *p);
  return formgpu_batch_create_mixed(params.data(), device, stream, n_sequences, out);
}

int formgpu_batch_create_mixed(const formgpu_params *params, int device, void *stream, size_t n_sequences,
                               formgpu_batch **out) {
  if (!params || !out || n_sequences == 0 || n_sequences > 4096) {
    g_batch_error = "formgpu_batch_create_mixed: bad argument";
    return FORMGPU_ERR_INVALID_ARG;
  }
  *out = nullptr;
  // every entry is checked before the first CUDA call, so a bad one fails on any machine
  for (size_t i = 0; i < n_sequences; ++i) {
    std::string msg;
    const int rc = validate_params(params[i], msg);
    if (rc != FORMGPU_OK) {
      g_batch_error = "formgpu_batch_create: params of sequence " + std::to_string(i) + ": " + msg;
      return rc;
    }
  }
  formgpu_batch *b = new (std::nothrow) formgpu_batch();
  if (!b) return FORMGPU_ERR_CAPACITY;
  b->device = device;
  b->stream = static_cast<cudaStream_t>(stream);
  if (const char *env = std::getenv("FORMGPU_MANY_ROWS_MIN")) b->many_rows_min = std::atoi(env);
  if (const char *env = std::getenv("FORMGPU_BATCH_TRACE")) b->trace.on = env[0] == '1';
  auto bail = [&](int rc, const std::string &msg) {
    g_batch_error = msg;
    formgpu_batch_destroy(b);
    return rc;
  };
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return bail(FORMGPU_ERR_CUDA, "no CUDA device available (there is no CPU fallback)");
  if (device < 0 || device >= ndev) return bail(FORMGPU_ERR_INVALID_ARG, "device index out of range");
  if (cudaSetDevice(device) != cudaSuccess) return bail(FORMGPU_ERR_CUDA, "cudaSetDevice failed");
  if (!b->stream) {
    if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess)
      return bail(FORMGPU_ERR_CUDA, "cudaStreamCreate failed");
    b->own_stream = true;
  }
  b->prof.stream = b->stream;
  {
    void *h = nullptr, *d = nullptr;
    if (cudaHostAlloc(&h, 64, cudaHostAllocMapped) != cudaSuccess || cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess)
      return bail(FORMGPU_ERR_CUDA, "cudaHostAlloc (completion word) failed");
    std::memset(h, 0, 64);
    b->h_done = static_cast<volatile uint32_t *>(h);
    b->d_done = reinterpret_cast<CUdeviceptr>(d);
  }
  for (size_t i = 0; i < n_sequences; ++i) {
    formgpu_ctx *c = nullptr;
    const int rc = formgpu_create(&params[i], device, b->stream, &c); // every context shares the batch stream
    if (rc != FORMGPU_OK)
      return bail(rc, "formgpu_create (sequence " + std::to_string(i) + "): " + formgpu_last_error(nullptr));
    c->moment_unit = kMomentUnit; // throughput-sized units (kernels.hpp)
    c->moment_cache = true;       // the batched stage 3 evaluates from the cache only
    b->ctx.push_back(c);
  }
  b->assoc_block_off.assign(n_sequences, kNoBlocks);
  b->lin_block_off.assign(n_sequences, kNoBlocks);
  b->assoc_plans.resize(n_sequences);
  b->extract_args.resize(n_sequences);
  b->commit_plans.resize(n_sequences);
  b->lin_indices.resize(n_sequences);
  b->lin_seqs.resize(n_sequences);
  *out = b;
  return FORMGPU_OK;
}

void formgpu_batch_destroy(formgpu_batch *b) {
  if (!b) return;
  if (b->stream) cudaStreamSynchronize(b->stream);
  if (b->trace.on && (b->trace.rounds[0] || b->trace.rounds[1])) {
    const formgpu_batch::Trace &t = b->trace;
    for (int k = 0; k < 2; ++k)
      if (t.rounds[k])
        std::fprintf(stderr, "[formgpu batch %p] %s rounds %zu: build %.1f us, in flight before wait %.1f us, collect %.1f us\n",
                     (void *)b, k ? "extract" : "other  ", t.rounds[k], t.build_us[k] / t.rounds[k],
                     t.flight_us[k] / t.rounds[k], t.collect_us[k] / t.rounds[k]);
    std::fprintf(stderr, "[formgpu batch %p] idle between rounds %.1f us/round; extract rounds: flag wait %.1f us, keypoint DMA %.1f us; block wait %.1f us/round; builds > 1.5 ms: %zu\n",
                 (void *)b, t.idle_us / (t.rounds[0] + t.rounds[1]), t.rounds[1] ? t.extract_wait_us / t.rounds[1] : 0.0,
                 t.rounds[1] ? t.dma_us / t.rounds[1] : 0.0, t.blocks_wait_us / (t.rounds[0] + t.rounds[1]), t.build_outliers);
  }
  for (formgpu_ctx *c : b->ctx) formgpu_destroy(c);
  if (b->h_args) cudaFreeHost(b->h_args);
  if (b->d_args) cudaFree(b->d_args);
  if (b->h_done) cudaFreeHost(const_cast<uint32_t *>(b->h_done));
  if (b->d_blocks) cudaFree(b->d_blocks);
  if (b->h_blocks) cudaFreeHost(b->h_blocks);
  b->prof.destroy();
  if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
  delete b;
}

size_t formgpu_batch_size(const formgpu_batch *b) { return b ? b->ctx.size() : 0; }

formgpu_ctx *formgpu_batch_ctx(formgpu_batch *b, size_t i) {
  return (b && i < b->ctx.size()) ? b->ctx[i] : nullptr;
}

int formgpu_batch_profile_enable(formgpu_batch *b, int on) {
  if (!b) return FORMGPU_ERR_INVALID_ARG;
  b->prof.collect();
  b->prof.timing = on != 0;
  return FORMGPU_OK;
}

int formgpu_batch_profile_read(formgpu_batch *b, double ms[FORMGPU_KG_COUNT],
                               uint64_t launches[FORMGPU_KG_COUNT]) {
  if (!b) return FORMGPU_ERR_INVALID_ARG;
  b->prof.collect();
  for (int g = 0; g < FORMGPU_KG_COUNT; ++g) {
    if (ms) ms[g] = b->prof.group[g].ms;
    if (launches) launches[g] = b->prof.group[g].launches;
    b->prof.group[g] = GroupProf();
  }
  return FORMGPU_OK;
}

uint64_t formgpu_batch_launch_count(const formgpu_batch *b) { return b ? b->prof.total_launches : 0; }

} // extern "C"

namespace {

// Build phase of a submission: validate, stage every group's argument blocks, ONE upload, queue
// every group's kernels.  Nothing is waited for.  An early return (bad request list, CUDA error)
// leaves the requests it did not reach untouched - the caller stamps them.
int submit_build(formgpu_batch *b, formgpu_request *reqs, size_t n) {
  BATCH_CUDA(b, cudaSetDevice(b->device));
  const size_t S = b->ctx.size();
  formgpu_batch::Pending &pend = b->pend;
  pend.reqs = reqs;
  pend.n = n;
  pend.first_error = FORMGPU_OK;
  pend.live_extract.clear();
  pend.live_assoc.clear();
  pend.live_lin[0].clear();
  pend.live_lin[1].clear();
  pend.live_commit.clear();
  std::vector<size_t> &live_extract = pend.live_extract, &live_assoc = pend.live_assoc,
                      &live_commit = pend.live_commit;
  std::vector<size_t>(&live_lin)[2] = pend.live_lin;
  int &first_error = pend.first_error;

  // ---- validate: known ops, one request per sequence ----
  std::vector<uint8_t> seen(S, 0);
  std::vector<size_t> by_op[FORMGPU_OP_COUNT];
  for (size_t r = 0; r < n; ++r) {
    formgpu_request &q = reqs[r];
    q.status = FORMGPU_OK;
    if (q.sequence >= S || q.op >= FORMGPU_OP_COUNT)
      return bfail(b, FORMGPU_ERR_INVALID_ARG, "formgpu_batch_submit: bad sequence index or op");
    if (seen[q.sequence])
      return bfail(b, FORMGPU_ERR_INVALID_ARG, "formgpu_batch_submit: two requests for one sequence");
    if (b->ctx[q.sequence]->shard_world > 1 || b->ctx[q.sequence]->comm)
      return bfail(b, FORMGPU_ERR_UNSUPPORTED,
                   "formgpu_batch_submit: point-sharded contexts (formgpu_set_shard) are not batched");
    seen[q.sequence] = 1;
    by_op[q.op].push_back(r);
  }
  // the previous submission's argument upload has been consumed before the ring restarts: its
  // completion word was waited for (formgpu_batch_wait), and the word is raised behind everything
  {
    const int rc = wait_done(b, 0, b->done_seq);
    if (rc) return rc;
  }
  b->blocks_used = 0;
  {
    // upper bound of the block words this submission can produce (sized before anything is staged:
    // the argument blocks carry pointers into d_blocks)
    size_t doubles = 0;
    for (size_t r : by_op[FORMGPU_OP_ASSOC_LIN]) doubles += 91 * (size_t)b->ctx[reqs[r].sequence]->W;
    for (size_t r : by_op[FORMGPU_OP_LINEARIZE]) doubles += 91 * reqs[r].n_pairs;
    const int rc = ensure_blocks(b, doubles);
    if (rc) return rc;
  }
  b->args_used = 0;
  auto set_status = [&](formgpu_request &q, int rc) {
    q.status = rc;
    if (rc != FORMGPU_OK && first_error == FORMGPU_OK) {
      first_error = rc;
      b->err = std::string("sequence ") + std::to_string(q.sequence) + ": " + formgpu_last_error(b->ctx[q.sequence]);
    }
  };

  // =====================================================================================
  // build phase: argument blocks of every group are staged in pinned memory; ONE upload
  // and then every group's kernels go onto the stream before the first wait
  // =====================================================================================
  std::vector<std::function<int()>> launchers;

  // ---- host-only: remove ----
  for (size_t r : by_op[FORMGPU_OP_REMOVE]) {
    formgpu_request &q = reqs[r];
    set_status(q, formgpu_remove_scans(b->ctx[q.sequence], q.scans, q.n_scans));
  }

  // ---- stage 1 ----
  std::function<int()> extract_launcher; // queued after every other group: extraction is the long pole
  // host scans of this submission: device buffer, source, bytes (each sequence's own point count)
  std::vector<std::tuple<void *, const void *, size_t>> scan_uploads;
  {
    std::vector<ExtractArgs> items;
    // raw clouds of this submission (FORMGPU_REQ_CLOUD): organised into their sequences' scan buffers
    // by one launch per kernel, queued right before the extraction
    std::vector<OrganizeArgs> cloud_items;
    std::vector<formgpu_ctx *> cloud_ctx;
    size_t max_records = 0, max_pixels = 0;
    for (size_t r : by_op[FORMGPU_OP_EXTRACT]) {
      formgpu_request &q = reqs[r];
      formgpu_ctx *ctx = b->ctx[q.sequence];
      const bool cloud = (q.flags & FORMGPU_REQ_CLOUD) != 0;
      if (cloud) {
        const int rc = cloud_check_request(ctx, q.scan, q.n_points, "extract (cloud)");
        if (rc) {
          set_status(q, rc);
          continue;
        }
      }
      if (!q.scan) {
        set_status(q, fail(ctx, FORMGPU_ERR_INVALID_ARG, "extract: null scan"));
        continue;
      }
      if (!cloud && q.n_points != ctx->n_points) {
        set_status(q, fail(ctx, FORMGPU_ERR_BAD_SCAN_SIZE,
                           "Provided scan does not match the expected size " +
                               std::to_string(ctx->n_points) + " != " + std::to_string(q.n_points)));
        continue;
      }
      const bool on_device = (q.flags & FORMGPU_REQ_SCAN_ON_DEVICE) != 0;
      const float4 *scan_dev = reinterpret_cast<const float4 *>(q.scan);
      formgpu_planar_feat *dp = nullptr;
      formgpu_point_feat *dq = nullptr;
      bool host_records = false;
      if (cloud) {
        const unsigned char *rec = reinterpret_cast<const unsigned char *>(q.scan);
        if (!on_device) {
          if (!(ctx->prefetched_cloud == q.scan && ctx->prefetched_cloud_n == q.n_points) && q.n_points)
            scan_uploads.emplace_back(ctx->d_records, q.scan, q.n_points * ctx->cloud.stride);
          rec = ctx->d_records;
        }
        ctx->prefetched_cloud = nullptr;
        ctx->prefetched_host = nullptr; // a prefetched organised scan is discarded, as for another pointer
        cloud_items.push_back(cloud_args(ctx, rec, q.n_points));
        cloud_ctx.push_back(ctx);
        ctx->cloud_last_n = q.n_points;
        max_records = std::max(max_records, q.n_points);
        max_pixels = std::max(max_pixels, ctx->n_points);
        scan_dev = ctx->d_scan;
      }
      if (!on_device) {
        if (cloud) {
          // organised on the device into d_scan (above)
        } else if (ctx->d_scan_next && ctx->prefetched_host == q.scan) {
          // uploaded ahead of this request (formgpu_batch_prefetch_scan, same stream): adopt the buffer
          std::swap(ctx->d_scan, ctx->d_scan_next);
        } else {
          scan_uploads.emplace_back(ctx->d_scan, q.scan, ctx->n_points * sizeof(float4));
        }
        ctx->prefetched_host = nullptr;
        scan_dev = ctx->d_scan;
        if (q.planar_out && q.point_out) {
          // f64 structs into device staging; a copy engine takes them to the caller (collect phase)
          if (!ctx->d_stage_planar) {
            BATCH_CUDA(b, cudaMalloc(reinterpret_cast<void **>(&ctx->d_stage_planar), ctx->kp_cap * sizeof(formgpu_planar_feat)));
            BATCH_CUDA(b, cudaMalloc(reinterpret_cast<void **>(&ctx->d_stage_point), ctx->kq_cap * sizeof(formgpu_point_feat)));
          }
          dp = ctx->d_stage_planar;
          dq = ctx->d_stage_point;
        } else {
          extract_direct_targets(ctx, q.planar_out, q.planar_cap, q.point_out, q.point_cap, dp, dq);
        }
        host_records = dp == nullptr && (q.planar_out || q.point_out);
      }
      ExtractArgs &a = b->extract_args[q.sequence];
      extract_prepare(ctx, scan_dev, q.scan_idx, host_records, dp, dq, a);
      ctx->cur_device_resident = on_device;
      items.push_back(a);
      live_extract.push_back(r);
    }
    if (!items.empty()) {
      // ONE launch per kernel whatever the mix of scan shapes (DESIGN.md 6): the grid covers the
      // largest rows, shared memory is the largest need; a homogeneous submission gets exactly the
      // grid and shared memory of a single-shape launch
      size_t off = 0;
      const int rc = stage_args(b, items.data(), items.size(), &off);
      if (rc) return rc;
      const ExtractLaunchShape shape = extract_launch_shape(items.data(), (int)items.size());
      const int n_items = (int)items.size();
      size_t off_cloud = 0;
      if (!cloud_items.empty()) {
        const int rc2 = stage_args(b, cloud_items.data(), cloud_items.size(), &off_cloud);
        if (rc2) return rc2;
      }
      const int n_cloud = (int)cloud_items.size();
      extract_launcher = [=]() -> int {
        // on the batch's own stream, right before the kernels that read them (every other group of
        // the submission is already queued ahead): no side stream, no event pair per submission
        for (const auto &u : scan_uploads)
          BATCH_CUDA(b, cudaMemcpyAsync(std::get<0>(u), std::get<1>(u), std::get<2>(u), cudaMemcpyHostToDevice,
                                        b->stream));
        if (n_cloud) {
          organize_batch_launch(staged<OrganizeArgs>(b, off_cloud), n_cloud, max_records, max_pixels, b->stream,
                                b->prof);
          BATCH_CUDA(b, cudaGetLastError());
          for (formgpu_ctx *c : cloud_ctx)
            BATCH_CUDA(b, cudaMemcpyAsync(c->h_cloud_stats, c->d_cloud_stats, kOrgStats * sizeof(unsigned),
                                          cudaMemcpyDeviceToHost, b->stream));
        }
        extract_batch_launch(shape, staged<ExtractArgs>(b, off), n_items, b->many_rows_min, b->stream, b->prof);
        BATCH_CUDA(b, cudaGetLastError());
        return FORMGPU_OK;
      };
    }
  }

  // ---- reparative map rebuild ----
  {
    std::vector<MapArgs> items;
    std::vector<MapClearRegion> regions;
    int max_points = 0;
    uint32_t max_hash = 0;
    size_t max_clear = 0;
    for (size_t r : by_op[FORMGPU_OP_MAP_REBUILD]) {
      formgpu_request &q = reqs[r];
      formgpu_ctx *ctx = b->ctx[q.sequence];
      if (q.n_poses && !q.poses) {
        set_status(q, fail(ctx, FORMGPU_ERR_INVALID_ARG, "map_rebuild: null poses"));
        continue;
      }
      MapArgs a[2];
      MapClearRegion clear;
      int rc = map_rebuild_prepare(ctx, q.poses, q.n_poses, b->stream, a, clear, false);
      if (rc) {
        set_status(q, rc);
        continue;
      }
      {
        // the request travels with the submission's arguments; the clear kernel puts it in place
        size_t off_req = 0;
        rc = stage_args(b, reinterpret_cast<const unsigned char *>(ctx->h_map_req), ctx->map_req_bytes, &off_req);
        if (rc) return rc;
        clear.copy_src_off = off_req;
        clear.copy_dst = ctx->d_map_req;
        clear.copy_bytes = ctx->map_req_bytes;
      }
      items.push_back(a[0]);
      items.push_back(a[1]);
      regions.push_back(clear);
      max_points = std::max(max_points, std::max(a[0].n_total, a[1].n_total));
      max_hash = std::max(max_hash, std::max(a[0].hash_mask, a[1].hash_mask) + 1);
      max_clear = std::max(max_clear, clear.bytes);
    }
    if (!regions.empty()) {
      size_t off_items = 0, off_regions = 0;
      int rc = stage_args(b, items.data(), items.size(), &off_items);
      if (rc) return rc;
      rc = stage_args(b, regions.data(), regions.size(), &off_regions);
      if (rc) return rc;
      const int n_items = (int)regions.size();
      launchers.push_back([=]() -> int {
        map_build_batch_launch(staged<MapArgs>(b, off_items), staged<MapClearRegion>(b, off_regions), b->d_args, n_items,
                               max_points, max_hash, max_clear, b->stream, b->prof);
        BATCH_CUDA(b, cudaGetLastError());
        return FORMGPU_OK;
      });
    }
  }

  // ---- association (+ fused linearisation of the current scan's pairs) ----
  {
    std::vector<AssocArgs> aitems;
    std::vector<SegmentArgs> sitems;
    std::vector<MomentArgs> mitems;
    int max_units = 0;
    std::vector<LinArgs> lin_ctx;
    std::vector<LinTask> &lin_tasks = b->tasks_scratch;
    lin_tasks.clear();
    int max_query = 0;
    for (int pass = 0; pass < 2; ++pass) {
      const int op = pass == 0 ? FORMGPU_OP_ASSOCIATE : FORMGPU_OP_ASSOC_LIN;
      for (size_t r : by_op[op]) {
        formgpu_request &q = reqs[r];
        formgpu_ctx *ctx = b->ctx[q.sequence];
        const formgpu_pose *pose_k = q.pose_k;
        if (op == FORMGPU_OP_ASSOC_LIN) {
          pose_k = nullptr;
          if (q.poses && q.out && ctx->have_current)
            for (size_t p = 0; p < q.n_poses; ++p)
              if (q.poses[p].scan == ctx->cur_scan) pose_k = &q.poses[p].pose;
        }
        if (!pose_k) {
          set_status(q, fail(ctx, FORMGPU_ERR_INVALID_ARG, "associate: missing pose / output argument"));
          continue;
        }
        AssocPlan &plan = b->assoc_plans[q.sequence];
        const bool want_blocks = op == FORMGPU_OP_ASSOC_LIN;
        const int rc = assoc_prepare(ctx, pose_k, want_blocks ? q.poses : nullptr, q.n_poses, want_blocks, plan);
        if (rc) {
          set_status(q, rc);
          continue;
        }
        live_assoc.push_back(r);
        b->assoc_block_off[q.sequence] = kNoBlocks;
        if (!plan.any_query) continue;
        aitems.push_back(plan.aa[0]);
        aitems.push_back(plan.aa[1]);
        sitems.push_back(plan.sa[0]);
        sitems.push_back(plan.sa[1]);
        mitems.push_back(plan.ma);
        max_units = std::max(max_units, plan.mom_units);
        max_query = std::max(max_query, std::max(plan.nq[0], plan.nq[1]));
        if (plan.fused && !plan.lin_tasks.empty()) {
          LinArgs la;
          lin_make_args(ctx, (int)plan.lin_tasks.size(), la);
          plan.lin_seq = la.seq;
          la.out_plain = b->d_blocks + b->blocks_used;
          b->assoc_block_off[q.sequence] = b->blocks_used;
          b->blocks_used += 91 * plan.lin_tasks.size();
          const uint32_t ci = (uint32_t)lin_ctx.size();
          lin_ctx.push_back(la);
          for (LinTask t : plan.lin_tasks) {
            t.ctx_index = ci;
            lin_tasks.push_back(t);
          }
        } else if (plan.fused) {
          LinArgs la;
          lin_make_args(ctx, 0, la); // no other scan has a pose: nothing to linearise
          plan.lin_seq = la.seq;
        }
      }
    }
    if (!aitems.empty()) {
      size_t off_a = 0, off_s = 0, off_m = 0;
      int rc = stage_args(b, aitems.data(), aitems.size(), &off_a);
      if (rc) return rc;
      rc = stage_args(b, sitems.data(), sitems.size(), &off_s);
      if (rc) return rc;
      rc = stage_args(b, mitems.data(), mitems.size(), &off_m);
      if (rc) return rc;
      const int n_items = (int)aitems.size() / 2;
      launchers.push_back([=]() -> int {
        assoc_batch_launch(staged<AssocArgs>(b, off_a), n_items, max_query, b->stream, b->prof);
        segment_build_batch_launch(staged<SegmentArgs>(b, off_s), n_items, max_query, b->stream, b->prof);
        moments_batch_launch(staged<MomentArgs>(b, off_m), n_items, max_units, b->stream, b->prof);
        BATCH_CUDA(b, cudaGetLastError());
        return FORMGPU_OK;
      });
      rc = stage_lin_groups(b, lin_ctx, lin_tasks, false, launchers);
      if (rc) return rc;
    }
  }

  // ---- linearisation / error of listed pairs ----
  for (int eo = 0; eo < 2; ++eo) {
    const int op = eo ? FORMGPU_OP_ERROR : FORMGPU_OP_LINEARIZE;
    const size_t per_pair = eo ? 1 : 91;
    std::vector<LinArgs> lin_ctx;
    std::vector<LinTask> &lin_tasks = b->tasks_scratch;
    std::vector<LinTask> tasks;
    lin_tasks.clear();
    for (size_t r : by_op[op]) {
      formgpu_request &q = reqs[r];
      formgpu_ctx *ctx = b->ctx[q.sequence];
      if (q.n_pairs == 0) {
        b->lin_indices[q.sequence].clear();
        live_lin[eo].push_back(r);
        b->lin_seqs[q.sequence] = 0;
        continue;
      }
      if (!q.pairs || !q.out || (q.n_poses && !q.poses)) {
        set_status(q, fail(ctx, FORMGPU_ERR_INVALID_ARG, "linearize: null argument"));
        continue;
      }
      const int rc = lin_build_tasks(ctx, q.pairs, q.n_pairs, q.poses, q.n_poses, per_pair, q.out, tasks,
                                     b->lin_indices[q.sequence]);
      if (rc) {
        set_status(q, rc);
        continue;
      }
      LinArgs la;
      lin_make_args(ctx, (int)tasks.size(), la);
      b->lin_seqs[q.sequence] = la.seq;
      live_lin[eo].push_back(r);
      if (!eo) b->lin_block_off[q.sequence] = kNoBlocks;
      if (tasks.empty()) continue;
      if (!eo) {
        la.out_plain = b->d_blocks + b->blocks_used; // task.out_index = position in q.pairs
        b->lin_block_off[q.sequence] = b->blocks_used;
        b->blocks_used += 91 * q.n_pairs;
      }
      const uint32_t ci = (uint32_t)lin_ctx.size();
      lin_ctx.push_back(la);
      for (LinTask &t : tasks) {
        t.ctx_index = ci;
        lin_tasks.push_back(t);
      }
    }
    const int rc = stage_lin_groups(b, lin_ctx, lin_tasks, eo != 0, launchers);
    if (rc) return rc;
  }
  // ---- commit ----
  {
    std::vector<CommitArgs> items;
    int max_query = 0;
    for (size_t r : by_op[FORMGPU_OP_COMMIT]) {
      formgpu_request &q = reqs[r];
      formgpu_ctx *ctx = b->ctx[q.sequence];
      CommitPlan &plan = b->commit_plans[q.sequence];
      const int rc = commit_prepare(ctx, plan);
      if (rc) {
        set_status(q, rc);
        continue;
      }
      live_commit.push_back(r);
      items.push_back(plan.ca[0]);
      items.push_back(plan.ca[1]);
      max_query = std::max(max_query, std::max(plan.ca[0].n_query, plan.ca[1].n_query));
    }
    if (!items.empty() && max_query > 0) {
      size_t off = 0;
      const int rc = stage_args(b, items.data(), items.size(), &off);
      if (rc) return rc;
      const int n_items = (int)items.size() / 2;
      launchers.push_back([=]() -> int {
        commit_batch_launch(staged<CommitArgs>(b, off), n_items, max_query, b->stream, b->prof);
        BATCH_CUDA(b, cudaGetLastError());
        return FORMGPU_OK;
      });
    }
  }
  // one upload for the whole submit, then every group's kernels
  if (b->args_used)
    BATCH_CUDA(b, cudaMemcpyAsync(b->d_args, b->h_args, b->args_used, cudaMemcpyHostToDevice, b->stream));
  for (auto &launch : launchers) {
    const int rc = launch();
    if (rc) return rc;
  }
  if (extract_launcher) {
    const int rc = extract_launcher();
    if (rc) return rc;
  }
  // every block of the submission goes home in ONE transfer, behind the last kernel (the collect
  // phase waits for the whole submission anyway), and the completion word behind that
  if (b->blocks_used)
    BATCH_CUDA(b, cudaMemcpyAsync(b->h_blocks, b->d_blocks, b->blocks_used * sizeof(double), cudaMemcpyDeviceToHost,
                                  b->stream));
  return queue_flag(b, 0, ++b->done_seq);
}

// Collect phase: wait for the results of the submission in flight (mapped-memory flags and
// tagged words, as the single-sequence calls) and fill the requests' output fields.
int submit_collect(formgpu_batch *b) {
  formgpu_batch::Pending &pend = b->pend;
  formgpu_request *reqs = pend.reqs;
  int &first_error = pend.first_error;
  auto set_status = [&](formgpu_request &q, int rc) {
    q.status = rc;
    if (rc != FORMGPU_OK && first_error == FORMGPU_OK) {
      first_error = rc;
      b->err = std::string("sequence ") + std::to_string(q.sequence) + ": " + formgpu_last_error(b->ctx[q.sequence]);
    }
  };
  const std::vector<size_t> &live_extract = pend.live_extract, &live_assoc = pend.live_assoc,
                            &live_commit = pend.live_commit;
  const std::vector<size_t>(&live_lin)[2] = pend.live_lin;
  bool dma_pending = false;
  const auto tc00 = std::chrono::steady_clock::now();
  {
    // ONE wait for the whole submission: the word is raised behind its last operation, so every
    // flag and tagged word the per-request code below looks at has already arrived
    const int rc = wait_done(b, 0, b->done_seq);
    if (rc) return rc;
  }
  const auto tc0 = std::chrono::steady_clock::now();
  for (size_t r : live_extract) {
    formgpu_request &q = reqs[r];
    formgpu_ctx *ctx = b->ctx[q.sequence];
    const ExtractArgs &a = b->extract_args[q.sequence];
    int rc = extract_finish(ctx, a, q.scan_idx);
    if (rc == FORMGPU_OK) {
      q.n_planar = (size_t)ctx->cur_n[0];
      q.n_point = (size_t)ctx->cur_n[1];
      if (a.host_planar || a.host_point) {
        rc = extract_widen(ctx, q.scan_idx, q.planar_out, q.planar_cap, q.point_out, q.point_cap);
      } else if (a.host_planar_f64 && a.host_planar_f64 == ctx->d_stage_planar) {
        // the counts are known now: exactly the written structs travel (the batch's stream is idle)
        if (q.n_planar > q.planar_cap || q.n_point > q.point_cap) {
          rc = fail(ctx, FORMGPU_ERR_CAPACITY, "formgpu_extract: output buffers too small");
        } else {
          dma_pending = true; // the stream is idle: the copies start at once
          if (q.n_planar)
            BATCH_CUDA(b, cudaMemcpyAsync(q.planar_out, ctx->d_stage_planar, q.n_planar * sizeof(formgpu_planar_feat),
                                          cudaMemcpyDeviceToHost, b->stream));
          if (q.n_point)
            BATCH_CUDA(b, cudaMemcpyAsync(q.point_out, ctx->d_stage_point, q.n_point * sizeof(formgpu_point_feat),
                                          cudaMemcpyDeviceToHost, b->stream));
        }
      }
    }
    set_status(q, rc);
  }
  const auto tc1 = std::chrono::steady_clock::now();
  if (dma_pending) {
    // keypoint copies queued above: their own completion word, polled without CUDA calls while
    // the remaining requests are collected
    const int rc = queue_flag(b, 1, ++b->kp_seq);
    if (rc) return rc;
  }
  if (b->trace.on) {
    b->trace.blocks_wait_us += std::chrono::duration<double, std::micro>(tc0 - tc00).count();
    b->trace.extract_wait_us += std::chrono::duration<double, std::micro>(tc1 - tc0).count();
  }
  for (size_t r : live_assoc) {
    formgpu_request &q = reqs[r];
    formgpu_ctx *ctx = b->ctx[q.sequence];
    AssocPlan &plan = b->assoc_plans[q.sequence];
    const bool want_blocks = q.op == FORMGPU_OP_ASSOC_LIN;
    const size_t off = want_blocks && plan.fused ? b->assoc_block_off[q.sequence] : kNoBlocks;
    set_status(q, assoc_finish(ctx, plan, q.poses, q.n_poses, q.counts_out, q.counts_cap, &q.n_counts,
                               want_blocks ? q.out : nullptr, off != kNoBlocks ? b->h_blocks + off : nullptr));
  }
  for (int eo = 0; eo < 2; ++eo)
    for (size_t r : live_lin[eo]) {
      formgpu_request &q = reqs[r];
      if (q.n_pairs == 0) continue;
      const std::vector<int> &indices = b->lin_indices[q.sequence];
      const size_t off = eo ? kNoBlocks : b->lin_block_off[q.sequence];
      if (off != kNoBlocks) {
        for (int p : indices)
          std::memcpy(q.out + 91 * (size_t)p, b->h_blocks + off + 91 * (size_t)p, 91 * sizeof(double));
        continue;
      }
      if (indices.empty()) continue;
      set_status(q, lin_collect(b->ctx[q.sequence], indices, b->lin_seqs[q.sequence], eo ? 1 : 91, q.out));
    }
  for (size_t r : live_commit) {
    formgpu_request &q = reqs[r];
    const CommitPlan &plan = b->commit_plans[q.sequence];
    commit_finish(b->ctx[q.sequence], plan);
    q.n_planar = plan.added[0];
    q.n_point = plan.added[1];
  }
  if (dma_pending) {
    const auto td0 = std::chrono::steady_clock::now();
    const int rc = wait_done(b, 1, b->kp_seq); // keypoints have landed
    if (rc) return rc;
    if (b->trace.on) b->trace.dma_us += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - td0).count();
  }
  if (b->prof.timing) b->prof.collect();
  return first_error;
}

} // namespace

extern "C" {

int formgpu_batch_submit_async(formgpu_batch *b, formgpu_request *reqs, size_t n) {
  if (!b) return FORMGPU_ERR_INVALID_ARG;
  if (b->pend.active)
    return bfail(b, FORMGPU_ERR_STATE, "formgpu_batch_submit_async: the previous submission has not been waited for");
  if (n == 0) return FORMGPU_OK;
  if (!reqs) return bfail(b, FORMGPU_ERR_INVALID_ARG, "formgpu_batch_submit: null requests");
  for (size_t r = 0; r < n; ++r) reqs[r].status = FORMGPU_OK;
  if (b->trace.on) {
    b->trace.t_submit = std::chrono::steady_clock::now();
    if (b->trace.have_done)
      b->trace.idle_us += std::chrono::duration<double, std::micro>(b->trace.t_submit - b->trace.t_done).count();
    b->trace.kind = 0;
    for (size_t r = 0; r < n; ++r)
      if (reqs[r].op == FORMGPU_OP_EXTRACT) b->trace.kind = 1;
  }
  const int rc = submit_build(b, reqs, n);
  if (b->trace.on) {
    b->trace.t_built = std::chrono::steady_clock::now();
    const double us = std::chrono::duration<double, std::micro>(b->trace.t_built - b->trace.t_submit).count();
    if (us < 1500.0) b->trace.build_us[b->trace.kind] += us; // first-use allocations are counted apart
    else b->trace.build_outliers += 1;
  }
  if (rc != FORMGPU_OK) {
    // aborted before the collect phase: no request may be taken for completed.  Whatever was
    // already queued is drained so that the caller can reuse its buffers.
    cudaStreamSynchronize(b->stream);
    for (size_t r = 0; r < n; ++r)
      if (reqs[r].status == FORMGPU_OK) reqs[r].status = rc;
    return rc;
  }
  b->pend.active = true;
  return FORMGPU_OK;
}

int formgpu_batch_wait(formgpu_batch *b) {
  if (!b) return FORMGPU_ERR_INVALID_ARG;
  if (!b->pend.active) return FORMGPU_OK;
  b->pend.active = false;
  if (!b->trace.on) return submit_collect(b);
  const auto t0 = std::chrono::steady_clock::now();
  const int rc = submit_collect(b);
  formgpu_batch::Trace &t = b->trace;
  t.t_done = std::chrono::steady_clock::now();
  t.have_done = true;
  t.flight_us[t.kind] += std::chrono::duration<double, std::micro>(t0 - t.t_built).count();
  t.collect_us[t.kind] += std::chrono::duration<double, std::micro>(t.t_done - t0).count();
  t.rounds[t.kind] += 1;
  return rc;
}

int formgpu_batch_done(formgpu_batch *b) {
  if (!b) return -FORMGPU_ERR_INVALID_ARG;
  if (!b->pend.active) return 1;
  if (b->h_done[0] == b->done_seq) return 1;
  // a caller that polls this in a loop must not enter the driver every time: the stream state is
  // looked at (so that a faulted kernel is noticed) once in 4096 polls
  if ((++b->done_polls & 0xfffu) != 0u) return 0;
  const cudaError_t e = cudaStreamQuery(b->stream);
  if (e == cudaSuccess || e == cudaErrorNotReady) return b->h_done[0] == b->done_seq ? 1 : 0;
  b->err = std::string("cudaStreamQuery: ") + cudaGetErrorString(e);
  return -FORMGPU_ERR_CUDA;
}

int formgpu_batch_prefetch_scan(formgpu_batch *b, size_t sequence, const formgpu_point4f *scan, size_t n_points) {
  if (!b || sequence >= b->ctx.size() || !scan) return bfail(b, FORMGPU_ERR_INVALID_ARG, "formgpu_batch_prefetch_scan: bad argument");
  formgpu_ctx *ctx = b->ctx[sequence];
  if (n_points != ctx->n_points)
    return bfail(b, FORMGPU_ERR_BAD_SCAN_SIZE, "formgpu_batch_prefetch_scan: scan does not match the expected size");
  BATCH_CUDA(b, cudaSetDevice(b->device));
  if (!ctx->d_scan_next) {
    BATCH_CUDA(b, cudaMalloc(reinterpret_cast<void **>(&ctx->d_scan_next), ctx->n_points * sizeof(float4)));
  }
  // d_scan_next is free: the extraction that last read it (as d_scan, before a swap) has been
  // waited for - a sequence has one request per submission and prefetches between them
  // on the batch's own stream: in order with the extraction that will read it, no event needed
  BATCH_CUDA(b, cudaMemcpyAsync(ctx->d_scan_next, scan, n_points * sizeof(float4), cudaMemcpyHostToDevice,
                                b->stream));
  ctx->prefetched_host = scan;
  return FORMGPU_OK;
}

int formgpu_batch_prefetch_cloud(formgpu_batch *b, size_t sequence, const void *records, size_t n) {
  if (!b || sequence >= b->ctx.size() || !records)
    return bfail(b, FORMGPU_ERR_INVALID_ARG, "formgpu_batch_prefetch_cloud: bad argument");
  formgpu_ctx *ctx = b->ctx[sequence];
  const int rc = cloud_check_request(ctx, records, n, "formgpu_batch_prefetch_cloud");
  if (rc) return bfail(b, rc, formgpu_last_error(ctx));
  BATCH_CUDA(b, cudaSetDevice(b->device));
  // d_records is free: the submission that last read it has been waited for; same stream as the
  // organisation that will read it, so no event is needed
  if (n)
    BATCH_CUDA(b, cudaMemcpyAsync(ctx->d_records, records, n * ctx->cloud.stride, cudaMemcpyHostToDevice, b->stream));
  ctx->prefetched_cloud = records;
  ctx->prefetched_cloud_n = n;
  return FORMGPU_OK;
}

int formgpu_batch_submit(formgpu_batch *b, formgpu_request *reqs, size_t n) {
  const int rc = formgpu_batch_submit_async(b, reqs, n);
  if (rc != FORMGPU_OK) return rc;
  return formgpu_batch_wait(b);
}

} // extern "C"
