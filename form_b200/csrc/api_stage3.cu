// C-ABI (include/formgpu.h): stage 3 - linearisation and error evaluation.
#include "api_common.hpp"

using namespace formgpu;

namespace formgpu {

// relative pose of scan j seen from scan i: R_i^T R_j and R_i^T (t_j - t_i)
void relative_pose(const formgpu_pose &Ti, const formgpu_pose &Tj, double rel[12]) {
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b)
      rel[3 * a + b] = Ti.R[a] * Tj.R[b] + Ti.R[3 + a] * Tj.R[3 + b] + Ti.R[6 + a] * Tj.R[6 + b];
  const double d[3] = {Tj.t[0] - Ti.t[0], Tj.t[1] - Ti.t[1], Tj.t[2] - Ti.t[2]};
  for (int a = 0; a < 3; ++a) rel[9 + a] = Ti.R[a] * d[0] + Ti.R[3 + a] * d[1] + Ti.R[6 + a] * d[2];
}

void lin_make_args(formgpu_ctx *ctx, int n_tasks, LinArgs &a) {
  a = LinArgs{};
  a.kp_cap = ctx->kp_cap;
  a.kq_cap = ctx->kq_cap;
  a.seg_planar = ctx->d_seg_planar;
  a.seg_point = ctx->d_seg_point;
  a.pair_row = ctx->d_pair;
  a.W = ctx->W;
  a.n_tasks = n_tasks;
  // CTAs per pair: as many as keep the launch within about one wave (2 CTAs per SM)
  a.cluster = kLinCluster;
  while (a.cluster > 1 && (size_t)a.cluster * (size_t)n_tasks > 2 * 148) a.cluster >>= 1;
  a.inv_sigma2 = 1.0 / (ctx->P.sigma * ctx->P.sigma);
  a.out = ctx->h_out;
  a.seq = ++ctx->seq;
  a.shard_rank = ctx->shard_rank;
  a.shard_world = ctx->shard_world;
  a.out_plain = nullptr;
  a.moments = ctx->d_moments;
}

int lin_launch(formgpu_ctx *ctx, const std::vector<LinTask> &tasks, bool error_only,
               unsigned long long *seq_out, double *out_plain) {
  LinArgs a;
  lin_make_args(ctx, (int)tasks.size(), a);
  a.out_plain = out_plain;
  *seq_out = a.seq;
  if (tasks.empty()) return FORMGPU_OK;
  const bool cached = use_moment_cache(ctx);
  if ((int)tasks.size() <= kLinInlineTasks) {
    // the whole request rides in the kernel parameters: no upload, no dependent loads
    static thread_local LinInline inl;
    std::memcpy(inl.tasks, tasks.data(), tasks.size() * sizeof(LinTask));
    if (cached) FORMGPU_CUDA(ctx, eval_launch(a, &inl, error_only, ctx->stream, ctx->prof));
    else FORMGPU_CUDA(ctx, linearize_launch(a, &inl, error_only, ctx->stream, ctx->prof));
  } else {
    // tasks, then (for the cached evaluation, whose kernel takes its argument block from
    // device memory) the argument block itself
    const size_t bytes = tasks.size() * sizeof(LinTask);
    FORMGPU_CUDA(ctx, cudaEventSynchronize(ctx->ev_upload));
    const int rc = ensure_upload(ctx, bytes + sizeof(LinArgs));
    if (rc) return rc;
    a.tasks = static_cast<const LinTask *>(ctx->d_request);
    std::memcpy(ctx->h_upload, tasks.data(), bytes);
    std::memcpy(static_cast<unsigned char *>(ctx->h_upload) + bytes, &a, sizeof(LinArgs));
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_request, ctx->h_upload, bytes + sizeof(LinArgs),
                                      cudaMemcpyHostToDevice, ctx->stream));
    FORMGPU_CUDA(ctx, cudaEventRecord(ctx->ev_upload, ctx->stream));
    if (cached) FORMGPU_CUDA(ctx, eval_launch(a, nullptr, error_only, ctx->stream, ctx->prof));
    else FORMGPU_CUDA(ctx, linearize_launch(a, nullptr, error_only, ctx->stream, ctx->prof));
  }
  return FORMGPU_OK;
}

int lin_wait(formgpu_ctx *ctx, const int *out_indices, size_t n, unsigned long long seq,
             size_t per_pair, double *dst) {
  // Each 8-byte word = 32 bits of payload | tag << 32; a word is fresh once its tag is
  // this call's.  Pairs (and words) complete in no particular order.
  const unsigned long long tag = seq & 0xffffffffull;
  const size_t words = 2 * per_pair; // words per pair in h_out: 182 (blocks) or 2 (errors)
  unsigned spins = 0;
  for (size_t k = 0; k < n; ++k) {
    volatile unsigned long long *w = ctx->h_out + (size_t)out_indices[k] * words;
    for (size_t e = 0; e < per_pair; ++e) {
      unsigned long long lo, hi;
      for (;;) {
        lo = w[2 * e];
        hi = w[2 * e + 1];
        if ((lo >> 32) == tag && (hi >> 32) == tag) break;
        if ((++spins & 0xfff) == 0) {
          const cudaError_t err = cudaStreamQuery(ctx->stream);
          if (err == cudaSuccess) {
            lo = w[2 * e];
            hi = w[2 * e + 1];
            if ((lo >> 32) == tag && (hi >> 32) == tag) break;
            return fail(ctx, FORMGPU_ERR_STATE, "linearize kernel finished without publishing a pair");
          }
          if (err != cudaErrorNotReady)
            return fail(ctx, FORMGPU_ERR_CUDA, std::string("linearize kernel failed: ") + cudaGetErrorString(err));
        }
        poll_relax(spins);
      }
      const unsigned long long bits = (lo & 0xffffffffull) | (hi << 32);
      std::memcpy(&dst[k * per_pair + e], &bits, sizeof(double));
    }
  }
  return FORMGPU_OK;
}

int lin_build_tasks(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                    const formgpu_scan_pose *poses, size_t n_poses, size_t per_pair, double *out,
                    std::vector<LinTask> &tasks, std::vector<int> &indices) {
  const int W = ctx->W;
  static thread_local std::vector<int> pose_idx;
  pose_idx.assign(W, -1);
  for (size_t p = 0; p < n_poses; ++p) {
    const int s = find_slot(ctx, poses[p].scan);
    if (s >= 0) pose_idx[s] = (int)p;
  }
  const int rc = ensure_out(ctx, n_pairs);
  if (rc) return rc;
  tasks.clear();
  indices.clear();
  for (size_t p = 0; p < n_pairs; ++p) {
    const int si = find_slot(ctx, pairs[p].i), sj = find_slot(ctx, pairs[p].j);
    const PairEntry *e = (si >= 0 && sj >= 0) ? &ctx->h_pair_table[(size_t)sj * W + si] : nullptr;
    if (!e || (e->n_planar == 0 && e->n_point == 0)) {
      // no correspondences (or unknown scans): zero block, never touched by a CTA
      std::memset(out + p * per_pair, 0, per_pair * sizeof(double));
      continue;
    }
    if (pose_idx[si] < 0 || pose_idx[sj] < 0)
      return fail(ctx, FORMGPU_ERR_INVALID_ARG,
                  "linearize: no pose given for a scan of pair (" + std::to_string(pairs[p].i) +
                      ", " + std::to_string(pairs[p].j) + ")");
    LinTask t{};
    relative_pose(poses[pose_idx[si]].pose, poses[pose_idx[sj]].pose, t.rel);
    t.off_planar = e->off_planar;
    t.n_planar = e->n_planar;
    t.off_point = e->off_point;
    t.n_point = e->n_point;
    t.slot_j = sj;
    t.slot_i = si;
    t.entry = ctx->d_moments + ((size_t)sj * W + si) * kMomentStride;
    t.out_index = (int)p;
    tasks.push_back(t);
    indices.push_back((int)p);
  }
  return FORMGPU_OK;
}

int lin_collect_comm(formgpu_ctx *ctx, size_t n_pairs, size_t per_pair, double *out) {
  const size_t count = n_pairs * per_pair;
  if (count == 0) return FORMGPU_OK;
  int rc = comm_allreduce_f64(ctx, ctx->d_red, count);
  if (rc) return rc;
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(ctx->h_red, ctx->d_red, count * sizeof(double), cudaMemcpyDeviceToHost,
                                    ctx->stream));
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  std::memcpy(out, ctx->h_red, count * sizeof(double));
  return FORMGPU_OK;
}

int lin_collect(formgpu_ctx *ctx, const std::vector<int> &indices, unsigned long long seq,
                size_t per_pair, double *out) {
  // decode into a dense scratch, then scatter to the pairs' positions
  static thread_local std::vector<double> dense;
  dense.resize(indices.size() * per_pair);
  const int rc = lin_wait(ctx, indices.data(), indices.size(), seq, per_pair, dense.data());
  if (rc) return rc;
  for (size_t k = 0; k < indices.size(); ++k)
    std::memcpy(out + (size_t)indices[k] * per_pair, dense.data() + k * per_pair, per_pair * sizeof(double));
  return FORMGPU_OK;
}

} // namespace formgpu

namespace {

// Shared body of formgpu_linearize / formgpu_error: one task per pair that has
// correspondences, one cluster per task, then poll the tagged words the kernel writes
// into mapped host memory.
int run(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs, const formgpu_scan_pose *poses,
        size_t n_poses, bool error_only, double *out) {
  const size_t per_pair = error_only ? 1 : 91;
  static thread_local std::vector<LinTask> tasks;
  static thread_local std::vector<int> indices;
  int rc = lin_build_tasks(ctx, pairs, n_pairs, poses, n_poses, per_pair, out, tasks, indices);
  if (rc) return rc;
  unsigned long long seq = 0;
  if (sharded_comm(ctx)) {
    // every rank evaluates the pairs from its partial moments into d_red (zeros for pairs without
    // a task), one all-reduce sums the blocks, the result is copied out
    rc = comm_ensure_reduce(ctx, n_pairs * per_pair);
    if (rc) return rc;
    FORMGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_red, 0, n_pairs * per_pair * sizeof(double), ctx->stream));
    rc = lin_launch(ctx, tasks, error_only, &seq, ctx->d_red);
    if (rc) return rc;
    return lin_collect_comm(ctx, n_pairs, per_pair, out);
  }
  rc = lin_launch(ctx, tasks, error_only, &seq);
  if (rc) return rc;
  return lin_collect(ctx, indices, seq, per_pair, out);
}

// device-output variants: blocks stay in device memory (zero-filled for empty pairs) and
// nothing is waited for - a collective queued on the same stream consumes them
int run_device(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs, const formgpu_scan_pose *poses,
               size_t n_poses, bool error_only, double *out_dev) {
  const size_t per_pair = error_only ? 1 : 91;
  static thread_local std::vector<LinTask> tasks;
  static thread_local std::vector<int> indices;
  static thread_local std::vector<double> sink;
  sink.resize(n_pairs * per_pair); // lin_build_tasks zero-fills the host slots of empty pairs
  int rc = lin_build_tasks(ctx, pairs, n_pairs, poses, n_poses, per_pair, sink.data(), tasks, indices);
  if (rc) return rc;
  FORMGPU_CUDA(ctx, cudaMemsetAsync(out_dev, 0, n_pairs * per_pair * sizeof(double), ctx->stream));
  unsigned long long seq = 0;
  return lin_launch(ctx, tasks, error_only, &seq, out_dev);
}

} // namespace

extern "C" {

int formgpu_set_shard(formgpu_ctx *ctx, int rank, int world) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (world < 1 || rank < 0 || rank >= world)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_set_shard: need 0 <= rank < world");
  ctx->shard_rank = rank;
  ctx->shard_world = world;
  return FORMGPU_OK;
}

int formgpu_linearize_device(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                             const formgpu_scan_pose *poses, size_t n_poses, double *out91_dev) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (n_pairs == 0) return FORMGPU_OK;
  if (!pairs || !out91_dev || (n_poses && !poses))
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_linearize_device: null argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  return run_device(ctx, pairs, n_pairs, poses, n_poses, false, out91_dev);
}

int formgpu_error_device(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                         const formgpu_scan_pose *poses, size_t n_poses, double *out_dev) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (n_pairs == 0) return FORMGPU_OK;
  if (!pairs || !out_dev || (n_poses && !poses))
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_error_device: null argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  return run_device(ctx, pairs, n_pairs, poses, n_poses, true, out_dev);
}

int formgpu_linearize(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                      const formgpu_scan_pose *poses, size_t n_poses, double *out91) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (n_pairs == 0) return FORMGPU_OK;
  if (!pairs || !out91 || (n_poses && !poses))
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_linearize: null argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  return run(ctx, pairs, n_pairs, poses, n_poses, false, out91);
}

int formgpu_error(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                  const formgpu_scan_pose *poses, size_t n_poses, double *out) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (n_pairs == 0) return FORMGPU_OK;
  if (!pairs || !out || (n_poses && !poses))
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_error: null argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  return run(ctx, pairs, n_pairs, poses, n_poses, true, out);
}

} // extern "C"
