// Helpers shared by the C-ABI translation units.
#pragma once

#include "ctx.hpp"
#include "kernels.hpp"

#include <cstdio>
#include <cstring>
#include <vector>

namespace formgpu {

inline int fail(const formgpu_ctx *ctx, int code, const std::string &msg) {
  if (ctx) ctx->err = msg;
  return code;
}

#define FORMGPU_CUDA(ctx, expr)                                                         \
  do {                                                                                  \
    cudaError_t e_ = (expr);                                                            \
    if (e_ != cudaSuccess)                                                              \
      return ::formgpu::fail((ctx), FORMGPU_ERR_CUDA,                                   \
                             std::string(#expr) + ": " + cudaGetErrorString(e_));      \
  } while (0)

/// Collects the event timings of an API call on scope exit (profiling mode only).
struct ProfScope {
  formgpu_ctx *ctx;
  explicit ProfScope(formgpu_ctx *c) : ctx(c) {}
  ~ProfScope() {
    if (ctx->prof.timing) ctx->prof.collect();
  }
};

template <typename T> inline cudaError_t dev_alloc(T **p, size_t count) {
  return cudaMalloc(reinterpret_cast<void **>(p), count * sizeof(T));
}

inline int find_slot(const formgpu_ctx *ctx, uint64_t scan) {
  auto it = ctx->slot_of.find(scan);
  return it == ctx->slot_of.end() ? -1 : it->second;
}

/// Spin until a kernel has published `seq` in the mapped flag.  Falls back to the
/// stream state every few thousand polls so a faulted kernel cannot hang the caller.
int wait_flag(formgpu_ctx *ctx, int which, unsigned long long seq);

/// One step of a result-polling loop: a pause, and - when FORMGPU_YIELD_WAIT=1 (more polling
/// host threads than cores, e.g. several batches per GPU on a box with two cores per GPU) - a
/// sched_yield() every 64 polls, so that a thread which is only waiting hands its core to one
/// that has a submit to build.  Without the variable the loop never enters the kernel.
void poll_relax(unsigned spins);
/// The parameter checks of formgpu_create that need no GPU: FORMGPU_OK, or an error code and `msg`.
int validate_params(const formgpu_params &P, std::string &msg);

/// Stage 3 building blocks (api_stage3.cu), also used by the fused association call.
void relative_pose(const formgpu_pose &Ti, const formgpu_pose &Tj, double rel[12]);
/// true: linearize / error of this context are evaluated from the pair-moment cache
inline bool use_moment_cache(const formgpu_ctx *ctx) { return ctx->moment_cache && ctx->shard_world == 1; }
/// true: the context is one rank of a point-sharded sequence (formgpu_comm_init)
inline bool sharded_comm(const formgpu_ctx *ctx) { return ctx->comm != nullptr && ctx->comm_world > 1; }
/// Launch one cluster per task - or, from the moment cache, one warp per task (no wait).
/// Assigns and returns the sequence number.
int lin_launch(formgpu_ctx *ctx, const std::vector<LinTask> &tasks, bool error_only,
               unsigned long long *seq_out, double *out_plain = nullptr);
/// Spin until every word of the listed pairs carries the call's tag, decoding them into
/// dst (per_pair = 91 doubles for blocks, 1 for errors; dst[k] belongs to out_indices[k]).
int lin_wait(formgpu_ctx *ctx, const int *out_indices, size_t n, unsigned long long seq,
             size_t per_pair, double *dst);

// ---- prepare / finish halves of the API calls (shared with the batched submit) ----

/// Stage 1: build the launch arguments of one scan (flips the keypoint ping-pong buffers,
/// assigns the completion sequence number) / wait for the pack kernel's flag and adopt
/// the scan as the context's current scan.
void extract_prepare(formgpu_ctx *ctx, const float4 *scan_dev, uint64_t scan_idx, bool host_records,
                     formgpu_planar_feat *direct_planar, formgpu_point_feat *direct_point,
                     ExtractArgs &a);
int extract_finish(formgpu_ctx *ctx, const ExtractArgs &a, uint64_t scan_idx);
void extract_direct_targets(formgpu_ctx *ctx, formgpu_planar_feat *planar_out, size_t planar_cap,
                            formgpu_point_feat *point_out, size_t point_cap,
                            formgpu_planar_feat *&dp, formgpu_point_feat *&dq);
int extract_widen(formgpu_ctx *ctx, uint64_t scan_idx, formgpu_planar_feat *planar_out, size_t planar_cap,
                  formgpu_point_feat *point_out, size_t point_cap);

/// The whole of stage 1 on a scan already in device memory (formgpu_extract after its upload).
int extract_run_scan(formgpu_ctx *ctx, const float4 *scan_dev, uint64_t scan_idx, bool host_records,
                     formgpu_planar_feat *direct_planar, formgpu_point_feat *direct_point);

/// Raw clouds (api_cloud.cu): the checks of formgpu_set_cloud_format; the boundary tables of rule R8
/// ([cols + 1] azimuth | [rows - 1] ascending beam midpoints; desc = beam table given top-down); the
/// argument block of one organisation into the context's scan buffer; the checks of one cloud request.
int check_cloud_format(const formgpu_cloud_format &f, int rows, int cols, std::string &msg);
void cloud_tables(const formgpu_cloud_format &f, int rows, int cols, std::vector<double2> &tab, int &desc);
OrganizeArgs cloud_args(formgpu_ctx *ctx, const unsigned char *records_dev, size_t n);
int cloud_check_request(formgpu_ctx *ctx, const void *records, size_t n, const char *who);

/// Reparative rebuild: uploads the request of this context on `stream` and fills the two
/// MapArgs and the region (cursor + hash tables) that must be zero before the build.
/// upload = false: the request is left in ctx->h_map_req (ctx->map_req_bytes) for the caller to
/// bring to ctx->d_map_req before the insert pass (batched submits stage it with their arguments).
int map_rebuild_prepare(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses,
                        cudaStream_t stream, MapArgs a[2], MapClearRegion &clear, bool upload = true);

/// Association (+ optionally the fused linearisation of the current scan's pairs).
struct AssocPlan {
  bool any_query = false; // the current scan has keypoints: kernels must run
  bool fused = false;     // lin_tasks are to be launched behind the scatter kernel
  int slot_k = -1;
  int nq[2] = {0, 0};
  int hbuf[2] = {0, 0};
  AssocArgs aa[2];
  SegmentArgs sa[2];
  unsigned long long assoc_seq = 0, lin_seq = 0;
  MomentArgs ma;      // pair moments of this association (queued behind the scatter kernel)
  int mom_units = 0;  // upper bound of the units (warps) the moment kernel needs
  std::vector<LinTask> lin_tasks;
  std::vector<int> lin_slots;
};
int assoc_prepare(formgpu_ctx *ctx, const formgpu_pose *pose_k, const formgpu_scan_pose *poses,
                  size_t n_poses, bool want_blocks, AssocPlan &plan);
/// dma_blocks != nullptr: the blocks of plan.lin_tasks ([task][91] plain doubles) are already in host
/// memory (batched submits); otherwise they are collected from the context's tagged words.
int assoc_finish(formgpu_ctx *ctx, AssocPlan &plan, const formgpu_scan_pose *poses, size_t n_poses,
                 formgpu_pair_count *counts_out, size_t counts_cap, size_t *n_counts, double *out91,
                 const double *dma_blocks);

/// Linearisation / error: argument block of a launch over `n_tasks` tasks of this context
/// (assigns the sequence number that tags the results).
void lin_make_args(formgpu_ctx *ctx, int n_tasks, LinArgs &a);
/// Tasks of formgpu_linearize / formgpu_error: one per listed pair with correspondences;
/// zero-fills the outputs of the others.  indices[k] = position of task k in `pairs`.
int lin_build_tasks(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                    const formgpu_scan_pose *poses, size_t n_poses, size_t per_pair, double *out,
                    std::vector<LinTask> &tasks, std::vector<int> &indices);
/// Wait for the tagged results of `indices` and scatter them to their pairs' positions.
int lin_collect(formgpu_ctx *ctx, const std::vector<int> &indices, unsigned long long seq,
                size_t per_pair, double *out);

/// Novel-keypoint commit.
struct CommitPlan {
  CommitArgs ca[2];
  size_t added[2] = {0, 0};
  int slots[2] = {-1, -1};
};
int commit_prepare(formgpu_ctx *ctx, CommitPlan &plan);
void commit_finish(formgpu_ctx *ctx, const CommitPlan &plan);

/// Point-sharded mode over NCCL (comm.cu): collectives queued on the context's stream.
int comm_allgather_matches(formgpu_ctx *ctx, int n_planar, int n_point);
int comm_allreduce_f64(formgpu_ctx *ctx, double *dev, size_t count);
int comm_ensure_reduce(formgpu_ctx *ctx, size_t doubles);
void comm_release(formgpu_ctx *ctx);
/// Blocks / errors of a request in point-sharded mode: d_red holds this rank's partial results
/// (n_pairs * per_pair doubles, zero for pairs without a task); all-reduce, copy out.
int lin_collect_comm(formgpu_ctx *ctx, size_t n_pairs, size_t per_pair, double *out);

/// Ensure the pinned upload / result staging buffers are large enough.
int ensure_upload(formgpu_ctx *ctx, size_t bytes);
int ensure_out(formgpu_ctx *ctx, size_t pairs);

} // namespace formgpu
