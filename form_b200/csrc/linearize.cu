// Stage 3 on sm_100a: residual / Jacobian linearisation reduced into per-pair
// 13x13 normal-equation blocks.
//
// Replaces PlanePoint/PointPoint::evaluateError + FeatureFactor::evaluateError
// (/root/reference/form/feature/factor.cpp:30-186) followed by
// DenseFactor::linearize / FastIsotropic whitening / HessianFactor(JacobianFactor)
// (/root/reference/form/optimization/gtsam.hpp:59-140).  Tolerance class
// (H/b rel <= 1e-5), so FMA contraction is allowed here.
//
// Arithmetic.  The reference materialises an (n+3m) x 13 dense Jacobian per pair
// and forms A^T A.  Here each correspondence is streamed once from HBM (coalesced
// SoA floats - the keypoints are float-exact) and reduced on the fly.  Working in
// the frame of scan i,
//     q = R_rel p_j + t_rel,   R_rel = R_i^T R_j,  t_rel = R_i^T (t_j - t_i)
// every row of [J_i J_j | -r] is LINEAR in a 7-vector of the correspondence, with
// coefficients that depend only on the pair's relative pose:
//     plane-point:  s = [ n x q,  n,  n.(q - p_i) ]
//     point-point:  z = [ p_i,  q - p_i,  1 ]     (3 rows, rotated by R_i^T, which
//                                                  leaves A^T A unchanged)
// so a thread accumulates only the 28 unique products of its 7-vector (56 registers
// instead of 182 for the 91 entries) and the 13x13 block is recovered per pair as
// sum_kl W_kl B_k^T B_l.
//
// Mapping.  One thread-block CLUSTER per scan pair (8 CTAs when the request has few
// pairs, down to 1 when it has thousands, so that one launch is about one wave): CTA r
// streams the r-th share of the pair's planar and point correspondences, reduces its 2 x 28 moments
// (butterfly-transpose warp reduction: 31 shuffles instead of 140), and leaves them
// in its shared memory; after cluster.sync() CTA 0 gathers the partial sums
// through distributed shared memory, expands the block and writes the 91 doubles
// straight into mapped pinned host memory as sequence-tagged words (32 bits of payload
// + 32 bits of tag per aligned 8-byte store), which the host polls.  There is no
// partial-sum traffic through global memory, no atomic, no second launch, no
// device->host memcpy and no system-wide fence.  Small requests travel in the kernel parameters (with
// the relative poses precomputed by the host), so the first instruction that
// touches memory is already a correspondence load.  The partition and every
// reduction order are fixed: results are run-to-run deterministic.
#include "lin_device.cuh"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace formgpu {

namespace {

// ---------------------------------------------------------------------------
// one cluster per pair
// ---------------------------------------------------------------------------
template <bool kErrorOnly>
__device__ __forceinline__ void lin_cluster_body(const LinArgs &a, const LinTask &task_in) {
  // ranges of the pair: given by the host, or - when the linearisation was queued right
  // behind the association that produces them - read from the device pair row
  struct {
    const double *rel;
    uint32_t off_planar, n_planar, off_point, n_point;
    int slot_j, out_index;
  } task = {task_in.rel, task_in.off_planar, task_in.n_planar, task_in.off_point, task_in.n_point,
            task_in.slot_j, task_in.out_index};
  if (task_in.dyn_slot_i_plus1) {
    const int si = (int)task_in.dyn_slot_i_plus1 - 1, nb = a.W + 1;
    task.off_planar = a.pair_row[0 * nb + si];
    task.n_planar = a.pair_row[1 * nb + si];
    task.off_point = a.pair_row[2 * nb + si];
    task.n_point = a.pair_row[3 * nb + si];
    if (task.n_planar + task.n_point == 0) return; // empty pair: the whole cluster leaves
  }
  const bool has_planar = task.n_planar > 0, has_point = task.n_point > 0;
  if (a.shard_world > 1) { // this rank's share of the pair
    uint32_t b0, c0;
    shard_range(task.n_planar, a.shard_rank, a.shard_world, b0, c0);
    task.off_planar += b0;
    task.n_planar = c0;
    shard_range(task.n_point, a.shard_rank, a.shard_world, b0, c0);
    task.off_point += b0;
    task.n_point = c0;
  }
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int kCluster = (int)cluster.num_blocks(); // 1, 2, 4 or 8: chosen per launch
  const int tid = threadIdx.x;
  __shared__ double s_warp[kWarps][28];
  __shared__ double s_sum[2][28];  // [planar | point] moments of this CTA (error: [0][0])
  __shared__ double s_total[2][28];

  __shared__ ExpandSmem s_exp;
  double acc[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) acc[k] = 0.0;
  double err_acc = 0.0;
  if (!kErrorOnly && rank == 0) build_basis(s_exp, task.rel);

  // ---- plane-point correspondences of this CTA's slice ----
  {
    const uint32_t lo = (uint32_t)(((unsigned long long)task.n_planar * rank) / kCluster);
    const uint32_t hi = (uint32_t)(((unsigned long long)task.n_planar * (rank + 1)) / kCluster);
    const float *s = a.seg_planar + (size_t)task.slot_j * 9 * a.kp_cap + task.off_planar;
    const size_t st = a.kp_cap;
#pragma unroll 2
    for (uint32_t c = lo + tid; c < hi; c += kThreads) {
      const double pix = s[0 * st + c], piy = s[1 * st + c], piz = s[2 * st + c];
      const double nx = s[3 * st + c], ny = s[4 * st + c], nz = s[5 * st + c];
      const double pjx = s[6 * st + c], pjy = s[7 * st + c], pjz = s[8 * st + c];
      double qx, qy, qz;
      apply_rel(task.rel, pjx, pjy, pjz, qx, qy, qz);
      const double r = nx * (qx - pix) + ny * (qy - piy) + nz * (qz - piz);
      if (kErrorOnly) {
        err_acc += r * r;
      } else {
        const double v[7] = {ny * qz - nz * qy, nz * qx - nx * qz, nx * qy - ny * qx, nx, ny, nz, r};
        int e = 0;
#pragma unroll
        for (int p = 0; p < 7; ++p)
#pragma unroll
          for (int q = p; q < 7; ++q) acc[e++] += v[p] * v[q];
      }
    }
  }
  if (!kErrorOnly) {
    block_reduce28(acc, s_warp, s_sum[0], tid);
#pragma unroll
    for (int k = 0; k < 32; ++k) acc[k] = 0.0;
  }
  // ---- point-point correspondences ----
  {
    const uint32_t lo = (uint32_t)(((unsigned long long)task.n_point * rank) / kCluster);
    const uint32_t hi = (uint32_t)(((unsigned long long)task.n_point * (rank + 1)) / kCluster);
    const float *s = a.seg_point + (size_t)task.slot_j * 6 * a.kq_cap + task.off_point;
    const size_t st = a.kq_cap;
#pragma unroll 2
    for (uint32_t c = lo + tid; c < hi; c += kThreads) {
      const double pix = s[0 * st + c], piy = s[1 * st + c], piz = s[2 * st + c];
      const double pjx = s[3 * st + c], pjy = s[4 * st + c], pjz = s[5 * st + c];
      double qx, qy, qz;
      apply_rel(task.rel, pjx, pjy, pjz, qx, qy, qz);
      const double ex = qx - pix, ey = qy - piy, ez = qz - piz;
      if (kErrorOnly) {
        err_acc += ex * ex + ey * ey + ez * ez;
      } else {
        const double v[7] = {pix, piy, piz, ex, ey, ez, 1.0};
        int e = 0;
#pragma unroll
        for (int p = 0; p < 7; ++p)
#pragma unroll
          for (int q = p; q < 7; ++q) acc[e++] += v[p] * v[q];
      }
    }
  }
  if (kErrorOnly) {
    const double w = warp_sum(err_acc);
    if ((tid & 31) == 0) s_warp[tid >> 5][0] = w;
    __syncthreads();
    if (tid == 0) {
      double v = 0.0;
#pragma unroll
      for (int k = 0; k < kWarps; ++k) v += s_warp[k][0];
      s_sum[0][0] = v;
    }
  } else {
    block_reduce28(acc, s_warp, s_sum[1], tid);
  }

  // ---- gather the CTA sums through distributed shared memory ----
  cluster.sync();
  if (rank == 0) {
    if (kErrorOnly) {
      if (tid == 0) {
        double v = 0.0;
        for (int r = 0; r < kCluster; ++r) v += *cluster.map_shared_rank(&s_sum[0][0], r);
        s_total[0][0] = 0.5 * v * a.inv_sigma2;
      }
    } else if (tid < 56) {
      const int which = tid / 28, e = tid % 28;
      double v = 0.0;
      for (int r = 0; r < kCluster; ++r) v += *cluster.map_shared_rank(&s_sum[which][e], r);
      s_total[which][e] = v;
    }
  }
  cluster.sync(); // the other CTAs' shared memory must outlive CTA 0's remote reads
  if (rank != 0) return;
  __syncthreads();
  // Publish straight into mapped pinned host memory.  Every 8-byte word carries the
  // call's sequence tag next to 32 bits of payload, so the host can tell a fresh word
  // from a stale one by itself: no system-wide fence (a ~3 us PCIe flush) and no
  // separate flag are needed - an aligned 8-byte store is a single atomic PCIe write.
  const unsigned long long tag = a.seq & 0xffffffffull;
  if (kErrorOnly) {
    if (tid == 0) {
      if (a.out_plain) a.out_plain[task.out_index] = s_total[0][0];
      else publish_tagged(a.out + 2 * (size_t)task.out_index, s_total[0][0], tag);
    }
  } else {
    expand_and_publish(s_exp, s_total[0], s_total[1], has_planar, has_point, a.inv_sigma2,
                       a.out + 182 * (size_t)task.out_index, tag,
                       a.out_plain ? a.out_plain + 91 * (size_t)task.out_index : nullptr);
  }
}

} // namespace

template <bool kErrorOnly>
__global__ void __launch_bounds__(kLinThreads) lin_inline_kernel(LinArgs a, LinInline req) {
  lin_cluster_body<kErrorOnly>(a, req.tasks[blockIdx.x / a.cluster]);
}

template <bool kErrorOnly>
__global__ void __launch_bounds__(kLinThreads) lin_global_kernel(LinArgs a) {
  __shared__ LinTask s_task;
  if (threadIdx.x < sizeof(LinTask) / sizeof(unsigned long long))
    reinterpret_cast<unsigned long long *>(&s_task)[threadIdx.x] =
        reinterpret_cast<const unsigned long long *>(a.tasks + blockIdx.x / a.cluster)[threadIdx.x];
  __syncthreads();
  lin_cluster_body<kErrorOnly>(a, s_task);
}

namespace {
template <typename... Args>
cudaError_t launch_cluster(void (*kernel)(Args...), int n_tasks, int cluster, cudaStream_t stream,
                           Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(n_tasks * cluster), 1, 1);
  cfg.blockDim = dim3(kLinThreads, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}
} // namespace

cudaError_t linearize_launch(const LinArgs &a, const LinInline *inline_req, bool error_only,
                             cudaStream_t stream, Profiler &prof) {
  if (a.n_tasks <= 0) return cudaSuccess;
  const int group = error_only ? FORMGPU_KG_ERR_CHUNK : FORMGPU_KG_LIN_CHUNK;
  prof.begin(group);
  cudaError_t e;
  if (inline_req) {
    e = error_only ? launch_cluster(lin_inline_kernel<true>, a.n_tasks, a.cluster, stream, a, *inline_req)
                   : launch_cluster(lin_inline_kernel<false>, a.n_tasks, a.cluster, stream, a, *inline_req);
  } else {
    e = error_only ? launch_cluster(lin_global_kernel<true>, a.n_tasks, a.cluster, stream, a)
                   : launch_cluster(lin_global_kernel<false>, a.n_tasks, a.cluster, stream, a);
  }
  prof.end(group, 1);
  return e;
}

} // namespace formgpu
