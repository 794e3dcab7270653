// C-ABI (include/formgpu.h): stage 2 - reparative map, association, commit.
#include "api_common.hpp"

#include <algorithm>
#include <cfloat>

using namespace formgpu;

namespace {

size_t next_pow2(size_t v) {
  size_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

void clear_pairs_of_slot(formgpu_ctx *ctx, int slot) {
  const int W = ctx->W;
  for (int i = 0; i < W; ++i) {
    ctx->h_pair_table[(size_t)slot * W + i] = PairEntry{0, 0, 0, 0};
    ctx->h_pair_table[(size_t)i * W + slot] = PairEntry{0, 0, 0, 0};
  }
}

/// The window's used slots in ascending scan id (rule R4): the order of map points, pair counts and
/// exported keypoints.
std::vector<int> slots_by_scan(const formgpu_ctx *ctx) {
  std::vector<int> order;
  for (int s = 0; s < ctx->W; ++s)
    if (ctx->slot_used[s]) order.push_back(s);
  std::sort(order.begin(), order.end(), [&](int a, int b) { return ctx->slot_scan[a] < ctx->slot_scan[b]; });
  return order;
}

/// scan id -> window slot, allocating one on first touch (KeypointMap::get,
/// map.tpp:98-110; ConstraintManager::get_constraints, constraints.cpp:39-64).
int ensure_slot(formgpu_ctx *ctx, uint64_t scan) {
  const int s = find_slot(ctx, scan);
  if (s >= 0) return s;
  for (int i = 0; i < ctx->W; ++i) {
    if (!ctx->slot_used[i]) {
      ctx->slot_used[i] = 1;
      ctx->slot_scan[i] = scan;
      ctx->store_n[0][i] = ctx->store_n[1][i] = 0;
      ctx->slot_of[scan] = i;
      clear_pairs_of_slot(ctx, i);
      return i;
    }
  }
  return -1;
}

// views into the pinned / device rebuild request
struct MapReq {
  double *pose;
  uint64_t *scan;
  int *off;   // [2][W+1]
  int *order; // [W]
  int *rank;  // [W] position of each slot in ascending scan-id order (rule R4, map rebuilds)
};
MapReq map_req_view(unsigned char *base, int W) {
  MapReq r;
  r.pose = reinterpret_cast<double *>(base);
  r.scan = reinterpret_cast<uint64_t *>(base + (size_t)W * 12 * sizeof(double));
  r.off = reinterpret_cast<int *>(base + (size_t)W * 12 * sizeof(double) + (size_t)W * sizeof(uint64_t));
  r.order = r.off + 2 * (W + 1);
  r.rank = r.order + W;
  return r;
}

} // namespace

extern "C" {

int formgpu_map_rebuild(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (n_poses && !poses) return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_map_rebuild: null poses");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  MapArgs a[2];
  MapClearRegion clear;
  const int rc = map_rebuild_prepare(ctx, poses, n_poses, ctx->stream, a, clear);
  if (rc) return rc;
  FORMGPU_CUDA(ctx, cudaMemsetAsync(clear.base, 0, clear.bytes, ctx->stream));
  map_build_launch(a[0], a[1], ctx->stream, ctx->prof);
  FORMGPU_CUDA(ctx, cudaGetLastError());
  return FORMGPU_OK;
}

} // extern "C"

namespace formgpu {

int map_rebuild_prepare(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses,
                        cudaStream_t stream, MapArgs a[2], MapClearRegion &clear, bool upload) {
  const int W = ctx->W;
  if (upload) FORMGPU_CUDA(ctx, cudaEventSynchronize(ctx->ev_upload));
  MapReq h = map_req_view(ctx->h_map_req, W);
  std::vector<uint8_t> has_pose(W, 0);
  for (size_t p = 0; p < n_poses; ++p) {
    const int s = find_slot(ctx, poses[p].scan);
    if (s < 0) continue; // a pose without stored keypoints (e.g. the current scan)
    std::memcpy(h.pose + 12 * s, &poses[p].pose, 12 * sizeof(double));
    has_pose[s] = 1;
  }
  // point-sharded mode: the map of this rank holds the scans of ITS window slots only
  const bool part = sharded_comm(ctx);
  for (int t = 0; t < 2; ++t) {
    int run = 0;
    for (int s = 0; s < W; ++s) {
      h.off[t * (W + 1) + s] = run;
      if (ctx->slot_used[s]) {
        if (ctx->store_n[t][s] > 0 && !has_pose[s])
          return fail(ctx, FORMGPU_ERR_INVALID_ARG,
                      "formgpu_map_rebuild: stored scan " + std::to_string(ctx->slot_scan[s]) +
                          " has no pose");
        if (!part || s % ctx->comm_world == ctx->comm_rank) run += ctx->store_n[t][s];
      }
    }
    h.off[t * (W + 1) + W] = run;
    ctx->map_n[t] = (size_t)run;
  }
  for (int s = 0; s < W; ++s) h.scan[s] = ctx->slot_scan[s];
  // the tie-break id of a map point is (rank of its scan, k): the scan id itself would need all 64
  // bits, and ranks (< W) order the scans exactly as their ids do
  {
    const std::vector<int> order = slots_by_scan(ctx);
    for (int s = 0; s < W; ++s) h.rank[s] = 0;
    for (size_t o = 0; o < order.size(); ++o) h.rank[order[o]] = (int)o;
  }
  if (upload) {
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_map_req, ctx->h_map_req, ctx->map_req_bytes,
                                      cudaMemcpyHostToDevice, stream));
    FORMGPU_CUDA(ctx, cudaEventRecord(ctx->ev_upload, stream));
  }

  // size the tables for this rebuild (load factor <= 0.5); cursor + both tables are one
  // contiguous region, cleared in one go by the caller
  size_t hs[2];
  for (int t = 0; t < 2; ++t) {
    hs[t] = std::min(ctx->hash_cap[t], next_pow2(std::max<size_t>(2 * ctx->map_n[t], 1024)));
    ctx->hash_mask[t] = (uint32_t)(hs[t] - 1);
  }
  ctx->d_hash[0] = reinterpret_cast<HashSlot *>(ctx->d_mapmem + 256);
  ctx->d_hash[1] = ctx->d_hash[0] + hs[0];
  clear.base = ctx->d_mapmem;
  clear.bytes = 256 + (hs[0] + hs[1]) * sizeof(HashSlot);
  clear.copy_src_off = 0;
  clear.copy_dst = nullptr;
  clear.copy_bytes = 0;
  MapReq d = map_req_view(ctx->d_map_req, W);
  for (int t = 0; t < 2; ++t) {
    a[t].type = t;
    a[t].W = W;
    a[t].kcap = t == 0 ? ctx->kp_cap : ctx->kq_cap;
    a[t].store = t == 0 ? (const void *)ctx->d_store_planar : (const void *)ctx->d_store_point;
    a[t].slot_off = d.off + t * (W + 1);
    a[t].slot_pose = d.pose;
    a[t].slot_rank = d.rank;
    a[t].n_total = (int)ctx->map_n[t];
    a[t].voxel_width = ctx->P.max_dist_matching; // form.cpp:61-65
    a[t].inv_voxel_width = 1.0 / ctx->P.max_dist_matching;
    a[t].hash = ctx->d_hash[t];
    a[t].hash_mask = ctx->hash_mask[t];
    a[t].world = ctx->d_world[t];
    a[t].world_src = ctx->d_world_src[t];
    a[t].cell_tab = ctx->d_cell_tab[t];
    a[t].scatter_src = ctx->d_scatter_src[t];
    a[t].cursor = reinterpret_cast<uint32_t *>(ctx->d_mapmem) + 16 * t;
    a[t].voxel_list = ctx->d_voxel_list[t];
  }
  ctx->map_built = true;
  return FORMGPU_OK;
}

// Matcher::match for both types; when `poses` is given, the linearisation of every pair
// (i, current scan) at those poses is queued right behind the association - its ranges are
// read on the device from the pair row the scatter kernel has just written - so the caller
// pays one device round trip instead of two per ICP iteration.
int assoc_prepare(formgpu_ctx *ctx, const formgpu_pose *pose_k, const formgpu_scan_pose *poses,
                  size_t n_poses, bool want_blocks, AssocPlan &plan) {
  if (!ctx->have_current) return fail(ctx, FORMGPU_ERR_STATE, "formgpu_associate: no current scan");
  if (!ctx->map_built) return fail(ctx, FORMGPU_ERR_STATE, "formgpu_associate: map not built");
  const int W = ctx->W;
  const int slot_k = ensure_slot(ctx, ctx->cur_scan);
  if (slot_k < 0) return fail(ctx, FORMGPU_ERR_CAPACITY, "window is full (max_window_scans)");
  plan.slot_k = slot_k;
  plan.nq[0] = ctx->cur_n[0];
  plan.nq[1] = ctx->cur_n[1];
  const int *nq = plan.nq;
  plan.any_query = nq[0] > 0 || nq[1] > 0;
  // fused linearisation: one dynamic task per window scan that has a pose (ascending scan
  // id = the order of the counts returned by assoc_finish)
  plan.fused = poses != nullptr && want_blocks && plan.any_query;
  plan.lin_tasks.clear();
  plan.lin_slots.clear();
  if (plan.fused) {
    int pk = -1;
    std::vector<int> pose_idx(W, -1);
    for (size_t p = 0; p < n_poses; ++p) {
      const int s = find_slot(ctx, poses[p].scan);
      if (s >= 0) pose_idx[s] = (int)p;
      if (poses[p].scan == ctx->cur_scan) pk = (int)p;
    }
    if (pk < 0) return fail(ctx, FORMGPU_ERR_INVALID_ARG, "associate_linearize: no pose for the current scan");
    std::vector<int> order;
    for (const int i : slots_by_scan(ctx))
      if (i != slot_k && pose_idx[i] >= 0) order.push_back(i);
    const int rc = ensure_out(ctx, order.size() + 1);
    if (rc) return rc;
    for (size_t n = 0; n < order.size(); ++n) {
      LinTask t{};
      relative_pose(poses[pose_idx[order[n]]].pose, poses[pk].pose, t.rel);
      t.slot_j = slot_k;
      t.slot_i = order[n];
      t.entry = ctx->d_moments + ((size_t)slot_k * W + order[n]) * kMomentStride;
      t.out_index = (int)n;
      t.dyn_slot_i_plus1 = (uint32_t)order[n] + 1u;
      plan.lin_tasks.push_back(t);
      plan.lin_slots.push_back(order[n]);
    }
  }
  if (!plan.any_query) return FORMGPU_OK;
  // per type: the counter buffer of this association (already cleared).  A type without
  // keypoints keeps its buffers untouched so that a stale match set stays committable.
  for (int t = 0; t < 2; ++t) {
    plan.hbuf[t] = nq[t] > 0 ? (ctx->hist_cur[t] ^ 1) : ctx->hist_cur[t];
    ctx->hist_cur[t] = plan.hbuf[t];
  }
  const int *hbuf = plan.hbuf;
  AssocArgs *aa = plan.aa;
  SegmentArgs *sa = plan.sa;
  plan.assoc_seq = ++ctx->seq; // published by the scatter kernel
  for (int t = 0; t < 2; ++t) {
    const void *queries = t == 0 ? (const void *)ctx->d_cur_planar : (const void *)ctx->d_cur_point;
    const size_t kcap = t == 0 ? ctx->kp_cap : ctx->kq_cap;
    aa[t].type = t;
    aa[t].n_query = nq[t];
    aa[t].q_begin = 0;
    aa[t].q_end = nq[t];
    aa[t].pack_rank = 0;
    aa[t].pad_rank = 0;
    aa[t].n_map = (int)ctx->map_n[t]; // point-sharded mode: this rank's sub-map
    aa[t].queries = queries;
    std::memcpy(aa[t].pose, pose_k, 12 * sizeof(double));
    aa[t].voxel_width = ctx->P.max_dist_matching;
    aa[t].inv_voxel_width = 1.0 / ctx->P.max_dist_matching;
    aa[t].hash = ctx->d_hash[t];
    aa[t].hash_mask = ctx->hash_mask[t];
    aa[t].cell_tab = ctx->d_cell_tab[t];
    aa[t].world = ctx->d_world[t];
    aa[t].world_src = ctx->d_world_src[t];
    aa[t].match = ctx->d_match[t];
    aa[t].W = W;
    aa[t].max_dist2 = ctx->P.max_dist_matching * ctx->P.max_dist_matching; // matcher.hpp:82
    aa[t].min_dist2 = ctx->P.min_dist_map * ctx->P.min_dist_map;           // map.tpp:158
    aa[t].hist_cnt = ctx->d_hist_cnt[hbuf[t]][t];
    sa[t].type = t;
    sa[t].W = W;
    sa[t].n_query = nq[t];
    sa[t].max_dist2 = ctx->P.max_dist_matching * ctx->P.max_dist_matching; // matcher.hpp:82
    sa[t].min_dist2 = ctx->P.min_dist_map * ctx->P.min_dist_map;           // map.tpp:158
    sa[t].kcap = kcap;
    sa[t].queries = queries;
    sa[t].store = t == 0 ? (const void *)ctx->d_store_planar : (const void *)ctx->d_store_point;
    sa[t].match = ctx->d_match[t];
    sa[t].hist_cnt = ctx->d_hist_cnt[hbuf[t]][t];
    sa[t].hist_next = ctx->d_hist_cnt[hbuf[t] ^ 1][t];
    sa[t].hist_bytes = nq[t] > 0 ? ctx->hist_bytes[t] : 0;
    sa[t].host_pair_off = ctx->h_pair + (size_t)(2 * t) * (W + 1);
    sa[t].host_pair_cnt = ctx->h_pair + (size_t)(2 * t + 1) * (W + 1);
    sa[t].dev_pair_off = ctx->d_pair + (size_t)(2 * t) * (W + 1);
    sa[t].dev_pair_cnt = ctx->d_pair + (size_t)(2 * t + 1) * (W + 1);
    sa[t].done_counter = ctx->d_counters + ctx->counter_cap + 1;
    sa[t].flag = ctx->h_flags + 1;
    sa[t].seq = plan.assoc_seq;
    sa[t].seg = t == 0 ? ctx->d_seg_planar + (size_t)slot_k * 9 * kcap
                       : ctx->d_seg_point + (size_t)slot_k * 6 * kcap;
  }
  // pair moments of (every map slot, current scan) at the poses of this association
  // (moments.cu): the kernel reads the pair row the scatter kernel leaves on the device
  MomentArgs &m = plan.ma;
  m = MomentArgs{};
  m.kp_cap = ctx->kp_cap;
  m.kq_cap = ctx->kq_cap;
  m.seg_planar = sa[0].seg;
  m.seg_point = sa[1].seg;
  m.pair_row = ctx->d_pair;
  m.slot_pose = reinterpret_cast<const double *>(ctx->d_map_req); // MapReq::pose, [W][12]
  std::memcpy(m.pose_k, pose_k, 12 * sizeof(double));
  m.moments = ctx->d_moments + (size_t)slot_k * W * kMomentStride;
  m.partials = ctx->d_mom_partials;
  m.tickets = ctx->d_mom_tickets;
  m.W = W;
  m.n_pairs = W;
  // formgpu_set_shard contexts stream their share at linearisation time (lin_launch) and keep
  // whole pairs here; ranks of a communicator accumulate their share of every pair
  m.shard_rank = sharded_comm(ctx) ? ctx->comm_rank : 0;
  m.shard_world = sharded_comm(ctx) ? ctx->comm_world : 1;
  for (int i = 0; i < W; ++i) m.slots[i] = (unsigned char)i;
  m.unit = ctx->moment_unit;
  plan.mom_units = std::min(ctx->mom_max_units, moment_max_units((size_t)nq[0] + (size_t)nq[1], W, m.unit));
  return FORMGPU_OK;
}

int assoc_finish(formgpu_ctx *ctx, AssocPlan &plan, const formgpu_scan_pose *poses, size_t n_poses,
                 formgpu_pair_count *counts_out, size_t counts_cap, size_t *n_counts, double *out91,
                 const double *dma_blocks) {
  const int W = ctx->W;
  const int slot_k = plan.slot_k;
  const int *nq = plan.nq;
  if (plan.any_query) {
    // the counts arrive through mapped memory as soon as CTA 0 of the scatter kernel
    // has summed the counters; the rest of the scatter keeps running behind (later
    // calls are ordered on the same stream)
    const int w = wait_flag(ctx, 1, plan.assoc_seq);
    if (w) return w;
    for (int t = 0; t < 2; ++t) {
      if (nq[t] == 0) continue; // Matcher::match returns early, state stays (matcher.hpp:72-74)
      const uint32_t *off = ctx->h_pair + (size_t)(2 * t) * (W + 1);
      const uint32_t *cnt = ctx->h_pair + (size_t)(2 * t + 1) * (W + 1);
      for (int i = 0; i < W; ++i) {
        PairEntry &e = ctx->h_pair_table[(size_t)slot_k * W + i];
        if (t == 0) {
          e.off_planar = off[i];
          e.n_planar = cnt[i];
        } else {
          e.off_point = off[i];
          e.n_point = cnt[i];
        }
      }
      ctx->match_n[t] = nq[t];
      ctx->match_scan[t] = ctx->cur_scan;
      ctx->match_queries[t] = t == 0 ? (const void *)ctx->d_cur_planar : (const void *)ctx->d_cur_point;
      ctx->match_novel[t] = cnt[W];
      ctx->match_hist[t] = ctx->d_hist_cnt[plan.hbuf[t]][t];
    }
  }
  // non-empty pairs of the current scan, ascending scan id (rule R7)
  std::vector<formgpu_pair_count> out;
  for (int i = 0; i < W; ++i) {
    const PairEntry &e = ctx->h_pair_table[(size_t)slot_k * W + i];
    if (ctx->slot_used[i] && (e.n_planar || e.n_point))
      out.push_back({ctx->slot_scan[i], e.n_planar, e.n_point});
  }
  std::sort(out.begin(), out.end(),
            [](const formgpu_pair_count &a, const formgpu_pair_count &b) { return a.i < b.i; });
  *n_counts = out.size();
  if (out.size() > counts_cap || (!counts_out && !out.empty()))
    return fail(ctx, FORMGPU_ERR_CAPACITY, "formgpu_associate: counts_out too small");
  if (!out.empty()) std::memcpy(counts_out, out.data(), out.size() * sizeof(formgpu_pair_count));
  if (out91) {
    if (plan.fused) {
      // the blocks of the non-empty pairs, in the order of `out`
      std::vector<int> idx;
      for (const auto &c : out) {
        const int s = find_slot(ctx, c.i);
        const auto it = std::find(plan.lin_slots.begin(), plan.lin_slots.end(), s);
        if (it == plan.lin_slots.end())
          return fail(ctx, FORMGPU_ERR_INVALID_ARG, "associate_linearize: no pose for a matched scan");
        idx.push_back((int)(it - plan.lin_slots.begin()));
      }
      if (dma_blocks) {
        // batched submits: the blocks of all plan.lin_tasks have arrived by DMA (api_batch.cu)
        for (size_t k = 0; k < idx.size(); ++k)
          std::memcpy(out91 + 91 * k, dma_blocks + 91 * (size_t)idx[k], 91 * sizeof(double));
      } else if (sharded_comm(ctx)) {
        // partial blocks of all plan.lin_tasks sit in d_red: all-reduce, then pick the non-empty pairs
        std::vector<double> all(91 * plan.lin_tasks.size());
        const int rc = lin_collect_comm(ctx, plan.lin_tasks.size(), 91, all.data());
        if (rc) return rc;
        for (size_t k = 0; k < idx.size(); ++k)
          std::memcpy(out91 + 91 * k, all.data() + 91 * (size_t)idx[k], 91 * sizeof(double));
      } else {
        const int rc = lin_wait(ctx, idx.data(), idx.size(), plan.lin_seq, 91, out91);
        if (rc) return rc;
      }
    } else if (!out.empty()) {
      // nothing was matched in this call (no keypoints): linearise what is there
      std::vector<formgpu_pair> pairs;
      for (const auto &c : out) pairs.push_back({c.i, ctx->cur_scan});
      return formgpu_linearize(ctx, pairs.data(), pairs.size(), poses, n_poses, out91);
    }
  }
  return FORMGPU_OK;
}

} // namespace formgpu

static int associate_impl(formgpu_ctx *ctx, const formgpu_pose *pose_k, const formgpu_scan_pose *poses,
                          size_t n_poses, formgpu_pair_count *counts_out, size_t counts_cap,
                          size_t *n_counts, double *out91) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (!pose_k || !n_counts)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_associate: null argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  static thread_local AssocPlan plan;
  int rc = assoc_prepare(ctx, pose_k, poses, n_poses, out91 != nullptr, plan);
  if (rc) return rc;
  if (plan.any_query) {
    if (sharded_comm(ctx)) {
      // every rank searches its sub-map for all queries; the candidates are all-gathered in
      // place and reduced with the rule-R5 key (+ the histogram) by the combine kernel
      AssocArgs part[2] = {plan.aa[0], plan.aa[1]};
      CombineArgs comb[2];
      const int stride = plan.nq[0] + plan.nq[1];
      for (int t = 0; t < 2; ++t) {
        const size_t off = t == 0 ? 0 : (size_t)plan.nq[0]; // a rank's block: [planar | point]
        part[t].hist_cnt = nullptr;
        part[t].pack_rank = 1;
        part[t].match = ctx->d_gather + (size_t)ctx->comm_rank * stride + off;
        comb[t].a = plan.aa[t];
        comb[t].gathered = ctx->d_gather + off;
        comb[t].slot_scan = reinterpret_cast<const uint64_t *>(ctx->d_map_req + (size_t)ctx->W * 12 * sizeof(double));
        comb[t].world = ctx->comm_world;
        comb[t].stride = stride;
      }
      assoc_launch(part[0], part[1], ctx->cell_search_single, ctx->stream, ctx->prof);
      rc = comm_allgather_matches(ctx, plan.nq[0], plan.nq[1]);
      if (rc) return rc;
      assoc_combine_launch(comb[0], comb[1], ctx->stream, ctx->prof);
    } else {
      assoc_launch(plan.aa[0], plan.aa[1], ctx->cell_search_single, ctx->stream, ctx->prof);
    }
    segment_build_launch(plan.sa[0], plan.sa[1], ctx->stream, ctx->prof);
    if (ctx->moment_cache) moments_launch(plan.ma, plan.mom_units, ctx->stream, ctx->prof);
    FORMGPU_CUDA(ctx, cudaGetLastError());
    if (plan.fused) {
      if (sharded_comm(ctx)) {
        rc = comm_ensure_reduce(ctx, 91 * (plan.lin_tasks.size() + 1));
        if (rc) return rc;
        FORMGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_red, 0, 91 * plan.lin_tasks.size() * sizeof(double), ctx->stream));
        rc = lin_launch(ctx, plan.lin_tasks, false, &plan.lin_seq, ctx->d_red);
      } else {
        rc = lin_launch(ctx, plan.lin_tasks, false, &plan.lin_seq);
      }
      if (rc) return rc;
    }
  }
  return assoc_finish(ctx, plan, poses, n_poses, counts_out, counts_cap, n_counts, out91, nullptr);
}

extern "C" {

int formgpu_associate(formgpu_ctx *ctx, const formgpu_pose *pose_k, formgpu_pair_count *counts_out,
                      size_t counts_cap, size_t *n_counts) {
  return associate_impl(ctx, pose_k, nullptr, 0, counts_out, counts_cap, n_counts, nullptr);
}

int formgpu_associate_linearize(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses,
                                formgpu_pair_count *counts_out, size_t counts_cap, size_t *n_counts,
                                double *out91) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (!poses || !out91)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_associate_linearize: null argument");
  if (!ctx->have_current) return fail(ctx, FORMGPU_ERR_STATE, "formgpu_associate_linearize: no current scan");
  const formgpu_pose *pose_k = nullptr;
  for (size_t p = 0; p < n_poses; ++p)
    if (poses[p].scan == ctx->cur_scan) pose_k = &poses[p].pose;
  if (!pose_k)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_associate_linearize: no pose for the current scan");
  return associate_impl(ctx, pose_k, poses, n_poses, counts_out, counts_cap, n_counts, out91);
}

int formgpu_get_matches(formgpu_ctx *ctx, int type, formgpu_match *out, size_t cap, size_t *n) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if ((type != 0 && type != 1) || !n)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_get_matches: bad argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t cnt = (size_t)ctx->match_n[type];
  *n = cnt;
  if (cnt == 0) return FORMGPU_OK;
  if (!out || cap < cnt) return fail(ctx, FORMGPU_ERR_CAPACITY, "formgpu_get_matches: buffer too small");
  std::vector<MatchRec> tmp(cnt);
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(tmp.data(), ctx->d_match[type], cnt * sizeof(MatchRec),
                                    cudaMemcpyDeviceToHost, ctx->stream));
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (size_t j = 0; j < cnt; ++j) {
    const bool found = tmp[j].slot != kNoSlot;
    out[j].scan = found ? ctx->slot_scan[tmp[j].slot] : 0;
    out[j].k = found ? tmp[j].k : 0;
    out[j].found = found ? 1u : 0u;
    out[j].dist_sqrd = found ? tmp[j].dist_sqrd : DBL_MAX;
  }
  return FORMGPU_OK;
}

int formgpu_commit_scan(formgpu_ctx *ctx, size_t *n_planar_added, size_t *n_point_added) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  CommitPlan plan;
  const int rc = commit_prepare(ctx, plan);
  if (rc) return rc;
  commit_launch(plan.ca[0], plan.ca[1], ctx->stream, ctx->prof);
  FORMGPU_CUDA(ctx, cudaGetLastError());
  commit_finish(ctx, plan);
  if (n_planar_added) *n_planar_added = plan.added[0];
  if (n_point_added) *n_point_added = plan.added[1];
  return FORMGPU_OK;
}

} // extern "C"

namespace formgpu {

int commit_prepare(formgpu_ctx *ctx, CommitPlan &plan) {
  CommitArgs *ca = plan.ca;
  for (int t = 0; t < 2; ++t) {
    plan.added[t] = 0;
    plan.slots[t] = -1;
    ca[t] = CommitArgs{};
    ca[t].type = t;
    ca[t].W = ctx->W;
    ca[t].n_query = 0;
    if (ctx->match_n[t] == 0) continue; // insert_matches: matches.empty() (map.tpp:152-154)
    // the scan is inferred from the matches themselves (map.tpp:155)
    const int slot = ensure_slot(ctx, ctx->match_scan[t]);
    if (slot < 0) return fail(ctx, FORMGPU_ERR_CAPACITY, "window is full (max_window_scans)");
    const size_t kcap = t == 0 ? ctx->kp_cap : ctx->kq_cap;
    if ((size_t)ctx->store_n[t][slot] + ctx->match_novel[t] > kcap)
      return fail(ctx, FORMGPU_ERR_CAPACITY, "keypoint store of a scan is full");
    plan.slots[t] = slot;
    plan.added[t] = ctx->match_novel[t];
    ca[t].n_query = ctx->match_n[t];
    ca[t].min_dist2 = ctx->P.min_dist_map * ctx->P.min_dist_map;
    ca[t].queries = ctx->match_queries[t];
    ca[t].match = ctx->d_match[t];
    ca[t].hist_cnt = ctx->match_hist[t];
    ca[t].store_dst = t == 0 ? (void *)(ctx->d_store_planar + (size_t)slot * kcap)
                             : (void *)(ctx->d_store_point + (size_t)slot * kcap);
    ca[t].dst_count = (uint32_t)ctx->store_n[t][slot];
  }
  return FORMGPU_OK;
}

void commit_finish(formgpu_ctx *ctx, const CommitPlan &plan) {
  for (int t = 0; t < 2; ++t)
    if (plan.slots[t] >= 0) ctx->store_n[t][plan.slots[t]] += (int)plan.added[t];
}

} // namespace formgpu

extern "C" {

int formgpu_remove_scans(formgpu_ctx *ctx, const uint64_t *scans, size_t n) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (n && !scans) return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_remove_scans: null scans");
  for (size_t s = 0; s < n; ++s) {
    const int slot = find_slot(ctx, scans[s]);
    if (slot < 0) continue; // KeypointMap::remove ignores unknown scans (map.tpp:114-117)
    ctx->slot_used[slot] = 0;
    ctx->store_n[0][slot] = ctx->store_n[1][slot] = 0;
    ctx->slot_of.erase(scans[s]);
    clear_pairs_of_slot(ctx, slot);
  }
  return FORMGPU_OK;
}

int formgpu_get_keypoints(formgpu_ctx *ctx, int type, uint64_t scan, void *out, size_t cap,
                          size_t *n) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if ((type != 0 && type != 1) || !n)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_get_keypoints: bad argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  const int slot = find_slot(ctx, scan);
  const size_t cnt = slot < 0 ? 0 : (size_t)ctx->store_n[type][slot];
  *n = cnt;
  if (!out || cnt == 0) return FORMGPU_OK;
  if (cap < cnt) return fail(ctx, FORMGPU_ERR_CAPACITY, "formgpu_get_keypoints: buffer too small");
  if (type == 0) {
    std::vector<PlanarRec> tmp(cnt);
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(tmp.data(), ctx->d_store_planar + (size_t)slot * ctx->kp_cap,
                                      cnt * sizeof(PlanarRec), cudaMemcpyDeviceToHost, ctx->stream));
    FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    auto *o = static_cast<formgpu_planar_feat *>(out);
    for (size_t i = 0; i < cnt; ++i)
      o[i] = formgpu_planar_feat{tmp[i].x, tmp[i].y, tmp[i].z, 0.0, tmp[i].nx, tmp[i].ny, tmp[i].nz, 0.0, scan};
  } else {
    std::vector<PointRec> tmp(cnt);
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(tmp.data(), ctx->d_store_point + (size_t)slot * ctx->kq_cap,
                                      cnt * sizeof(PointRec), cudaMemcpyDeviceToHost, ctx->stream));
    FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    auto *o = static_cast<formgpu_point_feat *>(out);
    for (size_t i = 0; i < cnt; ++i) o[i] = formgpu_point_feat{tmp[i].x, tmp[i].y, tmp[i].z, 0.0, scan};
  }
  return FORMGPU_OK;
}

int formgpu_world_keypoints(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses,
                            formgpu_planar_feat *planar_out, size_t planar_cap, size_t *n_planar,
                            formgpu_point_feat *point_out, size_t point_cap, size_t *n_point) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if ((n_poses && !poses) || !n_planar || !n_point)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_world_keypoints: null argument");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  const int W = ctx->W;
  FORMGPU_CUDA(ctx, cudaEventSynchronize(ctx->ev_upload));
  MapReq h = map_req_view(ctx->h_map_req, W);
  std::vector<uint8_t> has_pose(W, 0);
  for (size_t p = 0; p < n_poses; ++p) {
    const int s = find_slot(ctx, poses[p].scan);
    if (s < 0) continue;
    std::memcpy(h.pose + 12 * s, &poses[p].pose, 12 * sizeof(double));
    has_pose[s] = 1;
  }
  // slots in ascending scan id (rule R4)
  const std::vector<int> order = slots_by_scan(ctx);
  size_t total[2];
  for (int t = 0; t < 2; ++t) {
    int run = 0;
    for (int o = 0; o < W; ++o) {
      h.off[t * (W + 1) + o] = run;
      if (o < (int)order.size()) {
        const int s = order[o];
        if (ctx->store_n[t][s] > 0 && !has_pose[s])
          return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_world_keypoints: stored scan has no pose");
        run += ctx->store_n[t][s];
      }
    }
    h.off[t * (W + 1) + W] = run;
    total[t] = (size_t)run;
  }
  for (int o = 0; o < W; ++o) h.order[o] = o < (int)order.size() ? order[o] : 0;
  for (int s = 0; s < W; ++s) h.scan[s] = ctx->slot_scan[s];
  *n_planar = total[0];
  *n_point = total[1];
  if (total[0] > planar_cap || total[1] > point_cap || (total[0] && !planar_out) ||
      (total[1] && !point_out))
    return fail(ctx, FORMGPU_ERR_CAPACITY, "formgpu_world_keypoints: output buffers too small");
  const size_t bytes = total[0] * sizeof(formgpu_planar_feat) + total[1] * sizeof(formgpu_point_feat);
  if (bytes > ctx->export_bytes) {
    FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->d_export) cudaFree(ctx->d_export);
    ctx->d_export = nullptr;
    ctx->export_bytes = 0;
    FORMGPU_CUDA(ctx, cudaMalloc(&ctx->d_export, next_pow2(bytes)));
    ctx->export_bytes = next_pow2(bytes);
  }
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_map_req, ctx->h_map_req, ctx->map_req_bytes,
                                    cudaMemcpyHostToDevice, ctx->stream));
  FORMGPU_CUDA(ctx, cudaEventRecord(ctx->ev_upload, ctx->stream));
  MapReq d = map_req_view(ctx->d_map_req, W);
  unsigned char *out_dev = static_cast<unsigned char *>(ctx->d_export);
  for (int t = 0; t < 2; ++t) {
    WorldExportArgs a;
    a.type = t;
    a.W = W;
    a.kcap = t == 0 ? ctx->kp_cap : ctx->kq_cap;
    a.store = t == 0 ? (const void *)ctx->d_store_planar : (const void *)ctx->d_store_point;
    a.slot_off = d.off + t * (W + 1);
    a.order = d.order;
    a.slot_pose = d.pose;
    a.slot_scan = d.scan;
    a.n_total = (int)total[t];
    a.out = t == 0 ? out_dev : out_dev + total[0] * sizeof(formgpu_planar_feat);
    world_export_launch(a, ctx->stream, ctx->prof);
  }
  FORMGPU_CUDA(ctx, cudaGetLastError());
  if (total[0])
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(planar_out, out_dev, total[0] * sizeof(formgpu_planar_feat),
                                      cudaMemcpyDeviceToHost, ctx->stream));
  if (total[1])
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(point_out, out_dev + total[0] * sizeof(formgpu_planar_feat),
                                      total[1] * sizeof(formgpu_point_feat), cudaMemcpyDeviceToHost,
                                      ctx->stream));
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FORMGPU_OK;
}

} // extern "C"
