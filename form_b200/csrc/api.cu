// C-ABI (include/formgpu.h): lifecycle, instrumentation and stage 1.
#include "api_common.hpp"

#include <sched.h>
#include <cstdlib>

#include <algorithm>
#include <new>

using namespace formgpu;

namespace {
std::string g_create_error;

size_t next_pow2(size_t v) {
  size_t p = 1;
  while (p < v) p <<= 1;
  return p;
}
} // namespace

namespace formgpu {

int ensure_upload(formgpu_ctx *ctx, size_t bytes) {
  if (bytes <= ctx->h_upload_bytes) return FORMGPU_OK;
  // growing is rare (first full-window request); drain the stream first
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->h_upload) cudaFreeHost(ctx->h_upload);
  if (ctx->d_request) cudaFree(ctx->d_request);
  ctx->h_upload = nullptr;
  ctx->d_request = nullptr;
  const size_t cap = next_pow2(bytes);
  FORMGPU_CUDA(ctx, cudaHostAlloc(&ctx->h_upload, cap, cudaHostAllocDefault));
  FORMGPU_CUDA(ctx, cudaMalloc(&ctx->d_request, cap));
  ctx->h_upload_bytes = cap;
  ctx->request_bytes = cap;
  return FORMGPU_OK;
}

int ensure_out(formgpu_ctx *ctx, size_t pairs) {
  if (pairs <= ctx->out_cap) return FORMGPU_OK;
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->h_out) cudaFreeHost(const_cast<unsigned long long *>(ctx->h_out));
  if (ctx->d_counters) cudaFree(ctx->d_counters);
  ctx->h_out = nullptr;
  ctx->d_counters = nullptr;
  const size_t cap = next_pow2(pairs);
  // results are written by the kernels straight into this mapped pinned buffer
  FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(const_cast<unsigned long long **>(&ctx->h_out)),
                                  cap * 182 * sizeof(unsigned long long), cudaHostAllocMapped));
  for (size_t i = 0; i < cap * 182; ++i) ctx->h_out[i] = 0; // tag 0 is never used (seq starts at 1)
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_counters, cap + 8));
  FORMGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_counters, 0, (cap + 8) * sizeof(unsigned), ctx->stream));
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->counter_cap = cap;
  ctx->out_cap = cap;
  ctx->h_out_bytes = cap * 182 * sizeof(unsigned long long);
  return FORMGPU_OK;
}

int wait_flag(formgpu_ctx *ctx, int which, unsigned long long seq) {
  volatile unsigned long long *f = ctx->h_flags + which;
  for (unsigned spins = 0;; ++spins) {
    if (*f == seq) return FORMGPU_OK;
    if ((spins & 0xfff) == 0xfff) {
      const cudaError_t e = cudaStreamQuery(ctx->stream);
      if (e == cudaSuccess) {
        if (*f == seq) return FORMGPU_OK;
        return fail(ctx, FORMGPU_ERR_STATE, "kernel finished without publishing its results");
      }
      if (e != cudaErrorNotReady)
        return fail(ctx, FORMGPU_ERR_CUDA, std::string("kernel failed: ") + cudaGetErrorString(e));
    }
    poll_relax(spins);
  }
}

void poll_relax(unsigned spins) {
  static const bool yield_wait = [] {
    const char *e = std::getenv("FORMGPU_YIELD_WAIT");
    return e && e[0] == '1';
  }();
  if (yield_wait && (spins & 63u) == 63u) sched_yield();
#if defined(__x86_64__)
  __builtin_ia32_pause();
#endif
}

} // namespace formgpu

namespace formgpu {

int validate_params(const formgpu_params &P, std::string &msg) {
  auto bad = [&](int code, const char *m) {
    msg = m;
    return code;
  };
  if (P.neighbor_points < 1 || P.neighbor_points > 16)
    return bad(FORMGPU_ERR_UNSUPPORTED, "neighbor_points must be in [1, 16]");
  if (P.num_sectors < 1 || P.num_rows < 1 || P.num_columns < 2 * P.neighbor_points + 1 ||
      P.num_columns > 4096 || P.num_columns / P.num_sectors < 1)
    return bad(FORMGPU_ERR_UNSUPPORTED,
               "need 2*neighbor_points < num_columns <= 4096, num_rows >= 1, "
               "1 <= num_sectors <= num_columns");
  if (P.planar_feats_per_sector < 0 || P.point_feats_per_sector < 0 || P.min_points < 0)
    return bad(FORMGPU_ERR_INVALID_ARG, "negative feature counts");
  if (P.max_window_scans < 2 || P.max_window_scans > kMaxWindow)
    return bad(FORMGPU_ERR_UNSUPPORTED, "max_window_scans must be in [2, 128]");
  if (!(P.max_dist_matching > 0) || !(P.sigma > 0))
    return bad(FORMGPU_ERR_INVALID_ARG, "max_dist_matching and sigma must be positive");
  return FORMGPU_OK;
}

} // namespace formgpu

extern "C" {

int formgpu_abi_version(void) { return FORMGPU_ABI_VERSION; }

void formgpu_default_params(formgpu_params *p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->neighbor_points = 5;
  p->num_sectors = 6;
  p->planar_feats_per_sector = 50;
  p->point_feats_per_sector = 3;
  p->min_points = 5;
  p->num_columns = 1024;
  p->num_rows = 64;
  p->max_window_scans = 64;
  p->planar_threshold = 1.0;
  p->radius = 1.0;
  p->min_norm_squared = 1.0;
  p->max_norm_squared = 100.0 * 100.0;
  p->max_dist_matching = 0.8;
  p->min_dist_map = 0.1;
  p->sigma = 0.1;
  p->max_batch_scans = 1;
}

const char *formgpu_last_error(const formgpu_ctx *ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

static int create_impl(formgpu_ctx *ctx) {
  const formgpu_params &P = ctx->P;
  {
    std::string msg;
    const int rc = validate_params(P, msg);
    if (rc != FORMGPU_OK) return fail(ctx, rc, msg);
  }

  ctx->rows = P.num_rows;
  ctx->cols = P.num_columns;
  ctx->words = (ctx->cols + 31) / 32;
  ctx->W = P.max_window_scans;
  ctx->B = std::max(1, P.max_batch_scans);
  ctx->n_points = (size_t)ctx->rows * ctx->cols;
  // picks in one row are pairwise >= neighbor_points apart (suppression +-(np-1))
  ctx->qr_cap = (ctx->cols + P.neighbor_points - 1) / P.neighbor_points + 1;
  ctx->qr_cap = (ctx->qr_cap + 3) & ~3; // multiples of 4: every segment plane starts 16-byte aligned
  ctx->pr_cap = std::min(P.num_sectors * (P.planar_feats_per_sector + 1), ctx->qr_cap);
  ctx->pr_cap = (std::max(ctx->pr_cap, 1) + 3) & ~3;
  ctx->kp_cap = (size_t)ctx->rows * ctx->pr_cap;
  ctx->kq_cap = (size_t)ctx->rows * ctx->qr_cap;
  if (ctx->kp_cap >= (1u << 24) || ctx->kq_cap >= (1u << 24))
    return fail(ctx, FORMGPU_ERR_UNSUPPORTED, "more than 2^24 keypoints per scan");

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(ctx, FORMGPU_ERR_CUDA, "no CUDA device available (there is no CPU fallback)");
  if (ctx->device < 0 || ctx->device >= ndev)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "device index out of range");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  FORMGPU_CUDA(ctx, cudaGetDeviceProperties(&prop, ctx->device));
  if (prop.major < 10)
    return fail(ctx, FORMGPU_ERR_CUDA, "formgpu is built for sm_100a (Blackwell) only");
  if (!ctx->stream) {
    FORMGPU_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
  }
  ctx->prof.stream = ctx->stream;
  FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(const_cast<unsigned long long **>(&ctx->h_flags)),
                                  8 * sizeof(unsigned long long), cudaHostAllocMapped));
  for (int i = 0; i < 8; ++i) ctx->h_flags[i] = 0;

  const size_t B = ctx->B, R = ctx->rows, W = ctx->W;
  // stage 1
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_scan, B * ctx->n_points));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_valid_bits, B * R * ctx->words));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_row_box, B * R * ctx->words * 2));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_planar_cols, B * R * ctx->pr_cap));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_planar_cnt, B * R));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_point_cols, B * R * ctx->qr_cap));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_point_cnt, B * R));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_normals, B * R * ctx->pr_cap));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_keep_cnt, B * R));
  for (int i = 0; i < 2; ++i) {
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_cur_planar_buf[i], B * ctx->kp_cap));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_cur_point_buf[i], B * ctx->kq_cap));
  }
  ctx->d_cur_planar = ctx->d_cur_planar_buf[0];
  ctx->d_cur_point = ctx->d_cur_point_buf[0];
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_cur_counts, B * 2 + 8));
  FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_counts),
                                  (B * 2 + 8) * sizeof(int), cudaHostAllocMapped));
  FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_planar),
                                  ctx->kp_cap * sizeof(PlanarRec), cudaHostAllocMapped));
  FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_point),
                                  ctx->kq_cap * sizeof(PointRec), cudaHostAllocMapped));
  {
    ExtractArgs shape{};
    shape.cols = ctx->cols;
    shape.words = ctx->words;
    shape.cols_pad = ctx->words * 32;
    shape.num_sectors = ctx->P.num_sectors;
    shape.np = ctx->P.neighbor_points;
    shape.pps = ctx->cols / ctx->P.num_sectors;
    shape.planar_per_sector = ctx->P.planar_feats_per_sector;
    shape.point_per_sector = ctx->P.point_feats_per_sector;
    shape.pr_cap = ctx->pr_cap;
    shape.qr_cap = ctx->qr_cap;
    if (shape.num_sectors > kExtractMaxSectors)
      return fail(ctx, FORMGPU_ERR_INVALID_ARG, "num_sectors exceeds " + std::to_string(kExtractMaxSectors));
    FORMGPU_CUDA(ctx, extract_configure(shape));
  }
  if (const char *env = std::getenv("FORMGPU_SINGLE_CELL_SEARCH")) ctx->cell_search_single = env[0] == '1';

  // window / keypoint store
  ctx->slot_scan.assign(W, 0);
  ctx->slot_used.assign(W, 0);
  ctx->store_n[0].assign(W, 0);
  ctx->store_n[1].assign(W, 0);
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_store_planar, W * ctx->kp_cap));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_store_point, W * ctx->kq_cap));

  // world map: capacity for every store slot full
  const size_t cap[2] = {W * ctx->kp_cap, W * ctx->kq_cap};
  for (int t = 0; t < 2; ++t) {
    ctx->map_cap[t] = cap[t];
    ctx->hash_cap[t] = next_pow2(2 * cap[t]);
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_world[t], cap[t]));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_world_src[t], cap[t]));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_cell_tab[t], cap[t]));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_scatter_src[t], cap[t]));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_voxel_list[t], cap[t]));
  }
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_mapmem,
                              256 + (ctx->hash_cap[0] + ctx->hash_cap[1]) * sizeof(HashSlot)));
  ctx->map_req_bytes = W * 12 * sizeof(double) + W * sizeof(uint64_t) +
                       (2 * (W + 1) + 2 * W) * sizeof(int);
  ctx->map_req_bytes = (ctx->map_req_bytes + 7) / 8 * 8; // moved in 8-byte words by batched rebuilds
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_map_req, ctx->map_req_bytes));
  FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_map_req), ctx->map_req_bytes,
                                  cudaHostAllocDefault));
  FORMGPU_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_upload, cudaEventDisableTiming));

  // matches / correspondences
  // + 64: the in-place all-gather of point-sharded mode rounds every rank's share up
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_match[0], ctx->kp_cap + 64));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_match[1], ctx->kq_cap + 64));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_seg_planar, W * 9 * ctx->kp_cap));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_seg_point, W * 6 * ctx->kq_cap));
  for (int t = 0; t < 2; ++t) {
    const size_t n = ((t == 0 ? ctx->kp_cap : ctx->kq_cap) + 255) / 256 + 1;
    ctx->hist_bytes[t] = n * (W + 1) * sizeof(uint32_t);
    for (int b = 0; b < 2; ++b) {
      FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_hist_cnt[b][t], n * (W + 1)));
      FORMGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_hist_cnt[b][t], 0, ctx->hist_bytes[t], ctx->stream));
    }
  }
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_pair, 4 * (W + 1)));
  FORMGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_pair, 0, 4 * (W + 1) * sizeof(uint32_t), ctx->stream));
  // pair-moment cache + the scratch of the kernel that fills it
  if (const char *env = std::getenv("FORMGPU_STREAM_LINEARIZE")) ctx->moment_cache = env[0] != '1';
  ctx->moment_unit = kMomentUnitSingle;
  if (const char *env = std::getenv("FORMGPU_MOMENT_UNIT")) // tuning: 128 .. 4096, multiple of 32
    ctx->moment_unit = (uint32_t)std::min(4096, std::max(128, std::atoi(env) / 32 * 32));
  ctx->mom_max_units = moment_max_units(ctx->kp_cap + ctx->kq_cap, W, kMomentUnitSingle); // the smaller unit sizes the scratch
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_moments, (size_t)W * W * kMomentStride));
  FORMGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_moments, 0, (size_t)W * W * kMomentStride * sizeof(double), ctx->stream));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_mom_partials, (size_t)ctx->mom_max_units * kMomentPartial));
  FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_mom_tickets, (size_t)W));
  FORMGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_mom_tickets, 0, W * sizeof(unsigned), ctx->stream));
  ctx->h_pair_table.assign(W * W, PairEntry{0, 0, 0, 0});
  FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_pair), 4 * (W + 1) * sizeof(uint32_t),
                                  cudaHostAllocMapped));

  int rc = ensure_upload(ctx, 1 << 16);
  if (rc) return rc;
  rc = ensure_out(ctx, 64);
  if (rc) return rc;
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FORMGPU_OK;
}

int formgpu_create(const formgpu_params *p, int device, void *stream, formgpu_ctx **out) {
  if (!p || !out) {
    g_create_error = "formgpu_create: null argument";
    return FORMGPU_ERR_INVALID_ARG;
  }
  *out = nullptr;
  formgpu_ctx *ctx = new (std::nothrow) formgpu_ctx();
  if (!ctx) {
    g_create_error = "out of host memory";
    return FORMGPU_ERR_CAPACITY;
  }
  ctx->P = *p;
  ctx->device = device;
  ctx->stream = static_cast<cudaStream_t>(stream);
  const int rc = create_impl(ctx);
  if (rc != FORMGPU_OK) {
    g_create_error = ctx->err;
    formgpu_destroy(ctx);
    return rc;
  }
  *out = ctx;
  return FORMGPU_OK;
}

void formgpu_destroy(formgpu_ctx *ctx) {
  if (!ctx) return;
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  auto F = [](auto *&p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  auto H = [](auto *&p) {
    if (p) cudaFreeHost(p);
    p = nullptr;
  };
  F(ctx->d_scan); F(ctx->d_valid_bits); F(ctx->d_row_box); F(ctx->d_planar_cols); F(ctx->d_planar_cnt);
  F(ctx->d_point_cols); F(ctx->d_point_cnt); F(ctx->d_normals); F(ctx->d_closest);
  F(ctx->d_keep_cnt); F(ctx->d_cur_counts);
  for (int i = 0; i < 2; ++i) { F(ctx->d_cur_planar_buf[i]); F(ctx->d_cur_point_buf[i]); F(ctx->d_hist_cnt[i][0]); F(ctx->d_hist_cnt[i][1]); }
  F(ctx->d_dbg_valid); F(ctx->d_dbg_pvalid); F(ctx->d_dbg_curv);
  F(ctx->d_store_planar); F(ctx->d_store_point);
  for (int t = 0; t < 2; ++t) {
    F(ctx->d_world[t]); F(ctx->d_world_src[t]);
    F(ctx->d_cell_tab[t]); F(ctx->d_scatter_src[t]); F(ctx->d_voxel_list[t]); F(ctx->d_match[t]);
  }
  F(ctx->d_mapmem); F(ctx->d_map_req); F(ctx->d_export); H(ctx->h_map_req);
  if (ctx->ev_upload) cudaEventDestroy(ctx->ev_upload);
  F(ctx->d_seg_planar); F(ctx->d_seg_point); F(ctx->d_pair);
  F(ctx->d_request); F(ctx->d_counters);
  F(ctx->d_moments); F(ctx->d_mom_partials); F(ctx->d_mom_tickets);
  comm_release(ctx);
  F(ctx->d_stage_planar); F(ctx->d_stage_point);
  F(ctx->d_scan_next);
  F(ctx->d_records); F(ctx->d_pixel_keys); F(ctx->d_cloud_tab); F(ctx->d_cloud_stats); H(ctx->h_cloud_stats);
  if (ctx->ev_prefetch) cudaEventDestroy(ctx->ev_prefetch);
  if (ctx->h_flags) cudaFreeHost(const_cast<unsigned long long *>(ctx->h_flags));
  H(ctx->h_counts); H(ctx->h_planar); H(ctx->h_point); H(ctx->h_upload);
  if (ctx->h_out) cudaFreeHost(const_cast<unsigned long long *>(ctx->h_out));
  H(ctx->h_pair);
  ctx->prof.destroy();
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

void *formgpu_alloc_pinned(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void formgpu_free_pinned(void *p) {
  if (p) cudaFreeHost(p);
}

size_t formgpu_max_planar(const formgpu_ctx *ctx) { return ctx ? ctx->kp_cap : 0; }
size_t formgpu_max_point(const formgpu_ctx *ctx) { return ctx ? ctx->kq_cap : 0; }

// ---------------------------------------------------------------------------
// stage 1
// ---------------------------------------------------------------------------
static ExtractArgs make_extract_args(formgpu_ctx *ctx, const float4 *scan_dev, bool debug,
                                     bool host_records = false, bool publish = false) {
  const formgpu_params &P = ctx->P;
  ExtractArgs a{};
  a.host_planar_f64 = nullptr;
  a.host_point_f64 = nullptr;
  a.scan_idx = 0;
  a.rows = ctx->rows;
  a.cols = ctx->cols;
  a.words = ctx->words;
  a.cols_pad = ctx->words * 32;
  a.np = P.neighbor_points;
  a.num_sectors = P.num_sectors;
  a.pps = ctx->cols / P.num_sectors;
  a.planar_per_sector = P.planar_feats_per_sector;
  a.point_per_sector = P.point_feats_per_sector;
  a.min_points = P.min_points;
  a.pr_cap = ctx->pr_cap;
  a.qr_cap = ctx->qr_cap;
  a.kp_cap = ctx->kp_cap;
  a.kq_cap = ctx->kq_cap;
  a.min_norm2 = P.min_norm_squared;
  a.max_norm2 = P.max_norm_squared;
  a.planar_threshold = P.planar_threshold;
  a.radius = P.radius;
  a.scan = scan_dev;
  a.valid_bits = ctx->d_valid_bits;
  a.row_box = ctx->d_row_box;
  a.planar_cols = ctx->d_planar_cols;
  a.planar_cnt = ctx->d_planar_cnt;
  a.point_cols = ctx->d_point_cols;
  a.point_cnt = ctx->d_point_cnt;
  a.normals = ctx->d_normals;
  a.closest = debug ? ctx->d_closest : nullptr;
  a.keep_cnt = ctx->d_keep_cnt;
  a.cur_planar = ctx->d_cur_planar;
  a.cur_point = ctx->d_cur_point;
  a.cur_counts = ctx->d_cur_counts;
  a.dbg_valid = debug ? ctx->d_dbg_valid : nullptr;
  a.dbg_pvalid = debug ? ctx->d_dbg_pvalid : nullptr;
  a.dbg_curv = debug ? ctx->d_dbg_curv : nullptr;
  a.host_planar = host_records ? ctx->h_planar : nullptr;
  a.host_point = host_records ? ctx->h_point : nullptr;
  a.host_counts = ctx->h_counts;
  a.done_counter = ctx->d_counters + ctx->counter_cap + 2;
  a.flag = publish ? ctx->h_flags + 2 : nullptr;
  a.seq = publish ? ++ctx->seq : 0;
  a.done_target = (unsigned)ctx->rows; // one scan per launch item
  return a;
}

// runs the kernels on a device-resident scan and fetches the two counts
// device alias of a page-locked (cudaHostAlloc / cudaHostRegister, mapped) host pointer,
// nullptr for pageable memory
static void *mapped_alias(void *host_ptr) {
  if (!host_ptr) return nullptr;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, host_ptr) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return attr.type == cudaMemoryTypeHost ? attr.devicePointer : nullptr;
}

} // extern "C"

namespace formgpu {

// stage 1, split so that a batched submit can build the argument blocks of several
// contexts, launch once, and then complete each context
void extract_prepare(formgpu_ctx *ctx, const float4 *scan_dev, uint64_t scan_idx, bool host_records,
                     formgpu_planar_feat *direct_planar, formgpu_point_feat *direct_point,
                     ExtractArgs &a) {
  ctx->cur_buf ^= 1;
  ctx->d_cur_planar = ctx->d_cur_planar_buf[ctx->cur_buf];
  ctx->d_cur_point = ctx->d_cur_point_buf[ctx->cur_buf];
  // the pack kernel writes the counts (and, for host callers, the compact keypoint
  // records) into mapped pinned memory and raises a flag: no memcpy, no stream sync
  a = make_extract_args(ctx, scan_dev, false, host_records, true);
  a.host_planar_f64 = direct_planar;
  a.host_point_f64 = direct_point;
  a.scan_idx = scan_idx;
}

int extract_finish(formgpu_ctx *ctx, const ExtractArgs &a, uint64_t scan_idx) {
  const int w = wait_flag(ctx, 2, a.seq);
  if (w) return w;
  ctx->cur_n[0] = ctx->h_counts[0];
  ctx->cur_n[1] = ctx->h_counts[1];
  // a stale match set whose query buffer has just been overwritten is gone
  if (ctx->match_queries[0] == ctx->d_cur_planar && ctx->cur_n[0] > 0) ctx->match_n[0] = 0;
  if (ctx->match_queries[1] == ctx->d_cur_point && ctx->cur_n[1] > 0) ctx->match_n[1] = 0;
  ctx->cur_scan = scan_idx;
  ctx->have_current = true;
  return FORMGPU_OK;
}

// device aliases of page-locked caller buffers that can hold the worst case (the pack
// kernel then writes the f64 API structs itself); nullptr otherwise
void extract_direct_targets(formgpu_ctx *ctx, formgpu_planar_feat *planar_out, size_t planar_cap,
                            formgpu_point_feat *point_out, size_t point_cap,
                            formgpu_planar_feat *&dp, formgpu_point_feat *&dq) {
  dp = nullptr;
  dq = nullptr;
  if (planar_out && point_out && planar_cap >= ctx->kp_cap && point_cap >= ctx->kq_cap) {
    // probed on EVERY call (cudaPointerGetAttributes is a table lookup): a cached answer keyed
    // on the address would go stale when the caller frees its page-locked buffers and a
    // pageable allocation later lands at the same address
    ctx->direct_probe[0] = planar_out;
    ctx->direct_probe[1] = point_out;
    ctx->direct_alias[0] = mapped_alias(planar_out);
    ctx->direct_alias[1] = mapped_alias(point_out);
    if (ctx->direct_alias[0] && ctx->direct_alias[1]) {
      dp = static_cast<formgpu_planar_feat *>(ctx->direct_alias[0]);
      dq = static_cast<formgpu_point_feat *>(ctx->direct_alias[1]);
    }
  }
}

// widen the compact staging records (mapped pinned, written by the pack kernel) to the
// API's f64 structs
int extract_widen(formgpu_ctx *ctx, uint64_t scan_idx, formgpu_planar_feat *planar_out, size_t planar_cap,
                  formgpu_point_feat *point_out, size_t point_cap) {
  const size_t np = (size_t)ctx->cur_n[0], nq = (size_t)ctx->cur_n[1];
  if ((np && !planar_out) || (nq && !point_out) || np > planar_cap || nq > point_cap)
    return fail(ctx, FORMGPU_ERR_CAPACITY, "formgpu_extract: output buffers too small");
  for (size_t i = 0; i < np; ++i) {
    const PlanarRec &r = ctx->h_planar[i];
    formgpu_planar_feat &o = planar_out[i];
    o.x = r.x; o.y = r.y; o.z = r.z; o.pad = 0.0;
    o.nx = r.nx; o.ny = r.ny; o.nz = r.nz; o.npad = 0.0;
    o.scan = scan_idx;
  }
  for (size_t i = 0; i < nq; ++i) {
    const PointRec &r = ctx->h_point[i];
    formgpu_point_feat &o = point_out[i];
    o.x = r.x; o.y = r.y; o.z = r.z; o.pad = 0.0;
    o.scan = scan_idx;
  }
  return FORMGPU_OK;
}

} // namespace formgpu

static int extract_run(formgpu_ctx *ctx, const float4 *scan_dev, uint64_t scan_idx,
                       bool host_records, formgpu_planar_feat *direct_planar = nullptr,
                       formgpu_point_feat *direct_point = nullptr) {
  ExtractArgs a;
  extract_prepare(ctx, scan_dev, scan_idx, host_records, direct_planar, direct_point, a);
  extract_launch(a, 1, ctx->stream, ctx->prof);
  FORMGPU_CUDA(ctx, cudaGetLastError());
  return extract_finish(ctx, a, scan_idx);
}

int formgpu::extract_run_scan(formgpu_ctx *ctx, const float4 *scan_dev, uint64_t scan_idx, bool host_records,
                              formgpu_planar_feat *direct_planar, formgpu_point_feat *direct_point) {
  return extract_run(ctx, scan_dev, scan_idx, host_records, direct_planar, direct_point);
}

extern "C" {

int formgpu_extract(formgpu_ctx *ctx, const formgpu_point4f *scan, size_t n, uint64_t scan_idx,
                    formgpu_planar_feat *planar_out, size_t planar_cap, size_t *n_planar,
                    formgpu_point_feat *point_out, size_t point_cap, size_t *n_point) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (!scan || !n_planar || !n_point)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_extract: null argument");
  if (n != ctx->n_points)
    return fail(ctx, FORMGPU_ERR_BAD_SCAN_SIZE,
                "Provided scan does not match the expected size " +
                    std::to_string(ctx->n_points) + " != " + std::to_string(n));
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_scan, scan, n * sizeof(float4), cudaMemcpyHostToDevice,
                                    ctx->stream));
  // Page-locked caller buffers that can hold the worst case are written by the pack kernel
  // itself (f64 API structs straight over PCIe); pageable ones go through the compact
  // staging records and are widened here.
  formgpu_planar_feat *dp = nullptr;
  formgpu_point_feat *dq = nullptr;
  extract_direct_targets(ctx, planar_out, planar_cap, point_out, point_cap, dp, dq);
  const bool direct = dp != nullptr;
  const int rc = extract_run(ctx, ctx->d_scan, scan_idx, !direct, dp, dq);
  if (rc) return rc;
  ctx->cur_device_resident = false;
  *n_planar = (size_t)ctx->cur_n[0];
  *n_point = (size_t)ctx->cur_n[1];
  if (direct) return FORMGPU_OK;
  return extract_widen(ctx, scan_idx, planar_out, planar_cap, point_out, point_cap);
}

int formgpu_extract_device(formgpu_ctx *ctx, const formgpu_point4f *scan_dev, size_t n,
                           uint64_t scan_idx, size_t *n_planar, size_t *n_point) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (!scan_dev || !n_planar || !n_point)
    return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_extract_device: null argument");
  if (n != ctx->n_points)
    return fail(ctx, FORMGPU_ERR_BAD_SCAN_SIZE, "Provided scan does not match the expected size");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  // the kernels read the caller's device buffer in place; extract_debug is only
  // available after formgpu_extract (which keeps its own copy)
  const int rc = extract_run(ctx, reinterpret_cast<const float4 *>(scan_dev), scan_idx, false);
  ctx->cur_device_resident = true;
  if (rc) return rc;
  *n_planar = (size_t)ctx->cur_n[0];
  *n_point = (size_t)ctx->cur_n[1];
  return FORMGPU_OK;
}

int formgpu_extract_debug(formgpu_ctx *ctx, uint8_t *valid_mask, uint8_t *point_valid_mask,
                          float *curvature, uint32_t *planar_indices, uint8_t *planar_keep,
                          int32_t *closest_prev, int32_t *closest_next, size_t *n_planar_picks,
                          uint32_t *point_indices, size_t *n_point_picks) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (!ctx->have_current || ctx->cur_device_resident)
    return fail(ctx, FORMGPU_ERR_STATE, "formgpu_extract_debug needs a preceding formgpu_extract");
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t N = ctx->n_points, R = ctx->rows;
  if (!ctx->d_dbg_valid) {
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_dbg_valid, N));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_dbg_pvalid, N));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_dbg_curv, N));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_closest, R * ctx->pr_cap * 2));
  }
  // re-run stage 1 on the resident scan with the debug outputs switched on
  const ExtractArgs a = make_extract_args(ctx, ctx->d_scan, true);
  extract_launch(a, 1, ctx->stream, ctx->prof);
  FORMGPU_CUDA(ctx, cudaGetLastError());
  std::vector<int> pcnt(R), qcnt(R), closest(R * ctx->pr_cap * 2);
  std::vector<uint16_t> pcols(R * ctx->pr_cap), qcols(R * ctx->qr_cap);
  std::vector<float4> normals(R * ctx->pr_cap);
  cudaStream_t s = ctx->stream;
  if (valid_mask) FORMGPU_CUDA(ctx, cudaMemcpyAsync(valid_mask, ctx->d_dbg_valid, N, cudaMemcpyDeviceToHost, s));
  if (point_valid_mask) FORMGPU_CUDA(ctx, cudaMemcpyAsync(point_valid_mask, ctx->d_dbg_pvalid, N, cudaMemcpyDeviceToHost, s));
  if (curvature) FORMGPU_CUDA(ctx, cudaMemcpyAsync(curvature, ctx->d_dbg_curv, N * sizeof(float), cudaMemcpyDeviceToHost, s));
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(pcnt.data(), ctx->d_planar_cnt, R * sizeof(int), cudaMemcpyDeviceToHost, s));
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(qcnt.data(), ctx->d_point_cnt, R * sizeof(int), cudaMemcpyDeviceToHost, s));
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(pcols.data(), ctx->d_planar_cols, pcols.size() * sizeof(uint16_t), cudaMemcpyDeviceToHost, s));
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(qcols.data(), ctx->d_point_cols, qcols.size() * sizeof(uint16_t), cudaMemcpyDeviceToHost, s));
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(normals.data(), ctx->d_normals, normals.size() * sizeof(float4), cudaMemcpyDeviceToHost, s));
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(closest.data(), ctx->d_closest, closest.size() * sizeof(int), cudaMemcpyDeviceToHost, s));
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(s));
  size_t kp = 0, kq = 0;
  for (size_t r = 0; r < R; ++r) {
    for (int j = 0; j < pcnt[r]; ++j, ++kp) {
      const size_t e = r * ctx->pr_cap + j;
      if (planar_indices) planar_indices[kp] = (uint32_t)(r * ctx->cols + pcols[e]);
      if (planar_keep) planar_keep[kp] = normals[e].w != 0.0f;
      if (closest_prev) closest_prev[kp] = closest[2 * e];
      if (closest_next) closest_next[kp] = closest[2 * e + 1];
    }
    for (int j = 0; j < qcnt[r]; ++j, ++kq)
      if (point_indices) point_indices[kq] = (uint32_t)(r * ctx->cols + qcols[r * ctx->qr_cap + j]);
  }
  if (n_planar_picks) *n_planar_picks = kp;
  if (n_point_picks) *n_point_picks = kq;
  return FORMGPU_OK;
}

// ---------------------------------------------------------------------------
// instrumentation
// ---------------------------------------------------------------------------
int formgpu_profile_enable(formgpu_ctx *ctx, int on) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  ctx->prof.collect();
  ctx->prof.timing = on != 0;
  return FORMGPU_OK;
}

int formgpu_profile_read(formgpu_ctx *ctx, double ms[FORMGPU_KG_COUNT],
                         uint64_t launches[FORMGPU_KG_COUNT]) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  ctx->prof.collect();
  for (int g = 0; g < FORMGPU_KG_COUNT; ++g) {
    if (ms) ms[g] = ctx->prof.group[g].ms;
    if (launches) launches[g] = ctx->prof.group[g].launches;
    ctx->prof.group[g] = GroupProf();
  }
  return FORMGPU_OK;
}

uint64_t formgpu_launch_count(const formgpu_ctx *ctx) { return ctx ? ctx->prof.total_launches : 0; }

int formgpu_synchronize(formgpu_ctx *ctx) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FORMGPU_OK;
}

} // extern "C"
