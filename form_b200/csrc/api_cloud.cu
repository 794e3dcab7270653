// C-ABI (include/formgpu.h): raw sensor clouds - format, organisation (organize.cu), and
// extraction of a cloud.  The batched form (FORMGPU_REQ_CLOUD) is in api_batch.cu.
#include "api_common.hpp"

#include <algorithm>
#include <cmath>

using namespace formgpu;

namespace {

bool int_type(int t) { return t == FORMGPU_FIELD_U8 || t == FORMGPU_FIELD_U16 || t == FORMGPU_FIELD_U32; }
int type_bytes(int t) {
  switch (t) {
  case FORMGPU_FIELD_U8: return 1;
  case FORMGPU_FIELD_U16: return 2;
  case FORMGPU_FIELD_F64: return 8;
  default: return 4;
  }
}

} // namespace

namespace formgpu {

int check_cloud_format(const formgpu_cloud_format &f, int rows, int cols, std::string &msg) {
  auto bad = [&](int code, const std::string &m) {
    msg = "cloud format: " + m;
    return code;
  };
  if (rows < 1 || cols < 2) return bad(FORMGPU_ERR_INVALID_ARG, "the scan needs rows >= 1 and cols >= 2");
  if (f.stride == 0 || f.stride > 65536) return bad(FORMGPU_ERR_INVALID_ARG, "stride must be in [1, 65536] bytes");
  auto field = [&](const char *name, int off, int type, bool ok_type) -> int {
    if (!ok_type) return bad(FORMGPU_ERR_INVALID_ARG, std::string(name) + ": unsupported field type " + std::to_string(type));
    if (off < 0 || (int64_t)off + type_bytes(type) > (int64_t)f.stride)
      return bad(FORMGPU_ERR_INVALID_ARG, std::string(name) + ": offset " + std::to_string(off) + " does not fit a " +
                                              std::to_string(f.stride) + "-byte record");
    return FORMGPU_OK;
  };
  const bool xyz_ok = f.xyz_type == FORMGPU_FIELD_F32 || f.xyz_type == FORMGPU_FIELD_F64;
  int rc;
  if ((rc = field("x", f.off_x, f.xyz_type, xyz_ok)) || (rc = field("y", f.off_y, f.xyz_type, xyz_ok)) ||
      (rc = field("z", f.off_z, f.xyz_type, xyz_ok)))
    return rc;
  if (f.off_row != FORMGPU_CLOUD_ABSENT && (rc = field("row", f.off_row, f.row_type, int_type(f.row_type)))) return rc;
  if (f.off_col != FORMGPU_CLOUD_ABSENT && (rc = field("col", f.off_col, f.col_type, int_type(f.col_type)))) return rc;
  if (f.off_time != FORMGPU_CLOUD_ABSENT &&
      (rc = field("time", f.off_time, f.time_type,
                  f.time_type == FORMGPU_FIELD_F32 || f.time_type == FORMGPU_FIELD_F64 ||
                      f.time_type == FORMGPU_FIELD_U32_NS)))
    return rc;
  if (!(f.scan_period > 0.0) || !std::isfinite(f.scan_period))
    return bad(FORMGPU_ERR_INVALID_ARG, "scan_period must be a positive number of seconds");
  if (f.max_records == 0 || f.max_records > 0xffffffffull)
    return bad(FORMGPU_ERR_INVALID_ARG, "max_records must be in [1, 2^32 - 1]");
  switch (f.row_source) {
  case FORMGPU_ROW_FROM_FIELD:
    if (f.off_row == FORMGPU_CLOUD_ABSENT) return bad(FORMGPU_ERR_INVALID_ARG, "row source FIELD needs a ring / row field");
    break;
  case FORMGPU_ROW_FROM_ELEVATION: {
    if (!f.beam_elevations) return bad(FORMGPU_ERR_INVALID_ARG, "row source ELEVATION needs beam_elevations");
    const double *e = f.beam_elevations;
    for (int r = 0; r < rows; ++r)
      if (!(std::fabs(e[r]) < 1.5707963267948966))
        return bad(FORMGPU_ERR_INVALID_ARG, "beam elevation " + std::to_string(r) + " is not in (-pi/2, pi/2)");
    const bool up = rows < 2 || e[1] > e[0];
    for (int r = 1; r < rows; ++r)
      if (up ? !(e[r] > e[r - 1]) : !(e[r] < e[r - 1]))
        return bad(FORMGPU_ERR_INVALID_ARG, "beam elevations must be strictly monotonic (beam " + std::to_string(r) + ")");
    break;
  }
  default: return bad(FORMGPU_ERR_INVALID_ARG, "unknown row source " + std::to_string(f.row_source));
  }
  switch (f.col_source) {
  case FORMGPU_COL_FROM_FIELD:
    if (f.off_col == FORMGPU_CLOUD_ABSENT) return bad(FORMGPU_ERR_INVALID_ARG, "column source FIELD needs a col field");
    break;
  case FORMGPU_COL_FROM_TIME:
    if (f.off_time == FORMGPU_CLOUD_ABSENT) return bad(FORMGPU_ERR_INVALID_ARG, "column source TIME needs a time field");
    break;
  case FORMGPU_COL_FROM_AZIMUTH:
    if (f.azimuth_dir != 1 && f.azimuth_dir != -1) return bad(FORMGPU_ERR_INVALID_ARG, "azimuth_dir must be +1 or -1");
    if (!std::isfinite(f.azimuth_origin)) return bad(FORMGPU_ERR_INVALID_ARG, "azimuth_origin must be finite");
    break;
  default: return bad(FORMGPU_ERR_INVALID_ARG, "unknown column source " + std::to_string(f.col_source));
  }
  return FORMGPU_OK;
}

// The boundary tables of rule R8, host IEEE f64 and the C library's cos / sin (what
// tests/cloud_model.py computes with Python's math module):
//   azimuth: phi_b = origin + dir * (2 pi (b - 0.5) / cols), b = 0 .. cols
//   beams:   mu_j = (a_j + a_j+1) * 0.5 over the table in ascending order a
void cloud_tables(const formgpu_cloud_format &f, int rows, int cols, std::vector<double2> &tab, int &desc) {
  tab.assign((size_t)cols + 1 + (size_t)std::max(rows - 1, 0), double2{0.0, 0.0});
  for (int b = 0; b <= cols; ++b) {
    const double phi = f.azimuth_origin + (double)f.azimuth_dir * (2.0 * M_PI * ((double)b - 0.5) / (double)cols);
    tab[b] = double2{std::cos(phi), std::sin(phi)};
  }
  desc = 0;
  if (f.row_source != FORMGPU_ROW_FROM_ELEVATION) return;
  std::vector<double> asc(f.beam_elevations, f.beam_elevations + rows);
  if (rows > 1 && asc[1] < asc[0]) {
    desc = 1;
    std::reverse(asc.begin(), asc.end());
  }
  for (int j = 0; j + 1 < rows; ++j) {
    const double mu = (asc[j] + asc[j + 1]) * 0.5;
    tab[(size_t)cols + 1 + j] = double2{std::cos(mu), std::sin(mu)};
  }
}

OrganizeArgs cloud_args(formgpu_ctx *ctx, const unsigned char *records_dev, size_t n) {
  const formgpu_cloud_format &f = ctx->cloud;
  OrganizeArgs a{};
  a.records = records_dev;
  a.n = (unsigned)n;
  a.stride = f.stride;
  a.off_x = f.off_x;
  a.off_y = f.off_y;
  a.off_z = f.off_z;
  a.off_row = f.off_row;
  a.off_col = f.off_col;
  a.off_time = f.off_time;
  a.xyz_type = f.xyz_type;
  a.row_type = f.row_type;
  a.col_type = f.col_type;
  a.time_type = f.time_type;
  a.row_source = f.row_source;
  a.col_source = f.col_source;
  a.rows = ctx->rows;
  a.cols = ctx->cols;
  a.az_dir = f.azimuth_dir;
  a.el_desc = ctx->cloud_el_desc;
  a.scan_period = f.scan_period;
  a.az_tab = ctx->d_cloud_tab;
  a.el_tab = ctx->d_cloud_tab + ctx->cols + 1;
  a.keys = ctx->d_pixel_keys;
  a.scan = ctx->d_scan;
  a.stats = ctx->d_cloud_stats;
  return a;
}

int cloud_check_request(formgpu_ctx *ctx, const void *records, size_t n, const char *who) {
  if (!ctx->have_cloud)
    return fail(ctx, FORMGPU_ERR_STATE,
                std::string(who) + ": the context has no cloud format (formgpu_set_cloud_format)");
  if (!records && n) return fail(ctx, FORMGPU_ERR_INVALID_ARG, std::string(who) + ": null records");
  if (n > ctx->cloud.max_records)
    return fail(ctx, FORMGPU_ERR_CAPACITY,
                std::string(who) + ": " + std::to_string(n) + " records exceed the format's max_records " +
                    std::to_string(ctx->cloud.max_records));
  return FORMGPU_OK;
}

} // namespace formgpu

namespace {

void read_stats(const formgpu_ctx *ctx, formgpu_cloud_stats *s) {
  const unsigned *h = ctx->h_cloud_stats;
  s->records = ctx->cloud_last_n;
  s->placed = h[kOrgStatPlaced];
  s->pixels = h[kOrgStatPixels];
  s->dropped_nonfinite = h[kOrgStatNonfinite];
  s->dropped_zero = h[kOrgStatZero];
  s->dropped_time = h[kOrgStatTime];
  s->dropped_row = h[kOrgStatRow];
  s->dropped_col = h[kOrgStatCol];
}

// upload (host records) + the three kernels + the counters' copy, queued on the context's stream
int organize_queue(formgpu_ctx *ctx, const void *records, size_t n) {
  if (n)
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_records, records, n * ctx->cloud.stride, cudaMemcpyHostToDevice,
                                      ctx->stream));
  ctx->prefetched_cloud = nullptr;
  organize_launch(cloud_args(ctx, ctx->d_records, n), ctx->stream, ctx->prof);
  FORMGPU_CUDA(ctx, cudaGetLastError());
  FORMGPU_CUDA(ctx, cudaMemcpyAsync(ctx->h_cloud_stats, ctx->d_cloud_stats, kOrgStats * sizeof(unsigned),
                                    cudaMemcpyDeviceToHost, ctx->stream));
  ctx->cloud_last_n = n;
  return FORMGPU_OK;
}

} // namespace

extern "C" {

int formgpu_cloud_format_check(const formgpu_cloud_format *fmt, int rows, int cols, char *msg, size_t msg_cap) {
  std::string m;
  const int rc = fmt ? check_cloud_format(*fmt, rows, cols, m) : (m = "cloud format: null", FORMGPU_ERR_INVALID_ARG);
  if (msg && msg_cap) {
    const size_t k = std::min(m.size(), msg_cap - 1);
    std::memcpy(msg, m.data(), k);
    msg[k] = '\0';
  }
  return rc;
}

int formgpu_set_cloud_format(formgpu_ctx *ctx, const formgpu_cloud_format *fmt) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (!fmt) return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_set_cloud_format: null format");
  {
    std::string msg;
    const int rc = check_cloud_format(*fmt, ctx->rows, ctx->cols, msg);
    if (rc) return fail(ctx, rc, msg);
  }
  std::vector<double2> tab;
  int desc = 0;
  cloud_tables(*fmt, ctx->rows, ctx->cols, tab, desc);
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // no organisation of the old format in flight
  const size_t bytes = (size_t)fmt->max_records * fmt->stride;
  if (!ctx->have_cloud || bytes > (size_t)ctx->cloud.max_records * ctx->cloud.stride) {
    if (ctx->d_records) cudaFree(ctx->d_records);
    ctx->d_records = nullptr;
    ctx->have_cloud = false;
    FORMGPU_CUDA(ctx, cudaMalloc(reinterpret_cast<void **>(&ctx->d_records), bytes));
  }
  if (!ctx->d_pixel_keys) {
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_pixel_keys, ctx->n_points));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_cloud_tab, (size_t)ctx->cols + ctx->rows));
    FORMGPU_CUDA(ctx, dev_alloc(&ctx->d_cloud_stats, (size_t)kOrgStats));
    FORMGPU_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_cloud_stats), kOrgStats * sizeof(unsigned),
                                    cudaHostAllocDefault));
    std::memset(ctx->h_cloud_stats, 0, kOrgStats * sizeof(unsigned));
  }
  FORMGPU_CUDA(ctx, cudaMemcpy(ctx->d_cloud_tab, tab.data(), tab.size() * sizeof(double2), cudaMemcpyHostToDevice));
  ctx->cloud = *fmt;
  ctx->cloud.beam_elevations = nullptr;
  ctx->cloud_el_desc = desc;
  ctx->cloud_last_n = 0;
  ctx->prefetched_cloud = nullptr;
  ctx->have_cloud = true;
  return FORMGPU_OK;
}

int formgpu_organize(formgpu_ctx *ctx, const void *records, size_t n, formgpu_point4f *out,
                     formgpu_cloud_stats *stats) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  int rc = cloud_check_request(ctx, records, n, "formgpu_organize");
  if (rc) return rc;
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  rc = organize_queue(ctx, records, n);
  if (rc) return rc;
  // the scan buffer now holds this cloud, not the current scan's input: formgpu_extract_debug
  // needs a new formgpu_extract
  ctx->cur_device_resident = true;
  if (out)
    FORMGPU_CUDA(ctx, cudaMemcpyAsync(out, ctx->d_scan, ctx->n_points * sizeof(float4), cudaMemcpyDeviceToHost,
                                      ctx->stream));
  FORMGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (stats) read_stats(ctx, stats);
  return FORMGPU_OK;
}

int formgpu_extract_cloud(formgpu_ctx *ctx, const void *records, size_t n, uint64_t scan_idx,
                          formgpu_planar_feat *planar_out, size_t planar_cap, size_t *n_planar,
                          formgpu_point_feat *point_out, size_t point_cap, size_t *n_point) {
  if (!ctx) return FORMGPU_ERR_INVALID_ARG;
  if (!n_planar || !n_point) return fail(ctx, FORMGPU_ERR_INVALID_ARG, "formgpu_extract_cloud: null argument");
  int rc = cloud_check_request(ctx, records, n, "formgpu_extract_cloud");
  if (rc) return rc;
  FORMGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  ProfScope scope(ctx);
  rc = organize_queue(ctx, records, n);
  if (rc) return rc;
  // from here on formgpu_extract on the organised scan (stream order: the pack kernel's flag
  // is raised after the counters' copy has landed)
  formgpu_planar_feat *dp = nullptr;
  formgpu_point_feat *dq = nullptr;
  extract_direct_targets(ctx, planar_out, planar_cap, point_out, point_cap, dp, dq);
  const bool direct = dp != nullptr;
  rc = extract_run_scan(ctx, ctx->d_scan, scan_idx, !direct, dp, dq);
  if (rc) return rc;
  ctx->cur_device_resident = false;
  *n_planar = (size_t)ctx->cur_n[0];
  *n_point = (size_t)ctx->cur_n[1];
  if (direct) return FORMGPU_OK;
  return extract_widen(ctx, scan_idx, planar_out, planar_cap, point_out, point_cap);
}

int formgpu_cloud_stats_last(const formgpu_ctx *ctx, formgpu_cloud_stats *stats) {
  if (!ctx || !stats) return FORMGPU_ERR_INVALID_ARG;
  if (!ctx->have_cloud) return fail(ctx, FORMGPU_ERR_STATE, "formgpu_cloud_stats_last: the context has no cloud format");
  read_stats(ctx, stats);
  return FORMGPU_OK;
}

} // extern "C"
