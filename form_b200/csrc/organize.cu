// Raw sensor clouds -> organised row-major scans (rule R8, DESIGN.md §4).  Compiled with
// -fmad=false: the row / column decisions and the collision key are index work and must be the
// exact arithmetic that tests/cloud_model.py restates in numpy.
//
// Three kernels per organisation, each of them launched once per submission whatever the number
// of clouds in it (blockIdx.y = item, the item's argument block read from device memory as the
// batched extraction kernels do):
//   1. clear   - per-pixel u64 keys to ~0, the outcome counters to 0
//   2. scatter - one thread per record: decode, drop rules, row and column, 64-bit atomicMin of
//                (f32 bits of |p|^2) << 32 | record index; outcomes counted per warp
//   3. gather  - one thread per pixel: the winner's point, or (0, 0, 0, 0), into the scan buffer
#include "kernels.hpp"

namespace formgpu {
namespace {

constexpr int kOrgThreads = 256;
constexpr unsigned long long kNoKey = ~0ull;

__device__ __forceinline__ uint32_t ld_u32(const unsigned char *p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ unsigned long long ld_u64(const unsigned char *p) {
  return (unsigned long long)ld_u32(p) | ((unsigned long long)ld_u32(p + 4) << 32);
}
__device__ __forceinline__ float ld_coord(const unsigned char *p, int type) {
  if (type == FORMGPU_FIELD_F64) return (float)__longlong_as_double((long long)ld_u64(p)); // (float)v, as add_lidar
  return __uint_as_float(ld_u32(p));
}
__device__ __forceinline__ uint32_t ld_index(const unsigned char *p, int type) {
  if (type == FORMGPU_FIELD_U8) return p[0];
  if (type == FORMGPU_FIELD_U16) return (uint32_t)p[0] | ((uint32_t)p[1] << 8);
  return ld_u32(p);
}
__device__ __forceinline__ double ld_time(const unsigned char *p, int type) {
  if (type == FORMGPU_FIELD_F32) return (double)__uint_as_float(ld_u32(p));
  if (type == FORMGPU_FIELD_F64) return __longlong_as_double((long long)ld_u64(p));
  return (double)ld_u32(p) * 1e-9; // u32 nanoseconds
}

__device__ __forceinline__ void load_xyz(const OrganizeArgs &a, const unsigned char *rec, float &x, float &y,
                                         float &z) {
  x = ld_coord(rec + a.off_x, a.xyz_type);
  y = ld_coord(rec + a.off_y, a.xyz_type);
  z = ld_coord(rec + a.off_z, a.xyz_type);
}

// Nearest column centre by half-plane tests against the boundary lines az_tab[b] = (cos, sin) of
// phi_b = origin + dir * 2 pi (b - 1/2) / cols; column c spans [phi_c, phi_c+1).  "At or past
// boundary b" is dir * (y cos phi_b - x sin phi_b) >= 0, which orders the point against every
// boundary of the same half turn: the half is picked against boundaries 0 and cols/2, then a
// binary search runs inside it.
__device__ __forceinline__ bool past(const OrganizeArgs &a, double x, double y, int b) {
  const double2 cs = a.az_tab[b];
  double s = y * cs.x - x * cs.y;
  if (a.az_dir < 0) s = -s;
  return s >= 0.0;
}
__device__ int azimuth_column(const OrganizeArgs &a, float xf, float yf) {
  const double x = (double)xf, y = (double)yf;
  const int m = a.cols / 2;
  int lo = 0, hi = m;
  if (!(past(a, x, y, 0) && !past(a, x, y, m))) {
    lo = m;
    hi = a.cols;
  }
  while (hi - lo > 1) {
    const int mid = (lo + hi) / 2;
    if (past(a, x, y, mid)) lo = mid;
    else hi = mid;
  }
  return lo;
}

// Nearest beam: el_tab holds (cos, sin) of the rows - 1 midpoints of adjacent beams in ascending
// order; k = number of midpoints the point is at or above (z cos mu - rho sin mu >= 0, rho in f64).
__device__ int elevation_row(const OrganizeArgs &a, float xf, float yf, float zf) {
  const double x = (double)xf, y = (double)yf, z = (double)zf;
  const double rho = sqrt(x * x + y * y);
  int lo = 0, hi = a.rows - 1;
  while (lo < hi) {
    const int mid = (lo + hi) / 2;
    const double2 cs = a.el_tab[mid];
    if (z * cs.x - rho * cs.y >= 0.0) lo = mid + 1;
    else hi = mid;
  }
  return a.el_desc ? a.rows - 1 - lo : lo;
}

__device__ __forceinline__ void count_warp(unsigned *stats, int code) {
  // warp-aggregated outcome counters: one atomic per outcome present in the warp
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 1; k < kOrgStats; ++k) {
    if (k == kOrgStatPixels) continue;
    const unsigned m = __ballot_sync(0xffffffffu, code == k);
    if (m && lane == 0) atomicAdd(stats + k, (unsigned)__popc(m));
  }
}

__device__ __forceinline__ void clear_body(const OrganizeArgs &a, unsigned i) {
  if (i < (unsigned)(a.rows * a.cols)) a.keys[i] = kNoKey;
  if (i < (unsigned)kOrgStats) a.stats[i] = 0u;
}

__device__ __forceinline__ void scatter_body(const OrganizeArgs &a, unsigned i) {
  int code = 0;
  if (i < a.n) {
    const unsigned char *rec = a.records + (size_t)i * a.stride;
    float x, y, z;
    load_xyz(a, rec, x, y, z);
    const bool has_time = a.off_time >= 0;
    const double t = has_time ? ld_time(rec + a.off_time, a.time_type) : 0.0;
    if (!isfinite(x) || !isfinite(y) || !isfinite(z)) {
      code = kOrgStatNonfinite;
    } else if (x == 0.0f && y == 0.0f && z == 0.0f) {
      code = kOrgStatZero;
    } else if (has_time && !(t >= 0.0 && t < a.scan_period)) {
      code = kOrgStatTime;
    } else {
      int row;
      if (a.row_source == FORMGPU_ROW_FROM_FIELD) {
        const uint32_t v = ld_index(rec + a.off_row, a.row_type);
        row = v < (uint32_t)a.rows ? (int)v : -1;
      } else {
        row = elevation_row(a, x, y, z);
      }
      int col;
      if (a.col_source == FORMGPU_COL_FROM_FIELD) {
        const uint32_t v = ld_index(rec + a.off_col, a.col_type);
        col = v < (uint32_t)a.cols ? (int)v : -1;
      } else if (a.col_source == FORMGPU_COL_FROM_TIME) {
        const double q = (t * (double)a.cols) / a.scan_period;
        col = min((int)floor(q), a.cols - 1);
      } else {
        col = azimuth_column(a, x, y);
      }
      if (row < 0) {
        code = kOrgStatRow;
      } else if (col < 0) {
        code = kOrgStatCol;
      } else {
        code = kOrgStatPlaced;
        const float n2 = (x * x + z * z) + (y * y + 0.0f); // PointXYZf::squaredNorm
        const unsigned long long key = ((unsigned long long)__float_as_uint(n2) << 32) | (unsigned long long)i;
        atomicMin(a.keys + (size_t)row * a.cols + col, key);
      }
    }
  }
  count_warp(a.stats, code);
}

__device__ __forceinline__ void gather_body(const OrganizeArgs &a, unsigned i) {
  const unsigned npix = (unsigned)(a.rows * a.cols);
  bool filled = false;
  if (i < npix) {
    const unsigned long long key = a.keys[i];
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (key != kNoKey) {
      const unsigned char *rec = a.records + (size_t)(key & 0xffffffffull) * a.stride;
      load_xyz(a, rec, p.x, p.y, p.z);
      filled = true;
    }
    a.scan[i] = p;
  }
  const unsigned m = __ballot_sync(0xffffffffu, filled);
  if (m && (threadIdx.x & 31) == 0) atomicAdd(a.stats + kOrgStatPixels, (unsigned)__popc(m));
}

__global__ void __launch_bounds__(kOrgThreads) organize_clear_kernel(OrganizeArgs a) {
  clear_body(a, blockIdx.x * kOrgThreads + threadIdx.x);
}
__global__ void __launch_bounds__(kOrgThreads) organize_scatter_kernel(OrganizeArgs a) {
  if (blockIdx.x * kOrgThreads >= a.n) return;
  scatter_body(a, blockIdx.x * kOrgThreads + threadIdx.x);
}
__global__ void __launch_bounds__(kOrgThreads) organize_gather_kernel(OrganizeArgs a) {
  if (blockIdx.x * kOrgThreads >= (unsigned)(a.rows * a.cols)) return;
  gather_body(a, blockIdx.x * kOrgThreads + threadIdx.x);
}

// batched: blockIdx.y selects the item; CTAs past their own item's records / pixels exit whole
__global__ void __launch_bounds__(kOrgThreads) organize_clear_batch_kernel(const OrganizeArgs *items) {
  const OrganizeArgs &a = items[blockIdx.y];
  if (blockIdx.x * kOrgThreads >= (unsigned)max(a.rows * a.cols, kOrgStats)) return;
  clear_body(a, blockIdx.x * kOrgThreads + threadIdx.x);
}
__global__ void __launch_bounds__(kOrgThreads) organize_scatter_batch_kernel(const OrganizeArgs *items) {
  const OrganizeArgs &a = items[blockIdx.y];
  if (blockIdx.x * kOrgThreads >= a.n) return;
  scatter_body(a, blockIdx.x * kOrgThreads + threadIdx.x);
}
__global__ void __launch_bounds__(kOrgThreads) organize_gather_batch_kernel(const OrganizeArgs *items) {
  const OrganizeArgs &a = items[blockIdx.y];
  if (blockIdx.x * kOrgThreads >= (unsigned)(a.rows * a.cols)) return;
  gather_body(a, blockIdx.x * kOrgThreads + threadIdx.x);
}

unsigned blocks_for(size_t n) { return (unsigned)std::max<size_t>((n + kOrgThreads - 1) / kOrgThreads, 1); }

} // namespace

void organize_launch(const OrganizeArgs &a, cudaStream_t stream, Profiler &prof) {
  const size_t npix = (size_t)a.rows * a.cols;
  organize_clear_kernel<<<blocks_for(std::max<size_t>(npix, kOrgStats)), kOrgThreads, 0, stream>>>(a);
  if (a.n) organize_scatter_kernel<<<blocks_for(a.n), kOrgThreads, 0, stream>>>(a);
  organize_gather_kernel<<<blocks_for(npix), kOrgThreads, 0, stream>>>(a);
  prof.total_launches += a.n ? 3 : 2;
}

void organize_batch_launch(const OrganizeArgs *items_dev, int n_items, size_t max_records, size_t max_pixels,
                           cudaStream_t stream, Profiler &prof) {
  const dim3 clear(blocks_for(std::max<size_t>(max_pixels, kOrgStats)), (unsigned)n_items);
  organize_clear_batch_kernel<<<clear, kOrgThreads, 0, stream>>>(items_dev);
  if (max_records) {
    const dim3 scatter(blocks_for(max_records), (unsigned)n_items);
    organize_scatter_batch_kernel<<<scatter, kOrgThreads, 0, stream>>>(items_dev);
  }
  const dim3 gather(blocks_for(max_pixels), (unsigned)n_items);
  organize_gather_batch_kernel<<<gather, kOrgThreads, 0, stream>>>(items_dev);
  prof.total_launches += max_records ? 3 : 2;
}

} // namespace formgpu
