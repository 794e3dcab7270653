// Stage 2 on sm_100a: reparative map rebuild, voxel-hash nearest neighbour,
// correspondence segments and novel-keypoint commit.
//
// Replaces KeypointMap::to_voxel_map / VoxelMap::push_back / find_closest
// (/root/reference/form/mapping/map.tpp:34-165), Matcher::match
// (/root/reference/form/optimization/matcher.hpp:67-112) and
// KeypointMap::insert_matches (map.tpp:148-165).  Compiled with -fmad=false:
// world coordinates, voxel keys and squared distances are evaluated in the
// oracle's operation order (SURVEY A.2) so keys and neighbour ids are bit-exact.
//
// Data structure: tsl::robin_map<Vector3i, vector<Point>> becomes
//   * an open-addressing table of 16-byte slots {packed voxel key, start, count}
//     (linear probing, 64-bit CAS insert, load factor <= 0.5), and
//   * the world points (32 B: x, y, z f64 + tie-break id) stored contiguously
//     per voxel (CSR), so a bucket scan is a run of whole 32-byte sectors; buckets of
//     kCellMin..kCellMax points are ordered by 4x4x4 sub-cells and carry a cell table.
// Two searches: a single sequence's association shares one query between the 32 lanes of a warp
// (assoc_nn_body: whole buckets of the centre voxel and of the neighbour voxels of the reference's
// shift table, map.tpp:54-68, that the face bounds cannot rule out); batched submits give a query
// to one thread, which searches cell by cell (assoc_cells_body).  Both take the arg-min of the key
// (dist^2, shift rank, scan, k): rule R5, identical to the reference's strict-< visiting order.
#include "ctx.hpp"
#include "kernels.hpp"

#include <algorithm>
#include <cfloat>

namespace formgpu {

namespace {

// map.tpp:54-68: the 27 neighbour shifts in the reference's order.
// Packed 2 bits per entry as two's complement (0 -> 00, +1 -> 01, -1 -> 11), 16 voxels per
// 32-bit word, so a lane decodes a shift with a select, a left shift and an arithmetic right
// shift instead of a lane-divergent (serialised) constant-memory load.
constexpr uint32_t pack_axis(int axis, int half) {
  constexpr int T[27][3] = {
      {0, 0, 0},   {1, 0, 0},   {-1, 0, 0},  {0, 1, 0},   {0, -1, 0},  {0, 0, 1},   {0, 0, -1},
      {1, 1, 0},   {1, -1, 0},  {-1, 1, 0},  {-1, -1, 0}, {1, 0, 1},   {1, 0, -1},  {-1, 0, 1},
      {-1, 0, -1}, {0, 1, 1},   {0, 1, -1},  {0, -1, 1},  {0, -1, -1}, {1, 1, 1},   {1, 1, -1},
      {1, -1, 1},  {1, -1, -1}, {-1, 1, 1},  {-1, 1, -1}, {-1, -1, 1}, {-1, -1, -1}};
  uint32_t v = 0;
  for (int l = 0; l < 16; ++l)
    if (16 * half + l < 27) v |= ((uint32_t)T[16 * half + l][axis] & 3u) << (2 * l);
  return v;
}
constexpr uint32_t kShX0 = pack_axis(0, 0), kShX1 = pack_axis(0, 1), kShY0 = pack_axis(1, 0),
                   kShY1 = pack_axis(1, 1), kShZ0 = pack_axis(2, 0), kShZ1 = pack_axis(2, 1);
// shift of the voxel with rank v (0..31; ranks >= 27 decode to 0) along `axis` (compile-time)
__device__ __forceinline__ int lane_shift(int v, int axis) {
  const uint32_t lo = axis == 0 ? kShX0 : axis == 1 ? kShY0 : kShZ0;
  const uint32_t hi = axis == 0 ? kShX1 : axis == 1 ? kShY1 : kShZ1;
  const uint32_t w = (v & 16) ? hi : lo;
  return (int)(w << (30 - 2 * (v & 15))) >> 30;
}

// inverse of the table: rank of the shift (sx, sy, sz), 5 bits per entry, 12 entries per word
constexpr unsigned long long pack_rank(int word) {
  constexpr int T[27][3] = {
      {0, 0, 0},   {1, 0, 0},   {-1, 0, 0},  {0, 1, 0},   {0, -1, 0},  {0, 0, 1},   {0, 0, -1},
      {1, 1, 0},   {1, -1, 0},  {-1, 1, 0},  {-1, -1, 0}, {1, 0, 1},   {1, 0, -1},  {-1, 0, 1},
      {-1, 0, -1}, {0, 1, 1},   {0, 1, -1},  {0, -1, 1},  {0, -1, -1}, {1, 1, 1},   {1, 1, -1},
      {1, -1, 1},  {1, -1, -1}, {-1, 1, 1},  {-1, 1, -1}, {-1, -1, 1}, {-1, -1, -1}};
  unsigned long long v = 0;
  for (int r = 0; r < 27; ++r) {
    const int idx = (T[r][0] + 1) * 9 + (T[r][1] + 1) * 3 + (T[r][2] + 1);
    if (idx / 12 == word) v |= (unsigned long long)r << (5 * (idx % 12));
  }
  return v;
}
constexpr unsigned long long kRank0 = pack_rank(0), kRank1 = pack_rank(1), kRank2 = pack_rank(2);
__device__ __forceinline__ int shift_rank(int sx, int sy, int sz) {
  const int idx = (sx + 1) * 9 + (sy + 1) * 3 + (sz + 1);
  const unsigned long long wd = idx < 12 ? kRank0 : idx < 24 ? kRank1 : kRank2;
  return (int)((wd >> (5 * (idx % 12))) & 31ull);
}

constexpr unsigned long long kEmptyKey = 0ull; // table is cleared with memset(0)

// 21 bits per axis (two's complement wrap), bit 63 marks "occupied".
__device__ __forceinline__ unsigned long long pack_key(int x, int y, int z) {
  return (1ull << 63) | ((unsigned long long)(x & 0x1FFFFF) << 42) |
         ((unsigned long long)(y & 0x1FFFFF) << 21) | (unsigned long long)(z & 0x1FFFFF);
}

__device__ __forceinline__ uint32_t hash_key(unsigned long long k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ull;
  k ^= k >> 33;
  return (uint32_t)k;
}

// VoxelMap::computeCoords (map.tpp:34-38): floor(p / width) with an IEEE division.
// q = v * fl(1 / width) differs from the correctly rounded quotient by less than 3.4e-16 |q|
// (three roundings), so both have the same floor unless q lies within that distance of an
// integer; only then (about one coordinate in 1e13) is the division carried out.  Exact by
// construction: the result is always floor(fl(v / width)).
__device__ __forceinline__ int voxel_coord(double v, double width, double inv_width) {
  const double q = v * inv_width;
  const double f = floor(q);
  const double fr = q - f; // exact, in [0, 1)
  const double tol = 8.9e-16 * (fabs(q) + 1.0);
  if (fr < tol || fr > 1.0 - tol) return (int)floor(v / width);
  return (int)f;
}

// R p + t in the oracle's order ((r0 x + r1 y) + r2 z) + t
__device__ __forceinline__ void transform_point(const double *T, double x, double y, double z,
                                                double &ox, double &oy, double &oz) {
  ox = ((T[0] * x + T[1] * y) + T[2] * z) + T[9];
  oy = ((T[3] * x + T[4] * y) + T[5] * z) + T[10];
  oz = ((T[6] * x + T[7] * y) + T[8] * z) + T[11];
}

template <typename Rec> __device__ __forceinline__ void load_xyz(const Rec *r, double &x, double &y, double &z) {
  x = (double)r->x;
  y = (double)r->y;
  z = (double)r->z;
}

// global index -> (slot, k) through the exclusive prefix of the store counts
__device__ __forceinline__ int find_slot_of(const int *off, int W, int g) {
  int lo = 0, hi = W; // largest s with off[s] <= g
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (off[mid] <= g) lo = mid;
    else hi = mid;
  }
  return lo;
}

// Batched launches (blockIdx.z = item = one sequence) read their argument block from a
// device array [item][type]: one cooperative copy into shared memory per CTA.
template <typename T> __device__ __forceinline__ void load_item_args(T &dst, const T *src) {
  static_assert(sizeof(T) % 8 == 0, "argument blocks are copied in 8-byte words");
  for (int i = threadIdx.x; i < (int)(sizeof(T) / 8); i += blockDim.x)
    reinterpret_cast<unsigned long long *>(&dst)[i] = reinterpret_cast<const unsigned long long *>(src)[i];
  __syncthreads();
}

} // namespace

// ---------------------------------------------------------------------------
// map build, pass 1: transform + key + hash insert + per-voxel count
// ---------------------------------------------------------------------------
namespace {
__device__ __forceinline__ void map_insert_body(const MapArgs &a) {
  __shared__ int s_off[kMaxWindow + 1];
  for (int i = threadIdx.x; i <= a.W; i += blockDim.x) s_off[i] = a.slot_off[i];
  __syncthreads();
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.n_total) return;
  const int slot = find_slot_of(s_off, a.W, g);
  const int k = g - s_off[slot];
  double x, y, z;
  if (a.type == 0) load_xyz(reinterpret_cast<const PlanarRec *>(a.store) + (size_t)slot * a.kcap + k, x, y, z);
  else load_xyz(reinterpret_cast<const PointRec *>(a.store) + (size_t)slot * a.kcap + k, x, y, z);
  const double *T = a.slot_pose + 12 * slot;
  double wx, wy, wz;
  transform_point(T, x, y, z, wx, wy, wz);
  const unsigned long long key = pack_key(voxel_coord(wx, a.voxel_width, a.inv_voxel_width),
                                          voxel_coord(wy, a.voxel_width, a.inv_voxel_width),
                                          voxel_coord(wz, a.voxel_width, a.inv_voxel_width));
  uint32_t h = hash_key(key) & a.hash_mask;
  for (;;) {
    unsigned long long *kp = &a.hash[h].key;
    unsigned long long cur = *kp;
    if (cur == kEmptyKey) {
      cur = atomicCAS(kp, kEmptyKey, key);
      // this thread created the voxel: it also enters it in the list of occupied slots, so that
      // the later passes walk the voxels instead of the (mostly empty) table
      if (cur == kEmptyKey) a.voxel_list[atomicAdd(a.cursor + 1, 1u)] = h;
    }
    if (cur == kEmptyKey || cur == key) break;
    h = (h + 1) & a.hash_mask;
  }
  atomicAdd(&a.hash[h].count, 1u);
  a.world_src[g] = h;
  WorldPoint wp;
  wp.x = wx; wp.y = wy; wp.z = wz;
  wp.tie = ((unsigned long long)a.slot_rank[slot] << 24) | (unsigned long long)k; // rule R4 id
  a.world[g] = wp;
}
} // namespace
__global__ void __launch_bounds__(256) map_insert_kernel(MapArgs pa, MapArgs qa) {
  map_insert_body(blockIdx.y == 0 ? pa : qa);
}
__global__ void __launch_bounds__(256) map_insert_batch_kernel(const MapArgs *items) {
  __shared__ MapArgs s_a;
  load_item_args(s_a, items + 2 * blockIdx.z + blockIdx.y);
  pdl_wait();
  map_insert_body(s_a);
}

// pass 2: give every occupied voxel a contiguous range; start is left pointing
// one past the end and is walked down by the scatter pass
namespace {
__device__ __forceinline__ void map_alloc_body(const MapArgs &a) {
  if (a.n_total <= 0) return;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= __ldcg(a.cursor + 1)) return; // occupied voxels (<= points)
  const uint32_t h = a.voxel_list[i];
  const uint32_t cnt = a.hash[h].count;
  a.hash[h].start = atomicAdd(a.cursor, cnt) + cnt;
  // cell-ordered bucket (map_cells_body): the flag travels in the count's top bit, and the voxel
  // enters the list of cell-ordered voxels, which grows downwards from the end of voxel_list
  // (occupied + cell-ordered voxels <= points, so the two lists cannot meet)
  if (cnt >= kCellMin && cnt <= kCellMax) {
    a.hash[h].count = cnt | kCellFlag;
    a.voxel_list[(uint32_t)a.n_total - 1u - atomicAdd(a.cursor + 2, 1u)] = h;
  }
}
} // namespace
__global__ void __launch_bounds__(256) map_alloc_kernel(MapArgs pa, MapArgs qa) {
  map_alloc_body(blockIdx.y == 0 ? pa : qa);
}
__global__ void __launch_bounds__(256) map_alloc_batch_kernel(const MapArgs *items) {
  __shared__ MapArgs s_a;
  load_item_args(s_a, items + 2 * blockIdx.z + blockIdx.y);
  pdl_wait();
  map_alloc_body(s_a);
}

// pass 3: scatter into voxel-contiguous order (`cell_tab`, `scatter_src`)
namespace {
__device__ __forceinline__ void map_scatter_body(const MapArgs &a) {
  __shared__ int s_off[kMaxWindow + 1];
  for (int i = threadIdx.x; i <= a.W; i += blockDim.x) s_off[i] = a.slot_off[i];
  __syncthreads();
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.n_total) return;
  const uint32_t h = a.world_src[g];
  const uint32_t pos = atomicSub(&a.hash[h].start, 1u) - 1u;
  a.cell_tab[pos] = a.world[g];
  const int slot = find_slot_of(s_off, a.W, g);
  a.scatter_src[pos] = ((uint32_t)slot << 24) | (uint32_t)(g - s_off[slot]);
}
} // namespace
__global__ void __launch_bounds__(256) map_scatter_kernel(MapArgs pa, MapArgs qa) {
  map_scatter_body(blockIdx.y == 0 ? pa : qa);
}
__global__ void __launch_bounds__(256) map_scatter_batch_kernel(const MapArgs *items) {
  __shared__ MapArgs s_a;
  load_item_args(s_a, items + 2 * blockIdx.z + blockIdx.y);
  pdl_wait();
  map_scatter_body(s_a);
}

// pass 4 (cell-ordered buckets): copy every bucket from the scatter pass's output (`cell_tab`,
// `scatter_src`) into the final arrays (`world`, `world_src` - both dead once the scatter pass
// has run), ordering the buckets of kCellMin..kCellMax points by the kCellSub^3 cell code of
// their points, and leave the table of the cells' END offsets (64 x u16 = 128 B) in the first
// four records of `cell_tab` at the bucket's position - the source copy is dead by then, and a
// flagged bucket has at least kCellMin >= 4 records, so every voxel owns its table slot without
// any allocation.  One warp per voxel, any bucket size: histogram over the 64 cells (integer
// shared-memory atomics), exclusive prefix, scatter.  The order inside a cell is arbitrary, like
// the order inside a bucket before - rule R5's key does not depend on it.
namespace {
constexpr int kCellWarps = 8;
struct CellSmem { // one warp's voxel
  uint32_t hist[kCellSub * kCellSub * kCellSub];
  uint32_t cur[kCellSub * kCellSub * kCellSub];
};
static_assert(kCellSub * kCellSub * kCellSub == 64, "the table layout assumes 64 cells (two per lane)");

// cell of a coordinate relative to its voxel's lower corner (clamped: a point a rounding error
// outside its voxel lands in the edge cell, which the query-side margins cover)
__device__ __forceinline__ int cell_index(double rel, double inv_cw) {
  const int i = (int)floor(rel * inv_cw);
  return min(max(i, 0), kCellSub - 1);
}
__device__ __forceinline__ int unpack_coord(unsigned long long key, int shift) {
  const uint32_t v = (uint32_t)(key >> shift) & 0x1FFFFFu;
  return (int)(v << 11) >> 11; // sign-extend 21 bits
}

__device__ __forceinline__ void map_cells_body(const MapArgs &a) {
  __shared__ CellSmem s_cells[kCellWarps];
  if (a.n_total <= 0) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  CellSmem &S = s_cells[warp];
  const double w = a.voxel_width, inv_cw = (double)kCellSub * a.inv_voxel_width;
  // ---- small buckets (< kCellMin points): copied as they are, one THREAD per voxel ----
  const uint32_t n_vox = __ldcg(a.cursor + 1); // occupied voxels, listed by the insert pass
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_vox; i += gridDim.x * blockDim.x) {
    const HashSlot s = a.hash[a.voxel_list[i]];
    if (s.count & kCellFlag) continue;
    for (uint32_t k = 0; k < s.count; ++k) {
      a.world[s.start + k] = a.cell_tab[s.start + k];
      a.world_src[s.start + k] = a.scatter_src[s.start + k];
    }
  }
  // ---- cell-ordered buckets: one WARP per voxel ----
  const uint32_t n_tab = __ldcg(a.cursor + 2); // listed by the alloc pass
  const uint32_t n_warps = gridDim.x * kCellWarps;
  for (uint32_t j = blockIdx.x * kCellWarps + warp; j < n_tab; j += n_warps) {
    const HashSlot s = a.hash[a.voxel_list[(uint32_t)a.n_total - 1u - j]];
    const uint32_t start = s.start, cnt = s.count & ~kCellFlag;
    const double lx = (double)unpack_coord(s.key, 42) * w, ly = (double)unpack_coord(s.key, 21) * w,
                 lz = (double)unpack_coord(s.key, 0) * w;
    auto code_of = [&](const WorldPoint &p) {
      return (cell_index(p.x - lx, inv_cw) * kCellSub + cell_index(p.y - ly, inv_cw)) * kCellSub +
             cell_index(p.z - lz, inv_cw);
    };
    S.hist[lane] = 0u;
    S.hist[lane + 32] = 0u;
    __syncwarp();
    // buckets of up to 64 points (most): a lane keeps its one or two points in registers, so
    // the bucket is read once; larger ones are read twice
    const bool in_regs = cnt <= 64u;
    WorldPoint p0, p1;
    uint32_t src0 = 0u, src1 = 0u;
    int c0 = -1, c1 = -1;
    if (in_regs) {
      if ((uint32_t)lane < cnt) {
        p0 = a.cell_tab[start + lane];
        src0 = a.scatter_src[start + lane];
        c0 = code_of(p0);
        atomicAdd(&S.hist[c0], 1u);
      }
      if ((uint32_t)lane + 32u < cnt) {
        p1 = a.cell_tab[start + lane + 32];
        src1 = a.scatter_src[start + lane + 32];
        c1 = code_of(p1);
        atomicAdd(&S.hist[c1], 1u);
      }
    } else {
      for (uint32_t i = lane; i < cnt; i += 32) atomicAdd(&S.hist[code_of(a.cell_tab[start + i])], 1u);
    }
    __syncwarp();
    // exclusive prefix over the 64 bins, two per lane
    const uint32_t h0 = S.hist[2 * lane], h1 = S.hist[2 * lane + 1];
    uint32_t incl = h0 + h1;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const uint32_t excl = incl - (h0 + h1);
    S.cur[2 * lane] = excl;
    S.cur[2 * lane + 1] = excl + h0;
    __syncwarp();
    if (in_regs) {
      if (c0 >= 0) {
        const uint32_t pos = atomicAdd(&S.cur[c0], 1u);
        a.world[start + pos] = p0;
        a.world_src[start + pos] = src0;
      }
      if (c1 >= 0) {
        const uint32_t pos = atomicAdd(&S.cur[c1], 1u);
        a.world[start + pos] = p1;
        a.world_src[start + pos] = src1;
      }
    } else {
      for (uint32_t i = lane; i < cnt; i += 32) {
        const WorldPoint p = a.cell_tab[start + i];
        const uint32_t pos = atomicAdd(&S.cur[code_of(p)], 1u);
        a.world[start + pos] = p;
        a.world_src[start + pos] = a.scatter_src[start + i];
      }
    }
    __syncwarp(); // every read of the source bucket is done: its head becomes the table
    // END offsets of cells 2 lane and 2 lane + 1 as one 32-bit word
    reinterpret_cast<uint32_t *>(a.cell_tab + start)[lane] = (excl + h0) | ((excl + h0 + h1) << 16);
    __syncwarp();
  }
}
} // namespace
__global__ void __launch_bounds__(kCellWarps * 32) map_cells_kernel(MapArgs pa, MapArgs qa) {
  map_cells_body(blockIdx.y == 0 ? pa : qa);
}
__global__ void __launch_bounds__(kCellWarps * 32) map_cells_batch_kernel(const MapArgs *items) {
  __shared__ MapArgs s_a;
  load_item_args(s_a, items + 2 * blockIdx.z + blockIdx.y);
  pdl_wait();
  map_cells_body(s_a);
}

// clears the hash tables (and allocation cursors) of every item of a batched rebuild:
// regions[i] = {base, bytes}, bytes a multiple of 16
__global__ void __launch_bounds__(256) map_clear_batch_kernel(const MapClearRegion *regions, const unsigned char *ring) {
  const MapClearRegion r = regions[blockIdx.y];
  uint4 *p = reinterpret_cast<uint4 *>(r.base);
  const size_t n = r.bytes / sizeof(uint4);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    p[i] = make_uint4(0u, 0u, 0u, 0u);
  if (r.copy_bytes) { // the context's rebuild request, staged with the submission's arguments
    const unsigned long long *src = reinterpret_cast<const unsigned long long *>(ring + r.copy_src_off);
    unsigned long long *dst = reinterpret_cast<unsigned long long *>(r.copy_dst);
    const size_t m = r.copy_bytes / sizeof(unsigned long long);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (size_t)gridDim.x * blockDim.x)
      dst[i] = src[i];
  }
}

void map_build_launch(const MapArgs &pa, const MapArgs &qa, cudaStream_t stream, Profiler &prof) {
  const int n = max(pa.n_total, qa.n_total);
  if (n <= 0) return;
  prof.begin(FORMGPU_KG_MAP_BUILD);
  const dim3 gp((n + 255) / 256, 2);
  map_insert_kernel<<<gp, 256, 0, stream>>>(pa, qa);
  const int nt = max(pa.n_total, qa.n_total); // voxels <= points
  map_alloc_kernel<<<dim3((nt + 255) / 256, 2), 256, 0, stream>>>(pa, qa);
  map_scatter_kernel<<<gp, 256, 0, stream>>>(pa, qa);
  // grid-stride: a thread per small voxel, a warp per cell-ordered voxel (<= points / 16)
  const unsigned blocks = std::max(1u, std::min<unsigned>((unsigned)nt / (16u * kCellWarps) + 1u, 8 * 148));
  map_cells_kernel<<<dim3(blocks, 2), kCellWarps * 32, 0, stream>>>(pa, qa);
  prof.end(FORMGPU_KG_MAP_BUILD, 4);
}

void map_build_batch_launch(const MapArgs *items_dev, const MapClearRegion *regions_dev, const unsigned char *ring_dev,
                            int n_items, int max_points, uint32_t max_hash, size_t max_clear_bytes,
                            cudaStream_t stream, Profiler &prof) {
  if (n_items <= 0) return;
  prof.begin(FORMGPU_KG_MAP_BUILD);
  const unsigned clear_blocks = (unsigned)std::min<size_t>((max_clear_bytes / 16 + 255) / 256, 592);
  map_clear_batch_kernel<<<dim3(std::max(clear_blocks, 1u), n_items), 256, 0, stream>>>(regions_dev, ring_dev);
  int launches = 1;
  if (max_points > 0) {
    const dim3 gp((max_points + 255) / 256, 2, n_items);
    launch_pdl(map_insert_batch_kernel, gp, 256, 0, stream, items_dev);
    launch_pdl(map_alloc_batch_kernel, dim3((max_points + 255) / 256, 2, n_items), 256, 0, stream, items_dev);
    launch_pdl(map_scatter_batch_kernel, gp, 256, 0, stream, items_dev);
    const unsigned blocks = std::max(1u, std::min<unsigned>((unsigned)max_points / (16u * kCellWarps) + 1u, 512u));
    launch_pdl(map_cells_batch_kernel, dim3(blocks, 2, n_items), kCellWarps * 32, 0, stream, items_dev);
    launches += 4;
  }
  prof.end(FORMGPU_KG_MAP_BUILD, launches);
}

// ---------------------------------------------------------------------------
// nearest neighbour: one warp per query keypoint
// ---------------------------------------------------------------------------
// bin of a query: matched slot if dist^2 < max_dist^2 (matcher.hpp:104), else none.
// Bin W counts the keypoints that insert_matches would add (map.tpp:161).
__device__ __forceinline__ int match_bin(const MatchRec &m, double max_d2) {
  return (m.slot != kNoSlot && m.dist_sqrd < max_d2) ? (int)m.slot : -1;
}

// Read-only loads of the map go through the non-coherent path (the argument block lives in
// shared memory in the batched kernel, which hides from the compiler that these are global).
__device__ __forceinline__ HashSlot load_slot(const HashSlot *p) {
  const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
  HashSlot s;
  s.key = ((unsigned long long)v.y << 32) | v.x;
  s.start = v.z;
  s.count = v.w;
  return s;
}
// One 256-bit load per 32-byte map point (sm_100: LDG.E.256; the arrays come from cudaMalloc and the
// records are 32 bytes, so every point is 32-byte aligned): half the load instructions and half the
// L1 tag look-ups of the two 128-bit loads this replaces - every lane of a scan touches its own sector.
__device__ __forceinline__ WorldPoint load_world(const WorldPoint *p) {
  unsigned long long a, b, c, d;
  asm("ld.global.nc.v4.b64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
  WorldPoint w;
  w.x = __longlong_as_double((long long)a);
  w.y = __longlong_as_double((long long)b);
  w.z = __longlong_as_double((long long)c);
  w.tie = d;
  return w;
}
// bucket of the voxel `key`: linear probing (load <= 0.5); absent -> count stays 0
__device__ __forceinline__ void probe_voxel(const HashSlot *hash, uint32_t mask, unsigned long long key,
                                            uint32_t &start, uint32_t &count) {
  uint32_t h = hash_key(key) & mask;
  HashSlot s = load_slot(hash + h);
  while (s.key != key && s.key != kEmptyKey) {
    h = (h + 1) & mask;
    s = load_slot(hash + h);
  }
  if (s.key == key) {
    start = s.start;
    count = s.count;
  }
}

// One WARP per query: a single sequence's call (20 k queries) cannot fill the GPU either way and
// is latency-bound, so the 32 lanes of a warp share a query (shortest bucket scans).
//
// Order of the search: (1) the warp probes the CENTRE voxel and scans its bucket together;
// (2) lane v bounds the squared distance from the query to the box of the neighbour voxel with
// shift rank v (1..26; pure arithmetic on the distances to the six faces of the centre voxel) and
// keeps it if it can still hold a point at least as close as the centre's best - exact pruning:
// a skipped voxel cannot change the arg-min; (3) the surviving voxel ranks (typically one to four
// of 26) are compacted through shared memory so that lane s probes the s-th survivor; (4) the
// warp scans the survivors' buckets one after the other.  The arg-min key (dist^2, shift rank,
// scan, k) is rule R5, so neither the scan order nor the split over lanes matters.
constexpr int kNnWarps = 8; // queries per CTA (256 threads)

namespace {
__device__ __forceinline__ void assoc_nn_body(const AssocArgs &a) {
  constexpr int kDepth = 2;                  // bucket points a lane keeps in flight
  __shared__ unsigned char s_list[kNnWarps][28]; // compacted surviving voxel ranks
  __shared__ uint2 s_bucket[kNnWarps][27];       // their buckets {start, count}
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int q = blockIdx.x * (blockDim.x >> 5) + warp;
  const int nb = a.W + 1;
  const bool active = q >= a.q_begin && q < a.q_end; // the whole warp is active or not; shuffles need every lane
  const bool searchable = active && a.n_map > 0;
  double x = 0.0, y = 0.0, z = 0.0;
  if (active) {
    if (a.type == 0) load_xyz(reinterpret_cast<const PlanarRec *>(a.queries) + q, x, y, z);
    else load_xyz(reinterpret_cast<const PointRec *>(a.queries) + q, x, y, z);
  }
  double wx, wy, wz;
  transform_point(a.pose, x, y, z, wx, wy, wz); // kp->transform(init), matcher.hpp:89
  const double w = a.voxel_width, iw = a.inv_voxel_width;
  const int cx = voxel_coord(wx, w, iw), cy = voxel_coord(wy, w, iw), cz = voxel_coord(wz, w, iw);

  double best = DBL_MAX;                     // Match::dist_sqrd default (map.hpp:55)
  unsigned long long best_tie = ~0ull;
  int best_rank = 32;
  uint32_t best_pos = kNoSlot;
  auto consider = [&](const WorldPoint &p, uint32_t pos, int b) {
    // 4-lane double squared norm, lane 3 = 0 padding: (d0^2 + d2^2) + (d1^2 + 0)
    const double d0 = p.x - wx, d1 = p.y - wy, d2 = p.z - wz;
    const double dist = (d0 * d0 + d2 * d2) + (d1 * d1 + 0.0);
    // rule R5 key (dist, shift rank, tie)
    if (dist < best || (dist == best && (b < best_rank || (b == best_rank && p.tie < best_tie)))) {
      best = dist;
      best_tie = p.tie;
      best_rank = b;
      best_pos = pos;
    }
  };
  // the warp scans a bucket together, 32 consecutive 32-byte points per step; a lane requests its
  // next kDepth points before it looks at the first
  auto scan_bucket = [&](int b, uint32_t sb, uint32_t cb) {
    uint32_t i = lane;
    for (; i + (kDepth - 1) * 32 < cb; i += kDepth * 32) {
      WorldPoint p[kDepth];
#pragma unroll
      for (int u = 0; u < kDepth; ++u) p[u] = load_world(a.world + sb + i + u * 32);
#pragma unroll
      for (int u = 0; u < kDepth; ++u) consider(p[u], sb + i + u * 32, b);
    }
    for (; i < cb; i += 32) consider(load_world(a.world + sb + i), sb + i, b);
  };

  // (1) centre voxel: every lane probes the same slot (one broadcast load)
  {
    uint32_t s0 = 0u, c0 = 0u;
    if (searchable) probe_voxel(a.hash, a.hash_mask, pack_key(cx, cy, cz), s0, c0);
    c0 &= ~kCellFlag;
    scan_bucket(0, s0, c0);
  }
  double bound = best;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) bound = fmin(bound, __shfl_xor_sync(0xffffffffu, bound, off));

  // (2) squared distance from the query to the box of this lane's voxel, shrunk by a safety
  // margin that covers the rounding of floor(x / w) at the voxel faces.  All shifts are -1 / 0 /
  // +1 per axis, so the per-axis terms are the distances to the two faces of the centre voxel -
  // computed once per query, then three selects.
  double face2[3][2]; // [axis][0: towards -1, 1: towards +1], squared, margin applied
  {
    const double qq[3] = {wx, wy, wz};
    const int cc[3] = {cx, cy, cz};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double lo = (double)cc[k] * w, hi = lo + w;
      const double margin = 1e-9 * (1.0 + fabs(qq[k])) + 4e-16 * fabs(lo);
      const double dm = fmax(qq[k] - lo - margin, 0.0); // to the lower face (voxels with shift -1)
      const double dp = fmax(hi - qq[k] - margin, 0.0); // to the upper face (voxels with shift +1)
      face2[k][0] = dm * dm;
      face2[k][1] = dp * dp;
    }
  }
  bool keep = false;
  if (searchable && lane > 0 && lane < 27) {
    double lb = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int sh = lane_shift(lane, k);
      lb += sh == 0 ? 0.0 : sh < 0 ? face2[k][0] : face2[k][1];
    }
    keep = lb <= bound;
  }
  const unsigned survivors = __ballot_sync(0xffffffffu, keep); // bit v: voxel v must be searched

  // (3) compaction: the i-th surviving rank is probed by lane i, which leaves the bucket's
  // {start, count} in shared memory for the whole warp
  const int n_surv = __popc(survivors);
  if (keep) s_list[warp][__popc(survivors & ((1u << lane) - 1u))] = (unsigned char)lane;
  __syncwarp();
  if (lane < n_surv) {
    const int v = s_list[warp][lane];
    uint32_t st = 0u, ct = 0u;
    probe_voxel(a.hash, a.hash_mask,
                pack_key(cx + lane_shift(v, 0), cy + lane_shift(v, 1), cz + lane_shift(v, 2)), st, ct);
    s_bucket[warp][lane] = make_uint2(st, ct & ~kCellFlag);
  }
  __syncwarp();

  // (4) the survivors' non-empty buckets, one after the other
  for (int i = 0; i < n_surv; ++i) {
    const uint2 bk = s_bucket[warp][i];
    if (bk.y) scan_bucket(s_list[warp][i], bk.x, bk.y);
  }
  // arg-min over the lanes with the same key
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, best, off);
    const unsigned long long ot = __shfl_xor_sync(0xffffffffu, best_tie, off);
    const uint32_t op = __shfl_xor_sync(0xffffffffu, best_pos, off);
    const int orank = __shfl_xor_sync(0xffffffffu, best_rank, off);
    const bool take = (op != kNoSlot) &&
                      (best_pos == kNoSlot || od < best ||
                       (od == best && (orank < best_rank || (orank == best_rank && ot < best_tie))));
    if (take) {
      best = od;
      best_tie = ot;
      best_pos = op;
      best_rank = orank;
    }
  }
  if (active && lane == 0) {
    MatchRec m;
    if (best_pos == kNoSlot) {
      m.dist_sqrd = DBL_MAX;
      m.slot = kNoSlot;
      m.k = 0u;
    } else {
      const uint32_t src = a.world_src[best_pos];
      m.dist_sqrd = best;
      m.slot = src >> 24;
      if (a.pack_rank) m.slot |= (uint32_t)best_rank << 8;
      m.k = src & 0xFFFFFFu;
    }
    a.match[q] = m;
    // per-256-query histogram of the accepted matches by matched scan (+ novel count)
    if (a.hist_cnt) {
      const int bin = match_bin(m, a.max_dist2);
      if (bin >= 0) atomicAdd(&a.hist_cnt[(size_t)(q >> 8) * nb + bin], 1u);
      if (m.dist_sqrd > a.min_dist2) atomicAdd(&a.hist_cnt[(size_t)(q >> 8) * nb + a.W], 1u);
    }
  }
}
} // namespace
// ---------------------------------------------------------------------------
// association over cell-ordered buckets: one THREAD per query
// ---------------------------------------------------------------------------
// With the buckets ordered by 4x4x4 sub-cells (map_cells_body) a query whose nearest neighbour
// is a few centimetres away - the usual case: the map holds the same surfaces seen from the
// previous poses - has to look at the ~10 points of its own 20 cm cell and of the one to three
// adjacent cells that lie within its best distance, instead of the 100+ points of the whole
// 0.8 m voxel.  That is too little work to share between lanes (the cooperative kernel above
// spends its instructions on ballots, compaction and shuffles), so here a thread owns a query and
// runs the whole search by itself; a warp holds 32 consecutive keypoints, which are neighbours in
// space and mostly take the same path.
//   1. centre voxel probe; if its bucket is cell-ordered: scan the query's own cell, then the
//      adjacent cells whose box can hold a point at least as close as the best so far (per axis
//      only the directions whose cell face is that close are enumerated);
//   2. complete if the best is closer than one cell width (every cell that was not visited is at
//      least that far away) - otherwise, and for small or absent centre buckets, the exact
//      whole-voxel search: centre bucket + the neighbour voxels that survive the face bound.
// Same candidates' arg-min key (dist^2, shift rank, scan, k) = rule R5, so results are those of
// the cooperative kernel and of the reference, bit for bit.
namespace {
// per-256-query histogram of the accepted matches by matched scan (+ novel count), warp-aggregated;
// a warp covers 32 consecutive queries of one 256-query block.  Called by all 32 lanes.
__device__ __forceinline__ void hist_add(const AssocArgs &a, int q, int lane, bool counted, const MatchRec &m) {
  const int nb = a.W + 1;
  const int bin = counted ? match_bin(m, a.max_dist2) : -1;
  const bool novel = counted && m.dist_sqrd > a.min_dist2;
  const unsigned peers = __match_any_sync(0xffffffffu, bin);
  if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&a.hist_cnt[(size_t)(q >> 8) * nb + bin], (unsigned)__popc(peers));
  const unsigned nov = __ballot_sync(0xffffffffu, novel);
  if (nov && lane == __ffs(nov) - 1) atomicAdd(&a.hist_cnt[(size_t)(q >> 8) * nb + a.W], (unsigned)__popc(nov));
}
struct NnBest {
  double d = DBL_MAX; // Match::dist_sqrd default (map.hpp:55)
  unsigned long long tie = ~0ull;
  int rank = 32;
  uint32_t pos = kNoSlot;
};
__device__ __forceinline__ void nn_consider(NnBest &b, const WorldPoint &p, uint32_t pos, int rank, double wx,
                                            double wy, double wz) {
  // 4-lane double squared norm, lane 3 = 0 padding: (d0^2 + d2^2) + (d1^2 + 0)
  const double d0 = p.x - wx, d1 = p.y - wy, d2 = p.z - wz;
  const double dist = (d0 * d0 + d2 * d2) + (d1 * d1 + 0.0);
  // one comparison rejects nearly every candidate; the rule-R5 tie-break is off the hot path
  if (dist <= b.d) {
    if (dist < b.d || rank < b.rank || (rank == b.rank && p.tie < b.tie)) {
      b.d = dist;
      b.tie = p.tie;
      b.rank = rank;
      b.pos = pos;
    }
  }
}
__device__ __forceinline__ void nn_scan(NnBest &b, const WorldPoint *world, uint32_t lo, uint32_t n, int rank,
                                        double wx, double wy, double wz) {
  uint32_t i = 0;
  for (; i + 1 < n; i += 2) { // two points in flight
    const WorldPoint p0 = load_world(world + lo + i), p1 = load_world(world + lo + i + 1);
    nn_consider(b, p0, lo + i, rank, wx, wy, wz);
    nn_consider(b, p1, lo + i + 1, rank, wx, wy, wz);
  }
  if (i < n) nn_consider(b, load_world(world + lo + i), lo + i, rank, wx, wy, wz);
}
// point range of cell (ci) of a bucket: the whole bucket when it carries no table
__device__ __forceinline__ void cell_range(const AssocArgs &a, uint32_t start, uint32_t count_raw, int cix,
                                           int ciy, int ciz, uint32_t &lo, uint32_t &n) {
  if (count_raw & kCellFlag) {
    const int code = (cix * kCellSub + ciy) * kCellSub + ciz;
    const unsigned short *tab = reinterpret_cast<const unsigned short *>(a.cell_tab + start);
    const uint32_t b = code ? __ldg(tab + code - 1) : 0u, e = __ldg(tab + code);
    lo = start + b;
    n = e - b;
  } else {
    lo = start;
    n = count_raw;
  }
}

// bit v of kShiftMask[axis][0 / 1]: shift rank v moves by -1 / +1 along the axis
constexpr unsigned shift_mask(int axis, int dir) {
  constexpr int T[27][3] = {
      {0, 0, 0},   {1, 0, 0},   {-1, 0, 0},  {0, 1, 0},   {0, -1, 0},  {0, 0, 1},   {0, 0, -1},
      {1, 1, 0},   {1, -1, 0},  {-1, 1, 0},  {-1, -1, 0}, {1, 0, 1},   {1, 0, -1},  {-1, 0, 1},
      {-1, 0, -1}, {0, 1, 1},   {0, 1, -1},  {0, -1, 1},  {0, -1, -1}, {1, 1, 1},   {1, 1, -1},
      {1, -1, 1},  {1, -1, -1}, {-1, 1, 1},  {-1, 1, -1}, {-1, -1, 1}, {-1, -1, -1}};
  unsigned m = 0;
  for (int v = 1; v < 27; ++v)
    if (T[v][axis] == dir) m |= 1u << v;
  return m;
}
constexpr unsigned kShiftNeg[3] = {shift_mask(0, -1), shift_mask(1, -1), shift_mask(2, -1)};
constexpr unsigned kShiftPos[3] = {shift_mask(0, 1), shift_mask(1, 1), shift_mask(2, 1)};
__device__ __forceinline__ void assoc_cells_body(const AssocArgs &a) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool active = q >= a.q_begin && q < a.q_end;
  const bool searchable = active && a.n_map > 0;
  const double w = a.voxel_width, iw = a.inv_voxel_width;
  const double cw = w * (1.0 / kCellSub), inv_cw = (double)kCellSub * iw;
  NnBest best;
  double wx = 0.0, wy = 0.0, wz = 0.0;
  int c[3] = {0, 0, 0};
  uint32_t s0 = 0u, c0raw = 0u;
  if (searchable) {
    double x, y, z;
    if (a.type == 0) load_xyz(reinterpret_cast<const PlanarRec *>(a.queries) + q, x, y, z);
    else load_xyz(reinterpret_cast<const PointRec *>(a.queries) + q, x, y, z);
    transform_point(a.pose, x, y, z, wx, wy, wz); // kp->transform(init), matcher.hpp:89
    c[0] = voxel_coord(wx, w, iw);
    c[1] = voxel_coord(wy, w, iw);
    c[2] = voxel_coord(wz, w, iw);
    probe_voxel(a.hash, a.hash_mask, pack_key(c[0], c[1], c[2]), s0, c0raw);
  }
  // ---- phase 1: the query's own search unit - its CELL when the centre bucket is cell-ordered,
  // the whole centre VOXEL otherwise (small or absent bucket) ----
  const bool by_cell = (c0raw & kCellFlag) != 0u;
  const double qq[3] = {wx, wy, wz};
  int f0[3] = {0, 0, 0};
#pragma unroll
  for (int k = 0; k < 3; ++k)
    if (by_cell) f0[k] = cell_index(qq[k] - (double)c[k] * w, inv_cw);
  // squared distance from the query to the lower / upper face of its unit along axis k, shrunk by a
  // margin that covers the rounding of floor(x / w) at the voxel (and cell) faces.  Recomputed
  // where needed instead of kept: the far faces are only looked at by the rare far-side pass.
  auto faces = [&](const int k, double &lo2, double &hi2) -> double {
    const double vlo = (double)c[k] * w;
    const double margin = 1e-9 * (1.0 + fabs(qq[k])) + 4e-16 * fabs(vlo);
    const double ulo = by_cell ? vlo + (double)f0[k] * cw : vlo, uw = by_cell ? cw : w;
    const double dm = fmax(qq[k] - ulo - margin, 0.0), dp = fmax(ulo + uw - qq[k] - margin, 0.0);
    lo2 = dm * dm;
    hi2 = dp * dp;
    return margin;
  };
  {
    uint32_t lo = s0, n = c0raw & ~kCellFlag;
    if (by_cell) cell_range(a, s0, c0raw, f0[0], f0[1], f0[2], lo, n);
    nn_scan(best, a.world, lo, n, 0, wx, wy, wz);
  }
  // ---- phase 2: the adjacent units (cells, or voxels) that can hold a point at least as close
  // as the best so far.  (a) The seven units of the NEAR octant - per axis the unit behind the
  // closer face - in ascending order of their lower bound (sort of three face distances: a <= b
  // <= c gives a, b, {c, a+b}, a+c, b+c, a+b+c), leaving at the first bound above the best: a
  // query whose own unit is empty gets a finite best from its nearest neighbours first instead of
  // walking all 26 shifts against an infinite one, and a typical query stops after one or two
  // units.  (b) The 19 units with a component beyond a FAR face: six comparisons against the best
  // select the candidate shifts (usually none), the summed bound is tested when a shift is popped.
  // All pruning is against the best SO FAR with the margin-shrunk bounds: exact.
  auto visit = [&](const int sh0, const int sh1, const int sh2, const double lb) {
    const int sh[3] = {sh0, sh1, sh2};
    uint32_t lo = 0u, n = 0u;
    int rank = 0;
    if (lb <= best.d) {
      if (by_cell) {
        // the cell f0 + sh lies in the centre voxel or in the neighbour voxel `carry`
        int carry[3], ci[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int f = f0[k] + sh[k];
          carry[k] = f < 0 ? -1 : f >= kCellSub ? 1 : 0;
          ci[k] = f - kCellSub * carry[k];
        }
        rank = shift_rank(carry[0], carry[1], carry[2]);
        uint32_t st = s0, ctraw = c0raw;
        if (rank != 0) {
          st = 0u;
          ctraw = 0u;
          probe_voxel(a.hash, a.hash_mask, pack_key(c[0] + carry[0], c[1] + carry[1], c[2] + carry[2]), st, ctraw);
        }
        if (ctraw) cell_range(a, st, ctraw, ci[0], ci[1], ci[2], lo, n);
      } else {
        rank = shift_rank(sh0, sh1, sh2);
        uint32_t ct = 0u;
        probe_voxel(a.hash, a.hash_mask, pack_key(c[0] + sh0, c[1] + sh1, c[2] + sh2), lo, ct);
        n = ct & ~kCellFlag;
      }
    }
    nn_scan(best, a.world, lo, n, rank, wx, wy, wz);
  };
  bool unresolved = false;
  double margin_max = 0.0;
  if (searchable) {
    // near face per axis, then the three (bound, axis bit) pairs in ascending order
    double fa, fb, fc;
    unsigned nneg_bits = 0u; // bit k: the lower face of axis k is the near one
    {
      double lo2, hi2;
      margin_max = faces(0, lo2, hi2);
      if (lo2 <= hi2) nneg_bits |= 1u;
      fa = fmin(lo2, hi2);
      margin_max = fmax(margin_max, faces(1, lo2, hi2));
      if (lo2 <= hi2) nneg_bits |= 2u;
      fb = fmin(lo2, hi2);
      margin_max = fmax(margin_max, faces(2, lo2, hi2));
      if (lo2 <= hi2) nneg_bits |= 4u;
      fc = fmin(lo2, hi2);
    }
    unsigned ma = 1u, mb = 2u, mc = 4u;
    auto order2 = [](double &x, unsigned &mx, double &y, unsigned &my) {
      if (y < x) {
        const double t = x; x = y; y = t;
        const unsigned u = mx; mx = my; my = u;
      }
    };
    order2(fa, ma, fb, mb);
    order2(fb, mb, fc, mc);
    order2(fa, ma, fb, mb);
    // subsets of the sorted axes (bit 0 = a, 1 = b, 2 = c), three bits per step, first step lowest
    const unsigned seq = (fc <= fa + fb) ? 07653421u : 07654321u;
#pragma unroll 1
    for (int i = 0; i < 7; ++i) {
      const unsigned t = (seq >> (3 * i)) & 7u;
      const double lb = (((t & 1u) ? fa : 0.0) + ((t & 2u) ? fb : 0.0)) + ((t & 4u) ? fc : 0.0);
      if (!(lb <= best.d)) break; // ascending bounds: nothing later can qualify either
      const unsigned m = ((t & 1u) ? ma : 0u) | ((t & 2u) ? mb : 0u) | ((t & 4u) ? mc : 0u);
      visit((m & 1u) ? ((nneg_bits & 1u) ? -1 : 1) : 0, (m & 2u) ? ((nneg_bits & 2u) ? -1 : 1) : 0,
            (m & 4u) ? ((nneg_bits & 4u) ? -1 : 1) : 0, lb);
    }
    // shifts with a component beyond a far face, face-tested against the best so far
    constexpr unsigned neg[3] = {kShiftNeg[0], kShiftNeg[1], kShiftNeg[2]};
    constexpr unsigned pos[3] = {kShiftPos[0], kShiftPos[1], kShiftPos[2]};
    unsigned surv = 0u;
    double face2[3][2];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      faces(k, face2[k][0], face2[k][1]);
      surv |= ((nneg_bits >> k) & 1u) ? pos[k] : neg[k];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (!(face2[k][0] <= best.d)) surv &= ~neg[k];
      if (!(face2[k][1] <= best.d)) surv &= ~pos[k];
    }
    while (surv) {
      const int v = __ffs(surv) - 1;
      surv &= surv - 1u;
      const int sh[3] = {lane_shift(v, 0), lane_shift(v, 1), lane_shift(v, 2)};
      double lb = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) lb += sh[k] == 0 ? 0.0 : sh[k] < 0 ? face2[k][0] : face2[k][1];
      visit(sh[0], sh[1], sh[2], lb);
    }
  }
  if (by_cell && !unresolved) {
    // every cell that was not visited is at least one cell width away (along some axis) or was
    // pruned against a bound >= the final best: complete once the best is closer than that.
    // (A search by voxels is the reference's own 27-voxel search: complete by construction.)
    const double reach = cw - margin_max;
    unresolved = !(best.d < reach * reach);
  }
  // ---- phase 3: the exact whole-voxel search (the reference's 27 buckets, face-distance pruned)
  // for the few queries of this warp that are still unresolved, one after the other, ALL 32 LANES
  // on each: the lanes scan the centre bucket together, lane v bounds and probes neighbour voxel
  // v, the surviving buckets are scanned together, and a shuffle arg-min returns the result to
  // the owner.
  unsigned todo = __ballot_sync(0xffffffffu, unresolved);
  while (todo) {
    const int owner = __ffs(todo) - 1;
    todo &= todo - 1u;
    const double ox = __shfl_sync(0xffffffffu, wx, owner), oy = __shfl_sync(0xffffffffu, wy, owner),
                 oz = __shfl_sync(0xffffffffu, wz, owner);
    const int oc[3] = {__shfl_sync(0xffffffffu, c[0], owner), __shfl_sync(0xffffffffu, c[1], owner),
                       __shfl_sync(0xffffffffu, c[2], owner)};
    const uint32_t os0 = __shfl_sync(0xffffffffu, s0, owner);
    const uint32_t oc0 = __shfl_sync(0xffffffffu, c0raw, owner) & ~kCellFlag;
    NnBest mine; // this lane's share of the owner's candidates, seeded with the owner's best:
    mine.d = __shfl_sync(0xffffffffu, best.d, owner);       // it prunes, and ties resolve as if
    mine.tie = __shfl_sync(0xffffffffu, best.tie, owner);   // the point had been found here
    mine.rank = __shfl_sync(0xffffffffu, best.rank, owner);
    mine.pos = __shfl_sync(0xffffffffu, best.pos, owner);
    for (uint32_t i = lane; i < oc0; i += 32u) nn_consider(mine, load_world(a.world + os0 + i), os0 + i, 0, ox, oy, oz);
    double bound = mine.d;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) bound = fmin(bound, __shfl_xor_sync(0xffffffffu, bound, off));
    // lane v (1..26): neighbour voxel v of the owner
    uint32_t vst = 0u, vct = 0u;
    if (lane >= 1 && lane < 27) {
      const int sh[3] = {lane_shift(lane, 0), lane_shift(lane, 1), lane_shift(lane, 2)};
      const double oq[3] = {ox, oy, oz};
      double lb = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double vlo = (double)oc[k] * w;
        const double margin = 1e-9 * (1.0 + fabs(oq[k])) + 4e-16 * fabs(vlo);
        const double dm = fmax(oq[k] - vlo - margin, 0.0), dp = fmax(vlo + w - oq[k] - margin, 0.0);
        lb += sh[k] == 0 ? 0.0 : sh[k] < 0 ? dm * dm : dp * dp;
      }
      if (lb <= bound) {
        probe_voxel(a.hash, a.hash_mask, pack_key(oc[0] + sh[0], oc[1] + sh[1], oc[2] + sh[2]), vst, vct);
        vct &= ~kCellFlag;
      }
    }
    unsigned vox = __ballot_sync(0xffffffffu, vct != 0u);
    while (vox) {
      const int v = __ffs(vox) - 1;
      vox &= vox - 1u;
      const uint32_t st = __shfl_sync(0xffffffffu, vst, v), ct = __shfl_sync(0xffffffffu, vct, v);
      for (uint32_t i = lane; i < ct; i += 32u) nn_consider(mine, load_world(a.world + st + i), st + i, v, ox, oy, oz);
    }
    // arg-min over the lanes with the rule-R5 key
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, mine.d, off);
      const unsigned long long ot = __shfl_xor_sync(0xffffffffu, mine.tie, off);
      const uint32_t op = __shfl_xor_sync(0xffffffffu, mine.pos, off);
      const int orank = __shfl_xor_sync(0xffffffffu, mine.rank, off);
      const bool take = (op != kNoSlot) &&
                        (mine.pos == kNoSlot || od < mine.d ||
                         (od == mine.d && (orank < mine.rank || (orank == mine.rank && ot < mine.tie))));
      if (take) {
        mine.d = od;
        mine.tie = ot;
        mine.pos = op;
        mine.rank = orank;
      }
    }
    if (lane == owner) best = mine;
  }
  // ---- match record + per-256-query histogram by matched scan (warp-aggregated atomics) ----
  const bool mine = active;
  MatchRec m;
  m.dist_sqrd = DBL_MAX;
  m.slot = kNoSlot;
  m.k = 0u;
  if (mine && best.pos != kNoSlot) {
    const uint32_t src = a.world_src[best.pos];
    m.dist_sqrd = best.d;
    m.slot = src >> 24;
    if (a.pack_rank) m.slot |= (uint32_t)best.rank << 8;
    m.k = src & 0xFFFFFFu;
  }
  if (mine) a.match[q] = m;
  if (a.hist_cnt) hist_add(a, q, lane, mine, m);
}
} // namespace
// point-sharded mode: every rank searched ITS sub-map (the scans it owns) for every query; the
// all-gathered candidates are reduced here with the full rule-R5 key (dist^2, shift rank, scan,
// k) - the key the single-GPU search applies inside one map - so the winner is bit-identical
__global__ void __launch_bounds__(256) assoc_combine_kernel(CombineArgs pc, CombineArgs qc) {
  const CombineArgs &c = blockIdx.y == 0 ? pc : qc;
  const AssocArgs &a = c.a;
  if ((int)(blockIdx.x * blockDim.x) >= a.n_query) return;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = q < a.n_query;
  MatchRec best;
  best.dist_sqrd = DBL_MAX;
  best.slot = kNoSlot;
  best.k = 0u;
  int best_rank = 32;
  unsigned long long best_scan = ~0ull;
  if (active) {
    for (int r = 0; r < c.world; ++r) {
      const MatchRec m = c.gathered[(size_t)r * c.stride + q];
      if (m.slot == kNoSlot) continue;
      const uint32_t slot = m.slot & 0xffu;
      const int rank = (int)((m.slot >> 8) & 31u);
      const unsigned long long scan = c.slot_scan[slot];
      const bool take = m.dist_sqrd < best.dist_sqrd ||
                        (m.dist_sqrd == best.dist_sqrd &&
                         (rank < best_rank || (rank == best_rank && (scan < best_scan || (scan == best_scan && m.k < best.k)))));
      if (take) {
        best.dist_sqrd = m.dist_sqrd;
        best.slot = slot;
        best.k = m.k;
        best_rank = rank;
        best_scan = scan;
      }
    }
    a.match[q] = best;
  }
  hist_add(a, q, threadIdx.x & 31, active, best);
}
void assoc_combine_launch(const CombineArgs &pc, const CombineArgs &qc, cudaStream_t stream, Profiler &prof) {
  const int n = max(pc.a.n_query, qc.a.n_query);
  if (n <= 0) return;
  prof.begin(FORMGPU_KG_ASSOC_NN);
  assoc_combine_kernel<<<dim3((n + 255) / 256, 2), 256, 0, stream>>>(pc, qc);
  prof.end(FORMGPU_KG_ASSOC_NN, 1);
}

constexpr int kCellQueryThreads = 128;
__global__ void __launch_bounds__(kCellQueryThreads) assoc_cells_kernel(AssocArgs pa, AssocArgs qa) {
  assoc_cells_body(blockIdx.y == 0 ? pa : qa);
}
__global__ void __launch_bounds__(kCellQueryThreads) assoc_cells_batch_kernel(const AssocArgs *items) {
  __shared__ AssocArgs s_a;
  load_item_args(s_a, items + 2 * blockIdx.z + blockIdx.y);
  pdl_wait();
  if ((int)(blockIdx.x * kCellQueryThreads) >= s_a.n_query) return;
  assoc_cells_body(s_a);
}

__global__ void __launch_bounds__(kNnWarps * 32) assoc_nn_kernel(AssocArgs pa, AssocArgs qa) {
  assoc_nn_body(blockIdx.y == 0 ? pa : qa);
}

void assoc_launch(const AssocArgs &pa, const AssocArgs &qa, bool cell_search, cudaStream_t stream,
                  Profiler &prof) {
  const int n = max(pa.n_query, qa.n_query);
  if (n <= 0) return;
  prof.begin(FORMGPU_KG_ASSOC_NN);
  if (cell_search)
    assoc_cells_kernel<<<dim3((n + kCellQueryThreads - 1) / kCellQueryThreads, 2), kCellQueryThreads, 0, stream>>>(pa, qa);
  else
    assoc_nn_kernel<<<dim3((n + kNnWarps - 1) / kNnWarps, 2), kNnWarps * 32, 0, stream>>>(pa, qa);
  prof.end(FORMGPU_KG_ASSOC_NN, 1);
}

void assoc_batch_launch(const AssocArgs *items_dev, int n_items, int max_query, cudaStream_t stream, Profiler &prof) {
  if (n_items <= 0 || max_query <= 0) return;
  prof.begin(FORMGPU_KG_ASSOC_NN);
  launch_pdl(assoc_cells_batch_kernel, dim3((max_query + kCellQueryThreads - 1) / kCellQueryThreads, 2, n_items),
             kCellQueryThreads, 0, stream, items_dev);
  prof.end(FORMGPU_KG_ASSOC_NN, 1);
}

// ---------------------------------------------------------------------------
// correspondence segment of the current scan: stable counting sort of the
// accepted matches by the matched scan's slot (rule R6 order inside a pair).
// The NN kernel counts matches per (256-query block, matched slot) with integer atomics;
// every CTA here derives its own exclusive prefix from those counters (a few KB from
// L2), recomputes each query's stable rank inside its block and scatters.  CTA 0 also
// publishes the pair row to the host.
// ---------------------------------------------------------------------------
// Sums the per-256-query bin counters the NN kernel left behind: s_pre[b] = matches of
// bin b in earlier query blocks (exclusive prefix for this block), s_tot[b] = all of them.
// Integer shared-memory atomics: order-free, so the result is deterministic.
__device__ __forceinline__ void block_prefix(const uint32_t *hist_cnt, int nblocks, int nb, int blk,
                                             uint32_t *s_pre, uint32_t *s_tot) {
  for (int i = threadIdx.x; i < nb; i += blockDim.x) s_pre[i] = s_tot[i] = 0u;
  __syncthreads();
  const int total = nblocks * nb;
  // eight counters per thread are requested before the first is consumed (the loop was one L2
  // round trip per four counters: ncu, 43 % of the kernel's samples on the consuming compare)
  for (int i0 = threadIdx.x; i0 < total; i0 += 8 * blockDim.x) {
    uint32_t c[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * (int)blockDim.x;
      c[u] = i < total ? __ldcg(&hist_cnt[i]) : 0u;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (c[u]) {
        const int i = i0 + u * (int)blockDim.x;
        const int bb = i / nb, b = i - bb * nb;
        atomicAdd(&s_tot[b], c[u]);
        if (bb < blk) atomicAdd(&s_pre[b], c[u]);
      }
    }
  }
  __syncthreads();
}

namespace {
__device__ __forceinline__ void segment_scatter_body(const SegmentArgs &a) {
  __shared__ uint32_t s_warp[8][kMaxWindow];
  __shared__ uint32_t s_pre[kMaxWindow + 1], s_tot[kMaxWindow + 1], s_off[kMaxWindow + 1];
  // clear the other counter buffer for this type's next association (grid-stride; saves
  // a separate memset launch on the caller's critical path)
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.hist_bytes / sizeof(uint32_t);
       i += (size_t)gridDim.x * blockDim.x)
    a.hist_next[i] = 0u;
  const bool has_work = (int)(blockIdx.x * blockDim.x) < a.n_query;
  if (!has_work && blockIdx.x != 0) return; // block 0 always publishes the pair row
  const int nb = a.W + 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nblocks = (a.n_query + 255) / 256;
  for (int i = threadIdx.x; i < 8 * kMaxWindow; i += blockDim.x) (&s_warp[0][0])[i] = 0;
  block_prefix(a.hist_cnt, nblocks, nb, (int)blockIdx.x, s_pre, s_tot);
  if (threadIdx.x < 32) { // exclusive prefix over the bins = start of every pair in the segment
    uint32_t run = 0;
    for (int base = 0; base < a.W; base += 32) {
      const int b = base + lane;
      const uint32_t c = b < a.W ? s_tot[b] : 0u;
      uint32_t incl = c;
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (b < a.W) s_off[b] = run + incl - c;
      run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) s_off[a.W] = run; // total correspondences
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    // publish the pair row (offsets, counts, novel count) to the host without a memcpy
    for (int b = threadIdx.x; b <= a.W; b += blockDim.x) {
      a.host_pair_off[b] = s_off[b];
      a.host_pair_cnt[b] = s_tot[b]; // entry W = novel keypoints
      a.dev_pair_off[b] = s_off[b];
      a.dev_pair_cnt[b] = s_tot[b];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned d = atomicAdd(a.done_counter, 1u);
      if (d == 1u) { // both types published
        *a.done_counter = 0u;
        __threadfence_system();
        *a.flag = a.seq;
      }
    }
    if (!has_work) return;
  }
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  MatchRec m;
  m.slot = kNoSlot;
  m.dist_sqrd = DBL_MAX;
  m.k = 0;
  if (q < a.n_query) m = a.match[q];
  const int b = q < a.n_query ? match_bin(m, a.max_dist2) : -1;
  // stable rank inside the warp among lanes with the same bin
  const unsigned peers = __match_any_sync(0xffffffffu, b);
  const int rank_w = __popc(peers & ((1u << lane) - 1u));
  if (b >= 0 && rank_w == 0) s_warp[warp][b] = __popc(peers);
  __syncthreads();
  if (b < 0) return;
  uint32_t pos = s_off[b] + s_pre[b] + rank_w;
  for (int w = 0; w < warp; ++w) pos += s_warp[w][b];
  // correspondence = (map point in its own scan frame, current keypoint):
  // PlanePoint/PointPoint::push_back (factor.hpp:71-75, :113-116).  The map point
  // is the stored local keypoint (the reference's world->local round trip,
  // matcher.hpp:93-96, reproduces it to a few ulp).
  if (a.type == 0) {
    const PlanarRec pi = reinterpret_cast<const PlanarRec *>(a.store)[(size_t)m.slot * a.kcap + m.k];
    const PlanarRec pj = reinterpret_cast<const PlanarRec *>(a.queries)[q];
    float *s = a.seg;
    const size_t st = a.kcap;
    s[0 * st + pos] = pi.x;  s[1 * st + pos] = pi.y;  s[2 * st + pos] = pi.z;
    s[3 * st + pos] = pi.nx; s[4 * st + pos] = pi.ny; s[5 * st + pos] = pi.nz;
    s[6 * st + pos] = pj.x;  s[7 * st + pos] = pj.y;  s[8 * st + pos] = pj.z;
  } else {
    const PointRec pi = reinterpret_cast<const PointRec *>(a.store)[(size_t)m.slot * a.kcap + m.k];
    const PointRec pj = reinterpret_cast<const PointRec *>(a.queries)[q];
    float *s = a.seg;
    const size_t st = a.kcap;
    s[0 * st + pos] = pi.x; s[1 * st + pos] = pi.y; s[2 * st + pos] = pi.z;
    s[3 * st + pos] = pj.x; s[4 * st + pos] = pj.y; s[5 * st + pos] = pj.z;
  }
}
} // namespace
__global__ void __launch_bounds__(256) segment_scatter_kernel(SegmentArgs pa, SegmentArgs qa) {
  segment_scatter_body(blockIdx.y == 0 ? pa : qa);
}
__global__ void __launch_bounds__(256) segment_scatter_batch_kernel(const SegmentArgs *items) {
  __shared__ SegmentArgs s_a;
  load_item_args(s_a, items + 2 * blockIdx.z + blockIdx.y);
  pdl_wait();
  segment_scatter_body(s_a);
}

void segment_build_launch(const SegmentArgs &pa, const SegmentArgs &qa, cudaStream_t stream,
                          Profiler &prof) {
  const int n = max(pa.n_query, qa.n_query);
  if (n <= 0) return;
  prof.begin(FORMGPU_KG_SEGMENT);
  const dim3 g((n + 255) / 256, 2);
  segment_scatter_kernel<<<g, 256, 0, stream>>>(pa, qa);
  prof.end(FORMGPU_KG_SEGMENT, 1);
}

void segment_build_batch_launch(const SegmentArgs *items_dev, int n_items, int max_query,
                                cudaStream_t stream, Profiler &prof) {
  if (n_items <= 0 || max_query <= 0) return;
  prof.begin(FORMGPU_KG_SEGMENT);
  launch_pdl(segment_scatter_batch_kernel, dim3((max_query + 255) / 256, 2, n_items), 256, 0, stream, items_dev);
  prof.end(FORMGPU_KG_SEGMENT, 1);
}

// ---------------------------------------------------------------------------
// commit: append the novel keypoints (dist^2 > min_dist_map^2, unmatched
// included) to the scan's stored keypoints, in keypoint order (map.tpp:160-164)
// ---------------------------------------------------------------------------
namespace {
__device__ __forceinline__ void commit_body(const CommitArgs &a) {
  if ((int)(blockIdx.x * blockDim.x) >= a.n_query) return;
  __shared__ uint32_t s_warp[8];
  __shared__ uint32_t s_before; // novel keypoints in earlier query blocks
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_before = 0u;
  __syncthreads();
  {
    uint32_t mine = 0;
    for (int blk = threadIdx.x; blk < (int)blockIdx.x; blk += blockDim.x)
      mine += __ldcg(&a.hist_cnt[(size_t)blk * (a.W + 1) + a.W]);
    if (mine) atomicAdd(&s_before, mine);
  }
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  const bool novel = q < a.n_query && a.match[q].dist_sqrd > a.min_dist2;
  const unsigned bal = __ballot_sync(0xffffffffu, novel);
  if (lane == 0) s_warp[warp] = __popc(bal);
  __syncthreads();
  if (!novel) return;
  uint32_t pos = a.dst_count + s_before + __popc(bal & ((1u << lane) - 1u));
  for (int w = 0; w < warp; ++w) pos += s_warp[w];
  if (a.type == 0)
    reinterpret_cast<PlanarRec *>(a.store_dst)[pos] = reinterpret_cast<const PlanarRec *>(a.queries)[q];
  else
    reinterpret_cast<PointRec *>(a.store_dst)[pos] = reinterpret_cast<const PointRec *>(a.queries)[q];
}
} // namespace
__global__ void __launch_bounds__(256) commit_kernel(CommitArgs pa, CommitArgs qa) {
  commit_body(blockIdx.y == 0 ? pa : qa);
}
__global__ void __launch_bounds__(256) commit_batch_kernel(const CommitArgs *items) {
  __shared__ CommitArgs s_a;
  load_item_args(s_a, items + 2 * blockIdx.z + blockIdx.y);
  pdl_wait();
  commit_body(s_a);
}

void commit_launch(const CommitArgs &pa, const CommitArgs &qa, cudaStream_t stream, Profiler &prof) {
  const int n = max(pa.n_query, qa.n_query);
  if (n <= 0) return;
  prof.begin(FORMGPU_KG_COMMIT);
  commit_kernel<<<dim3((n + 255) / 256, 2), 256, 0, stream>>>(pa, qa);
  prof.end(FORMGPU_KG_COMMIT, 1);
}

void commit_batch_launch(const CommitArgs *items_dev, int n_items, int max_query, cudaStream_t stream,
                         Profiler &prof) {
  if (n_items <= 0 || max_query <= 0) return;
  prof.begin(FORMGPU_KG_COMMIT);
  launch_pdl(commit_batch_kernel, dim3((max_query + 255) / 256, 2, n_items), 256, 0, stream, items_dev);
  prof.end(FORMGPU_KG_COMMIT, 1);
}

// ---------------------------------------------------------------------------
// export: stored keypoints in the world frame as the API's f64 structs
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) world_export_kernel(WorldExportArgs a) {
  __shared__ int s_off[kMaxWindow + 1];
  for (int i = threadIdx.x; i <= a.W; i += blockDim.x) s_off[i] = a.slot_off[i];
  __syncthreads();
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.n_total) return;
  const int ord = find_slot_of(s_off, a.W, g); // position in scan-id order
  const int slot = a.order[ord];
  const int k = g - s_off[ord];
  const double *T = a.slot_pose + 12 * slot;
  if (a.type == 0) {
    const PlanarRec r = reinterpret_cast<const PlanarRec *>(a.store)[(size_t)slot * a.kcap + k];
    formgpu_planar_feat o;
    transform_point(T, (double)r.x, (double)r.y, (double)r.z, o.x, o.y, o.z);
    const double nx = r.nx, ny = r.ny, nz = r.nz;
    o.nx = (T[0] * nx + T[1] * ny) + T[2] * nz;
    o.ny = (T[3] * nx + T[4] * ny) + T[5] * nz;
    o.nz = (T[6] * nx + T[7] * ny) + T[8] * nz;
    o.pad = 0.0;
    o.npad = 0.0;
    o.scan = a.slot_scan[slot];
    reinterpret_cast<formgpu_planar_feat *>(a.out)[g] = o;
  } else {
    const PointRec r = reinterpret_cast<const PointRec *>(a.store)[(size_t)slot * a.kcap + k];
    formgpu_point_feat o;
    transform_point(T, (double)r.x, (double)r.y, (double)r.z, o.x, o.y, o.z);
    o.pad = 0.0;
    o.scan = a.slot_scan[slot];
    reinterpret_cast<formgpu_point_feat *>(a.out)[g] = o;
  }
}

void world_export_launch(const WorldExportArgs &a, cudaStream_t stream, Profiler &prof) {
  if (a.n_total <= 0) return;
  prof.begin(FORMGPU_KG_EXPORT);
  world_export_kernel<<<(a.n_total + 255) / 256, 256, 0, stream>>>(a);
  prof.end(FORMGPU_KG_EXPORT, 1);
}

} // namespace formgpu
