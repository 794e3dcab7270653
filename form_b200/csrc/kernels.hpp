// Kernel argument blocks and host-side launchers shared between the .cu files.
#pragma once

#include "ctx.hpp"

namespace formgpu {

// ---- programmatic dependent launch (batched submits) ----
// The kernels of a batched submission form one dependent chain per stream, and each is a short
// latency chain of its own, so the gap between one kernel's end and the next one's start is a sizeable
// share of each.  Kernels of the chain after the first are launched with programmatic stream
// serialisation: the launch of a kernel is prepared while its predecessor runs, the kernel copies its
// staged arguments (uploaded before the chain's first kernel) and then waits in pdl_wait until the
// predecessor has completed and its memory is visible, before it touches anything an earlier kernel
// writes or reads.  No kernel triggers its dependents early: CTAs waiting in pdl_wait hold SM
// resources that the other batches' kernels on other streams need (measured: -12 % batched
// throughput with a trigger at every kernel's start).  pdl_wait returns at once in a kernel launched
// without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
/// kernel<<<grid, block, smem, stream>>>(args...) with programmatic stream serialisation.  Every CTA
/// of the kernel calls pdl_wait before its first access to memory an earlier kernel of the stream
/// writes or reads, and before it exits: the kernel's successor then waits for all earlier kernels too
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- stage 1 (extract.cu, compiled with -fmad=false) ----
struct ExtractArgs {
  int rows, cols, cols_pad, words;
  int np, num_sectors, pps;
  int planar_per_sector, point_per_sector, min_points;
  int pr_cap, qr_cap;
  size_t kp_cap, kq_cap;
  double min_norm2, max_norm2, planar_threshold, radius;
  const float4 *scan;      // [B][rows*cols]
  uint32_t *valid_bits;    // [B][rows][words]
  float4 *row_box;         // [B][rows][words][2]  (lo, hi) of the valid points of a 32-column chunk
  uint16_t *planar_cols;   // [B][rows][pr_cap]
  int *planar_cnt;         // [B][rows]
  uint16_t *point_cols;    // [B][rows][qr_cap]
  int *point_cnt;          // [B][rows]
  float4 *normals;         // [B][rows][pr_cap]  (nx, ny, nz, keep)
  int *closest;            // [B][rows][pr_cap][2] or nullptr
  int *keep_cnt;           // [B][rows]
  PlanarRec *cur_planar;   // [B][kp_cap]
  PointRec *cur_point;     // [B][kq_cap]
  int *cur_counts;         // [B][2]
  uint8_t *dbg_valid, *dbg_pvalid; // [B][rows*cols] or nullptr
  float *dbg_curv;                 // [B][rows*cols] or nullptr
  // zero-copy results (mapped pinned host memory); host_planar/host_point may be null
  // when the caller only needs the counts (device-resident mode)
  PlanarRec *host_planar;
  PointRec *host_point;
  // ... or the caller's own page-locked buffers, filled with the API's f64 structs
  formgpu_planar_feat *host_planar_f64;
  formgpu_point_feat *host_point_f64;
  unsigned long long scan_idx;
  int *host_counts;                // [2]
  unsigned *done_counter;          // zero on entry, self-cleaning
  volatile unsigned long long *flag;
  unsigned long long seq;
  unsigned done_target;            // pack CTAs that share done_counter (rows x scans of the launch)
  unsigned pad_;
};

constexpr int kExtractMaxSectors = 64; // sectors per row the select kernel validates in order
/// Entries of a sector's speculative pick list in the select kernel (planar or point picks).
/// Picks of one sector are pairwise >= np columns apart (suppression +-(np-1)); the last sector is
/// the longest (it takes the remainder columns).
__host__ __device__ inline int extract_spec_cap(const ExtractArgs &a) {
  const int longest = a.cols - (a.num_sectors - 1) * a.pps;
  return (longest + a.np - 1) / a.np + 1;
}
cudaError_t extract_configure(const ExtractArgs &shape);
size_t extract_select_smem(int cols, int cols_pad, int words, int sectors, int spec_cap);
inline size_t extract_select_smem(const ExtractArgs &a) {
  return extract_select_smem(a.cols, a.cols_pad, a.words, a.num_sectors, extract_spec_cap(a));
}
size_t extract_normals_smem(int cols, int words, int pr_cap);
/// Launches the three stage-1 kernels.
void extract_launch(const ExtractArgs &a, int n_scans, cudaStream_t stream, Profiler &prof);
/// What a batched extraction launch needs of its items' geometry, which may differ from item to
/// item: the grid covers the largest `rows`, dynamic shared memory is the largest need of each
/// kernel, and the many-row choice counts the true sum of rows.
struct ExtractLaunchShape {
  int max_rows = 0;
  long long sum_rows = 0;
  size_t select_smem = 0, normals_smem = 0, pack_smem = 0;
};
ExtractLaunchShape extract_launch_shape(const ExtractArgs *items, int n_items);
/// Same three kernels for n_items scans of DIFFERENT contexts (one ExtractArgs each, in
/// device memory); `shape` comes from extract_launch_shape over the same items.
/// Launches with at least `many_rows_min` rows (summed over the items) use the many-row variants:
/// 128-thread select CTAs and the thread-per-pick normals kernel, which trade per-row latency for
/// rows in flight.
constexpr int kManyRowsMin = 1; // measured: +5 % batched throughput over switching at 2 x 148 rows
void extract_batch_launch(const ExtractLaunchShape &shape, const ExtractArgs *items_dev, int n_items,
                          int many_rows_min, cudaStream_t stream, Profiler &prof);

// ---- raw clouds -> organised scans (organize.cu, compiled with -fmad=false; rule R8) ----
// outcome counters of one organisation (formgpu_cloud_stats order; slot 0 is filled by the host)
constexpr int kOrgStatPlaced = 1, kOrgStatPixels = 2, kOrgStatNonfinite = 3, kOrgStatZero = 4,
              kOrgStatTime = 5, kOrgStatRow = 6, kOrgStatCol = 7, kOrgStats = 8;
struct OrganizeArgs {
  const unsigned char *records; // n records of `stride` bytes (device)
  unsigned n, stride;
  int off_x, off_y, off_z, off_row, off_col, off_time; // byte offsets, -1 = absent
  int xyz_type, row_type, col_type, time_type;         // FORMGPU_FIELD_*
  int row_source, col_source;                          // FORMGPU_ROW_FROM_* / FORMGPU_COL_FROM_*
  int rows, cols;
  int az_dir, el_desc; // column direction (+1 / -1); beam table given top-down
  double scan_period;
  const double2 *az_tab;    // [cols + 1] (cos, sin) of the column boundaries
  const double2 *el_tab;    // [rows - 1] (cos, sin) of the beam midpoints, ascending
  unsigned long long *keys; // [rows * cols] winner key per pixel
  float4 *scan;             // [rows * cols] organised output (the context's scan buffer)
  unsigned *stats;          // [kOrgStats]
};
/// clear + scatter + gather of one cloud on `stream`.
void organize_launch(const OrganizeArgs &a, cudaStream_t stream, Profiler &prof);
/// The same three kernels for n_items clouds of different contexts in one launch each; the grids
/// cover the largest record count and the largest pixel count of the items.
void organize_batch_launch(const OrganizeArgs *items_dev, int n_items, size_t max_records, size_t max_pixels,
                           cudaStream_t stream, Profiler &prof);

// ---- stage 2 (map_assoc.cu, compiled with -fmad=false) ----
struct MapArgs {
  int type;            // 0 planar, 1 point
  int W;
  size_t kcap;         // keypoints per slot in the store
  const void *store;   // PlanarRec* or PointRec*
  const int *slot_off; // [W+1] exclusive prefix of store counts (device)
  const double *slot_pose;   // [W][12]
  const int *slot_rank;      // [W] rank of the slot's scan id among the window's (tie-break, rule R4)
  int n_total;
  double voxel_width;
  double inv_voxel_width; // 1 / voxel_width (host, IEEE): fast path of voxel_coord
  HashSlot *hash;
  uint32_t hash_mask;
  // what the association reads, written by pass 4; passes 1-3 use the arrays as scratch
  WorldPoint *world;     // map points, voxel- and cell-ordered (pass 1: store order)
  uint32_t *world_src;   // (window slot << 24 | k) of every map point (pass 1: hash slot per point)
  WorldPoint *cell_tab;  // per-voxel cell tables (pass 3: the voxel-sorted points)
  uint32_t *scatter_src; // pass 3: (window slot << 24 | k) of the voxel-sorted points
  uint32_t *cursor;      // [0] allocation cursor, [1] occupied voxels (zeroed before the build)
  uint32_t *voxel_list;  // hash slots of the occupied voxels, in creation order (insert pass)
};
/// Cell-ordered buckets (map_assoc.cu, pass 4): a voxel holding kCellMin..kCellMax points gets
/// kCellFlag in its slot's count; its bucket is ordered by a kCellSub^3 cell code and has a
/// table of 64 u16 end offsets in cell_tab.
constexpr uint32_t kCellFlag = 0x80000000u;
constexpr uint32_t kCellMin = 16, kCellMax = 65535;
constexpr int kCellSub = 4;
void map_build_launch(const MapArgs &planar, const MapArgs &point, cudaStream_t stream, Profiler &prof);
struct MapClearRegion {
  void *base;   // 16-byte aligned
  size_t bytes; // multiple of 16
  // batched rebuilds: the request of the context (slot offsets, poses, scan ids) rides in the
  // submission's argument upload and the clear kernel - the first launch of the rebuild - moves it
  // to its place, instead of one upload + event pair per sequence (copy_bytes a multiple of 8)
  size_t copy_src_off; // offset of the staged request inside the submission's argument ring
  void *copy_dst;
  size_t copy_bytes;
};
/// Rebuild of n_items maps in one pass of four launches: items_dev = [item][type] MapArgs,
/// regions_dev[item] = the cursor + hash tables to clear first.
/// `ring_dev`: base of the argument ring the regions' copy_src_off refer to.
void map_build_batch_launch(const MapArgs *items_dev, const MapClearRegion *regions_dev, const unsigned char *ring_dev,
                            int n_items, int max_points, uint32_t max_hash, size_t max_clear_bytes,
                            cudaStream_t stream, Profiler &prof);

struct AssocArgs {
  int type;
  int n_query;
  int n_map;
  // queries this launch searches: [q_begin, q_end) (the whole scan)
  int q_begin, q_end;
  // point-sharded mode: the map holds only this rank's scans; the winner's shift rank travels in
  // bits 8..12 of MatchRec::slot so that assoc_combine can apply rule R5 across the ranks
  int pack_rank, pad_rank;
  const void *queries; // PlanarRec* / PointRec* of the current scan
  double pose[12];     // pose of the current scan
  double voxel_width;
  double inv_voxel_width; // 1 / voxel_width (host, IEEE): fast path of voxel_coord
  // the offset table of a flagged (cell-ordered) voxel whose bucket starts at `start` lives in
  // cell_tab[start .. start+3] (64 x u16 end offsets)
  const WorldPoint *cell_tab;
  const HashSlot *hash;
  uint32_t hash_mask;
  const WorldPoint *world;
  const uint32_t *world_src;
  MatchRec *match;
  // fused histogram: matches per (256-query block, matched slot), entry W = novel keypoints
  int W;
  double max_dist2, min_dist2;
  uint32_t *hist_cnt;      // [blocks256][W+1] atomic counters, zero on entry; nullptr: the
                           // histogram is built by assoc_hist_launch once all matches are there
};
/// Point-sharded mode: per query the rule-R5 minimum over the `world` candidate records the ranks
/// found in their sub-maps (gathered[r * n_query + q], shift rank packed into the slot), written to
/// a.match with the histogram the association kernels otherwise build themselves.
struct CombineArgs {
  AssocArgs a;                // n_query, match (output), hist_cnt, W, max / min dist
  const MatchRec *gathered;   // rank r's candidate of query q: gathered[r * stride + q]
  const uint64_t *slot_scan;  // [W] scan id of every window slot (tie-break, rule R4)
  int world;
  int stride;                 // records per rank (planar + point candidates of the scan)
};
void assoc_combine_launch(const CombineArgs &planar, const CombineArgs &point, cudaStream_t stream, Profiler &prof);
/// One sequence: `cell_search` = the one-thread-per-query search cell by cell (what batched submits
/// always use); otherwise one WARP per query scans whole buckets - the lower latency for a single
/// scan's ~30 k queries, which cannot fill the GPU either way.
void assoc_launch(const AssocArgs &planar, const AssocArgs &point, bool cell_search, cudaStream_t stream,
                  Profiler &prof);
/// Batched submits: the cell search, one thread per query.
void assoc_batch_launch(const AssocArgs *items_dev, int n_items, int max_query, cudaStream_t stream, Profiler &prof);

struct SegmentArgs {
  int type;
  int W;
  int n_query;
  double max_dist2;
  double min_dist2;
  size_t kcap;
  const void *queries;  // current scan keypoints
  const void *store;    // keypoint store
  const MatchRec *match;
  const uint32_t *hist_cnt; // [blocks256][W+1] counters filled by the NN kernel
  uint32_t *hist_next;      // the other counter buffer, cleared after this launch
  size_t hist_bytes;
  uint32_t *host_pair_off;  // [W+1] mapped pinned: start of every pair in the segment
  uint32_t *host_pair_cnt;  // [W+1] mapped pinned: counts (entry W = novel keypoints)
  uint32_t *dev_pair_off;   // device copies for a linearisation queued right behind
  uint32_t *dev_pair_cnt;
  unsigned *done_counter;   // zero on entry, self-cleaning
  volatile unsigned long long *flag; // mapped pinned: set to `seq` once both types are published
  unsigned long long seq;
  float *seg;           // segment base of the current slot: [9 or 6][kcap]
};
void segment_build_launch(const SegmentArgs &planar, const SegmentArgs &point, cudaStream_t stream, Profiler &prof);
void segment_build_batch_launch(const SegmentArgs *items_dev, int n_items, int max_query,
                                cudaStream_t stream, Profiler &prof);

struct CommitArgs {
  int type;
  int W;
  int n_query;
  double min_dist2;
  const void *queries;
  const MatchRec *match;
  const uint32_t *hist_cnt; // counters of the association the matches come from
  void *store_dst;   // store slot base of the scan being appended to
  uint32_t dst_count; // keypoints already stored there
};
void commit_launch(const CommitArgs &planar, const CommitArgs &point, cudaStream_t stream, Profiler &prof);
void commit_batch_launch(const CommitArgs *items_dev, int n_items, int max_query, cudaStream_t stream,
                         Profiler &prof);

struct WorldExportArgs {
  int type;
  int W;
  size_t kcap;
  const void *store;
  const int *slot_off;  // [W+1] prefix in scan-id order
  const int *order;     // [W] slot at each position of that order
  const double *slot_pose;
  const uint64_t *slot_scan;
  int n_total;
  void *out; // formgpu_planar_feat* / formgpu_point_feat* (device)
};
void world_export_launch(const WorldExportArgs &a, cudaStream_t stream, Profiler &prof);

// ---- stage 3 (linearize.cu, FMA allowed: tolerance class) ----
constexpr int kLinThreads = 256;   // threads per CTA
constexpr int kLinCluster = 8;     // largest cluster (CTAs per scan pair)
constexpr int kLinInlineTasks = 48; // pairs that travel in the kernel parameters (6 KB)

struct LinTask { // one scan pair with at least one correspondence (144 B)
  double rel[12];      // R_i^T R_j row-major, then R_i^T (t_j - t_i): precomputed by the host
  uint32_t off_planar, n_planar, off_point, n_point; // ranges inside the segment of slot_j
  int slot_j;
  int out_index;       // position of the pair in the caller's list
  uint32_t dyn_slot_i_plus1; // != 0: the ranges are read from the device pair row of slot_i
                             // (association and linearisation queued back to back)
  uint32_t ctx_index;        // batched launches: which context's LinArgs the task uses
  int slot_i;                // window slot of scan i: the pair's entry in the moment cache
  int pad_;
  const double *entry;       // the pair's cache entry (ctx->d_moments + (slot_j * W + slot_i) * kMomentStride):
                             // resolved by the host so that the evaluation kernel's first load is the entry itself
};
static_assert(sizeof(LinTask) == 144, "LinTask size");

struct LinInline {
  LinTask tasks[kLinInlineTasks];
};

struct LinArgs {
  size_t kp_cap, kq_cap;
  const float *seg_planar; // [W][9][kp_cap]
  const float *seg_point;  // [W][6][kq_cap]
  const LinTask *tasks;    // device copy of the request when it does not fit the parameters
  const uint32_t *pair_row; // device [type][off|cnt][W+1] written by the last association
  int W;
  int n_tasks;
  int cluster;             // CTAs per pair for this launch: 1, 2, 4 or 8
  double inv_sigma2;
  // mapped pinned host memory (zero-copy), sequence-tagged words: [n_pairs][182] for
  // blocks, [n_pairs][2] for errors; word = 32 bits of payload | (seq & 0xffffffff) << 32
  volatile unsigned long long *out;
  unsigned long long seq;
  // point-sharded mode (SURVEY 8e): this context reduces only the shard_rank-th of
  // shard_world contiguous shares of every pair's correspondences; the caller sums the
  // per-pair blocks over the ranks (NCCL all-reduce of 91 * P doubles)
  int shard_rank, shard_world;
  // != nullptr: blocks / errors are written as plain doubles into DEVICE memory
  // ([n_pairs][91] or [n_pairs]) instead of the tagged host words, so that a collective
  // queued on the same stream can consume them without a host round trip
  double *out_plain;
  // pair-moment cache of the context (moments.cu): [W(j)][W(i)][kMomentStride] doubles
  const double *moments;
};
static_assert(sizeof(LinArgs) % 8 == 0, "LinArgs: the evaluation kernels copy it in 8-byte words");
cudaError_t linearize_launch(const LinArgs &a, const LinInline *inline_req, bool error_only,
                             cudaStream_t stream, Profiler &prof);

// ---- stage 3, cached form (moments.cu, FMA allowed: tolerance class) ----
// Every association leaves, per pair (i, current scan), the POSE-INDEPENDENT second moments of
// its correspondences at a reference relative pose rel0 (header of moments.cu); a later
// linearisation / error evaluation at any poses is a 13x13 congruence of those moments - no
// correspondence is streamed again.
constexpr int kMomentPlanar = 91;    // packed upper triangle of sum phi phi^T, phi in R^13
constexpr int kMomentPoint = 28;     // packed upper triangle of sum zeta zeta^T, zeta in R^7
constexpr int kMomentStride = 132;   // doubles per entry: M_p[91] | M_q[28] | rel0[12] | counts (2 x u32)
constexpr int kMomentAcc = 73;       // distinct planar sums a thread accumulates
constexpr int kMomentPartial = 104;  // doubles per unit partial: 73 planar | 28 point | pad
// correspondences per warp-sized unit of work (MomentArgs::unit): batched submits amortise the
// per-unit reduction over 512 correspondences; a single sequence's association (~15 k accepted
// matches) would occupy ~40 warps of the GPU that way, so it is cut into units of 128
constexpr uint32_t kMomentUnit = 512, kMomentUnitSingle = 128;

struct MomentArgs { // one association of one context
  size_t kp_cap, kq_cap;
  const float *seg_planar;   // segment of the current slot: [9][kp_cap]
  const float *seg_point;    // [6][kq_cap]
  const uint32_t *pair_row;  // device [type][off|cnt][W+1] written by the scatter kernel just before
  const double *slot_pose;   // [W][12] poses of the last map rebuild (device)
  double pose_k[12];         // pose the current scan was associated at
  double *moments;           // cache row of the current slot: [W][kMomentStride]
  double *partials;          // [max_units][kMomentPartial]
  unsigned *tickets;         // [W], zero on entry, self-cleaning
  int W;
  int n_pairs;               // map slots listed in `slots`
  int shard_rank, shard_world;
  uint32_t unit, pad_unit;   // correspondences per unit (kMomentUnit or kMomentUnitSingle)
  unsigned char slots[kMaxWindow];
};
static_assert(sizeof(MomentArgs) % 8 == 0, "MomentArgs is copied in 8-byte words");
/// Upper bound of the units (= warps) one association with n_corr accepted matches over n_pairs
/// pairs can need.
inline int moment_max_units(size_t n_corr, int n_pairs, uint32_t unit) { return (int)(n_corr / unit) + n_pairs; }
void moments_launch(const MomentArgs &a, int max_units, cudaStream_t stream, Profiler &prof);
void moments_batch_launch(const MomentArgs *items_dev, int n_items, int max_units, cudaStream_t stream,
                          Profiler &prof);
/// Blocks / errors of the listed tasks from the moment cache: one warp per task.  Tasks travel in
/// the kernel parameters (inline_req, <= kLinInlineTasks) or in a.tasks (device memory).
cudaError_t eval_launch(const LinArgs &a, const LinInline *inline_req, bool error_only, cudaStream_t stream,
                        Profiler &prof);
cudaError_t eval_batch_launch(const LinArgs *ctx_args_dev, const LinTask *tasks_dev, int n_tasks,
                              bool error_only, cudaStream_t stream, Profiler &prof);

} // namespace formgpu
