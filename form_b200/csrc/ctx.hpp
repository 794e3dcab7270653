// Internal definition of the opaque formgpu_ctx (include/formgpu.h).
//
// Device memory layout (all allocated once in formgpu_create; nothing is
// allocated on the per-scan path):
//
//   scan staging   d_scan          [B][rows*cols] float4       input scans
//   stage 1        d_valid_bits    [B][rows][words] u32        validity masks
//                  d_planar_cols   [B][rows][pr_cap] u16       planar picks per row
//                  d_point_cols    [B][rows][qr_cap] u16       point picks per row
//                  d_normals       [B][rows][pr_cap] float4    normal + keep flag
//                  d_cur_planar    [B][kp_cap] PlanarRec (32B) packed keypoints
//                  d_cur_point     [B][kq_cap] PointRec  (16B)
//   keypoint store d_store_planar  [W][kp_cap] PlanarRec       scan-local, lossless f32
//                  d_store_point   [W][kq_cap] PointRec
//   world map      d_hash_*        open-addressing voxel hash (per type)
//                  d_world         voxel- and cell-ordered world points (32 B each)
//                  d_world_src     their (slot, k), d_cell_tab: cell tables
//   matches        d_match_*       per current keypoint: map id + dist^2
//   correspondences d_seg_planar   [W][9][kp_cap] float        SoA p_i,n_i,p_j
//                  d_seg_point     [W][6][kq_cap] float        SoA p_i,p_j
//                  d_pair_table    [W][W] PairEntry            offsets/counts per (k,i)
//
// W = max_window_scans slots; a scan id is mapped to a slot by the host side
// of the C-ABI (slot_of).  B = max_batch_scans.
#pragma once

#include "formgpu.h"

#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <unordered_map>
#include <vector>

namespace formgpu {

struct PlanarRec { // 32 B, one L2 sector
  float x, y, z;
  float nx, ny, nz;
  uint32_t pad0, pad1;
};
struct PointRec { // 16 B
  float x, y, z, w;
};
static_assert(sizeof(PlanarRec) == 32 && sizeof(PointRec) == 16, "record sizes");

struct WorldPoint { // 32 B: world coordinates (f64) + tie-break key
  double x, y, z;
  uint64_t tie; // (rank of the scan id << 24) | k  -> rule R4/R5 ordering
};
static_assert(sizeof(WorldPoint) == 32, "WorldPoint size");

struct HashSlot { // 16 B
  unsigned long long key; // packed voxel coords, EMPTY = ~0ull
  uint32_t start;
  uint32_t count;
};

struct MatchRec { // 16 B
  double dist_sqrd;
  uint32_t slot; // window slot of the matched point's scan (0xffffffff = none)
  uint32_t k;
};

struct PairEntry { // per (current slot k, map slot i)
  uint32_t off_planar, n_planar;
  uint32_t off_point, n_point;
};

constexpr int kMaxWindow = 128;
constexpr uint32_t kNoSlot = 0xffffffffu;

struct GroupProf {
  double ms = 0;
  uint64_t launches = 0;
};

/// Brackets kernel launches with CUDA events when timing is on; always counts launches.
struct Profiler {
  bool timing = false;
  cudaStream_t stream = nullptr;
  GroupProf group[FORMGPU_KG_COUNT];
  uint64_t total_launches = 0;
  struct Pending { int g; cudaEvent_t a, b; };
  std::vector<Pending> pending;
  std::vector<cudaEvent_t> pool;
  cudaEvent_t take() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
  void begin(int g) {
    if (!timing) return;
    Pending p{g, take(), take()};
    cudaEventRecord(p.a, stream);
    pending.push_back(p);
  }
  void end(int g, int launches) {
    group[g].launches += (uint64_t)launches;
    total_launches += (uint64_t)launches;
    if (!timing) return;
    cudaEventRecord(pending.back().b, stream);
  }
  /// after the work has been queued: wait and fold the event pairs into the sums
  void collect() {
    if (pending.empty()) return;
    cudaEventSynchronize(pending.back().b);
    for (auto &p : pending) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, p.a, p.b);
      group[p.g].ms += (double)ms;
      pool.push_back(p.a);
      pool.push_back(p.b);
    }
    pending.clear();
  }
  void destroy() {
    collect();
    for (cudaEvent_t e : pool) cudaEventDestroy(e);
    pool.clear();
  }
};

} // namespace formgpu

struct formgpu_ctx {
  formgpu_params P{};
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  mutable std::string err;

  // derived sizes
  int rows = 0, cols = 0, words = 0, W = 0, B = 1;
  int pr_cap = 0, qr_cap = 0;   // picks per row
  size_t kp_cap = 0, kq_cap = 0; // keypoints per scan
  size_t n_points = 0;

  // ---- stage 1 ----
  float4 *d_scan = nullptr;
  // batched submits, host scans: the NEXT scan of the sequence, uploaded ahead of its EXTRACT
  // request (formgpu_batch_prefetch_scan); swapped with d_scan when that request arrives
  float4 *d_scan_next = nullptr;
  const void *prefetched_host = nullptr; // host pointer the copy in d_scan_next came from
  cudaEvent_t ev_prefetch = nullptr;
  uint32_t *d_valid_bits = nullptr;
  float4 *d_row_box = nullptr; // [B][rows][words][2]
  uint16_t *d_planar_cols = nullptr;
  int *d_planar_cnt = nullptr;
  uint16_t *d_point_cols = nullptr;
  int *d_point_cnt = nullptr;
  float4 *d_normals = nullptr;
  int *d_closest = nullptr; // [B][rows][pr_cap][2]
  int *d_keep_cnt = nullptr;
  // current-scan keypoints, ping-pong: the previous scan's stay intact so that a
  // stale Matcher::matches (SURVEY A.3-12) can still be committed
  formgpu::PlanarRec *d_cur_planar_buf[2] = {nullptr, nullptr};
  formgpu::PointRec *d_cur_point_buf[2] = {nullptr, nullptr};
  int cur_buf = 0;
  formgpu::PlanarRec *d_cur_planar = nullptr; // = d_cur_planar_buf[cur_buf]
  formgpu::PointRec *d_cur_point = nullptr;
  int *d_cur_counts = nullptr; // [B][2]
  // debug (allocated lazily)
  uint8_t *d_dbg_valid = nullptr, *d_dbg_pvalid = nullptr;
  float *d_dbg_curv = nullptr;
  bool debug_extract = false;

  // pinned host staging
  int *h_counts = nullptr;               // [B][2] + misc
  formgpu::PlanarRec *h_planar = nullptr; // kp_cap
  formgpu::PointRec *h_point = nullptr;   // kq_cap
  void *h_upload = nullptr;              // request staging (poses, pairs, chunks)
  size_t h_upload_bytes = 0;
  // results, mapped pinned, written by the kernels as sequence-tagged words (182 per pair)
  volatile unsigned long long *h_out = nullptr;
  size_t h_out_bytes = 0;

  // batched host-scan extraction: the pack kernel leaves the f64 API structs here (device memory)
  // and a copy engine moves them to the caller's buffers - SM stores over PCIe kept the pack
  // kernel resident for ~30 us per scan (profiles/r03/e2e_probe.txt)
  formgpu_planar_feat *d_stage_planar = nullptr; // [kp_cap], allocated on first use
  formgpu_point_feat *d_stage_point = nullptr;   // [kq_cap]
  // caller output buffers last probed for page-locked-ness, and their device aliases
  void *direct_probe[2] = {nullptr, nullptr};
  void *direct_alias[2] = {nullptr, nullptr};

  // ---- raw clouds (formgpu_set_cloud_format; organize.cu writes the organised scan to d_scan) ----
  bool have_cloud = false;
  formgpu_cloud_format cloud{};          // beam_elevations is not kept (the tables below are)
  int cloud_el_desc = 0;
  unsigned char *d_records = nullptr;    // record staging, cloud.max_records * cloud.stride bytes
  unsigned long long *d_pixel_keys = nullptr; // [rows * cols]
  double2 *d_cloud_tab = nullptr;        // [cols + 1] azimuth boundaries | [rows - 1] beam midpoints
  unsigned *d_cloud_stats = nullptr;     // [8] outcome counters of the last organisation
  unsigned *h_cloud_stats = nullptr;     // pinned copy, queued behind the gather kernel
  size_t cloud_last_n = 0;
  const void *prefetched_cloud = nullptr; // formgpu_batch_prefetch_cloud: records already in d_records
  size_t prefetched_cloud_n = 0;

  // ---- current scan ----
  bool have_current = false;
  uint64_t cur_scan = 0;
  int cur_n[2] = {0, 0}; // planar, point keypoints of the current scan
  bool cur_device_resident = false;

  // ---- window / keypoint store ----
  std::unordered_map<uint64_t, int> slot_of; // scan id -> slot
  std::vector<uint64_t> slot_scan;           // slot -> scan id
  std::vector<uint8_t> slot_used;
  std::vector<int> store_n[2];               // keypoints stored per slot
  formgpu::PlanarRec *d_store_planar = nullptr;
  formgpu::PointRec *d_store_point = nullptr;

  // ---- world map (per type t) ----
  size_t hash_cap[2] = {0, 0}; // power of two, worst case
  // one allocation: [cursor (256 B)][hash planar][hash point]; the point table
  // starts right after the part of the planar table used by the last rebuild,
  // so one memset clears cursor + both tables
  unsigned char *d_mapmem = nullptr;
  formgpu::HashSlot *d_hash[2] = {nullptr, nullptr}; // views into d_mapmem (per rebuild)
  uint32_t hash_mask[2] = {0, 0};
  // as the association reads them; the rebuild's first passes use them as scratch (MapArgs)
  formgpu::WorldPoint *d_world[2] = {nullptr, nullptr};    // voxel- and cell-ordered map points
  uint32_t *d_world_src[2] = {nullptr, nullptr};           // (window slot << 24 | k) of every map point
  formgpu::WorldPoint *d_cell_tab[2] = {nullptr, nullptr}; // cell tables of the cell-ordered voxels
  uint32_t *d_scatter_src[2] = {nullptr, nullptr};         // rebuild scratch
  uint32_t *d_voxel_list[2] = {nullptr, nullptr}; // hash slots of the occupied voxels
  size_t map_n[2] = {0, 0};                       // points in the built map
  size_t map_cap[2] = {0, 0};
  // rebuild request, one H2D: [W][12] poses | [W] scan ids | [2][W+1] offsets | [W] order
  unsigned char *d_map_req = nullptr;
  unsigned char *h_map_req = nullptr; // pinned
  size_t map_req_bytes = 0;
  cudaEvent_t ev_upload = nullptr;    // guards reuse of the pinned request buffers
  bool map_built = false;
  // single-sequence associations: warp-per-query whole-bucket search (lowest latency, default) or,
  // with FORMGPU_SINGLE_CELL_SEARCH=1, the cell search of the batched submits (tests)
  bool cell_search_single = false;
  void *d_export = nullptr;           // lazily allocated world export buffer
  size_t export_bytes = 0;

  // ---- matches / correspondences ----
  formgpu::MatchRec *d_match[2] = {nullptr, nullptr};
  int match_n[2] = {0, 0};            // Matcher::matches.size() per type
  uint64_t match_scan[2] = {0, 0};    // matches.front().query.scan
  const void *match_queries[2] = {nullptr, nullptr}; // keypoint buffer the matches refer to
  uint32_t match_novel[2] = {0, 0};   // keypoints insert_matches would append
  float *d_seg_planar = nullptr; // [W][9][kp_cap]
  float *d_seg_point = nullptr;  // [W][6][kq_cap]
  // [ping-pong][blocks256][W+1] match counters per type: the NN kernel fills one buffer
  // while the other is being cleared for the next association
  uint32_t *d_hist_cnt[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  size_t hist_bytes[2] = {0, 0};
  int hist_cur[2] = {0, 0};                        // per type: buffer used by its last association
  const uint32_t *match_hist[2] = {nullptr, nullptr}; // counters the stored matches refer to
  uint32_t *h_pair = nullptr;     // mapped pinned [type][off|cnt][W+1], written by the scatter kernel
  uint32_t *d_pair = nullptr;     // device copy (read by a linearisation queued behind the association)
  std::vector<formgpu::PairEntry> h_pair_table; // host mirror [W(k)][W(i)]

  // ---- zero-copy completion signalling ----
  // mapped pinned page the kernels write their completion sequence numbers to
  volatile unsigned long long *h_flags = nullptr; // [8]: 0 lin/err, 1 assoc, 2 extract
  unsigned long long seq = 0;
  unsigned *d_counters = nullptr; // [pair tickets (cap) | done counters (8)]
  size_t counter_cap = 0;

  // ---- point-sharded mode (formgpu_set_shard) ----
  int shard_rank = 0, shard_world = 1;
  // ---- point-sharded mode over NCCL (formgpu_comm_init, comm.cu) ----
  void *comm = nullptr; // ncclComm_t
  int comm_rank = 0, comm_world = 1;
  double *d_red = nullptr, *h_red = nullptr; // blocks / errors of a request: all-reduced, then copied out
  size_t red_cap = 0;
  // [world][planar candidates | point candidates of the current scan]: one in-place all-gather
  formgpu::MatchRec *d_gather = nullptr;

  // ---- pair-moment cache (moments.cu) ----
  // [W(j)][W(i)][kMomentStride] doubles: moments of pair (i, j) left by scan j's last association
  double *d_moments = nullptr;
  double *d_mom_partials = nullptr; // [mom_max_units][kMomentPartial]
  unsigned *d_mom_tickets = nullptr; // [W], self-cleaning
  int mom_max_units = 0;
  uint32_t moment_unit = 128; // kMomentUnitSingle; contexts of a batch use kMomentUnit (api_batch.cu)
  // linearize / error are evaluated from the cache (default, and always in a batch) or, with
  // FORMGPU_STREAM_LINEARIZE=1 and always in point-sharded mode, by streaming the correspondences
  bool moment_cache = true;

  // ---- linearisation request ----
  void *d_request = nullptr;
  size_t request_bytes = 0;
  size_t out_cap = 0; // pairs

  // ---- instrumentation ----
  formgpu::Profiler prof;
};
