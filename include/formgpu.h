/*
 * formgpu.h - C-ABI of the B200 (sm_100a) implementation of FORM's per-scan
 * data-parallel hot path: scan-line feature extraction, voxel-hashed keypoint
 * association, and point-to-plane / point-to-point linearisation into per-pair
 * normal-equation blocks, plus the reparative map rebuild.
 *
 * This is the drop-in boundary.  Plain C types, caller-owned buffers, int status
 * codes; no exceptions, no C++ or torch types cross it.  Every entry point
 * names the reference interface it replaces (paths relative to the FORM
 * repository).  The C++ facade in form_b200/host/form/ (namespace form:
 * Estimator, FeatureExtractor, ...) sits on top of exactly these calls; see
 * INTEGRATION.md for the binding a FORM maintainer would add.
 *
 * Threading: one caller thread per context; contexts are independent (one per
 * sequence / GPU).  All work of a context is ordered on one CUDA stream.
 *
 * There is no CPU fallback: every compute entry point fails with
 * FORMGPU_ERR_CUDA when no CUDA device is usable.
 */
#ifndef FORMGPU_H
#define FORMGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FORMGPU_ABI_VERSION 1

/* ---- status codes ------------------------------------------------------- */
#define FORMGPU_OK 0
#define FORMGPU_ERR_INVALID_ARG 1 /* null pointer, bad enum, unknown scan id   */
#define FORMGPU_ERR_BAD_SCAN_SIZE 2 /* n != rows*cols (extraction.tpp:141-145) */
#define FORMGPU_ERR_CAPACITY 3    /* caller buffer or internal arena too small */
#define FORMGPU_ERR_CUDA 4        /* CUDA runtime error / no device            */
#define FORMGPU_ERR_STATE 5       /* call order violated (e.g. no current scan)*/
#define FORMGPU_ERR_UNSUPPORTED 6 /* parameter outside the supported range     */

/* ---- plain data --------------------------------------------------------- */

/* form::PointXYZf, form/utils.hpp:38-91.  Organised scans are row-major:
 * idx = row * num_columns + col (form/feature/extraction.tpp:155). */
typedef struct formgpu_point4f {
  float x, y, z, w;
} formgpu_point4f;

/* form::PointFeat, form/feature/features.hpp:31-86 (40 bytes). */
typedef struct formgpu_point_feat {
  double x, y, z, pad;
  uint64_t scan;
} formgpu_point_feat;

/* form::PlanarFeat, form/feature/features.hpp:89-163 (72 bytes). */
typedef struct formgpu_planar_feat {
  double x, y, z, pad;
  double nx, ny, nz, npad;
  uint64_t scan;
} formgpu_planar_feat;

/* gtsam::Pose3 as 12 doubles: row-major rotation then translation (96 bytes).
 * T * p = R p + t. */
typedef struct formgpu_pose {
  double R[9];
  double t[3];
} formgpu_pose;

/* Pose of one scan of the window: gtsam::Values entry X(scan). */
typedef struct formgpu_scan_pose {
  uint64_t scan;
  formgpu_pose pose;
} formgpu_scan_pose;

/* m_constraints[j][i], j > i (form/optimization/constraints.hpp:91-99). */
typedef struct formgpu_pair {
  uint64_t i;
  uint64_t j;
} formgpu_pair;

typedef struct formgpu_pair_count {
  uint64_t i;
  uint32_t n_planar;
  uint32_t n_point;
} formgpu_pair_count;

/* One nearest-neighbour result (form::Match, form/mapping/map.hpp:48-61).  The
 * matched map point is identified by its stable id (scan, k) = k-th stored
 * keypoint of that scan (rule R4).  found == 0 <=> dist_sqrd == DBL_MAX. */
typedef struct formgpu_match {
  uint64_t scan;
  uint32_t k;
  uint32_t found;
  double dist_sqrd;
} formgpu_match;

/* FeatureExtractor::Params (form/feature/extraction.hpp:59-88), MatcherParams
 * (form/optimization/matcher.hpp:32-41), KeypointMapParams
 * (form/mapping/map.hpp:97-100), planar_constraint_sigma
 * (form/optimization/constraints.hpp:60), plus arena capacities. */
typedef struct formgpu_params {
  int32_t neighbor_points;         /* 5   */
  int32_t num_sectors;             /* 6   */
  int32_t planar_feats_per_sector; /* 50  */
  int32_t point_feats_per_sector;  /* 3   */
  int32_t min_points;              /* 5   */
  int32_t num_columns;             /* 1024 */
  int32_t num_rows;                /* 64  */
  int32_t max_window_scans;        /* 64: scans resident at once (<= 1+10+50)   */
  double planar_threshold;         /* 1.0 */
  double radius;                   /* 1.0 */
  double min_norm_squared;         /* 1.0 */
  double max_norm_squared;         /* 1e4 */
  double max_dist_matching;        /* 0.8 (also the voxel width, form.cpp:61-65) */
  double min_dist_map;             /* 0.1 */
  double sigma;                    /* 0.1 */
  int32_t max_batch_scans;         /* 1: scans per formgpu_extract_batch call    */
  int32_t reserved;
} formgpu_params;

typedef struct formgpu_ctx formgpu_ctx;

/* ---- lifecycle ---------------------------------------------------------- */

/* Reference defaults (python/bindings.cpp:66-88). */
void formgpu_default_params(formgpu_params *p);

/* Estimator::Estimator(const Params&) (form/form.cpp:31-38).  `stream` is a
 * cudaStream_t to run on, or NULL to create a private non-blocking stream. */
int formgpu_create(const formgpu_params *p, int device, void *stream, formgpu_ctx **out);
void formgpu_destroy(formgpu_ctx *ctx);

/* Message of the last failing call on this context ("" if none).  With a NULL
 * context returns the message of the last failed formgpu_create. */
const char *formgpu_last_error(const formgpu_ctx *ctx);

int formgpu_abi_version(void);

/* ---- stage 1: feature extraction ---------------------------------------- */

/* FeatureExtractor::extract (form/feature/extraction.hpp:99-101,
 * extraction.tpp:29-132).  `scan` is a HOST buffer of n = rows*cols points.
 * Writes up to *_cap keypoints (rule R3 order) and the true counts; makes
 * scan_idx the context's "current scan".  FORMGPU_ERR_BAD_SCAN_SIZE when
 * n != rows*cols; FORMGPU_ERR_CAPACITY when a caller buffer is too small (the
 * counts are still written). */
int formgpu_extract(formgpu_ctx *ctx, const formgpu_point4f *scan, size_t n, uint64_t scan_idx,
                    formgpu_planar_feat *planar_out, size_t planar_cap, size_t *n_planar,
                    formgpu_point_feat *point_out, size_t point_cap, size_t *n_point);

/* Page-locked, device-mapped host memory (cudaHostAlloc) for callers that do not link
 * CUDA themselves.  Optional: when `scan` is page-locked the upload is a plain DMA, and
 * when planar_out / point_out are page-locked and sized formgpu_max_planar / _point the
 * kernels write the keypoint structs straight into them; pageable buffers work too and
 * go through a staging copy. */
void *formgpu_alloc_pinned(size_t bytes);
void formgpu_free_pinned(void *p);

/* Same, but `scan_dev` is a DEVICE pointer and nothing is copied back: only
 * the counts are returned (used to time the kernels with inputs resident). */
int formgpu_extract_device(formgpu_ctx *ctx, const formgpu_point4f *scan_dev, size_t n,
                           uint64_t scan_idx, size_t *n_planar, size_t *n_point);

/* Upper bounds for sizing caller buffers. */
size_t formgpu_max_planar(const formgpu_ctx *ctx);
size_t formgpu_max_point(const formgpu_ctx *ctx);

/* Intermediates of the last extraction, for parity tests (any pointer may be
 * NULL): validity masks (extraction.tpp:136-222), float curvature (:226-261),
 * planar picks before the normal drop with their keep flag and the
 * find_closest results (:402-420), point picks. */
int formgpu_extract_debug(formgpu_ctx *ctx, uint8_t *valid_mask, uint8_t *point_valid_mask,
                          float *curvature, uint32_t *planar_indices, uint8_t *planar_keep,
                          int32_t *closest_prev, int32_t *closest_next, size_t *n_planar_picks,
                          uint32_t *point_indices, size_t *n_point_picks);

/* ---- raw sensor clouds: organisation on the device ---------------------- */

/* A driver's point cloud (unordered records, missing returns absent) is turned into the
 * organised row-major scan the extraction reads, on the device (rule R8, DESIGN.md §4):
 *   - records that are dropped, counted by reason: a non-finite coordinate, the exact zero point,
 *     time outside [0, scan_period), row or column out of range;
 *   - row: the record's ring / row field, or the nearest beam of an elevation table (sign tests
 *     z cos(mu) - rho sin(mu) against the midpoints mu of adjacent beams);
 *   - column: the record's col field, floor(t * cols / scan_period) in f64 (clamped to cols - 1),
 *     or the nearest column centre origin + dir * 2 pi c / cols (half-plane sign tests
 *     y cos(phi) - x sin(phi) against a boundary table built once, no atan2);
 *   - collisions: the nearest point wins, key (f32 bits of |p|^2) << 32 | record index, ties to
 *     the lower index; pixels nobody claimed are (0, 0, 0, 0).
 * x, y, z in f64 are converted with (float)v. */
#define FORMGPU_CLOUD_ABSENT (-1)
#define FORMGPU_FIELD_F32 0
#define FORMGPU_FIELD_F64 1
#define FORMGPU_FIELD_U8 2
#define FORMGPU_FIELD_U16 3
#define FORMGPU_FIELD_U32 4
#define FORMGPU_FIELD_U32_NS 5 /* time: u32 nanoseconds since scan start */

#define FORMGPU_ROW_FROM_FIELD 0
#define FORMGPU_ROW_FROM_ELEVATION 1
#define FORMGPU_COL_FROM_FIELD 0
#define FORMGPU_COL_FROM_TIME 1
#define FORMGPU_COL_FROM_AZIMUTH 2

typedef struct formgpu_cloud_format {
  uint32_t stride;     /* bytes per record                                         */
  int32_t off_x, off_y, off_z; /* byte offsets inside a record                      */
  int32_t xyz_type;    /* FORMGPU_FIELD_F32 or _F64                                 */
  int32_t off_row;     /* ring / row field, FORMGPU_CLOUD_ABSENT if none            */
  int32_t row_type;    /* _U8, _U16 or _U32                                         */
  int32_t off_col;     /* column field, or FORMGPU_CLOUD_ABSENT                     */
  int32_t col_type;    /* _U16 or _U32                                              */
  int32_t off_time;    /* time since scan start, or FORMGPU_CLOUD_ABSENT            */
  int32_t time_type;   /* _F32 / _F64 seconds or _U32_NS                            */
  int32_t row_source;  /* FORMGPU_ROW_FROM_*                                        */
  int32_t col_source;  /* FORMGPU_COL_FROM_*                                        */
  int32_t azimuth_dir; /* +1: columns advance counter-clockwise, -1: clockwise      */
  double scan_period;  /* seconds, > 0                                              */
  double azimuth_origin; /* radians: centre of column 0                            */
  const double *beam_elevations; /* [num_rows] radians, strictly monotonic, |e| < pi/2
                                    (ROW_FROM_ELEVATION; copied by set_cloud_format) */
  uint64_t max_records; /* capacity: records of the largest cloud, < 2^32            */
} formgpu_cloud_format;

/* Outcome of the last organisation of a context: every record lands in exactly one of
 * placed / dropped_*; pixels = pixels that received a point (placed - pixels lost a collision). */
typedef struct formgpu_cloud_stats {
  uint64_t records;
  uint64_t placed;
  uint64_t pixels;
  uint64_t dropped_nonfinite;
  uint64_t dropped_zero;
  uint64_t dropped_time;
  uint64_t dropped_row;
  uint64_t dropped_col;
} formgpu_cloud_stats;

/* The checks of formgpu_set_cloud_format for a rows x cols scan, without a context or GPU.
 * Returns FORMGPU_OK or the error code, with a message in msg (may be NULL). */
int formgpu_cloud_format_check(const formgpu_cloud_format *fmt, int rows, int cols, char *msg, size_t msg_cap);

/* Give the context a cloud format (checked before any CUDA call).  Allocates, once, the record
 * staging buffer (max_records * stride bytes), the per-pixel keys and the boundary tables, so
 * nothing is allocated per scan.  Also valid on formgpu_batch_ctx(b, i).  A later call replaces
 * the format. */
int formgpu_set_cloud_format(formgpu_ctx *ctx, const formgpu_cloud_format *fmt);

/* Organise n records (HOST memory) into the context's scan buffer and, when out is not NULL,
 * copy the rows*cols scan to it; stats may be NULL.  FORMGPU_ERR_STATE without a format,
 * FORMGPU_ERR_CAPACITY when n > max_records.  The context's current scan (its keypoints and
 * matches) is unchanged; formgpu_extract_debug needs a new formgpu_extract afterwards. */
int formgpu_organize(formgpu_ctx *ctx, const void *records, size_t n, formgpu_point4f *out,
                     formgpu_cloud_stats *stats);

/* formgpu_extract with a raw cloud as input: organise, then extract the organised scan.  Same
 * outputs and "current scan" semantics. */
int formgpu_extract_cloud(formgpu_ctx *ctx, const void *records, size_t n, uint64_t scan_idx,
                          formgpu_planar_feat *planar_out, size_t planar_cap, size_t *n_planar,
                          formgpu_point_feat *point_out, size_t point_cap, size_t *n_point);

/* Counters of the context's last organisation (formgpu_organize, formgpu_extract_cloud or a
 * FORMGPU_REQ_CLOUD request of a batch). */
int formgpu_cloud_stats_last(const formgpu_ctx *ctx, formgpu_cloud_stats *stats);

/* ---- stage 2: reparative map + association ------------------------------ */

/* KeypointMap::to_voxel_map for both keypoint types (form/mapping/map.hpp:137,
 * map.tpp:128-146; called once per scan at form/form.cpp:61-65): transform all
 * stored keypoints by their scan's pose and rebuild the voxel hash with voxel
 * width max_dist_matching.  Every stored scan must appear in `poses`. */
int formgpu_map_rebuild(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses);

/* Matcher::match<0> + match<1> (form/optimization/matcher.hpp:67-112,
 * form/form.cpp:75-79) for the current scan at pose_k.  Replaces the current
 * scan's correspondences; writes one entry per non-empty pair. */
int formgpu_associate(formgpu_ctx *ctx, const formgpu_pose *pose_k,
                      formgpu_pair_count *counts_out, size_t counts_cap, size_t *n_counts);

/* formgpu_associate followed by formgpu_linearize of every non-empty pair (i, current
 * scan) at `poses` - what one ICP iteration does first (form/form.cpp:75-82: match, then
 * optimize(true) whose first step linearises exactly those FeatureFactors,
 * form/optimization/constraints.cpp:259-265) - as ONE device round trip: the
 * linearisation is queued behind the association and reads its ranges on the device.
 * The current scan is associated at its pose in `poses` (which must contain it).
 * out91 receives 91 doubles per entry of counts_out, in the same order; it must hold
 * 91 * counts_cap doubles. */
int formgpu_associate_linearize(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses,
                                formgpu_pair_count *counts_out, size_t counts_cap, size_t *n_counts,
                                double *out91);

/* Matcher::get_matches (matcher.hpp:114): per-keypoint results of the last
 * association; type 0 = planar, 1 = point. */
int formgpu_get_matches(formgpu_ctx *ctx, int type, formgpu_match *out, size_t cap, size_t *n);

/* KeypointMap::insert_matches for both types (form/mapping/map.hpp:142,
 * map.tpp:148-165; form/form.cpp:99-101). */
int formgpu_commit_scan(formgpu_ctx *ctx, size_t *n_planar_added, size_t *n_point_added);

/* KeypointMap::remove (map.hpp:130-133) + erase of all pairs touching the
 * scans (form/optimization/constraints.cpp:186-194). */
int formgpu_remove_scans(formgpu_ctx *ctx, const uint64_t *scans, size_t n);

/* Stored (scan-local) keypoints of one scan; type 0 planar -> formgpu_planar_feat,
 * 1 point -> formgpu_point_feat.  out may be NULL to query the count. */
int formgpu_get_keypoints(formgpu_ctx *ctx, int type, uint64_t scan, void *out, size_t cap,
                          size_t *n);

/* FORM::map() (python/bindings.cpp:96-119): all stored keypoints in the world
 * frame, ordered by (scan, k). */
int formgpu_world_keypoints(formgpu_ctx *ctx, const formgpu_scan_pose *poses, size_t n_poses,
                            formgpu_planar_feat *planar_out, size_t planar_cap, size_t *n_planar,
                            formgpu_point_feat *point_out, size_t point_cap, size_t *n_point);

/* ---- stage 3: linearisation --------------------------------------------- */

/* DenseFactor::linearize of FeatureFactor(X(i), X(j)) for every listed pair
 * (form/optimization/gtsam.hpp:67-86, form/feature/factor.cpp:30-186) under
 * the pair-set policy of ConstraintManager::get_graph
 * (form/optimization/constraints.cpp:252-308).  out91 receives 91 doubles per
 * pair: the row-major packed upper triangle of
 *   [[A^T A, A^T b], [b^T A, b^T b]],  A = [J_i J_j] / sigma,  b = -r / sigma,
 * variable order (xi_i, xi_j), tangent order [omega, v].  Pairs without
 * correspondences yield zeros. */
int formgpu_linearize(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                      const formgpu_scan_pose *poses, size_t n_poses, double *out91);

/* NoiseModelFactor::error = 0.5 |r / sigma|^2 per pair (LM trial steps). */
int formgpu_error(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                  const formgpu_scan_pose *poses, size_t n_poses, double *out);

/* ---- point-sharded mode: one dense sequence over several GPUs ------------ */

/* For very dense scans the correspondences of ONE sequence can be linearised by several
 * GPUs (SURVEY 8e, BASELINE.json configs[4]): every rank runs stages 1-2 on its own replica
 * of the context (same inputs, bit-identical state) and formgpu_set_shard(rank, world)
 * makes its stage-3 calls reduce only the rank-th of `world` contiguous shares of every
 * pair's correspondences.  The 13x13 blocks are additive in the correspondences, so the
 * block of a pair is the SUM of the ranks' blocks: the caller all-reduces 91 * n_pairs
 * doubles (errors: n_pairs).  rank = 0, world = 1 (the default) switches the mode off. */
int formgpu_set_shard(formgpu_ctx *ctx, int rank, int world);

/* formgpu_linearize / formgpu_error with the result left in DEVICE memory (91 doubles
 * per pair / one per pair, zeros for pairs without correspondences) and no wait: the work
 * is queued on the context's stream, so a collective queued on the same stream (NCCL
 * all-reduce over NVLink) consumes the blocks without a host round trip. */
int formgpu_linearize_device(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                             const formgpu_scan_pose *poses, size_t n_poses, double *out91_dev);
int formgpu_error_device(formgpu_ctx *ctx, const formgpu_pair *pairs, size_t n_pairs,
                         const formgpu_scan_pose *poses, size_t n_poses, double *out_dev);

/* Point-sharded mode over NCCL: the same dense sequence on `world` GPUs of one node, one process
 * (or thread) and one context per GPU, every context fed the same calls with the same inputs.
 * formgpu_comm_unique_id (any one rank; 128 bytes, to be handed to the other ranks by the caller's
 * own means) + formgpu_comm_init (every rank, collectively) attach a communicator to the context.
 * From then on
 *   - formgpu_map_rebuild builds, on rank r, the map of the scans whose window slot is congruent
 *     to r only (the map - 1.5 M points rebuilt every scan in configs[4] - is what is expensive);
 *     formgpu_associate / _associate_linearize search that sub-map for ALL keypoints, ONE in-place
 *     ncclAllGather (planar and point candidates together) and a combine kernel that applies the
 *     full rule-R5 key across the ranks return all matches to every rank, so pair counts,
 *     segments, formgpu_get_matches and formgpu_commit_scan stay replicated and bit-identical to
 *     a single GPU;
 *   - the pair moments (stage 3) are accumulated over this rank's share of every pair, and
 *     formgpu_linearize / formgpu_error / the blocks of formgpu_associate_linearize are the
 *     evaluation of those partial moments followed by ONE ncclAllReduce(sum, f64, 91 * n_pairs)
 *     on the context's stream - the only stage-3 bytes that cross NVLink.  Every rank receives
 *     the full result (equal across ranks; differs from one GPU by fp64 summation order only).
 * Extraction, segments and the commit are replicated.  NCCL is loaded at run time (libnccl.so.2);
 * FORMGPU_ERR_UNSUPPORTED when it is not there.  Contexts of a batch cannot be sharded. */
int formgpu_comm_unique_id(void *id128);
int formgpu_comm_init(formgpu_ctx *ctx, const void *id128, int rank, int world);
int formgpu_comm_destroy(formgpu_ctx *ctx);

/* ---- batched submit: many independent sequences per launch --------------- */
#define FORMGPU_KG_COUNT 12 /* kernel groups, listed under "instrumentation" below */

/* One sequence alone cannot fill a B200 (a per-scan request is < 1 MB and every call is a
 * dependent round trip).  A formgpu_batch owns `n_sequences` contexts - one per
 * independent sequence, i.e. one per form::Estimator - that share one CUDA stream.
 * formgpu_batch_submit executes at most ONE pending call per sequence; calls of the same
 * kind are executed by ONE launch per kernel (the grid's z / y index selects the
 * sequence).  The arithmetic is that of the single-sequence entry points, so results are
 * bit-identical to n separate contexts.  The call returns when every request has
 * completed; request i's status lands in reqs[i].status and the first failure is the
 * return value (the other requests still run).
 *
 * A request names the single-sequence call it stands for (the reference interfaces are
 * the ones cited at those entry points) and uses the fields that call takes:
 *   FORMGPU_OP_EXTRACT      formgpu_extract / formgpu_extract_device (flag
 *                           FORMGPU_REQ_SCAN_ON_DEVICE): scan, n_points, scan_idx,
 *                           planar_out/cap, point_out/cap -> n_planar, n_point
 *   FORMGPU_OP_MAP_REBUILD  formgpu_map_rebuild: poses, n_poses
 *   FORMGPU_OP_ASSOCIATE    formgpu_associate: pose_k, counts_out/cap -> n_counts
 *   FORMGPU_OP_ASSOC_LIN    formgpu_associate_linearize: poses, n_poses, counts_out/cap,
 *                           out (91 doubles per count) -> n_counts
 *   FORMGPU_OP_LINEARIZE    formgpu_linearize: pairs, n_pairs, poses, n_poses, out
 *   FORMGPU_OP_ERROR        formgpu_error: pairs, n_pairs, poses, n_poses, out
 *   FORMGPU_OP_COMMIT       formgpu_commit_scan -> n_planar, n_point (keypoints added)
 *   FORMGPU_OP_REMOVE       formgpu_remove_scans: scans, n_scans */
#define FORMGPU_OP_EXTRACT 0
#define FORMGPU_OP_MAP_REBUILD 1
#define FORMGPU_OP_ASSOCIATE 2
#define FORMGPU_OP_ASSOC_LIN 3
#define FORMGPU_OP_LINEARIZE 4
#define FORMGPU_OP_ERROR 5
#define FORMGPU_OP_COMMIT 6
#define FORMGPU_OP_REMOVE 7
#define FORMGPU_OP_COUNT 8

#define FORMGPU_REQ_SCAN_ON_DEVICE 1u /* `scan` is a device pointer; no keypoints copied back */
/* FORMGPU_OP_EXTRACT on a raw cloud (formgpu_extract_cloud): `scan` points at n_points records of
 * the sequence's cloud format.  The clouds of a submission are organised by one launch per kernel
 * ahead of the extraction.  With FORMGPU_REQ_SCAN_ON_DEVICE the records are in device memory. */
#define FORMGPU_REQ_CLOUD 2u

typedef struct formgpu_request {
  uint32_t sequence; /* index of the sequence inside the batch */
  uint32_t op;       /* FORMGPU_OP_* */
  uint32_t flags;    /* FORMGPU_REQ_* */
  int32_t status;    /* out: FORMGPU_OK or the error of this request */
  /* stage 1 */
  const formgpu_point4f *scan;
  size_t n_points;
  uint64_t scan_idx;
  formgpu_planar_feat *planar_out;
  size_t planar_cap;
  size_t n_planar; /* out */
  formgpu_point_feat *point_out;
  size_t point_cap;
  size_t n_point; /* out */
  /* stage 2 / 3 */
  const formgpu_scan_pose *poses;
  size_t n_poses;
  const formgpu_pose *pose_k;
  const formgpu_pair *pairs;
  size_t n_pairs;
  formgpu_pair_count *counts_out;
  size_t counts_cap;
  size_t n_counts; /* out */
  double *out;     /* 91 doubles per pair (blocks) or 1 per pair (errors) */
  const uint64_t *scans;
  size_t n_scans;
} formgpu_request;

typedef struct formgpu_batch formgpu_batch;

/* `stream`: cudaStream_t shared by all sequences of the batch, or NULL for a private one.
 * Every sequence is configured by `p`: formgpu_batch_create_mixed with p repeated. */
int formgpu_batch_create(const formgpu_params *p, int device, void *stream, size_t n_sequences,
                         formgpu_batch **out);
/* A batch whose sequence i is configured by params[i] (n_sequences entries): sensors of different
 * shapes and parameter variants share one launch per kernel.  Every field of formgpu_params may
 * differ from sequence to sequence.  Shared by the whole batch: `device` and `stream`.  The contexts
 * of a batch always evaluate linearisations and errors from their pair-moment caches
 * (FORMGPU_STREAM_LINEARIZE applies to single contexts only).  Every entry goes
 * through formgpu_create's parameter checks before any CUDA call; when one fails,
 * formgpu_batch_last_error(NULL) names the index of its sequence. */
int formgpu_batch_create_mixed(const formgpu_params *params, int device, void *stream, size_t n_sequences,
                               formgpu_batch **out);
void formgpu_batch_destroy(formgpu_batch *b);
size_t formgpu_batch_size(const formgpu_batch *b);
/* The context of sequence i, for the calls that are not batched (formgpu_get_matches,
 * formgpu_get_keypoints, formgpu_world_keypoints, ...); it runs on the batch's stream. */
formgpu_ctx *formgpu_batch_ctx(formgpu_batch *b, size_t i);
int formgpu_batch_submit(formgpu_batch *b, formgpu_request *reqs, size_t n);
/* The two halves of formgpu_batch_submit, for a host thread that drives SEVERAL batches (one
 * stream each) on one GPU: formgpu_batch_submit_async validates the requests, uploads their
 * arguments and queues every kernel, then returns; formgpu_batch_wait blocks until the results
 * have arrived and fills the output fields of the SAME reqs array (which, with every buffer it
 * points to, must stay alive and untouched in between).  One submission may be in flight per
 * batch (FORMGPU_ERR_STATE otherwise).  A thread that submits to each of its batches before it
 * waits for the first keeps as many rounds in flight as it owns batches.  If the build half fails
 * (bad request list, CUDA error) nothing stays in flight, and every request that was not
 * individually rejected carries the returned code in `status`.
 * formgpu_batch_done: 1 when formgpu_batch_wait would not block (or nothing is in flight), 0
 * while the submission is still running, < 0 (= -status code) on error. */
int formgpu_batch_submit_async(formgpu_batch *b, formgpu_request *reqs, size_t n);
int formgpu_batch_wait(formgpu_batch *b);
int formgpu_batch_done(formgpu_batch *b);
/* Upload ahead: `scan` (host memory, page-locked for a truly asynchronous copy) is the scan that
 * `sequence` will pass to its next FORMGPU_OP_EXTRACT - known early when recorded logs are
 * reprocessed, or when a driver thread receives the next revolution while the current one is being
 * registered (the reference copies nothing: extract() reads the caller's std::vector in place,
 * /root/reference/form/feature/extraction.tpp:29-45).  The copy starts now on the batch's copy
 * stream into the sequence's second scan buffer; the EXTRACT request that names the same pointer
 * finds its input on the device.  The scan must stay unmodified until that request has completed;
 * a different pointer in the request simply discards the prefetched copy.  Call it between
 * formgpu_batch_wait and the next submission of the batch. */
int formgpu_batch_prefetch_scan(formgpu_batch *b, size_t sequence, const formgpu_point4f *scan, size_t n_points);
/* The same for a raw cloud: the n records go ahead into the sequence's record staging buffer, and
 * the FORMGPU_REQ_CLOUD request that names the same pointer and count does not upload them again. */
int formgpu_batch_prefetch_cloud(formgpu_batch *b, size_t sequence, const void *records, size_t n);
const char *formgpu_batch_last_error(const formgpu_batch *b);
/* As formgpu_profile_enable / _read / formgpu_launch_count, for the batched launches. */
int formgpu_batch_profile_enable(formgpu_batch *b, int on);
int formgpu_batch_profile_read(formgpu_batch *b, double ms[FORMGPU_KG_COUNT],
                               uint64_t launches[FORMGPU_KG_COUNT]);
uint64_t formgpu_batch_launch_count(const formgpu_batch *b);

/* ---- instrumentation ---------------------------------------------------- */

/* Kernel groups of the hot path (one or a few kernels each). */
#define FORMGPU_KG_EXTRACT_SELECT 0  /* masks, curvature, sector sort, greedy picks */
#define FORMGPU_KG_EXTRACT_NORMALS 1 /* closest-row search + PCA normals            */
#define FORMGPU_KG_EXTRACT_PACK 2    /* keypoint compaction                         */
#define FORMGPU_KG_MAP_BUILD 3       /* transform + hash insert + alloc + scatter   */
#define FORMGPU_KG_ASSOC_NN 4        /* warp-cooperative voxel-hash NN              */
#define FORMGPU_KG_SEGMENT 5         /* correspondence segment (hist, scan, scatter)*/
#define FORMGPU_KG_LIN_CHUNK 6       /* streaming residual/Jacobian reduction       */
#define FORMGPU_KG_LIN_FINALIZE 7    /* per-pair 13x13 expansion                    */
#define FORMGPU_KG_ERR_CHUNK 8       /* streaming residual-only reduction           */
#define FORMGPU_KG_ERR_FINALIZE 9
#define FORMGPU_KG_COMMIT 10         /* novel keypoint append                       */
#define FORMGPU_KG_EXPORT 11         /* world-frame keypoint export                 */

/* When enabled every kernel group is bracketed by CUDA events on the context's
 * stream (the calls then synchronise once more at their end).
 * formgpu_profile_read returns the accumulated device milliseconds and launch
 * counts per group since the last read, then resets them.  Launches are counted
 * whether or not timing is enabled. */
int formgpu_profile_enable(formgpu_ctx *ctx, int on);
int formgpu_profile_read(formgpu_ctx *ctx, double ms[FORMGPU_KG_COUNT],
                         uint64_t launches[FORMGPU_KG_COUNT]);

/* Total kernels launched by this context since creation. */
uint64_t formgpu_launch_count(const formgpu_ctx *ctx);

/* Block the caller until all queued work of the context has finished. */
int formgpu_synchronize(formgpu_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* FORMGPU_H */
