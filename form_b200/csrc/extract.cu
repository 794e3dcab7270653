// Stage 1 on sm_100a: scan-line feature extraction.
//
// Replaces FeatureExtractor::extract (/root/reference/form/feature/
// extraction.tpp:29-132) and its helpers (:136-448).  Compiled with
// -fmad=false: every float/double operation below is evaluated in the same
// order, without contraction, as the CPU oracle (SURVEY A.2), so validity
// masks, curvature bits, feature indices, closest indices AND normals come out
// bit-identical.
//
// Mapping to the hardware: one CTA per scan row (rows are independent,
// extraction.tpp:44-68; suppression never crosses rows), grid.y = scan in the
// batch.  The 16-32 KB row is staged once in shared memory with coalesced
// 128-bit loads and every later access (11-tap curvature window, O(n^2) rank
// sort inside a sector, greedy walks) hits shared memory only.  The greedy
// selections are sequential by definition; they run on warp 0, 32 sorted
// candidates per step: candidates are fetched in parallel, conflicts inside
// the group are resolved with shuffles, and the row's "used" bitmask lives in
// shared memory.
#include "ctx.hpp"
#include "kernels.hpp"

#include <algorithm>
#include <cfloat>
#include <cstdlib>
#include <mutex>

namespace formgpu {

namespace {

__device__ __forceinline__ float diff_sqnorm4(const float4 a, const float4 b) {
  // (d0^2 + d2^2) + (d1^2 + d3^2): Eigen's 4-lane packet reduction (A.2)
  const float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z, d3 = a.w - b.w;
  return (d0 * d0 + d2 * d2) + (d1 * d1 + d3 * d3);
}

__device__ __forceinline__ bool get_bit(const uint32_t *m, int c) {
  return (m[c >> 5] >> (c & 31)) & 1u;
}

// clear bits [lo, hi] (inclusive) of a shared-memory bitmask, hi - lo < 32
__device__ __forceinline__ void clear_bits(uint32_t *m, int lo, int hi) {
  const int wl = lo >> 5, wh = hi >> 5;
  if (wl == wh) {
    const uint32_t width = (uint32_t)(hi - lo + 1);
    const uint32_t mask = (width >= 32 ? 0xffffffffu : ((1u << width) - 1u)) << (lo & 31);
    atomicAnd(&m[wl], ~mask);
  } else {
    atomicAnd(&m[wl], ~(0xffffffffu << (lo & 31)));
    atomicAnd(&m[wh], ~(0xffffffffu >> (31 - (hi & 31))));
  }
}

// Resolve the sequential "take it if still unused, then suppress +-(np-1)"
// rule inside a group of 32 candidates ordered by lane: lane l survives iff it
// is a candidate and no surviving earlier lane lies within np-1 columns.
// Each lane first collects the set of earlier candidate lanes it conflicts with (32
// independent shuffles); the survivors are then found by a short fixed-point iteration
// on ballots - the lowest undecided lane is always decidable, and in practice two or
// three rounds settle the whole group - instead of a 31-step dependent shuffle chain.
__device__ __forceinline__ bool resolve_group(bool cand, int col, int np, int lane) {
  const unsigned cand_bits = __ballot_sync(0xffffffffu, cand);
  if (cand_bits == 0) return false;
  unsigned conf = 0;
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const int ck = __shfl_sync(0xffffffffu, col, k);
    const int d = col - ck;
    if (d < np && d > -np) conf |= 1u << k;
  }
  conf &= cand_bits & ((1u << lane) - 1u); // earlier candidate lanes only
  unsigned undecided = cand_bits, alive_bits = 0;
  while (undecided) {
    const bool me = (undecided >> lane) & 1u;
    const bool kill = me && (conf & alive_bits);
    const bool ok = me && !kill && !(conf & undecided);
    const unsigned killb = __ballot_sync(0xffffffffu, kill);
    const unsigned okb = __ballot_sync(0xffffffffu, ok);
    alive_bits |= okb;
    undecided &= ~(killb | okb);
  }
  return (alive_bits >> lane) & 1u;
}

} // namespace

// ---------------------------------------------------------------------------
// K1: validity masks, curvature, per-sector sort, greedy planar + point picks
// ---------------------------------------------------------------------------
namespace {

// Batched launches (several sequences' scans in one grid) read the per-item argument
// block from a device array: one cooperative copy into shared memory per CTA.
__device__ __forceinline__ void load_item_args(ExtractArgs &dst, const ExtractArgs *src) {
  static_assert(sizeof(ExtractArgs) % 8 == 0, "ExtractArgs is copied in 8-byte words");
  for (int i = threadIdx.x; i < (int)(sizeof(ExtractArgs) / 8); i += blockDim.x)
    reinterpret_cast<unsigned long long *>(&dst)[i] = reinterpret_cast<const unsigned long long *>(src)[i];
  __syncthreads();
}

constexpr int kMaxSectors = kExtractMaxSectors;

// extract_planar (extraction.tpp:332-358) on ONE sector: 32 sorted candidates per step.  `mask` is
// the used-mask the walk reads and suppresses in (the row's shared mask, or a private copy); the
// picks go to out[0..], the return value is their number.  Called by all lanes of one warp.
__device__ __forceinline__ int planar_walk_sector(const ExtractArgs &a, const uint32_t *keys, const uint16_t *sorted,
                                                  uint32_t *mask, int s, int pps, int S, int cols, int np, int lane,
                                                  uint16_t *out) {
  const unsigned lt_mask = (1u << lane) - 1u;
  const int start = s * pps;
  const int len = ((s == S - 1) ? cols : start + pps) - start;
  int count = 0;
  bool done = false;
  for (int base = 0; base < len && !done; base += 32) {
    const int i = base + lane;
    const bool in = i < len;
    const int col = in ? (int)sorted[start + i] : 0;
    const float curv = in ? __uint_as_float(keys[col]) : FLT_MAX;
    const bool below = in && ((double)curv < a.planar_threshold);
    const bool cand = below && get_bit(mask, col);
    const bool alive = resolve_group(cand, col, np, lane);
    const unsigned sel = __ballot_sync(0xffffffffu, alive);
    const int rank = __popc(sel & lt_mask);
    // visited iff the count after all earlier visits is still <= cap (:354 '>')
    const bool accept = alive && (count + rank <= a.planar_per_sector);
    if (accept) {
      out[count + rank] = (uint16_t)col;
      clear_bits(mask, col - (np - 1), col + (np - 1));
    }
    count += __popc(__ballot_sync(0xffffffffu, accept));
    if (count > a.planar_per_sector) done = true;
    // sorted ascending: once one in-range lane is >= threshold nothing later qualifies
    if (__ballot_sync(0xffffffffu, below) != __ballot_sync(0xffffffffu, in)) done = true;
    __syncwarp();
  }
  return count;
}

// extract_point (extraction.tpp:360-399) on ONE sector; `mask` as above, `ulist_base` = the row's
// scratch list (the sector uses its own columns' slice of it).  Called by all lanes of one warp.
__device__ __forceinline__ int point_walk_sector(const ExtractArgs &a, uint32_t *mask, uint16_t *ulist_base, int s,
                                                 int pps, int S, int cols, int np, int pfps, int lane, uint16_t *out) {
  const unsigned lt_mask = (1u << lane) - 1u;
  const int start = s * pps;
  const int end = (s == S - 1) ? cols : start + pps;
  uint16_t *ulist = ulist_base + start;
  // unused_points (:371-376): ascending list of still-valid columns
  int U = 0;
  for (int base = start; base < end; base += 32) {
    const int c = base + lane;
    const bool bit = c < end && get_bit(mask, c);
    const unsigned bal = __ballot_sync(0xffffffffu, bit);
    if (bit) ulist[U + __popc(bal & lt_mask)] = (uint16_t)c;
    U += __popc(bal);
  }
  __syncwarp();
  const int factor = 1 + U / pfps; // :379
  // The reference visits u = offset + m * factor for offset = 0 .. factor-1 (outer) and
  // m = 0, 1, .. (inner), leaving the inner loop once count > pfps (:394-396).  Equivalently,
  // in that (offset, m) order: the first element of every pass is ALWAYS visited, a later
  // element (m > 0) is visited iff the running count is still <= pfps.  A pass holds at most
  // ceil(U / factor) <= pfps + 1 elements, so stepping pass by pass would keep 3-4 lanes of
  // the warp busy; instead 32 consecutive elements of the whole visiting sequence (several
  // passes) are resolved per step.  Pass `o` has n_full + 1 elements if o < rem, else n_full.
  const int n_full = U / factor, rem = U - n_full * factor;
  const int split = rem * (n_full + 1); // sequence index of the first element of pass `rem`
  auto pass_of = [&](int t, int &o, int &m) {
    if (t < split) {
      o = t / (n_full + 1);
      m = t - o * (n_full + 1);
    } else {
      const int t2 = t - split, d = t2 / n_full; // n_full > 0 whenever such a t exists
      o = rem + d;
      m = t2 - d * n_full;
    }
  };
  int count = 0;
  int offset = factor; // first pass the strided phase has not touched when it stops
  for (int base = 0; base < U && count <= pfps; base += 32) {
    const int t = base + lane;
    const bool in = t < U;
    int o = 0, m = 0;
    if (in) pass_of(t, o, m);
    const int col = in ? (int)ulist[o + m * factor] : 0;
    const bool cand = in && get_bit(mask, col);
    bool alive = resolve_group(cand, col, np, lane);
    unsigned sel = __ballot_sync(0xffffffffu, alive);
    // lanes whose count-before already exceeds pfps (a suffix of the group): their m > 0
    // candidates are not visited and must not suppress anything - resolve again without them
    // (the outcome of the lanes before the suffix does not depend on later lanes)
    const unsigned over_bits = __ballot_sync(0xffffffffu, count + __popc(sel & lt_mask) > pfps);
    if (over_bits) {
      const int first_over = __ffs(over_bits) - 1;
      const bool dropped = cand && m > 0 && lane >= first_over;
      if (__ballot_sync(0xffffffffu, dropped)) {
        alive = resolve_group(cand && !dropped, col, np, lane);
        sel = __ballot_sync(0xffffffffu, alive);
      }
    }
    if (alive) {
      out[count + __popc(sel & lt_mask)] = (uint16_t)col;
      clear_bits(mask, col - (np - 1), col + (np - 1));
    }
    count += __popc(sel);
    if (count > pfps) { // only the first element of every later pass is still visited
      int o_last, m_last;
      pass_of(min(base + 31, U - 1), o_last, m_last);
      offset = o_last + 1;
    }
    __syncwarp();
  }
  // Phase B: count > pfps, so every remaining pass visits only u = offset
  for (int base = offset; base < factor; base += 32) {
    const int o = base + lane;
    const bool in = o < factor && o < U;
    if (__ballot_sync(0xffffffffu, in) == 0) break;
    const int col = in ? (int)ulist[o] : 0;
    const bool cand = in && get_bit(mask, col);
    const bool alive = resolve_group(cand, col, np, lane);
    const unsigned sel = __ballot_sync(0xffffffffu, alive);
    const int rank = __popc(sel & lt_mask);
    if (alive) {
      out[count + rank] = (uint16_t)col;
      clear_bits(mask, col - (np - 1), col + (np - 1));
    }
    count += __popc(sel);
    __syncwarp();
  }
  return count;
}

__device__ __forceinline__ void extract_select_body(const ExtractArgs &a, const int row, const int b) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int cols = a.cols, words = a.words, np = a.np;
  float4 *pts = reinterpret_cast<float4 *>(smem_raw);
  // sort key = curvature bits (non-negative floats order like unsigned ints); the column
  // itself is the tie-break of rule R1, so 32 bits per point are enough
  uint32_t *keys = reinterpret_cast<uint32_t *>(pts + cols);
  uint16_t *sorted = reinterpret_cast<uint16_t *>(keys + a.cols_pad);
  uint16_t *ulist = sorted + a.cols_pad;
  uint32_t *m_range = reinterpret_cast<uint32_t *>(ulist + a.cols_pad);
  uint32_t *m_valid = m_range + words;
  uint32_t *m_pvalid = m_valid + words;
  uint32_t *m_used = m_pvalid + words;

  const int tid = threadIdx.x, lane = tid & 31;
  const size_t row_base = ((size_t)b * a.rows + row) * cols;
  const float4 *g = a.scan + row_base;

  for (int c = tid; c < cols; c += blockDim.x) pts[c] = __ldg(&g[c]);
  __syncthreads();

  // range test (extraction.tpp:167-168): float norm promoted to double
  for (int c0 = 0; c0 < words * 32; c0 += blockDim.x) {
    const int c = c0 + tid;
    bool ok = false;
    if (c < cols) {
      const float4 p = pts[c];
      const double r2 = (double)((p.x * p.x + p.z * p.z) + (p.y * p.y + p.w * p.w));
      ok = !(r2 < a.min_norm2 || r2 > a.max_norm2);
    }
    const unsigned bal = __ballot_sync(0xffffffffu, ok);
    if (lane == 0 && (c >> 5) < words) m_range[c >> 5] = bal;
  }
  __syncthreads();

  // validity masks (extraction.tpp:136-222) in closed form (SURVEY A.3-6):
  //   valid(c)  = !edge(c) && for all j in [c-np, c+np]: !edge(j) => range_ok(j)
  //   pvalid(c) = !edge(c) && range_ok(c)
  for (int c0 = 0; c0 < words * 32; c0 += blockDim.x) {
    const int c = c0 + tid;
    bool v = false, pv = false;
    if (c < cols && c >= np && c < cols - np) {
      pv = get_bit(m_range, c);
      v = true;
      const int lo = max(c - np, np), hi = min(c + np, cols - np - 1);
      for (int j = lo; j <= hi; ++j) v = v && get_bit(m_range, j);
    }
    const unsigned bv = __ballot_sync(0xffffffffu, v);
    const unsigned bp = __ballot_sync(0xffffffffu, pv);
    if (lane == 0 && (c >> 5) < words) {
      m_valid[c >> 5] = bv;
      m_used[c >> 5] = bv;
      m_pvalid[c >> 5] = bp;
      a.valid_bits[((size_t)b * a.rows + row) * words + (c >> 5)] = bv;
    }
  }
  __syncthreads();

  // bounding box of the VALID points of every 32-column chunk: lets the normals kernel
  // prune its exact adjacent-row search (find_closest only considers valid points)
  if (a.row_box) {
    const int warp = tid >> 5, nwarps = blockDim.x >> 5;
    for (int w = warp; w < words; w += nwarps) {
      const int c = w * 32 + lane;
      const bool v = c < cols && get_bit(m_valid, c);
      const float4 p = v ? pts[c] : make_float4(0.f, 0.f, 0.f, 0.f);
      float lo0 = v ? p.x : INFINITY, lo1 = v ? p.y : INFINITY, lo2 = v ? p.z : INFINITY;
      float hi0 = v ? p.x : -INFINITY, hi1 = v ? p.y : -INFINITY, hi2 = v ? p.z : -INFINITY;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        lo0 = fminf(lo0, __shfl_xor_sync(0xffffffffu, lo0, o));
        lo1 = fminf(lo1, __shfl_xor_sync(0xffffffffu, lo1, o));
        lo2 = fminf(lo2, __shfl_xor_sync(0xffffffffu, lo2, o));
        hi0 = fmaxf(hi0, __shfl_xor_sync(0xffffffffu, hi0, o));
        hi1 = fmaxf(hi1, __shfl_xor_sync(0xffffffffu, hi1, o));
        hi2 = fmaxf(hi2, __shfl_xor_sync(0xffffffffu, hi2, o));
      }
      if (lane == 0) {
        float4 *dst = a.row_box + (((size_t)b * a.rows + row) * words + w) * 2;
        dst[0] = make_float4(lo0, lo1, lo2, 0.f);
        dst[1] = make_float4(hi0, hi1, hi2, 0.f);
      }
    }
  }

  // curvature (extraction.tpp:226-261): double accumulation in the reference's
  // order, rounded to float; sort key = (float bits << 32) | column (rule R1)
  for (int c = tid; c < cols; c += blockDim.x) {
    float cf = FLT_MAX;
    if (get_bit(m_valid, c)) {
      const double k = -(2.0 * (double)np);
      const float4 p = pts[c];
      double dx = k * (double)p.x, dy = k * (double)p.y, dz = k * (double)p.z;
      for (int n = 1; n <= np; ++n) {
        const float4 pa = pts[c - n], pb = pts[c + n];
        dx = (dx + (double)pa.x) + (double)pb.x;
        dy = (dy + (double)pa.y) + (double)pb.y;
        dz = (dz + (double)pa.z) + (double)pb.z;
      }
      cf = (float)((dx * dx + dy * dy) + dz * dz);
    }
    keys[c] = __float_as_uint(cf);
    if (a.dbg_curv) a.dbg_curv[row_base + c] = cf;
    if (a.dbg_valid) {
      a.dbg_valid[row_base + c] = get_bit(m_valid, c);
      a.dbg_pvalid[row_base + c] = get_bit(m_pvalid, c);
    }
  }
  __syncthreads();

  // per-sector rank sort (std::sort at extraction.tpp:57-58 with rule R1)
  const int pps = a.pps, S = a.num_sectors;
  for (int c = tid; c < cols; c += blockDim.x) {
    const int s = min(c / pps, S - 1);
    const int start = s * pps;
    const int end = (s == S - 1) ? cols : start + pps;
    const uint32_t kc = keys[c];
    // rank under (key, column): columns before c count when <=, columns after c when <
    int rank = 0;
#pragma unroll 8
    for (int j = start; j < c; ++j) rank += keys[j] <= kc ? 1 : 0;
#pragma unroll 8
    for (int j = c + 1; j < end; ++j) rank += keys[j] < kc ? 1 : 0;
    sorted[start + rank] = (uint16_t)c;
  }
  __syncthreads();

  // ---- greedy walks.  The reference walks the sectors of a row one after the other on ONE mask
  // (extraction.tpp:44-68), so the walks are sequential by definition - but sectors interact only
  // through the np-1 columns at their boundaries: a pick near the end of sector s suppresses the
  // first columns of sector s+1.  So every warp walks a sector SPECULATIVELY on a private copy of
  // the mask, and warp 0 then validates the sectors in order on the shared mask:
  //   planar: a speculative result stands iff none of its picks has been suppressed by the
  //           sectors before it (then both walks take the same decisions candidate by candidate);
  //   point:  it stands iff the shared mask still equals the initial one on the sector's own
  //           columns (the list of unused points, and with it the pass structure, is built from
  //           exactly those bits);
  // a sector that fails is walked again on the shared mask, which then holds the true state
  // (CPU models of both rules against the reference's sequential form: tests/test_kernel_models.py).
  // The walk of one warp was 76 % of a row's latency (ncu, profiles/r04).
  const int warp = tid >> 5, nwarps = (int)blockDim.x >> 5;
  uint32_t *m_priv = m_used + words;            // [S][words] private masks
  uint32_t *m_pinit = m_priv + (size_t)S * words; // [words] point mask before any point pick
  uint16_t *spec_cols = reinterpret_cast<uint16_t *>(m_pinit + words); // [S][cap_spec]
  const int cap_spec = extract_spec_cap(a);
  __shared__ int s_spec_cnt[kMaxSectors];

  // ---- extract_planar (extraction.tpp:332-358) ----
  for (int s = warp; s < S; s += nwarps) {
    uint32_t *mask = m_priv + (size_t)s * words;
    for (int w = lane; w < words; w += 32) mask[w] = m_valid[w];
    __syncwarp();
    const int n = planar_walk_sector(a, keys, sorted, mask, s, pps, S, cols, np, lane, spec_cols + (size_t)s * cap_spec);
    if (lane == 0) s_spec_cnt[s] = n;
  }
  __syncthreads();
  uint16_t *out_pl = a.planar_cols + ((size_t)b * a.rows + row) * a.pr_cap;
  if (warp == 0) {
    int total = 0;
    for (int s = 0; s < S; ++s) {
      const int n = s_spec_cnt[s];
      const uint16_t *sc = spec_cols + (size_t)s * cap_spec;
      bool lost = false;
      for (int i = lane; i < n; i += 32) lost = lost || !get_bit(m_used, (int)sc[i]);
      int count = n;
      if (__ballot_sync(0xffffffffu, lost)) {
        count = planar_walk_sector(a, keys, sorted, m_used, s, pps, S, cols, np, lane, out_pl + total);
      } else {
        for (int i = lane; i < n; i += 32) {
          const int col = sc[i];
          out_pl[total + i] = (uint16_t)col;
          clear_bits(m_used, col - (np - 1), col + (np - 1));
        }
      }
      __syncwarp();
      total += count;
    }
    if (lane == 0) {
      a.planar_cnt[(size_t)b * a.rows + row] = total;
      a.keep_cnt[(size_t)b * a.rows + row] = 0; // accumulated by the normals kernel
    }
    // ---- point candidates (extraction.tpp:72-80): untouched by planar picks and
    // range-valid.  m_pvalid becomes the working mask of extract_point. ----
    for (int w = lane; w < words; w += 32) {
      const uint32_t v = ~(m_used[w] ^ m_valid[w]) & m_pvalid[w];
      m_pvalid[w] = v;
      m_pinit[w] = v;
    }
  }
  __syncthreads();

  // ---- extract_point (extraction.tpp:360-399) ----
  const int pfps = a.point_per_sector;
  uint16_t *out_pt = a.point_cols + ((size_t)b * a.rows + row) * a.qr_cap;
  if (pfps <= 0) {
    if (tid == 0) a.point_cnt[(size_t)b * a.rows + row] = 0;
    return;
  }
  for (int s = warp; s < S; s += nwarps) {
    uint32_t *mask = m_priv + (size_t)s * words;
    for (int w = lane; w < words; w += 32) mask[w] = m_pinit[w];
    __syncwarp();
    const int n = point_walk_sector(a, mask, ulist, s, pps, S, cols, np, pfps, lane, spec_cols + (size_t)s * cap_spec);
    if (lane == 0) s_spec_cnt[s] = n;
  }
  __syncthreads();
  if (warp != 0) return;
  int ptotal = 0;
  for (int s = 0; s < S; ++s) {
    const int start = s * pps;
    const int end = (s == S - 1) ? cols : start + pps;
    // does the shared mask still equal the initial one on the sector's own columns?
    bool differs = false;
    for (int w = (start >> 5) + lane; w <= ((end - 1) >> 5); w += 32) {
      uint32_t in = 0xffffffffu;
      if (w == (start >> 5)) in &= 0xffffffffu << (start & 31);
      if (w == ((end - 1) >> 5)) in &= 0xffffffffu >> (31 - ((end - 1) & 31));
      differs = differs || (((m_pvalid[w] ^ m_pinit[w]) & in) != 0u);
    }
    int count;
    if (__ballot_sync(0xffffffffu, differs)) {
      count = point_walk_sector(a, m_pvalid, ulist, s, pps, S, cols, np, pfps, lane, out_pt + ptotal);
    } else {
      count = s_spec_cnt[s];
      const uint16_t *sc = spec_cols + (size_t)s * cap_spec;
      for (int i = lane; i < count; i += 32) {
        const int col = sc[i];
        out_pt[ptotal + i] = (uint16_t)col;
        clear_bits(m_pvalid, col - (np - 1), col + (np - 1));
      }
    }
    __syncwarp();
    ptotal += count;
  }
  if (lane == 0) a.point_cnt[(size_t)b * a.rows + row] = ptotal;
}

} // namespace

__global__ void __launch_bounds__(512) extract_select_kernel(ExtractArgs a) {
  extract_select_body(a, blockIdx.x, blockIdx.y);
}

__global__ void __launch_bounds__(512) extract_select_batch_kernel(const ExtractArgs *items) {
  __shared__ ExtractArgs s_a;
  load_item_args(s_a, items + blockIdx.y);
  if ((int)blockIdx.x >= s_a.rows) return; // the grid covers the launch's largest scan
  extract_select_body(s_a, blockIdx.x, 0);
}

// ---------------------------------------------------------------------------
// K2: PCA normals of the planar picks (compute_normal, extraction.tpp:263-329)
// ---------------------------------------------------------------------------
namespace {

struct PickDesc {
  short c_prev, c_next; // closest column on the adjacent rows, -1 = none
  unsigned char n_plus, n_minus, pp, pm, np_, nm;
  unsigned char pad[2];
};

// find_neighbors (extraction.tpp:422-448): counts of consecutive in-radius
// neighbours in the + and - direction around column c of `rowp`.
__device__ __forceinline__ void neighbor_counts(const float4 *rowp, int c, int np, double r2,
                                                int lane, int &n_plus, int &n_minus) {
  bool flag = false;
  const float4 p = rowp[c];
  if (lane < np) flag = (double)diff_sqnorm4(rowp[c + lane + 1], p) < r2;
  else if (lane >= 16 && lane < 16 + np) flag = (double)diff_sqnorm4(rowp[c - (lane - 16) - 1], p) < r2;
  const unsigned bal = __ballot_sync(0xffffffffu, flag);
  n_plus = __ffs(~(bal & 0xffffu)) - 1;   // trailing ones = neighbours before the first miss
  n_minus = __ffs(~(bal >> 16)) - 1;
  if (n_plus > np) n_plus = np;
  if (n_minus > np) n_minus = np;
}

// find_closest (extraction.tpp:402-420), rule R2: arg-min (dist2, column) over the valid
// points of one row.  The reference scans the whole row for every pick; here the row's
// 32-column chunks carry the bounding box of their valid points (written by the select
// kernel).  The chunk at the pick's own azimuth is evaluated first (on an organised scan the
// closest point is nearly always there); any other chunk is evaluated only if its box can hold
// a point at least as close.  The pruning is exact: the float squared distance the
// reference computes differs from the true one by a few ulp, the box distance computed
// here likewise, and a chunk is skipped only when its bound exceeds the best so far by a
// 1e-5 relative margin - so every skipped point loses the (dist2, column) comparison.
__device__ __forceinline__ float box_dist2(const float4 lo, const float4 hi, const float4 p) {
  const float dx = fmaxf(fmaxf(lo.x - p.x, p.x - hi.x), 0.0f);
  const float dy = fmaxf(fmaxf(lo.y - p.y, p.y - hi.y), 0.0f);
  const float dz = fmaxf(fmaxf(lo.z - p.z, p.z - hi.z), 0.0f);
  return dx * dx + dy * dy + dz * dz; // +inf for an empty chunk (lo = +inf, hi = -inf)
}

__device__ __forceinline__ int closest_in_row_pruned(const float4 *rowp, const uint32_t *valid,
                                                     const float4 *box, const float4 p, int words,
                                                     int cols, int lane, int c_own) {
  float best = INFINITY;
  int bc = 0x7fffffff;
  auto eval = [&](int w) {
    const int c = w * 32 + lane;
    if (c < cols && ((valid[w] >> lane) & 1u)) {
      const float d2 = diff_sqnorm4(rowp[c], p);
      if (d2 < best || (d2 == best && c < bc)) {
        best = d2;
        bc = c;
      }
    }
  };
  auto warp_min = [](float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
  };
  // Seed: the chunk at the pick's own azimuth - on an organised scan the closest point of the
  // adjacent row is nearly always there, so its best distance prunes almost every other chunk
  // without first ranking all boxes.  (Any seed is valid: the pruning below is conservative.)
  int w_seed = c_own >> 5;
  eval(w_seed);
  float seed = warp_min(best);
  if (seed == INFINITY) {
    // nothing valid at that azimuth: seed with the nearest chunk by box distance (ties: lowest)
    float lb_min = INFINITY;
    int w_min = 0x7fffffff;
    for (int w = lane; w < words; w += 32) {
      const float lb = box_dist2(box[2 * w], box[2 * w + 1], p);
      if (lb < lb_min) {
        lb_min = lb;
        w_min = w;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ol = __shfl_xor_sync(0xffffffffu, lb_min, off);
      const int ow = __shfl_xor_sync(0xffffffffu, w_min, off);
      if (ol < lb_min || (ol == lb_min && ow < w_min)) {
        lb_min = ol;
        w_min = ow;
      }
    }
    if (w_min == 0x7fffffff) return -1; // no valid point in the row
    w_seed = w_min;
    eval(w_seed);
    seed = warp_min(best);
  }
  // every other chunk that the bound cannot exclude (empty chunks have an infinite bound)
  for (int w0 = 0; w0 < words; w0 += 32) {
    const int w = w0 + lane;
    bool need = false;
    if (w < words && w != w_seed) {
      const float lb = box_dist2(box[2 * w], box[2 * w + 1], p);
      need = lb < INFINITY && lb * (1.0f - 1e-5f) <= seed;
    }
    unsigned todo = __ballot_sync(0xffffffffu, need);
    while (todo) {
      eval(w0 + __ffs(todo) - 1);
      todo &= todo - 1u;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float od = __shfl_xor_sync(0xffffffffu, best, off);
    const int oc = __shfl_xor_sync(0xffffffffu, bc, off);
    if (od < best || (od == best && oc < bc)) {
      best = od;
      bc = oc;
    }
  }
  return bc == 0x7fffffff ? -1 : bc;
}

__device__ __forceinline__ float hypot_pos(float x, float y) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float p = ax > ay ? ax : ay;
  if (p == 0.0f) return 0.0f;
  const float q = ax > ay ? ay : ax;
  const float qp = q / p;
  return p * sqrtf(1.0f + qp * qp);
}

__device__ __forceinline__ void make_givens(float p, float q, float &c, float &s) {
  if (q == 0.0f) {
    c = p < 0.0f ? -1.0f : 1.0f;
    s = 0.0f;
  } else if (p == 0.0f) {
    c = 0.0f;
    s = q < 0.0f ? 1.0f : -1.0f;
  } else if (fabsf(p) > fabsf(q)) {
    const float t = q / p;
    float u = sqrtf(1.0f + t * t);
    if (p < 0.0f) u = -u;
    c = 1.0f / u;
    s = -t * c;
  } else {
    const float t = p / q;
    float u = sqrtf(1.0f + t * t);
    if (q < 0.0f) u = -u;
    s = -1.0f / u;
    c = -t * s;
  }
}

// SelfAdjointEigenSolver<Matrix3f> (iterative path), same operation order as
// oracle/oracle_extract.cpp::self_adjoint_eigen3f.  Returns the normalised
// eigenvector of the smallest eigenvalue.
__device__ void smallest_eigvec3f(float m00, float m10, float m11, float m20, float m21,
                                  float m22, float n[3]) {
  float scale = fabsf(m00);
  scale = fmaxf(scale, fabsf(m10));
  scale = fmaxf(scale, fabsf(m11));
  scale = fmaxf(scale, fabsf(m20));
  scale = fmaxf(scale, fabsf(m21));
  scale = fmaxf(scale, fabsf(m22));
  if (scale == 0.0f) scale = 1.0f;
  m00 = m00 / scale; m10 = m10 / scale; m11 = m11 / scale;
  m20 = m20 / scale; m21 = m21 / scale; m22 = m22 / scale;

  float diag[3], sub[2], Q[9];
  diag[0] = m00;
  const float v1norm2 = m20 * m20;
  if (v1norm2 <= FLT_MIN) {
    diag[1] = m11; diag[2] = m22; sub[0] = m10; sub[1] = m21;
    Q[0] = 1; Q[1] = 0; Q[2] = 0; Q[3] = 0; Q[4] = 1; Q[5] = 0; Q[6] = 0; Q[7] = 0; Q[8] = 1;
  } else {
    const float beta = sqrtf(m10 * m10 + v1norm2);
    const float invBeta = 1.0f / beta;
    const float m01 = m10 * invBeta;
    const float m02 = m20 * invBeta;
    const float q = 2.0f * m01 * m21 + m02 * (m22 - m11);
    diag[1] = m11 + m02 * q;
    diag[2] = m22 - m02 * q;
    sub[0] = beta;
    sub[1] = m21 - m01 * q;
    Q[0] = 1; Q[1] = 0; Q[2] = 0; Q[3] = 0; Q[4] = m01; Q[5] = m02; Q[6] = 0; Q[7] = m02; Q[8] = -m01;
  }
  int end = 2, start = 0, iter = 0;
  const float precision_inv = 1.0f / FLT_EPSILON;
  while (end > 0) {
    for (int i = start; i < end; ++i) {
      if (fabsf(sub[i]) < FLT_MIN) {
        sub[i] = 0.0f;
      } else {
        const float scaled = precision_inv * sub[i];
        if (scaled * scaled <= (fabsf(diag[i]) + fabsf(diag[i + 1]))) sub[i] = 0.0f;
      }
    }
    while (end > 0 && sub[end - 1] == 0.0f) end--;
    if (end <= 0) break;
    iter++;
    if (iter > 90) break;
    start = end - 1;
    while (start > 0 && sub[start - 1] != 0.0f) start--;

    const float td = (diag[end - 1] - diag[end]) * 0.5f;
    const float e = sub[end - 1];
    float mu = diag[end];
    if (td == 0.0f) {
      mu = mu - fabsf(e);
    } else if (e != 0.0f) {
      const float e2 = e * e;
      const float h = hypot_pos(td, e);
      if (e2 == 0.0f) mu = mu - e / ((td + (td > 0.0f ? h : -h)) / e);
      else mu = mu - e2 / (td + (td > 0.0f ? h : -h));
    }
    float x = diag[start] - mu;
    float z = sub[start];
    for (int k = start; k < end && z != 0.0f; ++k) {
      float c, s;
      make_givens(x, z, c, s);
      const float sdk = s * diag[k] + c * sub[k];
      const float dkp1 = s * sub[k] + c * diag[k + 1];
      diag[k] = c * (c * diag[k] - s * sub[k]) - s * (c * sub[k] - s * diag[k + 1]);
      diag[k + 1] = s * sdk + c * dkp1;
      sub[k] = c * sdk - s * dkp1;
      if (k > start) sub[k - 1] = c * sub[k - 1] - s * z;
      x = sub[k];
      if (k < end - 1) {
        z = -s * sub[k + 1];
        sub[k + 1] = c * sub[k + 1];
      }
      for (int r = 0; r < 3; ++r) {
        const float xi = Q[3 * r + k], yi = Q[3 * r + k + 1];
        Q[3 * r + k] = c * xi - s * yi;
        Q[3 * r + k + 1] = s * xi + c * yi;
      }
    }
  }
  // column of the smallest eigenvalue after the ascending selection sort:
  // the first minimum of diag (minCoeff returns the first occurrence)
  int k = 0;
  if (diag[1] < diag[k]) k = 1;
  if (diag[2] < diag[k]) k = 2;
  float n0 = Q[k], n1 = Q[3 + k], n2 = Q[6 + k];
  const float zz = n0 * n0 + (n1 * n1 + n2 * n2);
  if (zz > 0.0f) {
    const float s = sqrtf(zz);
    n0 = n0 / s; n1 = n1 / s; n2 = n2 / s;
  }
  n[0] = n0; n[1] = n1; n[2] = n2;
}

// Covariance of the gathered neighbours (own row +-, closest point of each adjacent row and its
// +-, extraction.tpp:275-305, :314-321) and the eigenvector of its smallest eigenvalue.
// Returns {n, 1} or all zero when the feature is dropped (:308-310).
__device__ __forceinline__ float4 pick_normal(const float4 *own, const float4 *prv, const float4 *nxt, int c,
                                              const PickDesc d, int min_points) {
  const float4 p = own[c];
  const int n = d.n_plus + d.n_minus + (d.c_prev >= 0 ? 1 + d.pp + d.pm : 0) +
                (d.c_next >= 0 ? 1 + d.np_ + d.nm : 0);
  const bool other = d.c_prev >= 0 || d.c_next >= 0;
  float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
  if (other && n >= min_points) {
    const float nf = (float)n;
    float c00 = 0.f, c10 = 0.f, c11 = 0.f, c20 = 0.f, c21 = 0.f, c22 = 0.f;
    auto acc = [&](const float4 q) {
      const float a0 = (q.x - p.x) / nf, a1 = (q.y - p.y) / nf, a2 = (q.z - p.z) / nf;
      c00 = c00 + a0 * a0;
      c10 = c10 + a1 * a0;
      c11 = c11 + a1 * a1;
      c20 = c20 + a2 * a0;
      c21 = c21 + a2 * a1;
      c22 = c22 + a2 * a2;
    };
    for (int i = 1; i <= d.n_plus; ++i) acc(own[c + i]);
    for (int i = 1; i <= d.n_minus; ++i) acc(own[c - i]);
    if (d.c_prev >= 0) {
      acc(prv[d.c_prev]);
      for (int i = 1; i <= d.pp; ++i) acc(prv[d.c_prev + i]);
      for (int i = 1; i <= d.pm; ++i) acc(prv[d.c_prev - i]);
    }
    if (d.c_next >= 0) {
      acc(nxt[d.c_next]);
      for (int i = 1; i <= d.np_; ++i) acc(nxt[d.c_next + i]);
      for (int i = 1; i <= d.nm; ++i) acc(nxt[d.c_next - i]);
    }
    float nrm[3];
    smallest_eigvec3f(c00, c10, c11, c20, c21, c22, nrm);
    out = make_float4(nrm[0], nrm[1], nrm[2], 1.0f);
  }
  return out;
}

} // namespace

// The search is arithmetic-bound (picks x 2 rows x cols distance evaluations) and a row
// alone gives one CTA per SM at best, so every row is shared by kNormalSplit CTAs that
// each stage the three rows and take a contiguous share of the row's picks.
constexpr int kNormalSplit = 4;

namespace {
__device__ __forceinline__ void extract_normals_body(const ExtractArgs &a, const int bx, const int b) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int cols = a.cols, words = a.words, np = a.np;
  float4 *own = reinterpret_cast<float4 *>(smem_raw);
  float4 *prv = own + cols;
  float4 *nxt = prv + cols;
  float4 *box_prv = nxt + cols;       // [words][2] chunk boxes of the adjacent rows
  float4 *box_nxt = box_prv + 2 * words;
  uint32_t *v_prv = reinterpret_cast<uint32_t *>(box_nxt + 2 * words);
  uint32_t *v_nxt = v_prv + words;
  PickDesc *desc = reinterpret_cast<PickDesc *>(v_nxt + words);
  __shared__ int s_keep;

  const int row = bx / kNormalSplit, part = bx % kNormalSplit;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const size_t rb = (size_t)b * a.rows + row;
  const int n_all = a.planar_cnt[rb];
  // this CTA's contiguous share [p_lo, p_hi) of the row's picks
  const int per = (n_all + kNormalSplit - 1) / kNormalSplit;
  const int p_lo = min(part * per, n_all), p_hi = min(p_lo + per, n_all);
  const int n_picks = p_hi - p_lo;
  if (tid == 0) s_keep = 0;
  if (n_picks == 0) return; // keep_cnt is zeroed by the select kernel and accumulated below
  const bool has_prev = row > 0, has_next = row < a.rows - 1;
  const float4 *g = a.scan + rb * cols;
  for (int c = tid; c < cols; c += blockDim.x) {
    own[c] = __ldg(&g[c]);
    if (has_prev) prv[c] = __ldg(&g[c - cols]);
    if (has_next) nxt[c] = __ldg(&g[c + cols]);
  }
  for (int w = tid; w < words; w += blockDim.x) {
    v_prv[w] = has_prev ? a.valid_bits[(rb - 1) * words + w] : 0u;
    v_nxt[w] = has_next ? a.valid_bits[(rb + 1) * words + w] : 0u;
  }
  for (int i = tid; i < 2 * words; i += blockDim.x) {
    if (has_prev) box_prv[i] = a.row_box[(rb - 1) * words * 2 + i];
    if (has_next) box_nxt[i] = a.row_box[(rb + 1) * words * 2 + i];
  }
  __syncthreads();

  const uint16_t *picks = a.planar_cols + rb * a.pr_cap + p_lo;
  const double r2 = a.radius * a.radius;

  // phase A: one warp per pick - closest points on the adjacent rows, then neighbour counts
  for (int pk = warp; pk < n_picks; pk += nwarps) {
    const int c = picks[pk];
    const float4 pp = own[c];
    const int cprev = has_prev ? closest_in_row_pruned(prv, v_prv, box_prv, pp, words, cols, lane, c) : -1;
    const int cnext = has_next ? closest_in_row_pruned(nxt, v_nxt, box_nxt, pp, words, cols, lane, c) : -1;
    int n_plus, n_minus, pp_ = 0, pm = 0, nq = 0, nm = 0;
    neighbor_counts(own, c, np, r2, lane, n_plus, n_minus);
    if (cprev >= 0) neighbor_counts(prv, cprev, np, r2, lane, pp_, pm);
    if (cnext >= 0) neighbor_counts(nxt, cnext, np, r2, lane, nq, nm);
    if (lane == 0) {
      PickDesc d;
      d.c_prev = (short)cprev; d.c_next = (short)cnext;
      d.n_plus = (unsigned char)n_plus; d.n_minus = (unsigned char)n_minus;
      d.pp = (unsigned char)pp_; d.pm = (unsigned char)pm;
      d.np_ = (unsigned char)nq; d.nm = (unsigned char)nm;
      d.pad[0] = d.pad[1] = 0;
      desc[pk] = d;
    }
  }
  __syncthreads();

  // phase B: one thread per pick - covariance + eigenvector (picks packed into as few warps as
  // possible: spreading them over all warps was measured 40 % more instructions, the eigen
  // solver being long and divergent)
  for (int pk = tid; pk < n_picks; pk += blockDim.x) {
    const int c = picks[pk];
    const PickDesc d = desc[pk];
    const float4 out = pick_normal(own, prv, nxt, c, d, a.min_points);
    if (out.w != 0.0f) atomicAdd(&s_keep, 1);
    a.normals[rb * a.pr_cap + p_lo + pk] = out;
    if (a.closest) {
      a.closest[(rb * a.pr_cap + p_lo + pk) * 2 + 0] = d.c_prev >= 0 ? (row - 1) * cols + d.c_prev : -1;
      a.closest[(rb * a.pr_cap + p_lo + pk) * 2 + 1] = d.c_next >= 0 ? (row + 1) * cols + d.c_next : -1;
    }
  }
  __syncthreads();
  if (tid == 0 && s_keep) atomicAdd(&a.keep_cnt[rb], s_keep); // integer count: order-free
}
} // namespace

__global__ void __launch_bounds__(256) extract_normals_kernel(ExtractArgs a) {
  extract_normals_body(a, blockIdx.x, blockIdx.y);
}

// ---------------------------------------------------------------------------
// K2 for many-row (batched) launches: one THREAD per pick, one CTA per row.
// The warp-per-pick search above spends ~450 warp instructions per pick, most of them the
// five-step shuffle reductions and ballots that hold 32 lanes together around a search which,
// after box pruning, touches one or two 32-column chunks (ncu: 620 warp instructions per pick,
// 13 of 32 lanes active on average).  With thousands of rows in flight there is no need to
// spread one pick over a warp: a thread walks the 32 chunk boxes (broadcast reads), evaluates
// the chunk at its own azimuth and the few the bound cannot exclude, counts its neighbours and
// goes straight on to its covariance and eigen solve - no shuffle, no barrier between the
// phases, 32 picks per warp.  Same arithmetic per candidate and the same (dist2, column) /
// first-miss rules, so the results are bit-identical to the warp-per-pick kernel.
// ---------------------------------------------------------------------------
namespace {

__device__ __forceinline__ int closest_in_row_thread(const float4 *rowp, const uint32_t *valid,
                                                     const float4 *box, const float4 p, int words, int c_own) {
  float best = INFINITY;
  int bc = 0x7fffffff;
  auto eval = [&](int w) {
    uint32_t m = valid[w];
    while (m) {
      const int c = w * 32 + __ffs(m) - 1;
      m &= m - 1u;
      const float d2 = diff_sqnorm4(rowp[c], p);
      if (d2 < best || (d2 == best && c < bc)) {
        best = d2;
        bc = c;
      }
    }
  };
  int w_seed = c_own >> 5; // the chunk at the pick's own azimuth
  eval(w_seed);
  if (best == INFINITY) {
    // nothing valid there: the nearest chunk by box distance (ties: lowest chunk)
    float lb_min = INFINITY;
    int w_min = -1;
    for (int w = 0; w < words; ++w) {
      const float lb = box_dist2(box[2 * w], box[2 * w + 1], p);
      if (lb < lb_min) {
        lb_min = lb;
        w_min = w;
      }
    }
    if (w_min < 0) return -1; // no valid point in the row
    w_seed = w_min;
    eval(w_seed);
  }
  // Every other chunk the bound cannot exclude.  The chunks are first COLLECTED (box tests against
  // the best of the seed chunk, 32 chunks per mask) and then evaluated from ONE loop: evaluating
  // inside the box loop left every thread of a warp at a different chunk index - the ~30-iteration
  // point loop then ran once per distinct index with a handful of lanes (ncu: 8 of 32).  Testing
  // against the seed's best instead of the running best is still exact (a chunk is skipped only
  // if each of its points loses to a best that can only improve); the bound is re-tested when
  // a chunk is popped.
  for (int w0 = 0; w0 < words; w0 += 32) {
    uint32_t need = 0u;
    const int wn = min(32, words - w0);
    for (int i = 0; i < wn; ++i) {
      const int w = w0 + i;
      const float lb = box_dist2(box[2 * w], box[2 * w + 1], p);
      if (w != w_seed && lb < INFINITY && lb * (1.0f - 1e-5f) <= best) need |= 1u << i;
    }
    while (need) {
      const int w = w0 + __ffs(need) - 1;
      need &= need - 1u;
      const float lb = box_dist2(box[2 * w], box[2 * w + 1], p);
      if (lb * (1.0f - 1e-5f) <= best) eval(w);
    }
  }
  return bc == 0x7fffffff ? -1 : bc;
}

// find_neighbors (extraction.tpp:422-448) around column c of `rowp`, sequential form
__device__ __forceinline__ void neighbor_counts_thread(const float4 *rowp, int c, int np, double r2,
                                                       int &n_plus, int &n_minus) {
  const float4 p = rowp[c];
  n_plus = 0;
  while (n_plus < np && (double)diff_sqnorm4(rowp[c + n_plus + 1], p) < r2) ++n_plus;
  n_minus = 0;
  while (n_minus < np && (double)diff_sqnorm4(rowp[c - n_minus - 1], p) < r2) ++n_minus;
}

__device__ __forceinline__ void extract_normals_thread_body(const ExtractArgs &a, const int row, const int b) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int cols = a.cols, words = a.words, np = a.np;
  float4 *own = reinterpret_cast<float4 *>(smem_raw);
  float4 *prv = own + cols;
  float4 *nxt = prv + cols;
  float4 *box_prv = nxt + cols; // [words][2] chunk boxes of the adjacent rows
  float4 *box_nxt = box_prv + 2 * words;
  uint32_t *v_prv = reinterpret_cast<uint32_t *>(box_nxt + 2 * words);
  uint32_t *v_nxt = v_prv + words;
  __shared__ int s_keep;

  const int tid = threadIdx.x;
  const size_t rb = (size_t)b * a.rows + row;
  const int n_picks = a.planar_cnt[rb];
  if (tid == 0) s_keep = 0;
  if (n_picks == 0) return; // keep_cnt was zeroed by the select kernel
  const bool has_prev = row > 0, has_next = row < a.rows - 1;
  const float4 *g = a.scan + rb * cols;
  for (int c = tid; c < cols; c += blockDim.x) {
    own[c] = __ldg(&g[c]);
    if (has_prev) prv[c] = __ldg(&g[c - cols]);
    if (has_next) nxt[c] = __ldg(&g[c + cols]);
  }
  for (int w = tid; w < words; w += blockDim.x) {
    v_prv[w] = has_prev ? a.valid_bits[(rb - 1) * words + w] : 0u;
    v_nxt[w] = has_next ? a.valid_bits[(rb + 1) * words + w] : 0u;
  }
  for (int i = tid; i < 2 * words; i += blockDim.x) {
    if (has_prev) box_prv[i] = a.row_box[(rb - 1) * words * 2 + i];
    if (has_next) box_nxt[i] = a.row_box[(rb + 1) * words * 2 + i];
  }
  __syncthreads();

  const uint16_t *picks = a.planar_cols + rb * a.pr_cap;
  const double r2 = a.radius * a.radius;
  int kept = 0;
  for (int pk = tid; pk < n_picks; pk += blockDim.x) {
    const int c = picks[pk];
    const float4 pp = own[c];
    const int cprev = has_prev ? closest_in_row_thread(prv, v_prv, box_prv, pp, words, c) : -1;
    const int cnext = has_next ? closest_in_row_thread(nxt, v_nxt, box_nxt, pp, words, c) : -1;
    int n_plus, n_minus, pp_ = 0, pm = 0, nq = 0, nm = 0;
    neighbor_counts_thread(own, c, np, r2, n_plus, n_minus);
    if (cprev >= 0) neighbor_counts_thread(prv, cprev, np, r2, pp_, pm);
    if (cnext >= 0) neighbor_counts_thread(nxt, cnext, np, r2, nq, nm);
    PickDesc d;
    d.c_prev = (short)cprev; d.c_next = (short)cnext;
    d.n_plus = (unsigned char)n_plus; d.n_minus = (unsigned char)n_minus;
    d.pp = (unsigned char)pp_; d.pm = (unsigned char)pm;
    d.np_ = (unsigned char)nq; d.nm = (unsigned char)nm;
    d.pad[0] = d.pad[1] = 0;
    const float4 out = pick_normal(own, prv, nxt, c, d, a.min_points);
    if (out.w != 0.0f) ++kept;
    a.normals[rb * a.pr_cap + pk] = out;
    if (a.closest) {
      a.closest[(rb * a.pr_cap + pk) * 2 + 0] = cprev >= 0 ? (row - 1) * cols + cprev : -1;
      a.closest[(rb * a.pr_cap + pk) * 2 + 1] = cnext >= 0 ? (row + 1) * cols + cnext : -1;
    }
  }
  if (kept) atomicAdd(&s_keep, kept);
  __syncthreads();
  if (tid == 0 && s_keep) atomicAdd(&a.keep_cnt[rb], s_keep); // integer count: order-free
}
} // namespace

__global__ void __launch_bounds__(256) extract_normals_batch_kernel(const ExtractArgs *items) {
  __shared__ ExtractArgs s_a;
  load_item_args(s_a, items + blockIdx.y);
  if ((int)blockIdx.x >= s_a.rows * kNormalSplit) return;
  extract_normals_body(s_a, blockIdx.x, 0);
}

__global__ void __launch_bounds__(256) extract_normals_rows_kernel(const ExtractArgs *items) {
  __shared__ ExtractArgs s_a;
  load_item_args(s_a, items + blockIdx.y);
  if ((int)blockIdx.x >= s_a.rows) return;
  extract_normals_thread_body(s_a, blockIdx.x, 0);
}

// ---------------------------------------------------------------------------
// K3: pack kept planar picks and point picks into the current-scan keypoint
// arrays in rule R3 order (row, sector, selection order; dropped normals removed)
// ---------------------------------------------------------------------------
namespace {
__device__ __forceinline__ void extract_pack_body(const ExtractArgs &a, const int row, const int b) {
  const int tid = threadIdx.x, lane = tid & 31;
  const size_t rb0 = (size_t)b * a.rows;
  __shared__ int s_off[2];
  __shared__ int s_tot[2];
  // exclusive prefix over earlier rows (and totals) - at most a few hundred ints
  if (tid < 32) {
    int offp = 0, offq = 0, totp = 0, totq = 0;
    for (int r = lane; r < a.rows; r += 32) {
      const int kp = a.keep_cnt[rb0 + r], kq = a.point_cnt[rb0 + r];
      totp += kp;
      totq += kq;
      if (r < row) {
        offp += kp;
        offq += kq;
      }
    }
    for (int o = 16; o > 0; o >>= 1) {
      offp += __shfl_xor_sync(0xffffffffu, offp, o);
      offq += __shfl_xor_sync(0xffffffffu, offq, o);
      totp += __shfl_xor_sync(0xffffffffu, totp, o);
      totq += __shfl_xor_sync(0xffffffffu, totq, o);
    }
    if (lane == 0) {
      s_off[0] = offp; s_off[1] = offq; s_tot[0] = totp; s_tot[1] = totq;
    }
  }
  __syncthreads();
  const size_t rb = rb0 + row;
  const float4 *g = a.scan + rb * a.cols;
  if (row == 0 && tid == 0) {
    a.cur_counts[2 * b + 0] = s_tot[0];
    a.cur_counts[2 * b + 1] = s_tot[1];
  }
  // planar: stable compaction of the keep flags by warp 0 into a list of kept picks
  extern __shared__ uint16_t s_kept[]; // [pr_cap]
  __shared__ int s_nkeep;
  const int n_picks = a.planar_cnt[rb];
  if (tid < 32) {
    int n = 0;
    for (int base = 0; base < n_picks; base += 32) {
      const int pk = base + lane;
      const bool keep = pk < n_picks && a.normals[rb * a.pr_cap + pk].w != 0.0f;
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (keep) s_kept[n + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)pk;
      n += __popc(bal);
    }
    if (lane == 0) s_nkeep = n;
  }
  __syncthreads();
  const int n_keep = s_nkeep;
  for (int j = tid; j < n_keep; j += blockDim.x) {
    const int pk = s_kept[j];
    const float4 nrm = a.normals[rb * a.pr_cap + pk];
    const int c = a.planar_cols[rb * a.pr_cap + pk];
    const float4 p = __ldg(&g[c]);
    PlanarRec r;
    r.x = p.x; r.y = p.y; r.z = p.z;
    r.nx = nrm.x; r.ny = nrm.y; r.nz = nrm.z;
    r.pad0 = (uint32_t)(row * a.cols + c);
    r.pad1 = 0;
    a.cur_planar[(size_t)b * a.kp_cap + s_off[0] + j] = r;
    if (a.host_planar) a.host_planar[s_off[0] + j] = r;
  }
  if (a.host_planar_f64) {
    // the caller's (page-locked, mapped) buffer receives the API's f64 structs directly:
    // consecutive threads write consecutive 8-byte words of the row's 72-byte records
    unsigned long long *dst = reinterpret_cast<unsigned long long *>(a.host_planar_f64) + (size_t)s_off[0] * 9;
    for (int i = tid; i < n_keep * 9; i += blockDim.x) {
      const int j = i / 9, f = i - 9 * j;
      const int pk = s_kept[j];
      unsigned long long bits = 0ull; // pad / npad
      if (f < 3) {
        const float4 p = __ldg(&g[a.planar_cols[rb * a.pr_cap + pk]]);
        bits = (unsigned long long)__double_as_longlong((double)(f == 0 ? p.x : f == 1 ? p.y : p.z));
      } else if (f >= 4 && f < 7) {
        const float4 nrm = a.normals[rb * a.pr_cap + pk];
        bits = (unsigned long long)__double_as_longlong((double)(f == 4 ? nrm.x : f == 5 ? nrm.y : nrm.z));
      } else if (f == 8) {
        bits = a.scan_idx;
      }
      dst[i] = bits;
    }
  }
  // points
  const int nq = a.point_cnt[rb];
  for (int j = tid; j < nq; j += blockDim.x) {
    const int c = a.point_cols[rb * a.qr_cap + j];
    const float4 p = __ldg(&g[c]);
    PointRec r;
    r.x = p.x; r.y = p.y; r.z = p.z;
    r.w = 0.0f;
    a.cur_point[(size_t)b * a.kq_cap + s_off[1] + j] = r;
    if (a.host_point) a.host_point[s_off[1] + j] = r;
  }
  if (a.host_point_f64) {
    unsigned long long *dst = reinterpret_cast<unsigned long long *>(a.host_point_f64) + (size_t)s_off[1] * 5;
    for (int i = tid; i < nq * 5; i += blockDim.x) {
      const int j = i / 5, f = i - 5 * j;
      unsigned long long bits = 0ull; // pad
      if (f < 3) {
        const float4 p = __ldg(&g[a.point_cols[rb * a.qr_cap + j]]);
        bits = (unsigned long long)__double_as_longlong((double)(f == 0 ? p.x : f == 1 ? p.y : p.z));
      } else if (f == 4) {
        bits = a.scan_idx;
      }
      dst[i] = bits;
    }
  }
  // publish: the last CTA to finish writes the counts and raises the host-visible flag
  if (a.flag) {
    if (a.host_planar || a.host_point || a.host_planar_f64 || a.host_point_f64)
      __threadfence_system(); // host records of this CTA first
    else __threadfence();
    __syncthreads();
    if (tid == 0) {
      const unsigned d = atomicAdd(a.done_counter, 1u);
      if (d == a.done_target - 1u) {
        *a.done_counter = 0u;
        a.host_counts[0] = s_tot[0];
        a.host_counts[1] = s_tot[1];
        __threadfence_system();
        *a.flag = a.seq;
      }
    }
  }
}
} // namespace

__global__ void __launch_bounds__(128) extract_pack_kernel(ExtractArgs a) {
  extract_pack_body(a, blockIdx.x, blockIdx.y);
}

__global__ void __launch_bounds__(128) extract_pack_batch_kernel(const ExtractArgs *items) {
  __shared__ ExtractArgs s_a;
  load_item_args(s_a, items + blockIdx.y);
  if ((int)blockIdx.x >= s_a.rows) return; // before the item's buffers and its done_counter
  extract_pack_body(s_a, blockIdx.x, 0);
}

// ---------------------------------------------------------------------------
// host-side launcher
// ---------------------------------------------------------------------------
size_t extract_select_smem(int cols, int cols_pad, int words, int sectors, int spec_cap) {
  // staged row, keys, sorted + unused lists, the four row masks; then the private masks of the
  // speculative walks ([sectors][words]), the initial point mask and the speculative pick lists
  return (size_t)cols * sizeof(float4) + (size_t)cols_pad * (sizeof(uint32_t) + 2 * sizeof(uint16_t)) +
         (size_t)words * 4 * sizeof(uint32_t) + (size_t)(sectors + 1) * words * sizeof(uint32_t) +
         ((size_t)sectors * spec_cap * sizeof(uint16_t) + 15) / 16 * 16;
}
size_t extract_normals_smem(int cols, int words, int pr_cap) {
  return (size_t)cols * 3 * sizeof(float4) + (size_t)words * 4 * sizeof(float4) +
         (size_t)words * 2 * sizeof(uint32_t) + (size_t)pr_cap * sizeof(PickDesc);
}

cudaError_t extract_configure(const ExtractArgs &shape) {
  // the attributes belong to the functions, not to a context: they only ever grow, so that contexts
  // of different scan shapes can live in one process (a 16x1800 context needs more normals shared
  // memory than a 64x1024 one created after it)
  static std::mutex mu;
  static size_t select_hi = 0, normals_hi = 0;
  std::lock_guard<std::mutex> lock(mu);
  select_hi = std::max(select_hi, extract_select_smem(shape));
  normals_hi = std::max(normals_hi, extract_normals_smem(shape.cols, shape.words, shape.pr_cap));
  cudaError_t e = cudaFuncSetAttribute(extract_select_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)select_hi);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(extract_select_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)select_hi);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(extract_normals_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)normals_hi);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(extract_normals_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)normals_hi);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(extract_normals_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)normals_hi);
}

ExtractLaunchShape extract_launch_shape(const ExtractArgs *items, int n_items) {
  ExtractLaunchShape sh;
  for (int i = 0; i < n_items; ++i) {
    const ExtractArgs &a = items[i];
    sh.max_rows = std::max(sh.max_rows, a.rows);
    sh.sum_rows += a.rows;
    sh.select_smem = std::max(sh.select_smem, extract_select_smem(a));
    sh.normals_smem = std::max(sh.normals_smem, extract_normals_smem(a.cols, a.words, a.pr_cap));
    sh.pack_smem = std::max(sh.pack_smem, (size_t)a.pr_cap * sizeof(uint16_t));
  }
  return sh;
}

void extract_batch_launch(const ExtractLaunchShape &sh, const ExtractArgs *items_dev, int n_items,
                          int many_rows_min, cudaStream_t stream, Profiler &prof) {
  // the items may differ in geometry (rows, cols, sectors, caps): the grid covers the largest rows
  // (CTAs past their own item's rows leave at once) and shared memory is the largest need
  const dim3 grid(sh.max_rows, n_items);
  prof.begin(FORMGPU_KG_EXTRACT_SELECT);
  // One warp of every CTA ends up walking the row's greedy selections alone, so what bounds a
  // many-row launch is how many rows are RESIDENT (registers: 2 CTAs of 512 threads per SM, 10
  // of 128).  Launches with more rows than fit at 512 threads use 128-thread CTAs: the parallel
  // part of a row takes four times longer, but five times as many serial walks overlap it.
  const bool many_rows = sh.sum_rows >= many_rows_min;
  // many rows: one warp per sector for the speculative walks (six sectors by default) and as many
  // rows resident as the registers allow; FORMGPU_SELECT_THREADS overrides it for tuning
  static const int select_many = [] {
    const char *e = std::getenv("FORMGPU_SELECT_THREADS");
    const int v = e ? std::atoi(e) : 0;
    return v >= 32 && v <= 512 && v % 32 == 0 ? v : 192;
  }();
  const int select_threads = many_rows ? select_many : 512;
  extract_select_batch_kernel<<<grid, select_threads, sh.select_smem, stream>>>(items_dev);
  prof.end(FORMGPU_KG_EXTRACT_SELECT, 1);
  prof.begin(FORMGPU_KG_EXTRACT_NORMALS);
  // many rows: one thread per pick (one CTA per row); few rows: one warp per pick, four CTAs
  // per row, which spreads a small launch over the whole GPU
  if (many_rows)
    extract_normals_rows_kernel<<<grid, 256, sh.normals_smem, stream>>>(items_dev);
  else
    extract_normals_batch_kernel<<<dim3(sh.max_rows * kNormalSplit, n_items), 256, sh.normals_smem, stream>>>(
        items_dev);
  prof.end(FORMGPU_KG_EXTRACT_NORMALS, 1);
  prof.begin(FORMGPU_KG_EXTRACT_PACK);
  extract_pack_batch_kernel<<<grid, 128, sh.pack_smem, stream>>>(items_dev);
  prof.end(FORMGPU_KG_EXTRACT_PACK, 1);
}

void extract_launch(const ExtractArgs &a, int n_scans, cudaStream_t stream, Profiler &prof) {
  const dim3 grid(a.rows, n_scans);
  prof.begin(FORMGPU_KG_EXTRACT_SELECT);
  extract_select_kernel<<<grid, 512, extract_select_smem(a), stream>>>(a);
  prof.end(FORMGPU_KG_EXTRACT_SELECT, 1);
  prof.begin(FORMGPU_KG_EXTRACT_NORMALS);
  extract_normals_kernel<<<dim3(a.rows * kNormalSplit, n_scans), 256,
                           extract_normals_smem(a.cols, a.words, a.pr_cap), stream>>>(a);
  prof.end(FORMGPU_KG_EXTRACT_NORMALS, 1);
  prof.begin(FORMGPU_KG_EXTRACT_PACK);
  extract_pack_kernel<<<grid, 128, (size_t)a.pr_cap * sizeof(uint16_t), stream>>>(a);
  prof.end(FORMGPU_KG_EXTRACT_PACK, 1);
}

} // namespace formgpu
