// Device helpers shared by the stage-3 kernels (linearize.cu: streaming reduction of the
// correspondences; moments.cu: pose-independent pair moments and their evaluation).
#pragma once

#include "ctx.hpp"
#include "kernels.hpp"

namespace formgpu {

namespace {

constexpr int kThreads = kLinThreads;
constexpr int kWarps = kThreads / 32;

__device__ __forceinline__ void apply_rel(const double *rel, double x, double y, double z,
                                          double &qx, double &qy, double &qz) {
  qx = rel[0] * x + rel[1] * y + rel[2] * z + rel[9];
  qy = rel[3] * x + rel[4] * y + rel[5] * z + rel[10];
  qz = rel[6] * x + rel[7] * y + rel[8] * z + rel[11];
}

// Butterfly-transpose reduction of 32 values per lane across the warp: at the step
// with offset o a lane keeps the half of its values selected by (lane & o) and adds
// the partner's copy of that half, so after 5 steps lane l holds the warp total of
// element l.  16+8+4+2+1 = 31 exchanges instead of 32 * 5.
template <int N> __device__ __forceinline__ void transpose_reduce(double (&v)[32], int lane) {
  if constexpr (N >= 1) {
    const bool upper = (lane & N) != 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const double keep = upper ? v[i + N] : v[i];
      const double send = upper ? v[i] : v[i + N];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, N);
    }
    transpose_reduce<N / 2>(v, lane);
  }
}

// CTA-wide sum of the 28 moments of every thread into out[28] (shared memory).
__device__ __forceinline__ void block_reduce28(double (&acc)[32], double (*s_warp)[28], double *out,
                                               int tid) {
  const int lane = tid & 31, warp = tid >> 5;
  transpose_reduce<16>(acc, lane);
  if (lane < 28) s_warp[warp][lane] = acc[0];
  __syncthreads();
  if (tid < 28) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) v += s_warp[w][tid];
    out[tid] = v;
  }
  __syncthreads();
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------
// expansion of the two 7x7 moment matrices to the 13x13 block (CTA 0 of a cluster)
// ---------------------------------------------------------------------------
struct ExpandSmem {
  double Wp[7][7], Wq[7][7];
  double Bp[7][13];    // plane-point basis rows
  double Bq[7][3][13]; // point-point basis (3 rows each)
  double Tp[7][13];    // W_p B_p
  double Tq[3][7][13]; // per residual row r: W_q B_q[.][r]
};

// entry (r, c) of the skew matrix [t]x
__device__ __forceinline__ double skew_entry(const double *t, int r, int c) {
  if (r == c) return 0.0;
  const double v = t[3 - r - c];
  return ((c - r + 3) % 3 == 1) ? -v : v;
}

__device__ __forceinline__ void zero_basis(ExpandSmem &S) {
  const int tid = (int)threadIdx.x, nthreads = (int)blockDim.x;
  for (int i = tid; i < 7 * 13; i += nthreads) (&S.Bp[0][0])[i] = 0.0;
  for (int i = tid; i < 7 * 3 * 13; i += nthreads) (&S.Bq[0][0][0])[i] = 0.0;
}

// The non-zero entries of the two bases, 39 independent work items (9 + 27 + 3) spread over the
// threads `first_thread + item` (a 3-thread version of this fill was 30 % of the evaluation
// kernel's stall samples: three serial chains while 125 threads waited at the barrier).
//   plane-point: row = [ u1, -u2, -R^T u1 - R^T [t]x u2, R^T u2, -r ]
//   point-point: rows = [ [P]x, -I, -[c]x R, R, -e ],  c = P + e - t
__device__ __forceinline__ void fill_basis(ExpandSmem &S, const double *rel, int first_thread = 0) {
  const int tid = (int)threadIdx.x - first_thread, nthreads = (int)blockDim.x;
  const double *R = rel, *t = rel + 9;
  for (int item = tid; item >= 0 && item < 39; item += nthreads) {
    if (item < 9) { // (k, c)
      const int k = item / 3, c = item % 3;
      S.Bp[k][6 + c] = -R[3 * k + c];    // -R^T u1
      S.Bp[3 + k][9 + c] = R[3 * k + c]; //  R^T u2
      double bt = 0.0, kr = 0.0;
      for (int b = 0; b < 3; ++b) {
        bt += R[3 * b + c] * skew_entry(t, b, k); // (R^T [t]x)[c][k]
        kr += skew_entry(t, k, b) * R[3 * b + c]; // ([t]x R)[k][c]
      }
      S.Bp[3 + k][6 + c] = -bt;   // -R^T [t]x u2
      S.Bq[6][k][6 + c] = kr;     // +[t]x R, the constant part of -[c]x R
      S.Bq[6][k][9 + c] = R[3 * k + c]; // R
    } else if (item < 36) { // (k, r, c): E_k = skew(e_k)
      const int j = item - 9, k = j / 9, r = (j / 3) % 3, c = j % 3;
      // skew(e_k)[x][y]: +-1 where 3 - x - y == k
      auto ek = [k](int x, int y) {
        return (x == y || 3 - x - y != k) ? 0.0 : (((y - x + 3) % 3 == 1) ? -1.0 : 1.0);
      };
      double er = 0.0; // (E_k R)[r][c]
      for (int b = 0; b < 3; ++b) er += ek(r, b) * R[3 * b + c];
      S.Bq[k][r][c] = ek(r, c); // [P]x
      S.Bq[k][r][6 + c] = -er;              // -[P]x R
      S.Bq[3 + k][r][6 + c] = -er;          // -[e]x R
    } else { // k
      const int k = item - 36;
      S.Bp[k][k] = 1.0;          // J_i rot   =  u1
      S.Bp[3 + k][3 + k] = -1.0; // J_i trans = -u2
      S.Bq[3 + k][k][12] = -1.0; // -e
      S.Bq[6][k][3 + k] = -1.0;  // -I
      if (k == 0) S.Bp[6][12] = -1.0; // b = -r
    }
  }
}

// The basis only depends on the relative pose, so CTA 0 builds it at kernel start while the
// rest of the CTA is already streaming correspondences (the first __syncthreads of the
// reduction publishes it).
__device__ __forceinline__ void build_basis(ExpandSmem &S, const double *rel) {
  zero_basis(S);
  __syncthreads();
  fill_basis(S, rel);
}

// out = B^T W B in two short unrolled passes: T = W B (7 MACs per entry, all threads),
// then B^T T (7 + 21 MACs per entry, 91 threads).  Every 8-byte word that leaves for the
// host carries the call's sequence tag in its upper half (see publish_tagged).
__device__ __forceinline__ void publish_tagged(volatile unsigned long long *dst, double v,
                                               unsigned long long tag) {
  const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
  dst[0] = (bits & 0xffffffffull) | (tag << 32);
  dst[1] = (bits >> 32) | (tag << 32);
}

__device__ __forceinline__ void expand_and_publish(ExpandSmem &S, const double *Wp28, const double *Wq28,
                                                   bool has_planar, bool has_point, double inv_sigma2,
                                                   volatile unsigned long long *out182,
                                                   unsigned long long tag, double *plain91 = nullptr) {
  const int tid = (int)threadIdx.x, nthreads = (int)blockDim.x;
  if (tid < 28) {
    int p = 0, e = tid; // upper-triangular index -> (p, q)
    while (e >= 7 - p) {
      e -= 7 - p;
      ++p;
    }
    const int q = p + e;
    S.Wp[p][q] = S.Wp[q][p] = Wp28[tid];
    S.Wq[p][q] = S.Wq[q][p] = Wq28[tid];
  }
  __syncthreads();
  for (int idx = tid; idx < 91 + 273; idx += nthreads) {
    double v = 0.0;
    if (idx < 91) {
      const int k = idx / 13, y = idx % 13;
#pragma unroll
      for (int l = 0; l < 7; ++l) v += S.Wp[k][l] * S.Bp[l][y];
      S.Tp[k][y] = v;
    } else {
      const int j = idx - 91, r = j / 91, k = (j % 91) / 13, y = j % 13;
#pragma unroll
      for (int l = 0; l < 7; ++l) v += S.Wq[k][l] * S.Bq[l][r][y];
      S.Tq[r][k][y] = v;
    }
  }
  __syncthreads();
  for (int o = tid; o < 91; o += nthreads) {
    int x = 0, e = o;
    while (e >= 13 - x) {
      e -= 13 - x;
      ++x;
    }
    const int y = x + e;
    double sum = 0.0;
    if (has_planar) {
#pragma unroll
      for (int k = 0; k < 7; ++k) sum += S.Bp[k][x] * S.Tp[k][y];
    }
    if (has_point) {
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = 0; k < 7; ++k) sum += S.Bq[k][r][x] * S.Tq[r][k][y];
    }
    if (plain91) plain91[o] = sum * inv_sigma2;
    else publish_tagged(out182 + 2 * o, sum * inv_sigma2, tag);
  }
}

// this rank's contiguous share of a pair's n correspondences (point-sharded mode; the whole
// range when shard_world == 1)
__device__ __forceinline__ void shard_range(uint32_t n, int shard_rank, int shard_world, uint32_t &begin,
                                            uint32_t &count) {
  const uint32_t lo = (uint32_t)(((unsigned long long)n * (unsigned)shard_rank) / (unsigned)shard_world);
  const uint32_t hi = (uint32_t)(((unsigned long long)n * (unsigned)(shard_rank + 1)) / (unsigned)shard_world);
  begin = lo;
  count = hi - lo;
}

} // namespace

} // namespace formgpu
