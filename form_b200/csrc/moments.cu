// Stage 3 on sm_100a, cached form: pose-independent pair moments and their evaluation.
//
// Replaces the same reference code as linearize.cu - PlanePoint/PointPoint::evaluateError +
// FeatureFactor::evaluateError (/root/reference/form/feature/factor.cpp:30-186) followed by
// DenseFactor::linearize / FastIsotropic / HessianFactor(JacobianFactor)
// (/root/reference/form/optimization/gtsam.hpp:59-140) - but organises the work around a fact
// of the reference's control flow: the correspondences of a pair (i, j) change only while j is
// the current scan (Matcher::match clears and refills m_constraints[j][*],
// /root/reference/form/optimization/matcher.hpp:78-80,103-111); afterwards the pair is
// re-linearised at new poses over and over (every LM iteration of every later scan,
// /root/reference/form/optimization/constraints.cpp:259-305) with the SAME correspondences.
//
// So each correspondence is streamed exactly once per association.  With a reference relative
// pose rel0 = (R0, t0) of the pair (the poses of the association) and q0 = R0 p_j + t0, keep
//     plane-point:  M_p = sum phi phi^T,   phi  = [ vec(n q0^T) (9, index 3a+b), n (3), r0 ],
//                                          r0 = n.(q0 - p_i)                        (13 x 13)
//     point-point:  M_q = sum zeta zeta^T, zeta = [ q0 (3), d0 = q0 - p_i (3), 1 ]  ( 7 x  7)
// For ANY later relative pose (R, t):  dR = R R0^T, dt = t - dR t0  =>  q = dR q0 + dt, and the
// 7-vectors of the streaming kernel (linearize.cu) are linear in phi / zeta,
//     s = [ n x q, n, n.(q - p_i) ] = S(dR, dt) phi,      z = [ p_i, q - p_i, 1 ] = Z(dR, dt) zeta,
// so its 7x7 moment matrices are the congruences W_p = S M_p S^T, W_q = Z M_q Z^T and the 13x13
// block follows from the same basis expansion (lin_device.cuh).  The result is exact in exact
// arithmetic for every (R, t).  Conditioning: the residual row of S is [vec(dR - I), dt, 1], i.e.
// r = n^T (dR - I) q0 + n.dt + r0 - the large coordinates |q0| <= 100 m enter the residual only
// multiplied by (dR - I), which is the (small) pose change since the association; measured
// against the oracle the blocks agree to <= 1e-11 (tests/test_moment_model.py, test_gpu_stages.py).
//
// Kernels:
//   moment_kernel      one WARP per unit of MomentArgs::unit correspondences of one pair (units are
//                      numbered pair by pair from the device-resident counts, so the launch needs
//                      no host knowledge of the association's outcome); a lane accumulates the 73
//                      distinct planar products of its correspondences, the warp reduces them with
//                      the butterfly transpose; pairs of several units are merged by the pair's
//                      last warp in unit order (ticket), which expands the 73 sums to the packed
//                      13x13 and stores the cache entry.  Fixed partition + fixed order =>
//                      run-to-run deterministic.
//   eval_kernel        one 128-thread CTA per pair: two small congruences, basis expansion, 91 tagged words
//                      to mapped host memory (or plain doubles to device memory); error-only
//                      variant: 0.5 (W_p[6][6] + tr W_q[3:6]) / sigma^2.
// model: tests/test_moment_model.py mirrors the index conventions below one to one.
#include "lin_device.cuh"

namespace formgpu {

namespace {

constexpr int kMomentThreads = 128; // 4 warps = 4 units per CTA
constexpr int kMomentWarps = kMomentThreads / 32;

// index of the symmetric pair (a, c), a, c in 0..2, among the six products
__host__ __device__ constexpr int sym3(int a, int c) {
  const int lo = a < c ? a : c, hi = a < c ? c : a;
  return lo * 3 - lo * (lo - 1) / 2 + (hi - lo);
}

// where entry (x, y), x <= y, of sum phi phi^T lives among the 73 accumulated sums
__device__ __forceinline__ int phi_pair_to_acc(int x, int y) {
  if (y < 9) return 6 * sym3(x / 3, y / 3) + sym3(x % 3, y % 3); // (n_a n_c)(q_b q_d)
  if (x < 9) {
    if (y < 12) return 36 + 3 * sym3(x / 3, y - 9) + x % 3; // (n_a n_c) q_b
    return 54 + x;                                         // n_a r0 q_b
  }
  if (x < 12) {
    if (y < 12) return 63 + sym3(x - 9, y - 9); // n_a n_c
    return 69 + (x - 9);                        // n_a r0
  }
  return 72; // r0^2
}

// butterfly transpose of 16 values per lane: the 8-4-2-1 steps leave element (lane & 15) summed
// over the 16 lanes that agree with this one in bit 4; the last exchange adds the other half
__device__ __forceinline__ void transpose_reduce16(double (&v)[16], int lane) {
#pragma unroll
  for (int N = 8; N >= 1; N >>= 1) {
    const bool upper = (lane & N) != 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const double keep = upper ? v[i + N] : v[i];
      const double send = upper ? v[i] : v[i + N];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, N);
    }
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 16);
}

struct MomentWarpSmem {
  double sum[kMomentPartial]; // this unit's (then the pair's) 73 + 28 sums
  double rel0[12];
};

// Sums of one unit: planar elements [p_lo, p_hi) and point elements [q_lo, q_hi) of the pair's
// ranges (absolute element indices inside the segment planes).
__device__ __forceinline__ void moment_unit(const MomentArgs &a, MomentWarpSmem &S, uint32_t p_lo,
                                            uint32_t p_hi, uint32_t q_lo, uint32_t q_hi, int lane) {
  const double *rel0 = S.rel0;
  // 73 sums in registers: two groups of 32 and one of 16 (9 used), each reduced by one butterfly
  double acc0[32], acc1[32], acc2[16];
#pragma unroll
  for (int k = 0; k < 32; ++k) acc0[k] = acc1[k] = 0.0;
#pragma unroll
  for (int k = 0; k < 16; ++k) acc2[k] = 0.0;
#define MOM_ACC(e) (*((e) < 32 ? &acc0[(e)&31] : (e) < 64 ? &acc1[(e)&31] : &acc2[(e)&15]))
  {
    const float *s = a.seg_planar;
    const size_t st = a.kp_cap;
    // the nine planes of the NEXT correspondence are requested before the current one is reduced:
    // the loop was stalled at the first conversion of a freshly loaded value (ncu: 58 % long
    // scoreboard), one L2 round trip per iteration on a warp that runs alone on its scheduler
    float cur[9], nxt[9];
    uint32_t c = p_lo + (uint32_t)lane;
    if (c < p_hi) {
#pragma unroll
      for (int pl = 0; pl < 9; ++pl) cur[pl] = __ldg(s + pl * st + c);
    }
#pragma unroll 1
    for (; c < p_hi; c += 32u) {
      if (c + 32u < p_hi) {
#pragma unroll
        for (int pl = 0; pl < 9; ++pl) nxt[pl] = __ldg(s + pl * st + c + 32u);
      }
      const double pix = cur[0], piy = cur[1], piz = cur[2];
      const double n[3] = {(double)cur[3], (double)cur[4], (double)cur[5]};
      double q[3];
      apply_rel(rel0, (double)cur[6], (double)cur[7], (double)cur[8], q[0], q[1], q[2]);
      const double r0 = n[0] * (q[0] - pix) + n[1] * (q[1] - piy) + n[2] * (q[2] - piz);
      double nn[6], qq[6];
      {
        int e = 0;
#pragma unroll
        for (int x = 0; x < 3; ++x)
#pragma unroll
          for (int y = x; y < 3; ++y) {
            nn[e] = n[x] * n[y];
            qq[e] = q[x] * q[y];
            ++e;
          }
      }
#pragma unroll
      for (int ac = 0; ac < 6; ++ac)
#pragma unroll
        for (int bd = 0; bd < 6; ++bd) MOM_ACC(6 * ac + bd) += nn[ac] * qq[bd];
#pragma unroll
      for (int ac = 0; ac < 6; ++ac)
#pragma unroll
        for (int b = 0; b < 3; ++b) MOM_ACC(36 + 3 * ac + b) += nn[ac] * q[b];
#pragma unroll
      for (int x = 0; x < 3; ++x) {
        const double nr = n[x] * r0;
#pragma unroll
        for (int b = 0; b < 3; ++b) MOM_ACC(54 + 3 * x + b) += nr * q[b];
        MOM_ACC(69 + x) += nr;
      }
#pragma unroll
      for (int ac = 0; ac < 6; ++ac) MOM_ACC(63 + ac) += nn[ac];
      MOM_ACC(72) += r0 * r0;
#pragma unroll
      for (int pl = 0; pl < 9; ++pl) cur[pl] = nxt[pl];
    }
  }
#undef MOM_ACC
  // warp totals: after the butterfly lane l holds element l of a group of 32 (l & 15 of the
  // group of 16, summed over the lanes that share bit 4; one more exchange completes it)
  transpose_reduce<16>(acc0, lane);
  transpose_reduce<16>(acc1, lane);
  transpose_reduce16(acc2, lane);
  S.sum[lane] = acc0[0];
  S.sum[32 + lane] = acc1[0];
  if (lane < kMomentAcc - 64) S.sum[64 + lane] = acc2[0];
  // point-point rows: zeta = [q0, q0 - p_i, 1], 28 products
#pragma unroll
  for (int k = 0; k < 32; ++k) acc0[k] = 0.0;
  {
    const float *s = a.seg_point;
    const size_t st = a.kq_cap;
#pragma unroll 1
    for (uint32_t c = q_lo + (uint32_t)lane; c < q_hi; c += 32u) {
      const double pix = s[0 * st + c], piy = s[1 * st + c], piz = s[2 * st + c];
      double qx, qy, qz;
      apply_rel(rel0, (double)s[3 * st + c], (double)s[4 * st + c], (double)s[5 * st + c], qx, qy, qz);
      const double v[7] = {qx, qy, qz, qx - pix, qy - piy, qz - piz, 1.0};
      int e = 0;
#pragma unroll
      for (int p = 0; p < 7; ++p)
#pragma unroll
        for (int r = p; r < 7; ++r) acc0[e++] += v[p] * v[r];
    }
  }
  transpose_reduce<16>(acc0, lane);
  if (lane < kMomentPoint) S.sum[kMomentAcc + lane] = acc0[0];
  __syncwarp();
}

__device__ __forceinline__ void moment_body(const MomentArgs &a, MomentWarpSmem &S) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int u = (int)blockIdx.x * kMomentWarps + warp; // unit id of this warp
  const int nb = a.W + 1;
  // ---- which pair does unit u belong to?  Units are numbered pair by pair. ----
  int my_pair = -1, my_rank = 0, my_units = 0;
  uint32_t off_p = 0, n_p = 0, off_q = 0, n_q = 0, raw = 0;
  int base = 0;
  for (int r0 = 0; r0 < a.n_pairs; r0 += 32) {
    const int p = r0 + lane;
    uint32_t op = 0, np = 0, oq = 0, nq = 0, total_raw = 0;
    int units = 0;
    if (p < a.n_pairs) {
      const int si = a.slots[p];
      op = __ldcg(&a.pair_row[0 * nb + si]);
      np = __ldcg(&a.pair_row[1 * nb + si]);
      oq = __ldcg(&a.pair_row[2 * nb + si]);
      nq = __ldcg(&a.pair_row[3 * nb + si]);
      total_raw = np + nq;
      if (a.shard_world > 1) { // this rank's share of the pair (point-sharded mode)
        uint32_t b0, c0;
        shard_range(np, a.shard_rank, a.shard_world, b0, c0);
        op += b0;
        np = c0;
        shard_range(nq, a.shard_rank, a.shard_world, b0, c0);
        oq += b0;
        nq = c0;
      }
      // a non-empty pair always gets a unit, so its entry is (re)written even when this
      // rank's share is empty
      if (total_raw) units = max(1, (int)((np + nq + a.unit - 1u) / a.unit));
    }
    int incl = units;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const int excl = base + incl - units;
    const unsigned bal = __ballot_sync(0xffffffffu, units > 0 && u >= excl && u < excl + units);
    if (bal) {
      const int owner = __ffs(bal) - 1;
      my_pair = r0 + owner;
      my_rank = u - __shfl_sync(0xffffffffu, excl, owner);
      my_units = __shfl_sync(0xffffffffu, units, owner);
      off_p = __shfl_sync(0xffffffffu, op, owner);
      n_p = __shfl_sync(0xffffffffu, np, owner);
      off_q = __shfl_sync(0xffffffffu, oq, owner);
      n_q = __shfl_sync(0xffffffffu, nq, owner);
      raw = __shfl_sync(0xffffffffu, total_raw, owner);
      break;
    }
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (my_pair < 0) return; // more warps than units
  const int si = a.slots[my_pair];
  // ---- reference relative pose of the pair: pose_i^-1 * pose_k ----
  if (lane < 12) {
    const double *Ti = a.slot_pose + 12 * si;
    double v = 0.0;
    if (lane < 9) {
      const int r = lane / 3, c = lane % 3; // (R_i^T R_k)[r][c]
      v = Ti[r] * a.pose_k[c] + Ti[3 + r] * a.pose_k[3 + c] + Ti[6 + r] * a.pose_k[6 + c];
    } else {
      const int r = lane - 9; // (R_i^T (t_k - t_i))[r]
      v = Ti[r] * (a.pose_k[9] - Ti[9]) + Ti[3 + r] * (a.pose_k[10] - Ti[10]) +
          Ti[6 + r] * (a.pose_k[11] - Ti[11]);
    }
    S.rel0[lane] = v;
  }
  __syncwarp();
  // ---- this unit's slice of the concatenated [planar | point] range ----
  const uint32_t lo = (uint32_t)my_rank * a.unit;
  const uint32_t hi = min(lo + a.unit, n_p + n_q);
  const uint32_t p_lo = min(lo, n_p), p_hi = min(hi, n_p);
  const uint32_t q_lo = max(lo, n_p) - n_p, q_hi = max(hi, n_p) - n_p;
  moment_unit(a, S, off_p + p_lo, off_p + p_hi, off_q + q_lo, off_q + q_hi, lane);
  if (my_units > 1) {
    // leave the partial sums, take a ticket; the pair's last warp adds them in unit order
    double *mine = a.partials + (size_t)u * kMomentPartial;
    for (int e = lane; e < kMomentAcc + kMomentPoint; e += 32) mine[e] = S.sum[e];
    __threadfence();
    __syncwarp();
    unsigned ticket = 0;
    if (lane == 0) ticket = atomicAdd(&a.tickets[my_pair], 1u);
    ticket = __shfl_sync(0xffffffffu, ticket, 0);
    if (ticket != (unsigned)(my_units - 1)) return;
    if (lane == 0) a.tickets[my_pair] = 0u; // self-cleaning for the next launch
    __threadfence();
    const double *all = a.partials + (size_t)(u - my_rank) * kMomentPartial;
    double v[4] = {0.0, 0.0, 0.0, 0.0}; // elements lane, lane + 32, lane + 64, lane + 96
    // four units' partial sums are requested together (16 loads in flight), added in unit order
    int r = 0;
    for (; r + 4 <= my_units; r += 4) {
      double t[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int k = 0; k < 4; ++k)
          t[u][k] = lane + 32 * k < kMomentAcc + kMomentPoint
                        ? __ldcg(&all[(size_t)(r + u) * kMomentPartial + lane + 32 * k])
                        : 0.0;
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] += t[u][k];
    }
    for (; r < my_units; ++r) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (lane + 32 * k < kMomentAcc + kMomentPoint) v[k] += __ldcg(&all[(size_t)r * kMomentPartial + lane + 32 * k]);
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (lane + 32 * k < kMomentAcc + kMomentPoint) S.sum[lane + 32 * k] = v[k];
    __syncwarp();
  }
  // ---- the pair's cache entry: M_p packed 13x13 | M_q packed 7x7 | rel0 | counts ----
  double *entry = a.moments + (size_t)si * kMomentStride;
  for (int o = lane; o < kMomentPlanar; o += 32) {
    int x = 0, e = o;
    while (e >= 13 - x) {
      e -= 13 - x;
      ++x;
    }
    entry[o] = S.sum[phi_pair_to_acc(x, x + e)];
  }
  if (lane < kMomentPoint) entry[kMomentPlanar + lane] = S.sum[kMomentAcc + lane];
  if (lane < 12) entry[kMomentPlanar + kMomentPoint + lane] = S.rel0[lane];
  if (lane == 12) {
    const unsigned long long counts = (unsigned long long)raw; // correspondences behind the entry
    entry[kMomentPlanar + kMomentPoint + 12] = __longlong_as_double((long long)counts);
  }
}

} // namespace

__global__ void __launch_bounds__(kMomentThreads, 2) moment_kernel(MomentArgs a) {
  __shared__ MomentWarpSmem s_w[kMomentWarps];
  moment_body(a, s_w[threadIdx.x >> 5]);
}

__global__ void __launch_bounds__(kMomentThreads, 2) moment_batch_kernel(const MomentArgs *items) {
  __shared__ MomentArgs s_a;
  __shared__ MomentWarpSmem s_w[kMomentWarps];
  for (int i = threadIdx.x; i < (int)(sizeof(MomentArgs) / 8); i += blockDim.x)
    reinterpret_cast<unsigned long long *>(&s_a)[i] =
        reinterpret_cast<const unsigned long long *>(items + blockIdx.z)[i];
  __syncthreads();
  pdl_wait();
  moment_body(s_a, s_w[threadIdx.x >> 5]);
}

// ---------------------------------------------------------------------------
// evaluation: one CTA of 128 threads per pair
// ---------------------------------------------------------------------------
// The work of a pair is ~7 k multiply-adds; what the kernel costs is its dependency chain (one
// warp per pair left every phase several rounds deep: 64 us for 10 k pairs, 17 us for 12).  With
// 128 threads every phase is one to three rounds, and the chain is kept short:
//   * the cache entry (and, for launches whose tasks live in device memory, the context's argument
//     block) is requested before anything else; while the loads are in flight the CTA zero-fills
//     the basis and coefficient matrices;
//   * the basis of the 13x13 expansion and the coefficient matrices S(dR, dt), Z(dR, dt) depend on
//     the two relative poses only and are filled in ONE phase, every thread deriving the entries
//     of dR / dt it needs itself (no dR -> dt -> coefficients barrier chain, no 3-thread fill);
//   * six barriers in all: loads | basis + coefficients | S M, Z M_q | congruences | W B | B^T (W B).
namespace {

constexpr int kEvalThreads = 128;

struct EvalSmem {
  double M[13][13];  // sum phi phi^T
  double Mq[7][7];   // sum zeta zeta^T
  double Sc[7][13];  // s = Sc phi
  double Zc[7][7];   // z = Zc zeta
  double T[7][13];   // Sc M
  double TZ[7][7];   // Zc Mq
  ExpandSmem exp;
  double Wp28[28], Wq28[28];
  double rel[12], rel0[12];
  LinTask task; // eval_global_kernel: the task / context blocks of this CTA
  LinArgs args;
};

__device__ __forceinline__ int eps3(int k, int a, int b) { // Levi-Civita symbol
  return (k == a || a == b || k == b) ? 0 : (((a - k + 3) % 3 == 1) ? 1 : -1);
}

// `a` may still be in flight when the body starts (eval_global_kernel loads it with the first
// phase): it is read after the first barrier only.
template <bool kErrorOnly>
__device__ __forceinline__ void eval_body(const LinArgs &a, const LinTask &task, EvalSmem &S) {
  const int tid = threadIdx.x;
  // ---- phase 0: the pair's cache entry into registers; zero fills while it travels ----
  const double *entry = task.entry;
  double ev = 0.0, r0v = 0.0;
  if (tid < kMomentPlanar + kMomentPoint) ev = __ldcg(entry + tid);
  if (tid < 12) r0v = __ldcg(entry + kMomentPlanar + kMomentPoint + tid);
  if (!kErrorOnly) zero_basis(S.exp);
  for (int i = tid; i < 7 * 13; i += kEvalThreads) (&S.Sc[0][0])[i] = 0.0;
  for (int i = tid; i < 7 * 7; i += kEvalThreads) (&S.Zc[0][0])[i] = 0.0;
  if (tid < kMomentPlanar) {
    int x = 0, e = tid;
    while (e >= 13 - x) {
      e -= 13 - x;
      ++x;
    }
    S.M[x][x + e] = ev;
    S.M[x + e][x] = ev;
  } else if (tid < kMomentPlanar + kMomentPoint) {
    int p = 0, e = tid - kMomentPlanar;
    while (e >= 7 - p) {
      e -= 7 - p;
      ++p;
    }
    S.Mq[p][p + e] = ev;
    S.Mq[p + e][p] = ev;
  }
  if (tid < 12) {
    S.rel0[tid] = r0v;
    S.rel[tid] = task.rel[tid];
  }
  __syncthreads();
  if (task.dyn_slot_i_plus1) {
    // queued right behind the association: an empty pair publishes nothing (the host learns
    // the counts from the association and does not wait for it)
    const int nb = a.W + 1, si = (int)task.dyn_slot_i_plus1 - 1;
    const uint32_t n = __ldcg(&a.pair_row[1 * nb + si]) + __ldcg(&a.pair_row[3 * nb + si]);
    if (n == 0) return; // CTA-uniform
  }
  // ---- phase 1: basis (threads 72..110) and coefficient matrices (threads 0..26, 32..40, 64..66,
  // 96; tests/test_moment_model.py: coeff_S, coeff_Z), both from rel / rel0 alone ----
  if (!kErrorOnly) fill_basis(S.exp, S.rel, 72);
  {
    const double *rel = S.rel, *rel0 = S.rel0;
    auto dR = [&](int r, int c) { // (R R0^T)[r][c]
      return rel[3 * r] * rel0[3 * c] + rel[3 * r + 1] * rel0[3 * c + 1] + rel[3 * r + 2] * rel0[3 * c + 2];
    };
    auto dt = [&](int k) { // t - dR t0
      return rel[9 + k] - (dR(k, 0) * rel0[9] + dR(k, 1) * rel0[10] + dR(k, 2) * rel0[11]);
    };
    if (tid < 27) { // (k, a, c): rows n x (dR q0)
      const int k = tid / 9, a_ = (tid / 3) % 3, c = tid % 3;
      double v = 0.0;
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        const int e = eps3(k, a_, b);
        if (e) v += (double)e * dR(b, c);
      }
      S.Sc[k][3 * a_ + c] = v;
    } else if (tid >= 32 && tid < 41) { // (k, a): rows n x dt, and the residual row
      const int k = (tid - 32) / 3, a_ = (tid - 32) % 3;
      double v = 0.0;
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        const int e = eps3(k, a_, b);
        if (e) v += (double)e * dt(b);
      }
      S.Sc[k][9 + a_] = v;
      const double d = dR(k, a_) - (k == a_ ? 1.0 : 0.0);
      S.Sc[6][3 * k + a_] = d;
      S.Zc[3 + k][a_] = d;
    } else if (tid >= 64 && tid < 67) {
      const int k = tid - 64;
      const double d = dt(k);
      S.Sc[3 + k][9 + k] = 1.0;
      S.Sc[6][9 + k] = d;
      S.Zc[k][k] = 1.0;
      S.Zc[k][3 + k] = -1.0;
      S.Zc[3 + k][3 + k] = 1.0;
      S.Zc[3 + k][6] = d;
    } else if (tid == 96) {
      S.Sc[6][12] = 1.0;
      S.Zc[6][6] = 1.0;
    }
  }
  __syncthreads();
  // ---- phase 2: T = Sc M (91 entries), TZ = Zc Mq (49 entries) ----
  for (int idx = tid; idx < 7 * 13 + 7 * 7; idx += kEvalThreads) {
    double v = 0.0;
    if (idx < 91) {
      const int k = idx / 13, y = idx % 13;
#pragma unroll
      for (int l = 0; l < 13; ++l) v += S.Sc[k][l] * S.M[l][y];
      S.T[k][y] = v;
    } else {
      const int j = idx - 91, k = j / 7, y = j % 7;
#pragma unroll
      for (int l = 0; l < 7; ++l) v += S.Zc[k][l] * S.Mq[l][y];
      S.TZ[k][y] = v;
    }
  }
  __syncthreads();
  // ---- phase 3: W_p = T Sc^T, W_q = TZ Zc^T (packed upper triangles, the order
  // expand_and_publish expects) ----
  if (tid < 56) {
    const int which = tid / 28;
    int p = 0, e = tid % 28;
    while (e >= 7 - p) {
      e -= 7 - p;
      ++p;
    }
    const int q = p + e;
    double v = 0.0;
    if (which == 0) {
#pragma unroll
      for (int y = 0; y < 13; ++y) v += S.T[p][y] * S.Sc[q][y];
      S.Wp28[tid] = v;
    } else {
#pragma unroll
      for (int y = 0; y < 7; ++y) v += S.TZ[p][y] * S.Zc[q][y];
      S.Wq28[tid - 28] = v;
    }
  }
  __syncthreads();
  const unsigned long long tag = a.seq & 0xffffffffull;
  if (kErrorOnly) {
    if (tid == 0) {
      // W_p[6][6] = sum r^2 (packed index 27), W_q[3][3], [4][4], [5][5] = sum |e|^2 (18, 22, 25)
      const double err = 0.5 * a.inv_sigma2 * (S.Wp28[27] + S.Wq28[18] + S.Wq28[22] + S.Wq28[25]);
      if (a.out_plain) a.out_plain[task.out_index] = err;
      else publish_tagged(a.out + 2 * (size_t)task.out_index, err, tag);
    }
    return;
  }
  // ---- phases 4-5: the 13x13 block ----
  expand_and_publish(S.exp, S.Wp28, S.Wq28, true, true, a.inv_sigma2, a.out + 182 * (size_t)task.out_index, tag,
                     a.out_plain ? a.out_plain + 91 * (size_t)task.out_index : nullptr);
}

} // namespace

template <bool kErrorOnly>
__global__ void __launch_bounds__(kEvalThreads) eval_inline_kernel(LinArgs a, LinInline req) {
  __shared__ EvalSmem s;
  eval_body<kErrorOnly>(a, req.tasks[blockIdx.x], s);
}

// tasks (and, for batched launches, the contexts' argument blocks) in device memory
template <bool kErrorOnly>
__global__ void __launch_bounds__(kEvalThreads)
eval_global_kernel(const LinArgs *ctx_args, const LinTask *tasks, int n_tasks) {
  __shared__ EvalSmem s;
  const int tid = threadIdx.x;
  if (tid < (int)(sizeof(LinTask) / 8))
    reinterpret_cast<unsigned long long *>(&s.task)[tid] =
        reinterpret_cast<const unsigned long long *>(tasks + blockIdx.x)[tid];
  // the context's argument block travels together with the cache entry (first phase of the body)
  if (tid >= 32 && tid < 32 + (int)(sizeof(LinArgs) / 8))
    reinterpret_cast<unsigned long long *>(&s.args)[tid - 32] =
        reinterpret_cast<const unsigned long long *>(ctx_args + tasks[blockIdx.x].ctx_index)[tid - 32];
  __syncthreads();
  pdl_wait(); // the cache entries come from the moment kernel queued before (batched submits)
  eval_body<kErrorOnly>(s.args, s.task, s);
}

void moments_launch(const MomentArgs &a, int max_units, cudaStream_t stream, Profiler &prof) {
  if (a.n_pairs <= 0 || max_units <= 0) return;
  prof.begin(FORMGPU_KG_LIN_CHUNK);
  moment_kernel<<<(max_units + kMomentWarps - 1) / kMomentWarps, kMomentThreads, 0, stream>>>(a);
  prof.end(FORMGPU_KG_LIN_CHUNK, 1);
}

void moments_batch_launch(const MomentArgs *items_dev, int n_items, int max_units, cudaStream_t stream,
                          Profiler &prof) {
  if (n_items <= 0 || max_units <= 0) return;
  prof.begin(FORMGPU_KG_LIN_CHUNK);
  launch_pdl(moment_batch_kernel, dim3((max_units + kMomentWarps - 1) / kMomentWarps, 1, n_items), kMomentThreads, 0,
             stream, items_dev);
  prof.end(FORMGPU_KG_LIN_CHUNK, 1);
}

cudaError_t eval_launch(const LinArgs &a, const LinInline *inline_req, bool error_only, cudaStream_t stream,
                        Profiler &prof) {
  if (a.n_tasks <= 0) return cudaSuccess;
  const int group = error_only ? FORMGPU_KG_ERR_FINALIZE : FORMGPU_KG_LIN_FINALIZE;
  const int grid = a.n_tasks;
  prof.begin(group);
  if (inline_req) {
    if (error_only) eval_inline_kernel<true><<<grid, kEvalThreads, 0, stream>>>(a, *inline_req);
    else eval_inline_kernel<false><<<grid, kEvalThreads, 0, stream>>>(a, *inline_req);
  } else {
    // the context's own argument block rides behind its tasks in the request buffer
    const LinArgs *args_dev = reinterpret_cast<const LinArgs *>(a.tasks + a.n_tasks);
    if (error_only) eval_global_kernel<true><<<grid, kEvalThreads, 0, stream>>>(args_dev, a.tasks, a.n_tasks);
    else eval_global_kernel<false><<<grid, kEvalThreads, 0, stream>>>(args_dev, a.tasks, a.n_tasks);
  }
  prof.end(group, 1);
  return cudaGetLastError();
}

cudaError_t eval_batch_launch(const LinArgs *ctx_args_dev, const LinTask *tasks_dev, int n_tasks,
                              bool error_only, cudaStream_t stream, Profiler &prof) {
  if (n_tasks <= 0) return cudaSuccess;
  const int group = error_only ? FORMGPU_KG_ERR_FINALIZE : FORMGPU_KG_LIN_FINALIZE;
  const int grid = n_tasks;
  prof.begin(group);
  const cudaError_t e =
      error_only ? launch_pdl(eval_global_kernel<true>, grid, kEvalThreads, 0, stream, ctx_args_dev, tasks_dev, n_tasks)
                 : launch_pdl(eval_global_kernel<false>, grid, kEvalThreads, 0, stream, ctx_args_dev, tasks_dev, n_tasks);
  prof.end(group, 1);
  return e != cudaSuccess ? e : cudaGetLastError();
}

} // namespace formgpu
