// The canonical fp64 distance of the core-set stage.  Every kernel that computes d(i,c) — the row norms, the passes,
// the segment filter and the candidate x candidate tiles of coreset.cu, the re-score of the tcgen05 initialisation in
// tc_dist.cu — builds it from the functions below, so d(i,c) has the same bits wherever it is computed.  The planner's
// replay of a pass, the pruning test and the screen's "fmin(m_old, d) == m_old" all rest on that.
#pragma once

#include "common.cuh"

namespace vatlq {

// ---- the fp64 tensor-core tile --------------------------------------------------------------
// mma.sync.m8n8k4.f64 (DMMA; measured 18.5 T FMA/s on B200, tools/micro/fp64_rate.cu): a warp
// computes 8 rows x 8 centers per instruction with ONE A and ONE B operand per lane, so the
// register tile is tiny (2 doubles per 8x8 block) and shared-memory traffic is 1/8 of a scalar
// DFMA register tile.  Lane (g = lane>>2, kk = lane&3) owns row g of an 8-row block and feeds,
// for super-step s (16 features), the float4 x[row][16s+4kk .. +3]; element e of that float4
// is k-slot kk of MMA e, i.e. feature 16s+4kk+e.  The B operand of lane (g, kk) is center g
// at the same feature.  Output: lane holds (row g, centers 2kk and 2kk+1).
//
// CANONICAL DOT: the feature axis is cut into kSeg = 8 segments of ceil(nss/8) super-steps.
// Inside a segment, element e (0..3) of every float4 feeds its own sequential DMMA chain
// (four independent chains hide the dependent-issue latency of DMMA), and
//   P_seg = (c_0 + c_1) + (c_2 + c_3),   dot = ((P0 + P1) + (P2 + P3)) + ((P4 + P5) + (P6 + P7)).
// Every kernel (norms, pass, candidate pairs, pairwise) evaluates exactly this, so d(i,c) has
// the same bits wherever it is computed and dot(x,x) == xx (d(c,c) == 0).  In the pass the eight
// segments of a block are computed by eight warps in parallel (split-K): a warp then only ever
// needs 1/8 of every centre, which fits its REGISTERS (see pass_kernel_tma).
constexpr int kSeg = 8;
constexpr int kSteps = 16;                    // super-steps per segment at the fast width
constexpr int kFastD = kSeg * kSteps * 16;    // 2048: the width of the register-resident centre slices

// ELEMENT TYPES of X (VATLQ_F32 / F16 / BF16): every kernel that reads X is a template on the element type T and
// reads it a quad (four consecutive features: a float4 in fp32, a uint2 in 16 bits, common.cuh) at a time, widened
// exactly to fp32 at the load; from there on the fp64 arithmetic is the same instruction sequence in every type, so
// a 16-bit X gives every output of its fp32 upcast bit for bit.
template <typename T>
using quad_t = typename QuadOf<T>::type;
template <typename T>
__device__ __forceinline__ float4 ldg_q(const quad_t<T>* p) { return quad_f32(__ldg(p), (const T*)nullptr); }

__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c[0]), "+d"(c[1])
      : "d"(a), "d"(b));
}

__device__ __forceinline__ double combine4(double p0, double p1, double p2, double p3) {
  return __dadd_rn(__dadd_rn(p0, p1), __dadd_rn(p2, p3));
}
__device__ __forceinline__ double combine8(const double* p, int stride) {
  return __dadd_rn(combine4(p[0], p[stride], p[2 * stride], p[3 * stride]),
                   combine4(p[4 * stride], p[5 * stride], p[6 * stride], p[7 * stride]));
}

// d(i,c)^2 and d(i,c) from the canonical dot, in sklearn's order: (-2 x.c + |x|^2) + |c|^2
__device__ __forceinline__ double sq_from_dot(double dot, double xxi, double xxc) {
  double t = __dmul_rn(-2.0, dot);
  t = __dadd_rn(t, xxi);
  return __dadd_rn(t, xxc);
}
__device__ __forceinline__ double dist_from_dot(double dot, double xxi, double xxc) {
  return sqrt(fmax(sq_from_dot(dot, xxi, xxc), 0.0));
}

// ---- the fast width (d == kFastD): warp `seg` of a CTA computes K-segment seg, kSteps super-steps, for 8 rows
// against 8 centres; the split-K exchange (seg_partial, then combine8 over the 8 warps) finishes the dots.
// Lane (g, kk)'s B operands: its 1/8 of centre `row` of X (d4 quads per row), held in registers for a whole pass.
template <typename T>
__device__ __forceinline__ void centre_slice(const T* X, int d4, long long row, int seg, int kk, double (&b)[kSteps][4]) {
  const quad_t<T>* cp = reinterpret_cast<const quad_t<T>*>(X) + (size_t)row * d4 + seg * (kSteps * 4) + kk;
#pragma unroll
  for (int s = 0; s < kSteps; ++s) {
    const float4 v = ldg_q<T>(cp + 4 * s);
    b[s][0] = (double)v.x;
    b[s][1] = (double)v.y;
    b[s][2] = (double)v.z;
    b[s][3] = (double)v.w;
  }
}
// one super-step: element e of the lane's A quad x and of its B operands feeds chain c[e]
__device__ __forceinline__ void seg_step(double (&c)[4][2], const float4& x, const double (&b)[4]) {
  dmma(c[0], (double)x.x, b[0]);
  dmma(c[1], (double)x.y, b[1]);
  dmma(c[2], (double)x.z, b[2]);
  dmma(c[3], (double)x.w, b[3]);
}
__device__ __forceinline__ void seg_step(double (&c)[4][2], const float4& x, const float4& b) {
  dmma(c[0], (double)x.x, (double)b.x);
  dmma(c[1], (double)x.y, (double)b.y);
  dmma(c[2], (double)x.z, (double)b.z);
  dmma(c[3], (double)x.w, (double)b.w);
}
// the segment's partial dots of (row g, centres 2kk and 2kk+1), as a warp stores them for the split-K exchange
__device__ __forceinline__ double2 seg_partial(const double (&c)[4][2]) {
  return make_double2(combine4(c[0][0], c[1][0], c[2][0], c[3][0]), combine4(c[0][1], c[1][1], c[2][1], c[3][1]));
}

// The pruning test (coreset.cu, "pruning (exact)"): no row of a segment (anchor a with |a|^2 = xxa, radius R, largest
// min_d M of its rows) can get closer to a group of centres whose nearest squared canonical distance to a is d2min and
// whose largest squared norm is cn_max.  The margin is orders of magnitude above the rounding of the canonical
// distances, so a skipped segment keeps every min_d bit for bit.
__device__ __forceinline__ bool segment_skip(double d2min, double R, double M, double xxa, double cn_max) {
  const double margin = 1e-6 * (1.0 + sqrt(xxa) + sqrt(cn_max));
  return isfinite(M) && sqrt(fmax(d2min, 0.0)) - R - M >= margin;
}

}  // namespace vatlq
