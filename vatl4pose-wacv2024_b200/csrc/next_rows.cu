// SURVEY.md §8f "next" rows on the device:
//   * pose-level uncertainties HP and TPC from the scan's outputs  (ActiveLearning.py:329-344,736-745)
//   * heat-map Entropy as one more streaming pass                  (ActiveLearning.py:790-796)
//   * Influence / Diversity: row sums of the cosine-distance matrix (ActiveLearning.py:467-483,581-590)
//   * the uncertainty / representativeness blend                   (ActiveLearning.py:517-521)
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace vatlq {

// ------------------------------------------------------------------------------------
// HP and TPC.  One thread per frame; everything comes from the scan's outputs.
//   HP  = float(-np.sum(pose_scores))                      (:329-330)  fp32, numpy's pairwise order
//   TPC = #joints with |p_t - p_adj|_2 > thresh, p_adj decoded from frame t-1 / t+1's heat maps
//         with frame t's crop box; x2 rule like THC         (:333-344, compute_tpc :736-745)
// ------------------------------------------------------------------------------------
// np.add.reduce over n contiguous fp32 values, n < 128: eight strided accumulators over the
// leading multiple of 8, combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail.
__device__ __forceinline__ float np_sum_f32(const float* a, int stride, int n) {
  if (n < 8) {
    float res = 0.f;
    for (int i = 0; i < n; ++i) res = __fadd_rn(res, a[(size_t)i * stride]);
    return res;
  }
  float r[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = a[(size_t)k * stride];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = __fadd_rn(r[k], a[(size_t)(i + k) * stride]);
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __fadd_rn(res, a[(size_t)i * stride]);
  return res;
}

struct Affine {  // inverse crop transform of transforms.py:753-792 (rot = 0), see scan_finalize
  double a, c, e, f;
};
__device__ __forceinline__ Affine affine_of(const float* bbox, int h, int w) {
  const double xmin = bbox[0], ymin = bbox[1], xmax = bbox[2], ymax = bbox[3];
  const double bw = __dsub_rn(xmax, xmin), bh = __dsub_rn(ymax, ymin);
  const double cxd = __dadd_rn(xmin, __dmul_rn(bw, 0.5)), cyd = __dadd_rn(ymin, __dmul_rn(bh, 0.5));
  const float X0 = (float)cxd, Y0 = (float)cyd;
  const float Y1 = (float)__dadd_rn(cyd, __dmul_rn(bw, -0.5));
  const float dY = __fsub_rn(Y0, Y1);
  const float X2 = __fsub_rn(X0, dY);
  const double W2 = 0.5 * (double)w, H2 = 0.5 * (double)h;
  Affine t;
  t.a = __ddiv_rn(__dsub_rn((double)X0, (double)X2), W2);
  t.c = (double)X2;
  t.e = __ddiv_rn(__dsub_rn((double)Y0, (double)Y1), W2);
  t.f = __dsub_rn((double)Y1, __dmul_rn(t.e, __dsub_rn(H2, W2)));
  return t;
}

__global__ void __launch_bounds__(128)
pose_unc_kernel(const float* __restrict__ coords_hm, const float* __restrict__ kpts, const float* __restrict__ bbox,
                const uint8_t* __restrict__ is_prev, const uint8_t* __restrict__ is_next, int64_t n, int J, int h,
                int w, const float* __restrict__ halo_prev_xy, const float* __restrict__ halo_next_xy,
                float* __restrict__ hp, float* __restrict__ tpc) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  if (hp) hp[t] = -np_sum_f32(kpts + (size_t)t * J * 3 + 2, 3, J);
  if (!tpc) return;
  const bool has_p = is_prev && is_prev[t] && (t > 0 || halo_prev_xy);
  const bool has_n = is_next && is_next[t] && (t < n - 1 || halo_next_xy);
  int cnt = 0;
  if (has_p || has_n) {
    const float* b = bbox + (size_t)t * 4;
    const Affine T = affine_of(b, h, w);
    // thresh = 0.01 * sqrt((x2-x1)*(y2-y1)) on python floats (:334)
    const double thresh = __dmul_rn(0.01, sqrt(__dmul_rn(__dsub_rn((double)b[2], (double)b[0]),
                                                         __dsub_rn((double)b[3], (double)b[1]))));
    const float* cur = coords_hm + (size_t)t * J * 2;
    for (int side = 0; side < 2; ++side) {
      if (!(side ? has_n : has_p)) continue;
      const float* adj = side ? (t < n - 1 ? cur + (size_t)J * 2 : halo_next_xy)
                              : (t > 0 ? cur - (size_t)J * 2 : halo_prev_xy);
      for (int j = 0; j < J; ++j) {
        const float cx = (float)__dadd_rn(__dmul_rn(T.a, (double)cur[2 * j]), T.c);
        const float cy = (float)__dadd_rn(__dmul_rn(T.e, (double)cur[2 * j + 1]), T.f);
        const float ax = (float)__dadd_rn(__dmul_rn(T.a, (double)adj[2 * j]), T.c);
        const float ay = (float)__dadd_rn(__dmul_rn(T.e, (double)adj[2 * j + 1]), T.f);
        // np.linalg.norm(axis=1) on float32: sqrt(dx*dx + dy*dy) in fp32; the comparison with the
        // float64 threshold promotes to float64
        const float dx = __fsub_rn(cx, ax), dy = __fsub_rn(cy, ay);
        const float dist = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
        cnt += ((double)dist > thresh) ? 1 : 0;
      }
    }
    if (has_p != has_n) cnt *= 2;   // only one neighbour: doubled (:340-343)
  }
  tpc[t] = (float)cnt;
}

// ------------------------------------------------------------------------------------
// Entropy (:790-796): per joint scipy.stats.entropy(map.flatten()) = sum(entr(p)), p = x / sum(x)
// in fp32 (entr(p) = -p log p for p > 0, 0 at 0, -inf below 0); summed over the joints.
// One warp per (frame, joint) map: the map is read from HBM once and kept in registers between
// the sum and the entr pass when it is a 64x48 map (24 float4 per lane).
// ------------------------------------------------------------------------------------
// entr(p) with the MUFU logarithm (lg2 * ln 2: relative error ~1e-7 on log p, far inside the 1e-5
// budget).  Branch-free: tiny p (MUFU flushes denormals) are scaled by 2^64 first.
__device__ __forceinline__ float entr_f32(float p) {
  const bool tiny = p < 1e-30f;
  const float l2 = __log2f(p * (tiny ? 18446744073709551616.f : 1.f)) - (tiny ? 64.f : 0.f);
  float e = -p * (l2 * 0.69314718055994531f);     // p < 0: NaN here, fixed below; NaN p stays NaN
  e = (p == 0.f) ? 0.f : e;
  e = (p < 0.f) ? -INFINITY : e;
  return e;
}

// NV quads per lane when the map is NV*128 pixels, 0: generic (second read from L2).  T: fp32, or a 16-bit type read
// as 8-byte quads and converted exactly in registers (same pixels per lane and chain: the bits of the fp32 upcast).
template <int NV, typename T>
__global__ void __launch_bounds__(256, 2)
entropy_kernel(const T* __restrict__ H, int64_t maps, int npx, float* __restrict__ per_map) {
  const int lane = threadIdx.x & 31;
  const int64_t mi = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (mi >= maps) return;
  const T* mp = H + (size_t)mi * npx;
  double acc = 0.0;
  float e;
  if (NV > 0) {
    float4 v[NV > 0 ? NV : 1];
#pragma unroll
    for (int q = 0; q < NV; ++q) v[q] = ldg_stream_quad(mp, q * 32 + lane);
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
      s += (v[q].x + v[q].y) + (v[q].z + v[q].w);
      if ((q & 3) == 3) {  // bound the fp32 run length
        acc += (double)s;
        s = 0.f;
      }
    }
    acc += (double)s;
    const float S = (float)warp_sum(acc);   // np.sum(pk) is fp32
    if (S > 1e-10f && S < 1e30f) {
      // ordinary map (positive finite sum; a NaN pixel makes S NaN and takes the other branch):
      //   sum_i entr(x_i / S) = ln S - (ln 2 / S) * sum_i x_i lg2 x_i        (sum_i x_i / S = 1 to fp32 rounding)
      // one MUFU + four ALU instructions per pixel instead of twelve; within 2e-7 of the elementwise form
      // (checked against scipy on the golden maps).  Any negative pixel makes the reference's sum -inf.
      double ta = 0.0;
      float vmin = INFINITY;
#pragma unroll
      for (int q = 0; q < NV; ++q) {
        const float4 x = v[q];
        const float t0 = x.x > 1e-30f ? x.x * __log2f(x.x) : 0.f, t1 = x.y > 1e-30f ? x.y * __log2f(x.y) : 0.f;
        const float t2 = x.z > 1e-30f ? x.z * __log2f(x.z) : 0.f, t3 = x.w > 1e-30f ? x.w * __log2f(x.w) : 0.f;
        vmin = fminf(vmin, fminf(fminf(x.x, x.y), fminf(x.z, x.w)));
        ta += (double)((t0 + t1) + (t2 + t3));
      }
      const double T = warp_sum(ta);
#pragma unroll
      for (int o = 16; o; o >>= 1) vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
      const double ln2 = 0.69314718055994531;
      e = (vmin < 0.f) ? -INFINITY : (float)((double)__log2f(S) * ln2 - (ln2 / (double)S) * T);
    } else {
      // p = x / S as x * (1/S) when 1/S is a normal number (within 1 ulp of numpy's quotient), else
      // the IEEE division (S == 0 -> inf / NaN exactly like numpy)
      const float rS = __frcp_rn(S);
      const bool mul = fabsf(rS) > 1e-30f && fabsf(rS) < 1e30f;
      double ea = 0.0;
#pragma unroll
      for (int q = 0; q < NV; ++q) {
        float4 p;
        if (mul) p = make_float4(v[q].x * rS, v[q].y * rS, v[q].z * rS, v[q].w * rS);
        else p = make_float4(__fdiv_rn(v[q].x, S), __fdiv_rn(v[q].y, S), __fdiv_rn(v[q].z, S), __fdiv_rn(v[q].w, S));
        const float e4 = (entr_f32(p.x) + entr_f32(p.y)) + (entr_f32(p.z) + entr_f32(p.w));
        ea += (double)e4;
      }
      e = (float)warp_sum(ea);
    }
  } else {
    for (int i = lane; i < npx; i += 32) acc += (double)to_f32(mp[i]);
    const float S = (float)warp_sum(acc);
    double ea = 0.0;
    for (int i = lane; i < npx; i += 32) ea += (double)entr_f32(__fdiv_rn(to_f32(mp[i]), S));
    e = (float)warp_sum(ea);
  }
  if (lane == 0) per_map[mi] = e;
}

// The same arithmetic with the scan's staging (heatmap_scan.cu): one warp walks a run of consecutive 64x48 maps, each
// map fetched by ONE 12 288-byte cp.async.bulk (TMA, UBLKCP) into the warp's own two-stage shared-memory ring, so the
// next map is in flight while this one is summed and turned into entr() — no occupancy-bound register staging.
constexpr int kEntWarps = 8, kEntStages = 2, kEntNV = 24, kEntPix = kEntNV * 128;
constexpr size_t kEntSmem = (size_t)kEntWarps * kEntStages * kEntPix * 4 + (size_t)kEntWarps * kEntStages * 8;
__global__ void __launch_bounds__(kEntWarps * 32, 1)
entropy_tma_kernel(const float* __restrict__ H, int64_t maps, int run_len, float* __restrict__ per_map) {
  extern __shared__ __align__(128) unsigned char ent_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t a = ((int64_t)blockIdx.x * kEntWarps + warp) * run_len;
  if (a >= maps) return;
  const int64_t count = min((int64_t)run_len, maps - a);
  float* stage0 = reinterpret_cast<float*>(ent_smem) + (size_t)warp * kEntStages * kEntPix;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ent_smem + (size_t)kEntWarps * kEntStages * kEntPix * 4) + warp * kEntStages;
  if (lane == 0) {
    for (int st = 0; st < kEntStages; ++st) mbar_init(&bars[st], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int st = 0; st < kEntStages && st < count; ++st) {
      mbar_expect_tx(&bars[st], kEntPix * 4);
      tma_load_1d(stage0 + (size_t)st * kEntPix, H + (size_t)(a + st) * kEntPix, kEntPix * 4, &bars[st]);
    }
  }
  __syncwarp();
  for (int64_t i = 0; i < count; ++i) {
    const int st = (int)(i % kEntStages);
    mbar_wait(&bars[st], (uint32_t)((i / kEntStages) & 1));
    const float4* m4 = reinterpret_cast<const float4*>(stage0 + (size_t)st * kEntPix);
    float4 v[kEntNV];
#pragma unroll
    for (int q = 0; q < kEntNV; ++q) v[q] = m4[q * 32 + lane];
    // the stage is free as soon as the map sits in registers: refill it now (maximum lead time)
    __syncwarp();
    if (lane == 0 && i + kEntStages < count) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(&bars[st], kEntPix * 4);
      tma_load_1d(stage0 + (size_t)st * kEntPix, H + (size_t)(a + i + kEntStages) * kEntPix, kEntPix * 4, &bars[st]);
    }
    double acc = 0.0;
    float sm = 0.f;
#pragma unroll
    for (int q = 0; q < kEntNV; ++q) {       // (identical order to entropy_kernel<24, float>: same bits)
      sm += (v[q].x + v[q].y) + (v[q].z + v[q].w);
      if ((q & 3) == 3) {
        acc += (double)sm;
        sm = 0.f;
      }
    }
    acc += (double)sm;
    const float S = (float)warp_sum(acc);
    const float rS = __frcp_rn(S);
    const bool mul = fabsf(rS) > 1e-30f && fabsf(rS) < 1e30f;
    double ea = 0.0;
#pragma unroll
    for (int q = 0; q < kEntNV; ++q) {
      float4 p;
      if (mul) p = make_float4(v[q].x * rS, v[q].y * rS, v[q].z * rS, v[q].w * rS);
      else p = make_float4(__fdiv_rn(v[q].x, S), __fdiv_rn(v[q].y, S), __fdiv_rn(v[q].z, S), __fdiv_rn(v[q].w, S));
      const float e4 = (entr_f32(p.x) + entr_f32(p.y)) + (entr_f32(p.z) + entr_f32(p.w));
      ea += (double)e4;
    }
    const float e = (float)warp_sum(ea);
    if (lane == 0) per_map[a + i] = e;
  }
}

// entropy_value += entropy(heatmap) over the joints, in joint order (:793-795)
__global__ void __launch_bounds__(256)
entropy_frames_kernel(const float* __restrict__ per_map, int64_t n, int J, float* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  double tot = 0.0;
  for (int j = 0; j < J; ++j) tot += (double)per_map[(size_t)t * J + j];
  out[t] = (float)tot;
}

// ------------------------------------------------------------------------------------
// Influence / Diversity.  KNeighborsTransformer(mode='distance', metric='cosine',
// n_neighbors=m-1).fit_transform(X_sub) holds every pairwise cosine distance, and the score is
// its row sum: sum_j (1 - xh_i . xh_j) = m - xh_i . S with S = sum_j xh_j, xh = x / |x|
// (sklearn normalize: a zero row stays zero; its self-distance is the zeroed diagonal, so its row
// sum is m - 1 — for pools small enough that sklearn's pairwise_distances_chunked takes one chunk,
// which is where `X is Y` holds; zero embeddings do not occur after ReLU + average pooling except
// for the reference's all-zero fvecs_matrix, :270,283, where the normalised score is 0/0 either
// way).  O(m d) instead of O(m^2 d), two streaming
// passes over the rows, fp64 accumulation.
//   colsum: every warp walks rows, keeps its share of S in registers (d <= 2048: 16 float4
//           columns per lane), CTA partials land in the workspace and are added in a fixed order.
//   rowsum: out_i = m_total - (x_i . S) / |x_i|.
// ------------------------------------------------------------------------------------
constexpr int kCosNV = 16;        // float4 per lane per row: d <= 2048
constexpr int kCosThreads = 256;
constexpr int kCosRows = kCosThreads / 32;   // rows per tile: one per warp

__device__ __forceinline__ const float4* cos_row(const float* X, int d, const int64_t* rows, int64_t i) {
  const int64_t r = rows ? rows[i] : i;
  return reinterpret_cast<const float4*>(X + (size_t)r * d);
}

// column sums of the normalised rows.  A CTA takes tiles of 8 rows: warp w loads row w (streamed
// through shared memory, the squared norm reduced on the way), then every thread adds the 8
// scaled rows into the (up to two) float4 columns it owns.  CTA partials -> workspace.
__global__ void __launch_bounds__(kCosThreads, 2)
cos_colsum_kernel(const float* __restrict__ X, int d, const int64_t* __restrict__ rows, int64_t m,
                  double* __restrict__ partial /* gridDim.x x d */) {
  extern __shared__ __align__(16) unsigned char cos_smem[];
  float4* s_x = reinterpret_cast<float4*>(cos_smem);   // kCosRows x d4
  __shared__ double s_inv[kCosRows];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int d4 = d >> 2;
  double acc[2][4] = {{0.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 0.0}};
  const int64_t tiles = (m + kCosRows - 1) / kCosRows;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t i = tile * kCosRows + warp;
    double nn = 0.0;
    if (i < m) {
      const float4* rp = cos_row(X, d, rows, i);
#pragma unroll 8
      for (int q = 0; q < kCosNV; ++q) {
        const int c = q * 32 + lane;
        if (c < d4) {
          const float4 v = ldg_stream(rp + c);
          s_x[warp * d4 + c] = v;
          nn = fma((double)v.x, (double)v.x, nn);
          nn = fma((double)v.y, (double)v.y, nn);
          nn = fma((double)v.z, (double)v.z, nn);
          nn = fma((double)v.w, (double)v.w, nn);
        }
      }
    }
    nn = warp_sum(nn);
    // rows past the end scale whatever the stage holds by 0 (it holds finite leftovers or zeros)
    if (lane == 0) s_inv[warp] = (i < m) ? (nn > 0.0 ? 1.0 / sqrt(nn) : 1.0) : 0.0;
    __syncthreads();
    const int nr = (int)min((int64_t)kCosRows, m - tile * kCosRows);
    for (int r = 0; r < nr; ++r) {
      const double inv = s_inv[r];
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int c = threadIdx.x + hh * kCosThreads;
        if (c < d4) {
          const float4 v = s_x[r * d4 + c];
          acc[hh][0] = fma((double)v.x, inv, acc[hh][0]);
          acc[hh][1] = fma((double)v.y, inv, acc[hh][1]);
          acc[hh][2] = fma((double)v.z, inv, acc[hh][2]);
          acc[hh][3] = fma((double)v.w, inv, acc[hh][3]);
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    const int c = threadIdx.x + hh * kCosThreads;
    if (c < d4) {
      double* o = partial + (size_t)blockIdx.x * d + (size_t)c * 4;
      o[0] = acc[hh][0]; o[1] = acc[hh][1]; o[2] = acc[hh][2]; o[3] = acc[hh][3];
    }
  }
}

__global__ void __launch_bounds__(256)
cos_colsum_reduce_kernel(const double* __restrict__ partial, int parts, int d, double* __restrict__ S) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= d) return;
  double s = 0.0;
  for (int p = 0; p < parts; ++p) s += partial[(size_t)p * d + col];
  S[col] = s;
}

// out_i = m_total - (x_i . S) / |x_i|: one warp per row, S in shared memory
__global__ void __launch_bounds__(kCosThreads)
cos_rowsum_kernel(const float* __restrict__ X, int d, const int64_t* __restrict__ rows, int64_t m,
                  const double* __restrict__ S, double m_total, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char cos_smem[];
  double* s_S = reinterpret_cast<double*>(cos_smem);   // d doubles
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int d4 = d >> 2;
  for (int c = threadIdx.x; c < d; c += blockDim.x) s_S[c] = S[c];
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * nw + warp; i < m; i += (int64_t)gridDim.x * nw) {
    const float4* rp = cos_row(X, d, rows, i);
    double nn = 0.0, dot = 0.0;
#pragma unroll
    for (int q0 = 0; q0 < kCosNV; q0 += 8) {
      float4 v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int c = (q0 + q) * 32 + lane;
        v[q] = (c < d4) ? ldg_stream(rp + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int c = (q0 + q) * 32 + lane;
        if (c < d4) {
          const double2 sa = *reinterpret_cast<const double2*>(s_S + (size_t)c * 4);
          const double2 sb = *reinterpret_cast<const double2*>(s_S + (size_t)c * 4 + 2);
          nn = fma((double)v[q].x, (double)v[q].x, nn);
          nn = fma((double)v[q].y, (double)v[q].y, nn);
          nn = fma((double)v[q].z, (double)v[q].z, nn);
          nn = fma((double)v[q].w, (double)v[q].w, nn);
          dot = fma((double)v[q].x, sa.x, dot);
          dot = fma((double)v[q].y, sa.y, dot);
          dot = fma((double)v[q].z, sb.x, dot);
          dot = fma((double)v[q].w, sb.y, dot);
        }
      }
    }
    nn = warp_sum(nn);
    dot = warp_sum(dot);
    // a zero row has cosine distance 1 to every other row and 0 to itself (sklearn zeroes the
    // diagonal when the graph is built over the fitted rows themselves): m_total - 1
    if (lane == 0) out[i] = nn > 0.0 ? m_total - dot / sqrt(nn) : m_total - 1.0;
  }
}

// min / -max of a float64 vector over the rows with mask != 0 (same layout as fuse stats2)
__device__ __forceinline__ void atomic_min_f64_(double* addr, double val) {
  unsigned long long* a = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *a;
  while (true) {
    const double cur = __longlong_as_double((long long)old);
    if (cur <= val) return;
    const unsigned long long prev = atomicCAS(a, old, (unsigned long long)__double_as_longlong(val));
    if (prev == old) return;
    old = prev;
  }
}

__global__ void __launch_bounds__(256)
minmax_stats_f64_kernel(const double* __restrict__ v, const uint8_t* __restrict__ mask, int64_t n, double* stats2) {
  __shared__ double s[2][8];
  double lo = INFINITY, nhi = INFINITY;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (mask && !mask[i]) continue;
    const double x = v[i];
    if (x != x) lo = nhi = -INFINITY;   // a NaN makes np.min / np.max NaN: (min, -max) = (-inf, -inf) turns every score into NaN
    lo = fmin(lo, x);
    nhi = fmin(nhi, -x);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    nhi = fmin(nhi, __shfl_xor_sync(0xffffffffu, nhi, o));
  }
  if ((threadIdx.x & 31) == 0) {
    s[0][threadIdx.x >> 5] = lo;
    s[1][threadIdx.x >> 5] = nhi;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    double r = s[threadIdx.x][0];
    for (int k = 1; k < (int)(blockDim.x >> 5); ++k) r = fmin(r, s[threadIdx.x][k]);
    atomic_min_f64_(stats2 + threadIdx.x, r);
  }
}

// total = cw * unc + (1 - cw) * influence  (:519), 0 on labelled rows; every step one IEEE op
__global__ void __launch_bounds__(256)
blend_kernel(const double* __restrict__ unc, const double* __restrict__ infl, const uint8_t* __restrict__ mask,
             int64_t n, double cw, double* __restrict__ out) {
  const double ncw = __dsub_rn(1.0, cw);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (mask && !mask[i]) out[i] = 0.0;
    else out[i] = __dadd_rn(__dmul_rn(cw, unc[i]), __dmul_rn(ncw, infl[i]));
  }
}

static unsigned grid_1d(long long n) {
  long long g = (n + 255) / 256;
  const long long cap = (long long)sm_count() * 8;
  return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace vatlq

using namespace vatlq;

extern "C" int vatlq_pose_unc(const float* coords_hm, const float* kpts, const float* bbox_xyxy,
                              const uint8_t* is_prev, const uint8_t* is_next, int64_t n, int J, int h, int w,
                              const float* halo_prev_xy, const float* halo_next_xy, float* hp, float* tpc,
                              vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(n >= 0 && J > 0 && J < 128 && h > 0 && w > 0, "bad shape");
  VQ_REQUIRE(hp == nullptr || kpts != nullptr, "HP needs kpts");
  VQ_REQUIRE(tpc == nullptr || (coords_hm != nullptr && bbox_xyxy != nullptr), "TPC needs coords_hm and bbox_xyxy");
  if (n == 0 || (!hp && !tpc)) return 0;
  pose_unc_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(coords_hm, kpts, bbox_xyxy, is_prev, is_next, n, J,
                                                                   h, w, halo_prev_xy, halo_next_xy, hp, tpc);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_heatmap_entropy_dt(const void* H_, int dtype, int64_t n, int J, int h, int w, float* entropy,
                                        void* ws, size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(n >= 0 && J > 0 && h > 0 && w > 0, "bad shape");
  VQ_REQUIRE(dtype_size(dtype) != 0, "unknown dtype (VATLQ_F32, VATLQ_F16 or VATLQ_BF16)");
  if (n == 0) return 0;
  VQ_REQUIRE(H_ && entropy, "null pointer");
  const int64_t maps = n * J;
  VQ_REQUIRE(ws != nullptr && ws_bytes >= (size_t)maps * sizeof(float), "workspace must hold n*J floats");
  VQ_REQUIRE((maps + 7) / 8 <= 2147483647LL, "grid too large");
  const int npx = h * w;
  const unsigned grid = (unsigned)((maps + 7) / 8);
  if (dtype != VATLQ_F32) {
    // the TMA variant below is fp32 only: 16-bit maps take the register-staged kernel whatever VATLQ_ENTROPY_TMA says
    VQ_REQUIRE(npx != 24 * 128 || quad_aligned(H_, dtype), "16-bit H must be 8-byte aligned");
    const int rc = with_dtype(dtype, [&](auto tag) {
      using T = std::remove_const_t<std::remove_pointer_t<decltype(tag)>>;
      if (npx == 24 * 128) entropy_kernel<24, T><<<grid, 256, 0, stream>>>((const T*)H_, maps, npx, (float*)ws);
      else entropy_kernel<0, T><<<grid, 256, 0, stream>>>((const T*)H_, maps, npx, (float*)ws);
      VQ_LAUNCHED();
      return 0;
    });
    if (rc != 0) return rc;
    entropy_frames_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>((const float*)ws, n, J, entropy);
    VQ_LAUNCHED();
    return 0;
  }
  const float* H = (const float*)H_;
  // Measured on B200 (tools/time_next_rows.py, 40 000 frames): the TMA-staged variant runs at 2.5 TB/s, the
  // register-staged one at 3.9 TB/s — the kernel is bound by the ~1.4 k instructions per lane and map (MUFU.LG2 chain),
  // and 8 warps per SM (196 KB of stages) hide less of that than 16 resident warps do.  Kept for experiments only.
  static const bool use_tma = []() {
    const char* e = getenv("VATLQ_ENTROPY_TMA");
    return e && e[0] == '1';
  }();
  if (npx == kEntPix && ((uintptr_t)H & 15) == 0 && use_tma && maps >= 4096) {
    static bool cfg = false;
    if (!cfg) {
      VQ_CUDA(cudaFuncSetAttribute(entropy_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEntSmem));
      cfg = true;
    }
    // runs long enough to amortise the ring fill, short enough for ~4 waves of warps over the SMs
    const int64_t warps = (int64_t)sm_count() * kEntWarps * 4;
    const int run_len = (int)std::max<int64_t>(4, std::min<int64_t>(64, (maps + warps - 1) / warps));
    const int64_t tasks = (maps + run_len - 1) / run_len;
    entropy_tma_kernel<<<(unsigned)((tasks + kEntWarps - 1) / kEntWarps), kEntWarps * 32, kEntSmem, stream>>>(H, maps, run_len, (float*)ws);
  } else if (npx == 24 * 128 && ((uintptr_t)H & 15) == 0)
    entropy_kernel<24, float><<<grid, 256, 0, stream>>>(H, maps, npx, (float*)ws);
  else
    entropy_kernel<0, float><<<grid, 256, 0, stream>>>(H, maps, npx, (float*)ws);
  VQ_LAUNCHED();
  entropy_frames_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>((const float*)ws, n, J, entropy);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_heatmap_entropy(const float* H, int64_t n, int J, int h, int w, float* entropy,
                                     void* ws, size_t ws_bytes, vatlq_stream_t stream) {
  return vatlq_heatmap_entropy_dt(H, VATLQ_F32, n, J, h, w, entropy, ws, ws_bytes, stream);
}

static int cos_grid(int64_t m) {
  const int nw = kCosThreads / 32;
  int64_t g = (m + nw - 1) / nw;
  const int64_t cap = (int64_t)sm_count() * 2;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

extern "C" size_t vatlq_cosine_workspace_bytes(int d) {
  if (d <= 0) return 0;
  return (size_t)sm_count() * 2 * (size_t)d * sizeof(double);
}

extern "C" int vatlq_cosine_colsum(const float* X, int64_t n, int d, const int64_t* rows, int64_t m,
                                   double* S, void* ws, size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(X && S && n >= 0 && m >= 0, "null pointer");
  VQ_REQUIRE(d > 0 && (d & 3) == 0 && d <= kCosNV * 128, "d must be a multiple of 4 and <= 2048");
  VQ_REQUIRE(((uintptr_t)X & 15) == 0, "X must be 16-byte aligned");
  VQ_REQUIRE(rows != nullptr || m == n, "m must equal n without a row list");
  VQ_REQUIRE(ws != nullptr && ws_bytes >= vatlq_cosine_workspace_bytes(d), "workspace too small");
  if (m == 0) {
    VQ_CUDA(cudaMemsetAsync(S, 0, (size_t)d * sizeof(double), stream));
    return 0;
  }
  const int grid = cos_grid(m);
  const size_t smem = (size_t)kCosRows * d * sizeof(float);
  static bool cfg = false;
  if (!cfg) {
    VQ_CUDA(cudaFuncSetAttribute(cos_colsum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCosRows * kCosNV * 128 * 4));
    cfg = true;
  }
  cos_colsum_kernel<<<grid, kCosThreads, smem, stream>>>(X, d, rows, m, (double*)ws);
  VQ_LAUNCHED();
  cos_colsum_reduce_kernel<<<(d + 255) / 256, 256, 0, stream>>>((const double*)ws, grid, d, S);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_cosine_rowsum(const float* X, int64_t n, int d, const int64_t* rows, int64_t m,
                                   const double* S, double m_total, double* out, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(X && S && out && n >= 0 && m >= 0, "null pointer");
  VQ_REQUIRE(d > 0 && (d & 3) == 0 && d <= kCosNV * 128, "d must be a multiple of 4 and <= 2048");
  VQ_REQUIRE(((uintptr_t)X & 15) == 0, "X must be 16-byte aligned");
  VQ_REQUIRE(rows != nullptr || m == n, "m must equal n without a row list");
  if (m == 0) return 0;
  const int grid = (int)std::min<int64_t>((m + kCosRows - 1) / kCosRows, (int64_t)sm_count() * 6);
  cos_rowsum_kernel<<<grid, kCosThreads, (size_t)d * sizeof(double), stream>>>(X, d, rows, m, S, m_total, out);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_minmax_stats_f64(const double* v, const uint8_t* mask, int64_t n, double* stats2,
                                      vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(v && stats2 && n >= 0, "null pointer");
  if (int e = fill_f64(stats2, 2, INFINITY, stream)) return e;
  if (n == 0) return 0;
  minmax_stats_f64_kernel<<<grid_1d(n), 256, 0, stream>>>(v, mask, n, stats2);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_fuse_blend(const double* unc, const double* infl, const uint8_t* mask, int64_t n,
                                double combine_weight, double* out, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(unc && infl && out && n >= 0, "null pointer");
  if (n == 0) return 0;
  blend_kernel<<<grid_1d(n), 256, 0, stream>>>(unc, infl, mask, n, combine_weight, out);
  VQ_LAUNCHED();
  return 0;
}
