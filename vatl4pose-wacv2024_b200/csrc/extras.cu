// Round-2 rows next to the hot path:
//   * OKS of every item against its ground-truth pose (active_learning/al_metric.py:42-69): the
//     controller derives moks_queried (the core-set's score weights, ActiveLearning.py:815-821,858)
//     and the stopping criteria (:707-725) from it.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>

#include "common.cuh"

namespace vatlq {

// np.add.reduce over n contiguous fp64 values, n < 128 (numpy's pairwise sum: sequential below 8,
// else eight strided accumulators over the leading multiple of 8, fixed combine tree, then the tail)
__device__ __forceinline__ double np_sum_f64(const double* a, int n) {
  if (n < 8) {
    double res = 0.0;   // (numpy starts from a[0]; 0 + a[0] is exact)
    for (int i = 0; i < n; ++i) res = __dadd_rn(res, a[i]);
    return res;
  }
  double r[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = a[k];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], a[i + k]);
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __dadd_rn(res, a[i]);
  return res;
}

__constant__ double c_oks_vars[17];

// one thread per item; fp64 like the reference (python floats / numpy float64)
__global__ void __launch_bounds__(128) oks_kernel(const float* __restrict__ kpts, const float* __restrict__ gt,
                                                  const float* __restrict__ bbox_xyxy, long long n, double* __restrict__ oks) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* d = kpts + i * 51;
  const float* g = gt + i * 51;
  const float* b = bbox_xyxy + i * 4;
  // bbox_xyxy_to_xywh (alphapose/utils/bbox.py:91-97)
  const double bx = b[0], by = b[1];
  const double bw = __dadd_rn(__dsub_rn((double)b[2], (double)b[0]), 1.0);
  const double bh = __dadd_rn(__dsub_rn((double)b[3], (double)b[1]), 1.0);
  int k1 = 0;
  for (int j = 0; j < 17; ++j) k1 += (g[3 * j + 2] > 0.f) ? 1 : 0;
  const double x0 = __dsub_rn(bx, bw), x1 = __dadd_rn(bx, __dmul_rn(bw, 2.0));
  const double y0 = __dsub_rn(by, bh), y1 = __dadd_rn(by, __dmul_rn(bh, 2.0));
  const double area = __dadd_rn(__dmul_rn(bw, bh), 2.220446049250313e-16);   // + np.spacing(1)
  double e[17];
  int m = 0;
  for (int j = 0; j < 17; ++j) {
    const double xd = d[3 * j], yd = d[3 * j + 1];
    double dx, dy;
    if (k1 > 0) {
      dx = __dsub_rn(xd, (double)g[3 * j]);
      dy = __dsub_rn(yd, (double)g[3 * j + 1]);
    } else {
      dx = __dadd_rn(fmax(0.0, __dsub_rn(x0, xd)), fmax(0.0, __dsub_rn(xd, x1)));
      dy = __dadd_rn(fmax(0.0, __dsub_rn(y0, yd)), fmax(0.0, __dsub_rn(yd, y1)));
    }
    double v = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    v = __ddiv_rn(v, c_oks_vars[j]);
    v = __ddiv_rn(v, area);
    v = __dmul_rn(v, 0.5);
    if (k1 == 0 || g[3 * j + 2] > 0.f) e[m++] = exp(-v);
  }
  oks[i] = __ddiv_rn(np_sum_f64(e, m), (double)m);
}

// ------------------------------------------------------------------------------------
// MPE and Margin (ActiveLearning.py:762-788): both need skimage.feature.peak_local_max(heatmap,
// min_distance=5, num_peaks=5) of every joint map.  One warp per map, staged in shared memory:
//   11 x 11 maximum filter with edge replication ('nearest'), separable (rows, then columns);
//   mask = (pixel == window max) & (pixel > map minimum), empty when EVERY pixel equals its window
//   maximum, border of 5 pixels excluded;
//   up to five rounds of "best remaining mask pixel" (largest value, lowest row-major index on ties —
//   np.argsort(-v, kind='stable') over np.nonzero order), each accepted peak clearing the mask within
//   Chebyshev distance < 5 (ensure_spacing, p_norm = inf).
//   MPE    += entropy(softmax(peaks))   (fp32, scipy.special.softmax / scipy.stats.entropy)
//   Margin += |peaks[0] - peaks[1]|     when at least two peaks exist
// ------------------------------------------------------------------------------------
constexpr int kPeakWarps = 4;
constexpr int kPeakMinDist = 5;

// MPE / Margin of one map from its <= 5 peaks in descending order (one thread)
__device__ __forceinline__ void peak_scores(const float (&peaks)[5], int npk, float* mpe_out, float* margin_out) {
  float mpe = 0.f, margin = 0.f;
  if (npk > 0) {
    // scipy.special.softmax (fp32): exp(x - max) / sum; scipy.stats.entropy: pk / sum(pk), sum(entr(pk))
    float e[5], ssum = 0.f;
    for (int k = 0; k < npk; ++k) {
      e[k] = expf(peaks[k] - peaks[0]);          // peaks[0] is the maximum (descending order)
      ssum = __fadd_rn(ssum, e[k]);
    }
    float psum = 0.f;
    for (int k = 0; k < npk; ++k) {
      e[k] = __fdiv_rn(e[k], ssum);
      psum = __fadd_rn(psum, e[k]);
    }
    for (int k = 0; k < npk; ++k) {
      const float pk = __fdiv_rn(e[k], psum);
      mpe = __fadd_rn(mpe, pk > 0.f ? -pk * logf(pk) : 0.f);
    }
  }
  if (npk > 1) margin = fabsf(peaks[0] - peaks[1]);
  *mpe_out = mpe;
  *margin_out = margin;
}

// CH / CW > 0: compile-time map shape (64 x 48: index arithmetic without runtime divisions), else the arguments.
// T: fp32, or a 16-bit type converted exactly while the map is staged into the fp32 image.
template <int CH, int CW, typename T>
__device__ __forceinline__ void peak_map_generic(const T* __restrict__ H, long long mi, int h_, int w_, float* __restrict__ mpe_map,
                                                 float* __restrict__ margin_map, float* img, int lane) {
  const int h = CH > 0 ? CH : h_, w = CW > 0 ? CW : w_;
  const int npx = h * w;
  float* aux = img + npx;                         // row maxima, then the peak mask (as 0 / 1); img: the map
  const T* src = H + (size_t)mi * npx;
  float vmin = INFINITY;
  if (CH > 0 && (reinterpret_cast<uintptr_t>(src) & (4 * sizeof(T) - 1)) == 0) {
    float4* d4 = reinterpret_cast<float4*>(img);
#pragma unroll 4
    for (int i = lane; i < npx / 4; i += 32) {
      const float4 v = ldg_stream_quad(src, i);
      d4[i] = v;
      vmin = fminf(vmin, fminf(fminf(v.x, v.y), fminf(v.z, v.w)));
    }
  } else {
    for (int i = lane; i < npx; i += 32) {
      const float v = ldg_f32(src + i);
      img[i] = v;
      vmin = fminf(vmin, v);
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
  __syncwarp();
  for (int i = lane; i < npx; i += 32) {           // row pass
    const int y = i / w, x = i - y * w;
    float m = -INFINITY;
    for (int dx = -kPeakMinDist; dx <= kPeakMinDist; ++dx) m = fmaxf(m, img[y * w + min(max(x + dx, 0), w - 1)]);
    aux[i] = m;
  }
  __syncwarp();
  int n_eq = 0;
  unsigned keep_bits[4] = {0u, 0u, 0u, 0u};        // this lane's mask bits (pixel i = lane + 32 q, q < 128)
  for (int i = lane, q = 0; i < npx; i += 32, ++q) {   // column pass + mask
    const int y = i / w, x = i - y * w;
    float m = -INFINITY;
    for (int dy = -kPeakMinDist; dy <= kPeakMinDist; ++dy) m = fmaxf(m, aux[min(max(y + dy, 0), h - 1) * w + x]);
    const float v = img[i];
    const bool eq = v == m;
    n_eq += eq ? 1 : 0;
    const bool interior = y >= kPeakMinDist && y < h - kPeakMinDist && x >= kPeakMinDist && x < w - kPeakMinDist;
    if (eq && v > vmin && interior) keep_bits[q >> 5] |= 1u << (q & 31);
  }
  n_eq = warp_sum(n_eq);
  __syncwarp();
  const bool trivial = n_eq == npx;                // every pixel equals its window maximum: no peak at all
  for (int i = lane, q = 0; i < npx; i += 32, ++q)
    aux[i] = (!trivial && ((keep_bits[q >> 5] >> (q & 31)) & 1u)) ? 1.f : 0.f;
  __syncwarp();
  float peaks[5];
  int npk = 0;
  for (int r = 0; r < 5; ++r) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = lane; i < npx; i += 32)
      if (aux[i] != 0.f) {
        const float v = img[i];
        if (v > bv || (v == bv && i < bi)) {
          bv = v;
          bi = i;
        }
      }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
      const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
      if (v2 > bv || (v2 == bv && i2 < bi)) {
        bv = v2;
        bi = i2;
      }
    }
    if (bi == 0x7fffffff) break;
    peaks[npk++] = bv;
    const int py = bi / w, px = bi - py * w;
    // clear the mask within Chebyshev distance < 5 of the accepted peak (itself included)
    for (int t = lane; t < (2 * kPeakMinDist - 1) * (2 * kPeakMinDist - 1); t += 32) {
      const int yy = py + t / (2 * kPeakMinDist - 1) - (kPeakMinDist - 1), xx = px + t % (2 * kPeakMinDist - 1) - (kPeakMinDist - 1);
      if (yy >= 0 && yy < h && xx >= 0 && xx < w) aux[yy * w + xx] = 0.f;
    }
    __syncwarp();
  }
  if (lane == 0) peak_scores(peaks, npk, mpe_map + mi, margin_map + mi);
}

template <int CH, int CW, typename T>
__global__ void __launch_bounds__(kPeakWarps * 32)
peak_unc_kernel(const T* __restrict__ H, long long maps, int h_, int w_, float* __restrict__ mpe_map,
                float* __restrict__ margin_map) {
  extern __shared__ __align__(16) float s_peak[];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const long long mi = (long long)blockIdx.x * kPeakWarps + wp;
  if (mi >= maps) return;
  const int npx = (CH > 0 ? CH : h_) * (CW > 0 ? CW : w_);
  peak_map_generic<CH, CW, T>(H, mi, h_, w_, mpe_map, margin_map, s_peak + (size_t)wp * 2 * npx, lane);
}

// the generic 64 x 48 routine on a list of maps (the fast path's overflow cases); grid-stride over the list
template <typename T>
__global__ void __launch_bounds__(kPeakWarps * 32)
peak_unc_redo_kernel(const T* __restrict__ H, const unsigned int* __restrict__ redo_count, const int* __restrict__ redo_list,
                     float* __restrict__ mpe_map, float* __restrict__ margin_map) {
  extern __shared__ __align__(16) float s_peak[];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const unsigned total = *redo_count;
  for (unsigned slot = blockIdx.x * kPeakWarps + wp; slot < total; slot += gridDim.x * kPeakWarps) {
    peak_map_generic<64, 48, T>(H, redo_list[slot], 64, 48, mpe_map, margin_map, s_peak + (size_t)wp * 2 * 64 * 48, lane);
    __syncwarp();
  }
}


// ---- 64 x 48 fast path.  The generic kernel above spends ~10 k instructions per lane and map on the two 11-tap
// window passes (22 shared loads + clamps per pixel) and on five full-map scans for the peaks.  Here:
//   * the map sits in shared memory with 5 replicated columns on each side (row stride 59: conflict-free when the
//     lanes walk different rows), the row maxima with 5 replicated rows above and below (row stride 49);
//   * a lane takes whole rows (then whole columns) into REGISTERS and gets the 11-wide maxima by doubling
//     (w2 = max(p[i], p[i+1]), w4, w8, out[x] = max(w8[x], w8[x+3])): 4 max ops per element, no clamps;
//   * mask pixels (a few dozen per map) are appended to a candidate list; the five rounds of "best remaining
//     peak + Chebyshev-< 5 suppression" run on the list.  A list overflow (large plateaus) is flagged and the map
//     is redone by the generic kernel.
constexpr int kPfW = 48, kPfH = 64, kPfPad = kPeakMinDist;
constexpr int kPfPS = kPfW + 2 * kPfPad + 1;            // 59: padded image row stride
constexpr int kPfRS = kPfW + 1;                         // 49: row-maxima row stride
constexpr int kPfRows = kPfH + 2 * kPfPad;              // 74 rows of row maxima
constexpr int kPfCand = 256;
constexpr int kPfWarps = 7;
constexpr size_t kPfSmemWarp = (size_t)(kPfH * kPfPS + kPfRows * kPfRS) * 4 + kPfCand * 8 + 16;

template <int N>
__device__ __forceinline__ void window11(float (&p)[N]) {   // p[i] <- max(p[i .. i+10]) for i < N - 10, in place
#pragma unroll
  for (int i = 0; i < N - 1; ++i) p[i] = fmaxf(p[i], p[i + 1]);      // width 2
#pragma unroll
  for (int i = 0; i < N - 3; ++i) p[i] = fmaxf(p[i], p[i + 2]);      // width 4
#pragma unroll
  for (int i = 0; i < N - 7; ++i) p[i] = fmaxf(p[i], p[i + 4]);      // width 8
#pragma unroll
  for (int i = 0; i < N - 10; ++i) p[i] = fmaxf(p[i], p[i + 3]);     // width 11
}

// the <= 5 peaks of a map from its candidate list (mask pixels: value, row-major index): five rounds of "best remaining
// candidate (largest value, lowest index on ties), then drop everything within Chebyshev distance < 5 of it"; one warp
__device__ __forceinline__ void peak_select(const float* cval, const int* cidx, int ncand, int lane, float* mpe_out, float* margin_out) {
  float v8[kPfCand / 32];
  int i8[kPfCand / 32];
#pragma unroll
  for (int j = 0; j < kPfCand / 32; ++j) {
    const int q = lane + 32 * j;
    v8[j] = q < ncand ? cval[q] : -INFINITY;
    i8[j] = q < ncand ? cidx[q] : 0x7fffffff;
  }
  float peaks[5];
  int npk = 0;
  for (int r = 0; r < 5; ++r) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < kPfCand / 32; ++j)
      if (i8[j] != 0x7fffffff && (v8[j] > bv || (v8[j] == bv && i8[j] < bi))) {
        bv = v8[j];
        bi = i8[j];
      }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
      const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
      if (i2 != 0x7fffffff && (bi == 0x7fffffff || v2 > bv || (v2 == bv && i2 < bi))) {
        bv = v2;
        bi = i2;
      }
    }
    if (bi == 0x7fffffff) break;
    peaks[npk++] = bv;
    const int py = bi / kPfW, px = bi - py * kPfW;
#pragma unroll
    for (int j = 0; j < kPfCand / 32; ++j)
      if (i8[j] != 0x7fffffff) {
        const int yy = i8[j] / kPfW, xx = i8[j] - yy * kPfW;
        if (abs(yy - py) < kPeakMinDist && abs(xx - px) < kPeakMinDist) i8[j] = 0x7fffffff;
      }
  }
  if (lane == 0) peak_scores(peaks, npk, mpe_out, margin_out);
}

__global__ void __launch_bounds__(kPfWarps * 32, 1)
peak_unc_fast_kernel(const float* __restrict__ H, long long maps, float* __restrict__ mpe_map, float* __restrict__ margin_map,
                     unsigned int* __restrict__ redo_count, int* __restrict__ redo_list) {
  extern __shared__ __align__(16) unsigned char pf_smem[];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const long long mi = (long long)blockIdx.x * kPfWarps + wp;
  if (mi >= maps) return;
  float* P = reinterpret_cast<float*>(pf_smem + (size_t)wp * kPfSmemWarp);     // [64][59]
  float* R = P + kPfH * kPfPS;                                                  // [74][49]
  float* cval = R + kPfRows * kPfRS;                                            // [256]
  int* cidx = reinterpret_cast<int*>(cval + kPfCand);                           // [256]
  int* ccount = cidx + kPfCand;
  const float4* src = reinterpret_cast<const float4*>(H + (size_t)mi * (kPfH * kPfW));
  float vmin = INFINITY;
  if (lane == 0) *ccount = 0;
#pragma unroll 4
  for (int i = lane; i < kPfH * kPfW / 4; i += 32) {       // 12 float4 per row
    const float4 v = ldg_stream(src + i);
    const int y = i / 12, x = (i - y * 12) * 4;
    float* d = P + y * kPfPS + kPfPad + x;
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    vmin = fminf(vmin, fminf(fminf(v.x, v.y), fminf(v.z, v.w)));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
  __syncwarp();
  // row pass: lane takes rows lane and lane + 32 into registers (edge columns replicated)
#pragma unroll 1
  for (int rr = 0; rr < 2; ++rr) {
    const int y = lane + 32 * rr;
    float p[kPfW + 2 * kPfPad];
    const float* row = P + y * kPfPS;
#pragma unroll
    for (int i = 0; i < kPfW; ++i) p[kPfPad + i] = row[kPfPad + i];
#pragma unroll
    for (int i = 0; i < kPfPad; ++i) {
      p[i] = p[kPfPad];
      p[kPfPad + kPfW + i] = p[kPfPad + kPfW - 1];
    }
    window11(p);
    float* out = R + (y + kPfPad) * kPfRS;
#pragma unroll
    for (int x = 0; x < kPfW; ++x) out[x] = p[x];
    if (y == 0) {
#pragma unroll 1
      for (int e = 0; e < kPfPad; ++e)
#pragma unroll
        for (int x = 0; x < kPfW; ++x) R[e * kPfRS + x] = p[x];
    }
    if (y == kPfH - 1) {
#pragma unroll 1
      for (int e = 0; e < kPfPad; ++e)
#pragma unroll
        for (int x = 0; x < kPfW; ++x) R[(kPfH + kPfPad + e) * kPfRS + x] = p[x];
    }
  }
  __syncwarp();
  // column pass: lane takes columns lane and lane + 32 (< 48); mask and candidates
  int n_eq = 0;
#pragma unroll 1
  for (int cc = 0; cc < 2; ++cc) {
    const int x = lane + 32 * cc;
    if (x < kPfW) {
      float c[kPfRows];
#pragma unroll
      for (int i = 0; i < kPfRows; ++i) c[i] = R[i * kPfRS + x];
      window11(c);
      const bool xin = x >= kPfPad && x < kPfW - kPfPad;
#pragma unroll
      for (int y = 0; y < kPfH; ++y) {
        const float v = P[y * kPfPS + kPfPad + x];
        const bool eq = v == c[y];
        n_eq += eq ? 1 : 0;
        if (eq && xin && y >= kPfPad && y < kPfH - kPfPad && v > vmin) {
          const int pos = atomicAdd(ccount, 1);
          if (pos < kPfCand) {
            cval[pos] = v;
            cidx[pos] = y * kPfW + x;
          }
        }
      }
    }
  }
  n_eq = warp_sum(n_eq);
  __syncwarp();
  int ncand = *ccount;
  if (n_eq == kPfH * kPfW) ncand = 0;                       // trivial image: no peak at all
  if (ncand > kPfCand) {                                     // large plateaus: the generic kernel redoes this map
    if (lane == 0) redo_list[atomicAdd(redo_count, 1u)] = (int)mi;
    return;
  }
  peak_select(cval, cidx, ncand, lane, mpe_map + mi, margin_map + mi);
}

// ---- 64 x 48 register path (the default).  No staging of the map at all: lane l reads rows 2l and 2l+1 straight from
// global memory (96 contiguous floats), gets their 11-wide row maxima by doubling in registers, and the 11-tall column
// maxima from its neighbours' row maxima with six shuffles per column: rows 2l-4 .. 2l+5 are the row pairs of lanes
// l-2 .. l+2 (pair maximum m), row 2l-5 is the second row of lane l-3, row 2l+6 the first row of lane l+3.  Source
// lanes are clamped to 0 .. 31: a clamped lane only repeats rows that are inside the window already, which is exactly
// what edge replication does to a maximum.  The originals are read a second time (L1 / L2) for the mask test.
// Shared memory: the candidate list only -> occupancy is set by registers (12 warps per SM instead of 7).
// T: fp32, or a 16-bit type read as 8-byte quads (same rows per lane) and converted exactly in registers.
constexpr int kPrWarps = 4;
template <typename T>
__global__ void __launch_bounds__(kPrWarps * 32, 3)
peak_unc_reg_kernel(const T* __restrict__ H, long long maps, float* __restrict__ mpe_map, float* __restrict__ margin_map,
                    unsigned int* __restrict__ redo_count, int* __restrict__ redo_list) {
  __shared__ float s_cval[kPrWarps][kPfCand];
  __shared__ int s_cidx[kPrWarps][kPfCand];
  __shared__ int s_cnt[kPrWarps];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const long long mi = (long long)blockIdx.x * kPrWarps + wp;
  if (mi >= maps) return;
  float* cval = s_cval[wp];
  int* cidx = s_cidx[wp];
  int* ccount = &s_cnt[wp];
  if (lane == 0) *ccount = 0;
  const T* src = H + (size_t)mi * (kPfH * kPfW) + (size_t)lane * (2 * kPfW);
  float a[kPfW], b[kPfW];           // row maxima of rows 2l / 2l+1, then their window maxima
  float vmin = INFINITY;
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    float p[kPfW + 2 * kPfPad];
#pragma unroll
    for (int q = 0; q < kPfW / 4; ++q) {
      const float4 v = ldg_quad(src, rr * (kPfW / 4) + q);
      p[kPfPad + 4 * q] = v.x; p[kPfPad + 4 * q + 1] = v.y; p[kPfPad + 4 * q + 2] = v.z; p[kPfPad + 4 * q + 3] = v.w;
      vmin = fminf(vmin, fminf(fminf(v.x, v.y), fminf(v.z, v.w)));
    }
#pragma unroll
    for (int i = 0; i < kPfPad; ++i) {
      p[i] = p[kPfPad];
      p[kPfPad + kPfW + i] = p[kPfPad + kPfW - 1];
    }
    window11(p);
#pragma unroll
    for (int x = 0; x < kPfW; ++x) {
      if (rr == 0) a[x] = p[x];
      else b[x] = p[x];
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
  const int lu1 = max(lane - 1, 0), lu2 = max(lane - 2, 0), lu3 = max(lane - 3, 0);
  const int ld1 = min(lane + 1, 31), ld2 = min(lane + 2, 31), ld3 = min(lane + 3, 31);
#pragma unroll
  for (int x = 0; x < kPfW; ++x) {
    const float m = fmaxf(a[x], b[x]);
    const float u1 = __shfl_sync(0xffffffffu, m, lu1), u2 = __shfl_sync(0xffffffffu, m, lu2);
    const float d1 = __shfl_sync(0xffffffffu, m, ld1), d2 = __shfl_sync(0xffffffffu, m, ld2);
    const float eu = __shfl_sync(0xffffffffu, b[x], lu3), ed = __shfl_sync(0xffffffffu, a[x], ld3);
    const float m5 = fmaxf(fmaxf(m, fmaxf(u1, u2)), fmaxf(d1, d2));
    a[x] = fmaxf(m5, eu);
    b[x] = fmaxf(m5, ed);
  }
  __syncwarp();
  int n_eq = 0;
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    const int y = 2 * lane + rr;
    const bool yin = y >= kPfPad && y < kPfH - kPfPad;
#pragma unroll
    for (int q = 0; q < kPfW / 4; ++q) {
      const float4 v4 = ldg_quad(src, rr * (kPfW / 4) + q);
      const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int x = 4 * q + e;
        const float wm = rr == 0 ? a[x] : b[x];
        const bool eq = vv[e] == wm;
        n_eq += eq ? 1 : 0;
        if (eq && yin && x >= kPfPad && x < kPfW - kPfPad && vv[e] > vmin) {
          const int pos = atomicAdd(ccount, 1);
          if (pos < kPfCand) {
            cval[pos] = vv[e];
            cidx[pos] = y * kPfW + x;
          }
        }
      }
    }
  }
  n_eq = warp_sum(n_eq);
  __syncwarp();
  int ncand = *ccount;
  if (n_eq == kPfH * kPfW) ncand = 0;                       // trivial image: no peak at all
  if (ncand > kPfCand) {                                     // large plateaus: the generic kernel redoes this map
    if (lane == 0) redo_list[atomicAdd(redo_count, 1u)] = (int)mi;
    return;
  }
  peak_select(cval, cidx, ncand, lane, mpe_map + mi, margin_map + mi);
}

// per-frame sums over the joints, in joint order
__global__ void __launch_bounds__(256) peak_frames_kernel(const float* __restrict__ mpe_map, const float* __restrict__ margin_map,
                                                          long long n, int J, float* __restrict__ mpe, float* __restrict__ margin) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  float a = 0.f, b = 0.f;
  for (int j = 0; j < J; ++j) {
    a = __fadd_rn(a, mpe_map[t * J + j]);
    b = __fadd_rn(b, margin_map[t * J + j]);
  }
  if (mpe) mpe[t] = a;
  if (margin) margin[t] = b;
}

// ------------------------------------------------------------------------------------
// candidate ordering (ActiveLearning.py:527-538, 587-589): ids of the masked-in rows by descending (or ascending)
// score, ties in ascending id order — what `sorted(dict.items(), key=score, reverse=True)` yields for a dict built in
// ascending id order (Python's sort is stable; reverse=True keeps equal keys in their original order).
// Order-preserving 64-bit keys + a stable LSD radix sort (cub::DeviceRadixSort); masked-out rows sort last.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rank_keys_kernel(const double* __restrict__ score, const uint8_t* __restrict__ mask, long long n,
                                                        int descending, unsigned long long* __restrict__ keys, long long* __restrict__ vals) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long k = 0xFFFFFFFFFFFFFFFFULL;
  if (!mask || mask[i]) {
    double s = score[i];
    if (s == 0.0) s = 0.0;                                       // -0.0 and +0.0 compare equal in Python
    unsigned long long b = (unsigned long long)__double_as_longlong(s);
    b = (b >> 63) ? ~b : (b | 0x8000000000000000ULL);            // ascending order of the doubles
    k = descending ? ~b : b;
    if (k == 0xFFFFFFFFFFFFFFFFULL) k -= 1;                      // (keep the sentinel unique to masked-out rows)
  }
  keys[i] = k;
  vals[i] = i;
}

// ------------------------------------------------------------------------------------
// fp64 tensor-core peak, measured on the device the library runs on: the roofline denominator of the core-set
// pass once it is bound by the DMMA pipe (MEASURED_PEAKS.json only carries the HBM and bf16 figures).
// 8 independent accumulator chains per warp, 8 warps per CTA, 4 CTAs per SM: the pipe is saturated.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters, double a, double b) {
  double c[8][2];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    c[k][0] = threadIdx.x * 1e-9;
    c[k][1] = k;
  }
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 8; ++k)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[k][0]), "+d"(c[k][1])
                   : "d"(a), "d"(b));
  }
  double s = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) s += c[k][0] + c[k][1];
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace vatlq

using namespace vatlq;

extern "C" int vatlq_measure_fp64_mma(double* host_fma_per_s, void* ws, size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  const int grid = sm_count() * 4, iters = 4096;
  VQ_REQUIRE(host_fma_per_s && ws && ws_bytes >= (size_t)grid * 256 * 8, "workspace must hold 4*SMs*256 doubles");
  cudaEvent_t e0, e1;
  VQ_CUDA(cudaEventCreate(&e0));
  VQ_CUDA(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {          // first repetition warms up; best of the rest
    cudaEventRecord(e0, stream);
    dmma_peak_kernel<<<grid, 256, 0, stream>>>((double*)ws, iters, 1.0000001, 0.9999999);
    cudaEventRecord(e1, stream);
    VQ_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    // one m8n8k4 DMMA = 8*8*4 = 256 FMA per warp
    const double fma = (double)grid * 8.0 * iters * 8.0 * 256.0;
    if (rep > 0 && ms > 0.f) best = std::max(best, fma / (ms * 1e-3));
  }
  g_launches.fetch_add(4);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *host_fma_per_s = best;
  return 0;
}

extern "C" size_t vatlq_rank_workspace_bytes(int64_t n) {
  if (n <= 0) return 0;
  size_t cb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cb, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                  (const long long*)nullptr, (long long*)nullptr, (int)n);
  return align_up(cb, 256) + 3 * align_up((size_t)n * 8, 256);
}

extern "C" int vatlq_rank_scores(const double* score, const uint8_t* mask, int64_t n, int descending, int64_t* out_idx,
                                 void* ws, size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(n >= 0 && n < (1LL << 31), "n out of range");
  if (n == 0) return 0;
  VQ_REQUIRE(score && out_idx && ws, "null pointer");
  VQ_REQUIRE(ws_bytes >= vatlq_rank_workspace_bytes(n), "workspace too small (vatlq_rank_workspace_bytes)");
  char* w = (char*)ws;
  const size_t seg = align_up((size_t)n * 8, 256);
  unsigned long long* k_in = (unsigned long long*)w;
  unsigned long long* k_out = (unsigned long long*)(w + seg);
  long long* v_in = (long long*)(w + 2 * seg);
  void* tmp = w + 3 * seg;
  size_t cb = ws_bytes - 3 * seg;
  rank_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(score, mask, (long long)n, descending, k_in, v_in);
  VQ_LAUNCHED();
  VQ_CUDA(cub::DeviceRadixSort::SortPairs(tmp, cb, k_in, k_out, v_in, (long long*)out_idx, (int)n, 0, 64, stream));
  g_launches.fetch_add(1);
  return 0;
}

extern "C" size_t vatlq_peak_workspace_bytes(int64_t n, int J, int h, int w) {
  if (n <= 0 || J <= 0) return 0;
  const size_t maps = (size_t)n * J;
  // two floats per map; the 64 x 48 fast path adds its overflow list (a counter + one int per map)
  return maps * 8 + ((h == kPfH && w == kPfW) ? 16 + maps * 4 : 0);
}

template <typename T>
static int launch_peak_unc(const T* H, int64_t n, int J, int h, int w, float* mpe, float* margin, void* ws, size_t smem,
                           cudaStream_t stream) {
  const long long maps = (long long)n * J;
  static size_t configured = 0;
  if (smem > configured) {
    VQ_CUDA(cudaFuncSetAttribute((peak_unc_kernel<0, 0, T>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VQ_CUDA(cudaFuncSetAttribute((peak_unc_kernel<64, 48, T>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VQ_CUDA(cudaFuncSetAttribute(peak_unc_redo_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)((size_t)kPeakWarps * 2 * kPfH * kPfW * sizeof(float))));
    if (std::is_same<T, float>::value)
      VQ_CUDA(cudaFuncSetAttribute(peak_unc_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kPfWarps * kPfSmemWarp)));
    configured = smem;
  }
  float* mm = (float*)ws;
  const bool no_fast = getenv("VATLQ_PEAK_GENERIC") != nullptr;     // measurement / test switch (read per call)
  if (h == kPfH && w == kPfW && !no_fast && (reinterpret_cast<uintptr_t>(H) & (4 * sizeof(T) - 1)) == 0) {
    unsigned int* redo_count = (unsigned int*)((char*)ws + (size_t)maps * 8);
    int* redo_list = (int*)((char*)ws + (size_t)maps * 8 + 16);
    VQ_CUDA(cudaMemsetAsync(redo_count, 0, 16, stream));
    // the shared-memory-staged variant (measurement switch) is fp32 only: 16-bit maps take the register kernel
    // whatever VATLQ_PEAK_SMEM says
    if (std::is_same<T, float>::value && getenv("VATLQ_PEAK_SMEM") != nullptr)
      peak_unc_fast_kernel<<<(unsigned)((maps + kPfWarps - 1) / kPfWarps), kPfWarps * 32, kPfWarps * kPfSmemWarp, stream>>>(
          (const float*)H, maps, mm, mm + maps, redo_count, redo_list);
    else
      peak_unc_reg_kernel<T><<<(unsigned)((maps + kPrWarps - 1) / kPrWarps), kPrWarps * 32, 0, stream>>>(H, maps, mm, mm + maps,
                                                                                                  redo_count, redo_list);
    VQ_LAUNCHED();
    const unsigned rgrid = (unsigned)std::min<long long>((maps + kPeakWarps - 1) / kPeakWarps, (long long)sm_count() * 4);
    peak_unc_redo_kernel<T><<<rgrid, kPeakWarps * 32, (size_t)kPeakWarps * 2 * kPfH * kPfW * sizeof(float), stream>>>(
        H, redo_count, redo_list, mm, mm + maps);
    VQ_LAUNCHED();
  } else {
    const unsigned pgrid = (unsigned)((maps + kPeakWarps - 1) / kPeakWarps);
    if (h == 64 && w == 48) peak_unc_kernel<64, 48, T><<<pgrid, kPeakWarps * 32, smem, stream>>>(H, maps, h, w, mm, mm + maps);
    else peak_unc_kernel<0, 0, T><<<pgrid, kPeakWarps * 32, smem, stream>>>(H, maps, h, w, mm, mm + maps);
    VQ_LAUNCHED();
  }
  peak_frames_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(mm, mm + maps, (long long)n, J, mpe, margin);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_peak_unc_dt(const void* H, int dtype, int64_t n, int J, int h, int w, float* mpe, float* margin, void* ws,
                                 size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(n >= 0 && J > 0 && h > 2 * kPeakMinDist && w > 2 * kPeakMinDist, "bad shape");
  VQ_REQUIRE(dtype_size(dtype) != 0, "unknown dtype (VATLQ_F32, VATLQ_F16 or VATLQ_BF16)");
  if (n == 0) return 0;
  VQ_REQUIRE(H && ws && (mpe || margin), "null pointer");
  VQ_REQUIRE(h * w <= 128 * 32 * 4, "map too large (<= 16384 pixels)");
  const long long maps = (long long)n * J;
  VQ_REQUIRE(maps < (1LL << 31), "too many maps per call (n*J < 2^31)");
  VQ_REQUIRE(ws_bytes >= vatlq_peak_workspace_bytes(n, J, h, w), "workspace too small (vatlq_peak_workspace_bytes)");
  // (fp32 keeps its generic fallback for a misaligned H; the 16-bit forms are new and ask for the alignment instead)
  VQ_REQUIRE(dtype == VATLQ_F32 || h != kPfH || w != kPfW || quad_aligned(H, dtype), "16-bit H must be 8-byte aligned");
  const size_t smem = (size_t)kPeakWarps * 2 * h * w * sizeof(float);
  VQ_REQUIRE(smem <= 200 * 1024, "map too large for the shared-memory staging");
  return with_dtype(dtype, [&](auto tag) {
    using T = std::remove_const_t<std::remove_pointer_t<decltype(tag)>>;
    return launch_peak_unc<T>((const T*)H, n, J, h, w, mpe, margin, ws, smem, stream);
  });
}

extern "C" int vatlq_peak_unc(const float* H, int64_t n, int J, int h, int w, float* mpe, float* margin, void* ws,
                              size_t ws_bytes, vatlq_stream_t stream) {
  return vatlq_peak_unc_dt(H, VATLQ_F32, n, J, h, w, mpe, margin, ws, ws_bytes, stream);
}

extern "C" int vatlq_oks(const float* kpts, const float* gt_kpts, const float* bbox_ann_xyxy, int64_t n, double* oks,
                         vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(n >= 0, "n must be >= 0");
  if (n == 0) return 0;
  VQ_REQUIRE(kpts && gt_kpts && bbox_ann_xyxy && oks, "null pointer");
  static bool init = false;
  if (!init) {   // OKS_vars = (OKS_sigmas * 2) ** 2, OKS_sigmas = [...] / 10.0   (al_metric.py:38-39)
    const double s[17] = {.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89};
    double v[17];
    for (int j = 0; j < 17; ++j) {
      const double t = (s[j] / 10.0) * 2.0;
      v[j] = t * t;
    }
    VQ_CUDA(cudaMemcpyToSymbol(c_oks_vars, v, sizeof(v)));
    init = true;
  }
  oks_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(kpts, gt_kpts, bbox_ann_xyxy, (long long)n, oks);
  VQ_LAUNCHED();
  return 0;
}
