// Heat-map scan: THC + local-peak statistics + argmax / quarter-pixel coordinates in ONE
// streaming pass over the (n,J,h,w) pool, fp32, fp16 or bf16 (16-bit maps are converted exactly at the load:
// every output equals the fp32 scan of the upcast, bit for bit).  See include/vatlq.h for the reference
// functions this replaces and DESIGN.md §scan for the data flow.
//
// Work decomposition (fast path): one warp walks a run of consecutive frames of one joint.
// Maps land in shared memory by 1-D TMA bulk copies and are pulled into registers, where frame
// t-1 stays for the |H_t - H_{t-1}| term, so every byte of H is fetched from HBM exactly once
// (plus one halo map per run).  Only the few pixels that reach half of the map maximum ever
// look at their 3x3 neighbourhood in shared memory:
//   * the largest peak of a map is its global maximum whenever that maximum is > 0, and
//     when it is <= 0 the 0.5*max threshold rejects everything but exact zeros
//     (local_peak.py:5-10), so "kept peak" == "pixel >= 0.5*gmax that is a 3x3 (zero-padded)
//     maximum" — no full 3x3 filter is needed.
#include "common.cuh"

namespace vatlq {

constexpr int kScanThreads = 256;
constexpr int kWarps = kScanThreads / 32;

struct ScanOut {
  double* pair_sum;  // [(n+1)*J]  sum |H_t - H_{t-1}| of joint j, t = 0..n
  float* psum;       // [n*J] kept-peak value sum
  int* pcnt;         // [n*J] kept-peak count
  float* maxv;       // [n*J] map maximum
  float* hmxy;       // [n*J*2] heat-map-space coordinates
};

__device__ __forceinline__ bool pair_wanted(int64_t t, int64_t n, const uint8_t* __restrict__ is_prev,
                                            const uint8_t* __restrict__ is_next, bool has_hp, bool has_hn) {
  // pair t couples frame t-1 and frame t (t = 0 uses halo_prev, t = n uses halo_next)
  if (t == 0 && !has_hp) return false;
  if (t == n && !has_hn) return false;
  bool want = false;
  if (t < n && is_prev && is_prev[t]) want = true;
  if (t > 0 && is_next && is_next[t - 1]) want = true;
  return want;
}

// 3x3 zero-padded maximum test of pixel (y,x) against the map in shared memory
template <int HM_H, int HM_W, typename T>
__device__ __forceinline__ bool is_local_max(const T* __restrict__ s_map, int y, int x, float val,
                                             int h_rt, int w_rt) {
  const int hh = HM_H > 0 ? HM_H : h_rt, ww = HM_W > 0 ? HM_W : w_rt;
  bool ok = true;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      if (dy == 0 && dx == 0) continue;
      const int yy = y + dy, xx = x + dx;
      const float nb = (yy >= 0 && yy < hh && xx >= 0 && xx < ww) ? to_f32(s_map[yy * ww + xx]) : 0.0f;
      ok = ok && (val >= nb);
    }
  }
  return ok;
}

// quarter-pixel shift of transforms.py:560-566 (strictly interior pixels only; sign(0) = 0)
template <typename T>
__device__ __forceinline__ void quarter_shift(const T* __restrict__ s_map, int y, int x, int hh, int ww,
                                              float gmax, float& fx, float& fy) {
  if (!(gmax > 0.0f)) {  // get_max_pred zeroes the coordinates (transforms.py:723-726)
    fx = 0.0f;
    fy = 0.0f;
    return;
  }
  fx = (float)x;
  fy = (float)y;
  if (x > 1 && x < ww - 1 && y > 1 && y < hh - 1) {
    const float dx = to_f32(s_map[y * ww + x + 1]) - to_f32(s_map[y * ww + x - 1]);
    const float dy = to_f32(s_map[(y + 1) * ww + x]) - to_f32(s_map[(y - 1) * ww + x]);
    fx += (dx > 0.0f) ? 0.25f : ((dx < 0.0f) ? -0.25f : 0.0f);
    fy += (dy > 0.0f) ? 0.25f : ((dy < 0.0f) ? -0.25f : 0.0f);
  }
}

constexpr int FH = 64, FW = 48, FPIX = FH * FW, FQ = FPIX / 4;  // 3072 px, 768 float4 per map

// ------------------------------------------------------------------------------------
// fast path, 64x48 maps (every config of the reference): one WARP owns a run of consecutive frames of one joint.
// Lane 0 keeps kStages-1 maps in flight with cp.async.bulk (1-D TMA bulk copy, 12 288 B each in fp32, 6 144 B in 16 bits,
// completion counted on an mbarrier per stage); the warp pulls the landed map into registers
// (24 float4 per lane, converted from 24 8-byte quads in 16 bits), where it stays to serve as frame t-1 of the next step, so every byte
// of H crosses HBM once and shared memory is only a landing zone + the 3x3 neighbourhood
// lookups of the few pixels above half of the map maximum.  No __syncthreads anywhere: all
// reductions are warp shuffles, warps of a CTA only share the launch.
// ------------------------------------------------------------------------------------
#ifndef VQ_SCAN_WARPS
#define VQ_SCAN_WARPS 8
#endif
#ifndef VQ_SCAN_STAGES
#define VQ_SCAN_STAGES 2
#endif
// 16-bit maps (6 144 B per stage): 2, 3 and 4 stages measured within 0.5 % of each other on B200 (170 000 frames,
// tools/time_heatmap_dtypes.py --stage-libs): the 16-bit scan is not bound by bytes in flight (DESIGN.md §4.1), so it
// keeps the fp32 kernel's two stages and half its shared memory
#ifndef VQ_SCAN_STAGES16
#define VQ_SCAN_STAGES16 2
#endif
constexpr int kTmaWarps = VQ_SCAN_WARPS;
constexpr int kLaneQ = FQ / 32;                  // 24 quads per lane
template <typename T> struct ScanStages { static constexpr int value = VQ_SCAN_STAGES16; };
template <> struct ScanStages<float> { static constexpr int value = VQ_SCAN_STAGES; };
template <typename T>
constexpr size_t tma_smem() {
  return (size_t)kTmaWarps * ScanStages<T>::value * (FPIX * sizeof(T)) + (size_t)kTmaWarps * ScanStages<T>::value * 8;
}

template <typename T>
__global__ void __launch_bounds__(kTmaWarps * 32, 1)
scan_tma_64x48(const T* __restrict__ H, const uint8_t* __restrict__ is_prev,
               const uint8_t* __restrict__ is_next, int64_t n, int J,
               const T* __restrict__ halo_prev, const T* __restrict__ halo_next,
               int run_len, int64_t n_runs, ScanOut out) {
  constexpr int kStages = ScanStages<T>::value;
  constexpr int kMapBytes = FPIX * sizeof(T);    // 12 288 (fp32) / 6 144 (16-bit)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t task = (int64_t)blockIdx.x * kTmaWarps + warp;   // task = run * J + joint
  if (task >= n_runs * J) return;
  const int j = (int)(task % J);
  const int64_t a = (task / J) * run_len;
  const int64_t b = min(n, a + (int64_t)run_len);
  T* stage0 = reinterpret_cast<T*>(smem_raw) + (size_t)warp * kStages * FPIX;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kTmaWarps * kStages * kMapBytes) + warp * kStages;
  const bool has_hp = halo_prev != nullptr, has_hn = halo_next != nullptr;

  // frames this warp streams: [first, last]; first == a-1 only feeds the |H_a - H_{a-1}| term,
  // last == n (the halo that follows the pool) only closes the final pair
  const int64_t first = pair_wanted(a, n, is_prev, is_next, has_hp, has_hn) ? a - 1 : a;
  const bool tail_pair = (b == n) && pair_wanted(n, n, is_prev, is_next, has_hp, has_hn);
  const int64_t last = tail_pair ? n : b - 1;
  const int64_t count = last - first + 1;
  auto src_of = [&](int64_t f) -> const T* {
    if (f < 0) return halo_prev + (size_t)j * FPIX;
    if (f >= n) return halo_next + (size_t)j * FPIX;
    return H + ((size_t)f * J + j) * FPIX;
  };
  if (lane == 0) {
    for (int s = 0; s < kStages; ++s) mbar_init(&bars[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int s = 0; s < kStages && s < count; ++s) {
      mbar_expect_tx(&bars[s], kMapBytes);
      tma_load_1d(stage0 + (size_t)s * FPIX, src_of(first + s), kMapBytes, &bars[s]);
    }
  }
  __syncwarp();

  float4 pv[kLaneQ];   // frame f-1 (registers)
#pragma unroll
  for (int r = 0; r < kLaneQ; ++r) pv[r] = make_float4(0.f, 0.f, 0.f, 0.f);

  for (int64_t i = 0; i < count; ++i) {
    const int64_t f = first + i;
    const int s = (int)(i % kStages);
    const T* cur = stage0 + (size_t)s * FPIX;
    mbar_wait(&bars[s], (uint32_t)((i / kStages) & 1));
    const bool want = (f >= a) && pair_wanted(f, n, is_prev, is_next, has_hp, has_hn);

    // ---- pass 1: pull the map into registers; map maximum and |H_f - H_{f-1}|
    // (four independent chains each: a lone warp per scheduler has no other latency hiding)
    float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY), sm = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < kLaneQ; ++r) {
      const float4 c = load_quad(cur, r * 32 + lane);   // LDS.128 (fp32) / LDS.64 + exact conversion
      if (want) {
        sm.x += fabsf(c.x - pv[r].x);
        sm.y += fabsf(c.y - pv[r].y);
        sm.z += fabsf(c.z - pv[r].z);
        sm.w += fabsf(c.w - pv[r].w);
      }
      mx.x = fmaxf(mx.x, c.x);
      mx.y = fmaxf(mx.y, c.y);
      mx.z = fmaxf(mx.z, c.z);
      mx.w = fmaxf(mx.w, c.w);
      pv[r] = c;
    }
    float sum = (sm.x + sm.y) + (sm.z + sm.w);
    const float lmax = fmaxf(fmaxf(mx.x, mx.y), fmaxf(mx.z, mx.w));
    if (f >= a) {
      sum = warp_sum(sum);
      if (lane == 0) out.pair_sum[(size_t)f * J + j] = want ? (double)sum : 0.0;
    }
    if (f >= a && f < n) {
      const float gmax = warp_max(lmax);
      // ---- pass 2: only pixels >= 0.5*gmax can be kept peaks; only pixels == gmax the argmax
      const float thr = 0.5f * gmax;
      float ps = 0.0f, cx = 0.f, cy = 0.f;
      int pc = 0, cand = 0x7fffffff;
      unsigned hot = 0;   // which of this lane's float4 hold a pixel >= thr (or the maximum)
#pragma unroll
      for (int r = 0; r < kLaneQ; ++r) {
        const float m4 = fmaxf(fmaxf(pv[r].x, pv[r].y), fmaxf(pv[r].z, pv[r].w));
        if (m4 >= thr || m4 == gmax) hot |= 1u << r;  // (a negative maximum is below its own half: thr > gmax)
      }
      while (hot) {        // rolled on purpose: a handful of float4 per map, small code
        const int r = __ffs(hot) - 1;
        hot &= hot - 1;
        const int q = r * 32 + lane;
        const int y = q / (FW / 4), x0 = (q % (FW / 4)) * 4;
        const float4 c4 = load_quad(cur, q);
        const float e[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (e[c] >= thr && is_local_max<FH, FW>(cur, y, x0 + c, e[c], FH, FW)) {
            ps += e[c];
            pc += 1;
          }
          if (e[c] == gmax && cand == 0x7fffffff) {
            cand = q * 4 + c;
            quarter_shift(cur, y, x0 + c, FH, FW, gmax, cx, cy);
          }
        }
      }
      const int best = __reduce_min_sync(0xffffffffu, cand);   // first flat argmax (np.argmax)
      ps = warp_sum(ps);
      pc = warp_sum(pc);
      const size_t o = (size_t)f * J + j;
      if (lane == 0) {
        out.psum[o] = ps;
        out.pcnt[o] = pc;
        out.maxv[o] = gmax;
      }
      if (cand == best) {
        out.hmxy[o * 2 + 0] = cx;
        out.hmxy[o * 2 + 1] = cy;
      }
    }
    // ---- the stage is free: refill it with frame f + kStages
    __syncwarp();
    if (lane == 0 && i + kStages < count) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(&bars[s], kMapBytes);
      tma_load_1d(stage0 + (size_t)s * FPIX, src_of(f + kStages), kMapBytes, &bars[s]);
    }
  }
  if (b == n && !tail_pair && lane == 0) out.pair_sum[(size_t)n * J + j] = 0.0;
}

// ------------------------------------------------------------------------------------
// generic path: any (h,w) with h*w*4 bytes of shared memory; one CTA per (frame, joint).
// Reads the previous frame from global memory again (2x traffic) — used for odd shapes only.
// 16-bit maps are converted while they are staged into the fp32 s_map.
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kScanThreads)
scan_generic(const T* __restrict__ H, const uint8_t* __restrict__ is_prev,
             const uint8_t* __restrict__ is_next, int64_t n, int J, int h, int w,
             const T* __restrict__ halo_prev, const T* __restrict__ halo_next, ScanOut out) {
  extern __shared__ float s_dyn[];
  float* s_map = s_dyn;
  __shared__ float s_wmax[kWarps];
  __shared__ float s_wsum[kWarps];
  __shared__ float s_wps[kWarps];
  __shared__ int s_wpc[kWarps];
  __shared__ int s_arg;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int j = blockIdx.y;
  const int64_t t = blockIdx.x;  // 0..n  (t == n: trailing pair only)
  const int npx = h * w;
  const bool has_hp = halo_prev != nullptr, has_hn = halo_next != nullptr;
  const bool want = pair_wanted(t, n, is_prev, is_next, has_hp, has_hn);
  const T* cur = (t < n) ? H + ((size_t)t * J + j) * npx : (has_hn ? halo_next + (size_t)j * npx : nullptr);
  const T* prv = (t > 0) ? H + ((size_t)(t - 1) * J + j) * npx : (has_hp ? halo_prev + (size_t)j * npx : nullptr);
  if (tid == 0) s_arg = 0x7fffffff;
  float lmax = -INFINITY, s = 0.0f;
  if (cur) {
    for (int p = tid; p < npx; p += kScanThreads) {
      const float val = to_f32(cur[p]);
      s_map[p] = val;
      lmax = fmaxf(lmax, val);
      if (want) s += fabsf(val - to_f32(prv[p]));
    }
  }
  lmax = warp_max(lmax);
  s = warp_sum(s);
  if (lane == 0) {
    s_wmax[warp] = lmax;
    s_wsum[warp] = s;
  }
  __syncthreads();
  float gmax = s_wmax[0];
  for (int k = 1; k < kWarps; ++k) gmax = fmaxf(gmax, s_wmax[k]);
  if (tid == 0) {
    double ps = 0.0;
    for (int k = 0; k < kWarps; ++k) ps += (double)s_wsum[k];
    out.pair_sum[(size_t)t * J + j] = want ? ps : 0.0;
  }
  if (t >= n) return;
  const float thr = 0.5f * gmax;
  float ps = 0.0f, cx = 0.f, cy = 0.f;
  int pc = 0, cand = 0x7fffffff;
  for (int p = tid; p < npx; p += kScanThreads) {
    const float val = s_map[p];
    if (val >= thr || val == gmax) {
      const int y = p / w, x = p % w;
      if (val >= thr && is_local_max<0, 0>(s_map, y, x, val, h, w)) {
        ps += val;
        pc += 1;
      }
      if (val == gmax && cand == 0x7fffffff) {
        cand = p;
        quarter_shift(s_map, y, x, h, w, gmax, cx, cy);
      }
    }
  }
  if (cand != 0x7fffffff) atomicMin(&s_arg, cand);
  ps = warp_sum(ps);
  pc = warp_sum(pc);
  if (lane == 0) {
    s_wps[warp] = ps;
    s_wpc[warp] = pc;
  }
  __syncthreads();
  const size_t o = (size_t)t * J + j;
  if (tid == 0) {
    float tps = 0.0f;
    int tpc = 0;
    for (int k = 0; k < kWarps; ++k) {
      tps += s_wps[k];
      tpc += s_wpc[k];
    }
    out.psum[o] = tps;
    out.pcnt[o] = tpc;
    out.maxv[o] = gmax;
  }
  if (cand != 0x7fffffff && cand == s_arg) {
    out.hmxy[o * 2 + 0] = cx;
    out.hmxy[o * 2 + 1] = cy;
  }
}

// ------------------------------------------------------------------------------------
// per-frame epilogue: x2 rule, peak mean, heat-map -> image coordinates
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
scan_finalize(int64_t n, int J, int h, int w, const uint8_t* __restrict__ is_prev,
              const uint8_t* __restrict__ is_next, bool has_hp, bool has_hn,
              const float* __restrict__ bbox, ScanOut in, float* __restrict__ thc,
              float* __restrict__ peak_sum, int32_t* __restrict__ peak_cnt, float* __restrict__ peak_mean,
              float* __restrict__ coords_hm, float* __restrict__ kpts) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  if (thc) {
    // ActiveLearning.py:345-363: add the pair terms that exist, double when only one does
    const bool hp = is_prev && is_prev[t] && (t > 0 || has_hp);
    const bool hn = is_next && is_next[t] && (t < n - 1 || has_hn);
    double sp = 0.0, sn = 0.0;
    for (int j = 0; j < J; ++j) {
      sp += in.pair_sum[(size_t)t * J + j];
      sn += in.pair_sum[(size_t)(t + 1) * J + j];
    }
    double acc = 0.0;
    if (hp) acc += sp / (double)J;
    if (hn) acc += sn / (double)J;
    if (hp != hn) acc *= 2.0;
    thc[t] = (float)acc;
  }
  if (peak_sum || peak_cnt || peak_mean) {
    double s = 0.0;
    int c = 0;
    for (int j = 0; j < J; ++j) {
      s += (double)in.psum[(size_t)t * J + j];
      c += in.pcnt[(size_t)t * J + j];
    }
    if (peak_sum) peak_sum[t] = (float)s;
    if (peak_cnt) peak_cnt[t] = c;
    if (peak_mean) peak_mean[t] = (c > 0) ? (float)(s / (double)c) : __int_as_float(0x7fc00000);
  }
  if (coords_hm) {
    for (int j = 0; j < 2 * J; ++j) coords_hm[(size_t)t * 2 * J + j] = in.hmxy[(size_t)t * 2 * J + j];
  }
  if (kpts) {
    // inverse affine of transforms.py:568-581,753-792 in closed form.  The reference builds
    // three float32 point pairs and lets cv2.getAffineTransform solve them in double; with
    // rot = 0 the solution is a = (X1-X2)/(w/2), c = X2, e = (Y0-Y1)/(w/2),
    // f = Y1 - e*(h/2 - w/2) (b = d = 0), evaluated here on the same float32-rounded points.
    const double xmin = bbox[t * 4 + 0], ymin = bbox[t * 4 + 1], xmax = bbox[t * 4 + 2], ymax = bbox[t * 4 + 3];
    const double bw = __dsub_rn(xmax, xmin), bh = __dsub_rn(ymax, ymin);
    const double cxd = __dadd_rn(xmin, __dmul_rn(bw, 0.5)), cyd = __dadd_rn(ymin, __dmul_rn(bh, 0.5));
    const float X0 = (float)cxd, Y0 = (float)cyd;
    const float Y1 = (float)__dadd_rn(cyd, __dmul_rn(bw, -0.5));
    const float dY = __fsub_rn(Y0, Y1);   // get_3rd_point works on the float32 arrays
    const float X2 = __fsub_rn(X0, dY);
    const double W2 = 0.5 * (double)w, H2 = 0.5 * (double)h;
    const double a = __ddiv_rn(__dsub_rn((double)X0, (double)X2), W2);
    const double e = __ddiv_rn(__dsub_rn((double)Y0, (double)Y1), W2);
    const double f = __dsub_rn((double)Y1, __dmul_rn(e, __dsub_rn(H2, W2)));
    for (int j = 0; j < J; ++j) {
      const size_t o = (size_t)t * J + j;
      const double x = in.hmxy[o * 2 + 0], y = in.hmxy[o * 2 + 1];
      kpts[o * 3 + 0] = (float)__dadd_rn(__dmul_rn(a, x), (double)X2);
      kpts[o * 3 + 1] = (float)__dadd_rn(__dmul_rn(e, y), f);
      kpts[o * 3 + 2] = in.maxv[o];
    }
  }
}

// strict three-tensor THC: one CTA per frame, every tensor read once
template <typename T>
__global__ void __launch_bounds__(256)
thc3_kernel(const T* __restrict__ cur, const T* __restrict__ prev, const T* __restrict__ next,
            const uint8_t* __restrict__ is_prev, const uint8_t* __restrict__ is_next, int64_t n, int J,
            int npx, float* __restrict__ thc) {
  __shared__ double s_p[8], s_n[8];
  const int64_t t = blockIdx.x;
  const bool hp = is_prev && is_prev[t] && prev, hn = is_next && is_next[t] && next;
  const size_t fl = (size_t)J * npx;
  const T* c = cur + t * fl;
  float sp = 0.f, sn = 0.f;
  double dp = 0.0, dn = 0.0;
  if (hp || hn) {
    const T* p = prev ? prev + t * fl : nullptr;
    const T* q = next ? next + t * fl : nullptr;
    if ((fl & 3) == 0) {
      int cnt = 0;
      for (size_t i = threadIdx.x; i < fl / 4; i += blockDim.x) {
        const float4 x = ldg_stream_quad(c, i);
        if (hp) {
          const float4 y = ldg_stream_quad(p, i);
          sp += fabsf(x.x - y.x) + fabsf(x.y - y.y) + fabsf(x.z - y.z) + fabsf(x.w - y.w);
        }
        if (hn) {
          const float4 y = ldg_stream_quad(q, i);
          sn += fabsf(x.x - y.x) + fabsf(x.y - y.y) + fabsf(x.z - y.z) + fabsf(x.w - y.w);
        }
        if (++cnt == 16) {  // bound the fp32 run length
          dp += sp; dn += sn; sp = sn = 0.f; cnt = 0;
        }
      }
    } else {
      for (size_t i = threadIdx.x; i < fl; i += blockDim.x) {
        if (hp) dp += fabsf(to_f32(c[i]) - to_f32(p[i]));
        if (hn) dn += fabsf(to_f32(c[i]) - to_f32(q[i]));
      }
    }
    dp += sp;
    dn += sn;
  }
  dp = warp_sum(dp);
  dn = warp_sum(dn);
  if ((threadIdx.x & 31) == 0) {
    s_p[threadIdx.x >> 5] = dp;
    s_n[threadIdx.x >> 5] = dn;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) {
      a += s_p[k];
      b += s_n[k];
    }
    double acc = 0.0;
    if (hp) acc += a / (double)J;
    if (hn) acc += b / (double)J;
    if (hp != hn) acc *= 2.0;
    thc[t] = (float)acc;
  }
}

}  // namespace vatlq

using namespace vatlq;

extern "C" size_t vatlq_heatmap_scan_workspace_bytes(int64_t n, int J) {
  if (n < 0 || J <= 0) return 0;
  size_t nj = (size_t)n * J;
  return align_up((size_t)(n + 1) * J * sizeof(double), 256) + 3 * align_up(nj * 4, 256) +
         align_up(nj * 8, 256);
}

template <typename T>
static int launch_scan(const T* H, const uint8_t* is_prev, const uint8_t* is_next, int64_t n, int J, int h, int w,
                       const T* halo_prev, const T* halo_next, const ScanOut& so, cudaStream_t stream) {
  const bool fast = (h == FH && w == FW) && (halo_prev == nullptr || ((uintptr_t)halo_prev & 15) == 0) &&
                    (halo_next == nullptr || ((uintptr_t)halo_next & 15) == 0);
  if (fast) {
    // one warp per (run, joint) task, ~4 tasks per warp slot so that CTAs finishing early are
    // replaced; runs no shorter than 8 frames keep the halo re-read <= 1/8 of the traffic.
    // fp32: 8 warps x 2 stages per SM measured best (6.8 TB/s; 6x3 5.3, 4x4 3.7: tools/tune_scan.py);
    // 16-bit: 8 warps x VQ_SCAN_STAGES16 stages
    const int64_t slots = (int64_t)sm_count() * kTmaWarps;
    int64_t runs = (slots * 4 + J - 1) / J;
    int64_t run_len = (n + runs - 1) / runs;
    if (run_len < 8) run_len = 8;
    if (run_len > n) run_len = n;
    runs = (n + run_len - 1) / run_len;
    const int64_t tasks = runs * J;
    static bool cfg = false;
    if (!cfg) {
      VQ_CUDA(cudaFuncSetAttribute(scan_tma_64x48<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tma_smem<T>()));
      cfg = true;
    }
    VQ_REQUIRE((tasks + kTmaWarps - 1) / kTmaWarps <= 2147483647LL, "grid too large");
    scan_tma_64x48<T><<<(unsigned)((tasks + kTmaWarps - 1) / kTmaWarps), kTmaWarps * 32, tma_smem<T>(), stream>>>(
        H, is_prev, is_next, n, J, halo_prev, halo_next, (int)run_len, runs, so);
    VQ_LAUNCHED();
  } else {
    const size_t smem = (size_t)h * w * sizeof(float);
    VQ_REQUIRE(smem <= 200 * 1024, "map too large for the generic path");
    VQ_REQUIRE(n + 1 <= 2147483647LL && J <= 65535, "grid too large");
    if (smem > 48 * 1024)
      VQ_CUDA(cudaFuncSetAttribute(scan_generic<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)(n + 1), (unsigned)J);
    scan_generic<T><<<grid, kScanThreads, smem, stream>>>(H, is_prev, is_next, n, J, h, w, halo_prev, halo_next, so);
    VQ_LAUNCHED();
  }
  return 0;
}

extern "C" int vatlq_heatmap_scan_dt(const void* H, int dtype, const uint8_t* is_prev, const uint8_t* is_next,
                                     int64_t n, int J, int h, int w, const void* halo_prev,
                                     const void* halo_next, const float* bbox_xyxy, float* thc,
                                     float* peak_sum, int32_t* peak_cnt, float* peak_mean,
                                     float* coords_hm, float* kpts, void* ws, size_t ws_bytes,
                                     vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(n >= 0 && J > 0 && h > 0 && w > 0, "bad shape");
  VQ_REQUIRE(dtype_size(dtype) != 0, "unknown dtype (VATLQ_F32, VATLQ_F16 or VATLQ_BF16)");
  if (n == 0) return 0;
  VQ_REQUIRE(H != nullptr, "H is null");
  VQ_REQUIRE(((uintptr_t)H & 15) == 0, "H must be 16-byte aligned");
  VQ_REQUIRE(dtype == VATLQ_F32 || ((((uintptr_t)halo_prev | (uintptr_t)halo_next) & 7) == 0),
             "16-bit halos must be 8-byte aligned");
  VQ_REQUIRE(kpts == nullptr || bbox_xyxy != nullptr, "kpts needs bbox_xyxy");
  VQ_REQUIRE(ws != nullptr && ws_bytes >= vatlq_heatmap_scan_workspace_bytes(n, J), "workspace too small");
  const size_t nj = (size_t)n * J;
  char* p = (char*)ws;
  ScanOut so;
  so.pair_sum = (double*)p; p += align_up((size_t)(n + 1) * J * sizeof(double), 256);
  so.psum = (float*)p;      p += align_up(nj * 4, 256);
  so.pcnt = (int*)p;        p += align_up(nj * 4, 256);
  so.maxv = (float*)p;      p += align_up(nj * 4, 256);
  so.hmxy = (float*)p;

  const int rc = with_dtype(dtype, [&](auto tag) {
    using T = std::remove_const_t<std::remove_pointer_t<decltype(tag)>>;
    return launch_scan<T>((const T*)H, is_prev, is_next, n, J, h, w, (const T*)halo_prev, (const T*)halo_next, so, stream);
  });
  if (rc != 0) return rc;
  const int fb = 128;
  scan_finalize<<<(unsigned)((n + fb - 1) / fb), fb, 0, stream>>>(
      n, J, h, w, is_prev, is_next, halo_prev != nullptr, halo_next != nullptr, bbox_xyxy, so, thc,
      peak_sum, peak_cnt, peak_mean, coords_hm, kpts);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_heatmap_scan(const float* H, const uint8_t* is_prev, const uint8_t* is_next,
                                  int64_t n, int J, int h, int w, const float* halo_prev,
                                  const float* halo_next, const float* bbox_xyxy, float* thc,
                                  float* peak_sum, int32_t* peak_cnt, float* peak_mean,
                                  float* coords_hm, float* kpts, void* ws, size_t ws_bytes,
                                  vatlq_stream_t stream) {
  return vatlq_heatmap_scan_dt(H, VATLQ_F32, is_prev, is_next, n, J, h, w, halo_prev, halo_next, bbox_xyxy, thc, peak_sum,
                               peak_cnt, peak_mean, coords_hm, kpts, ws, ws_bytes, stream);
}

extern "C" int vatlq_thc3_dt(const void* cur, const void* prev, const void* next, int dtype, const uint8_t* is_prev,
                             const uint8_t* is_next, int64_t n, int J, int h, int w, float* thc,
                             vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(n >= 0 && J > 0 && h > 0 && w > 0, "bad shape");
  VQ_REQUIRE(dtype_size(dtype) != 0, "unknown dtype (VATLQ_F32, VATLQ_F16 or VATLQ_BF16)");
  if (n == 0) return 0;
  VQ_REQUIRE(cur && thc, "null pointer");
  VQ_REQUIRE(n <= 2147483647LL, "n too large");
  const size_t fl = (size_t)J * h * w;
  if ((fl & 3) == 0)
    VQ_REQUIRE(quad_aligned((const void*)((uintptr_t)cur | (uintptr_t)prev | (uintptr_t)next), dtype),
               dtype == VATLQ_F32 ? "tensors must be 16-byte aligned" : "16-bit tensors must be 8-byte aligned");
  return with_dtype(dtype, [&](auto tag) {
    using T = std::remove_const_t<std::remove_pointer_t<decltype(tag)>>;
    thc3_kernel<T><<<(unsigned)n, 256, 0, stream>>>((const T*)cur, (const T*)prev, (const T*)next, is_prev, is_next, n, J,
                                                    h * w, thc);
    VQ_LAUNCHED();
    return 0;
  });
}

extern "C" int vatlq_thc3(const float* cur, const float* prev, const float* next, const uint8_t* is_prev,
                          const uint8_t* is_next, int64_t n, int J, int h, int w, float* thc,
                          vatlq_stream_t stream) {
  return vatlq_thc3_dt(cur, prev, next, VATLQ_F32, is_prev, is_next, n, J, h, w, thc, stream);
}
