// Labelled-set initialisation of the core-set (min_d[i] = min over the labelled centres of d(i,c),
// ActiveLearning.py:802-814,841 — sklearn materialises the N x L distance matrix) on the 5th-generation
// tensor cores:  a TF32 tcgen05 GEMM with a PROVED error bound decides which (row, centre) pairs can
// possibly be the minimum; only those are re-scored with the canonical fp64 arithmetic.
//
//   sweep 1  tcgen05.mma kind::tf32 (operands fp32 in shared memory via 2-D TMA, 128B swizzle; fp32
//            accumulators in TMEM, double buffered; 128 x 256 tiles, K = 2048 in 64 blocks of 32):
//            t~(i,c) = |x_i|^2 + |c|^2 - 2 S~(i,c)  and its running minimum per row (one epilogue thread
//            per row = TMEM lane, so the minimum lives in a register).
//   sweep 2  the same GEMM again for the same 128 rows: every (row, group of 8 centres) with
//            t~(i,c) <= t~min(i) + 2 E(i) is appended to a list.
//   rescore  the list, sorted by centre group, goes through the canonical fp64 DMMA tile the exact
//            passes of coreset.cu use (canonical.cuh: 8 centres as register-resident B operands, 8
//            listed rows per tile) and min_d is lowered with atomicMin on the bit pattern of the
//            (non-negative) distance.
//
// Error bound.  kind::tf32 uses the upper 19 bits of each fp32 operand (relative error <= 2^-10 per
// operand, whether truncated or rounded), products are accumulated in fp32 over K = 2048.  With
// u = 2^-8 (a factor 2 above 2*2^-10 + 2^-20 + 2048*2^-24 relative to sum_k |x_k c_k| <= |x||c|):
//      |S~ - S| <= u |x_i| |c|,   |t~ - t| <= E(i) := 2 u |x_i| max_c |c| + 2^-20 (|x_i|^2 + max|c|^2)
// (the second term covers the fp32 epilogue arithmetic).  If c* minimises the exact t(i,.) then
// t~(i,c*) <= t(i,c*) + E <= t(i,c) + E <= t~(i,c) + 2E for every c, so c* is always listed and
// min over the listed pairs of the canonical value == min over ALL centres, bit for bit.
// flags & 1 additionally checks t~ against the bound on a sample of the entries (tests).
#include <cuda.h>
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "canonical.cuh"

namespace vatlq {

constexpr int TC_BM = 128;          // rows per tile (UMMA M, one TMEM lane per row)
constexpr int TC_BN = 256;          // centres per tile (UMMA N)
constexpr int TC_BK = 32;           // fp32 per k-block: 128 bytes = one 128B-swizzle atom row
constexpr int TC_STAGES = 4;
constexpr int TC_D = 2048;
static_assert(TC_D == kFastD, "the re-score keeps 1/8 of a centre in registers (canonical.cuh)");
constexpr int TC_KB = TC_D / TC_BK; // 64 k-blocks
constexpr int TC_A_BYTES = TC_BM * TC_BK * 4;    // 16 KB
constexpr int TC_B_BYTES = TC_BN * TC_BK * 4;    // 32 KB
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr int TC_THREADS = 192;     // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue
constexpr size_t TC_SMEM = (size_t)TC_STAGES * TC_STAGE_BYTES + 1024 /*alignment slack*/ + 2 * TC_BN * 4 + 256;
constexpr double TC_U = 1.0 / 256.0;

__device__ __forceinline__ void tc_tma_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(bar)
               : "memory");
}
// K-major operand tile, 128-byte swizzle: rows of 128 bytes, 8-row atoms 1024 bytes apart (SBO), LBO unused
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);          // start address
  d |= (uint64_t)0 << 16;                              // leading byte offset (one atom along K)
  d |= (uint64_t)((1024 >> 4) & 0x3FFF) << 32;         // stride byte offset between 8-row atoms
  d |= (uint64_t)1 << 46;                              // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                              // SWIZZLE_128B
  return d;
}
// kind::tf32, D = F32, A/B = TF32, both K-major, M = 128, N = 256
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);

__device__ __forceinline__ void tc_mma(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_c), "l"(da), "l"(db), "r"(TC_IDESC), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct TcArgs {
  const double* xx;        // canonical squared norms of every row of X
  const long long* centers;  // labelled row indices (global)
  const float* cnorm2;     // |c|^2 per centre (fp32), TC_BN-padded with +inf
  long long lo, hi;        // owned rows
  int L;                   // centres
  double cmax;             // max_c |c|
  int* pair_group;         // out: (centre group, row) pairs
  int* pair_row;
  unsigned int* pair_count;   // [0] pairs written (may exceed cap -> overflow), [1] bound violations (verify)
  unsigned int cap;
  int verify;              // check |t~ - t| <= E against fp64 on a sample of the entries
  const float* X;          // (verify only)
  float* tmin_out;         // optional: t~min per owned row (tests)
};

__global__ void __launch_bounds__(TC_THREADS, 1)
tc_prefilter_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, TcArgs a) {
  extern __shared__ unsigned char smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;       // swizzle-128B tiles need 1024-byte alignment
  unsigned char* gen = smem_raw + (base - smem_u32(smem_raw));
  float* s_cn = reinterpret_cast<float*>(gen + (size_t)TC_STAGES * TC_STAGE_BYTES);   // [2][TC_BN] centre norms
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_cn + 2 * TC_BN);
  uint64_t* full = bars;                    // [TC_STAGES] TMA -> MMA
  uint64_t* empty = bars + TC_STAGES;       // [TC_STAGES] MMA -> TMA
  uint64_t* tfull = bars + 2 * TC_STAGES;   // [2] MMA -> epilogue
  uint64_t* tempty = tfull + 2;             // [2] epilogue -> MMA
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(tempty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 4);             // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {                           // TMEM: all 512 columns (two 128 x 256 fp32 accumulators)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *s_tmem;

  const long long own = a.hi - a.lo;
  const int num_m = (int)((own + TC_BM - 1) / TC_BM);
  const int nblk = (a.L + TC_BN - 1) / TC_BN;
  const int iters_per_m = 2 * nblk;          // sweep 1 then sweep 2 over the same centre blocks

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int st = 0;
      unsigned ph = 0;
      for (int m = blockIdx.x; m < num_m; m += gridDim.x) {
        for (int it = 0; it < iters_per_m; ++it) {
          const int nb = it % nblk;
          for (int kb = 0; kb < TC_KB; ++kb) {
            mbar_wait(&empty[st], ph ^ 1u);
            const uint32_t sa = base + st * TC_STAGE_BYTES, sb = sa + TC_A_BYTES;
            mbar_expect_tx(&full[st], (uint32_t)TC_STAGE_BYTES);
            tc_tma_2d(sa, &tmA, kb * TC_BK, m * TC_BM, smem_u32(&full[st]));
            tc_tma_2d(sb, &tmB, kb * TC_BK, nb * TC_BN, smem_u32(&full[st]));
            if (++st == TC_STAGES) {
              st = 0;
              ph ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (one thread)
    if (lane == 0) {
      int st = 0, acc = 0;
      unsigned ph = 0, aph = 0;
      for (int m = blockIdx.x; m < num_m; m += gridDim.x) {
        for (int it = 0; it < iters_per_m; ++it) {
          mbar_wait(&tempty[acc], aph ^ 1u);                 // the epilogue has drained this accumulator
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t tacc = tmem + (uint32_t)(acc * TC_BN);
          for (int kb = 0; kb < TC_KB; ++kb) {
            mbar_wait(&full[st], ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa = base + st * TC_STAGE_BYTES, sb = sa + TC_A_BYTES;
            const uint64_t da = tc_smem_desc(sa), db = tc_smem_desc(sb);
#pragma unroll
            for (int k = 0; k < TC_BK / 8; ++k)               // UMMA K = 8 tf32 = 32 bytes: advance inside the atom
              tc_mma(tacc, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), (kb | k) != 0 ? 1u : 0u);
            tc_commit(smem_u32(&empty[st]));                  // frees the stage when these MMAs retire
            if (++st == TC_STAGES) {
              st = 0;
              ph ^= 1u;
            }
          }
          tc_commit(smem_u32(&tfull[acc]));                   // accumulator complete
          if (++acc == 2) {
            acc = 0;
            aph ^= 1u;
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: one thread per row (TMEM lane)
    const int q = warp & 3;                                   // TMEM lane group this warp may read
    const int r = q * 32 + lane;                              // row inside the tile
    const int et = threadIdx.x - 64;                          // 0..127
    int acc = 0;
    unsigned aph = 0;
    for (int m = blockIdx.x; m < num_m; m += gridDim.x) {
      const long long i = a.lo + (long long)m * TC_BM + r;
      const bool live = i < a.hi;
      const double xxi_d = live ? a.xx[i] : 0.0;
      const float xxi = (float)xxi_d;
      // E(i): see the header; evaluated in fp64, rounded up into fp32
      const double E = 2.0 * TC_U * sqrt(xxi_d) * a.cmax + ldexp(xxi_d + a.cmax * a.cmax, -20);
      const float twoE = (float)(2.0 * E * (1.0 + 1e-6));
      float tmin = INFINITY;
      for (int it = 0; it < iters_per_m; ++it) {
        const int nb = it % nblk;
        const bool emit = it >= nblk;
        // this block's centre norms (double buffered with the accumulators; +inf beyond L)
        float* cn = s_cn + acc * TC_BN;
        for (int c = et; c < TC_BN; c += 128) {
          const int gc = nb * TC_BN + c;
          cn[c] = gc < a.L ? a.cnorm2[gc] : INFINITY;
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");        // the 4 epilogue warps
        mbar_wait(&tfull[acc], aph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * TC_BN);
#pragma unroll 1
        for (int c0 = 0; c0 < TC_BN; c0 += 32) {
          uint32_t v[32];
          tc_ld32(trow + (uint32_t)c0, v);
          if (!emit) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float t = (xxi + cn[c0 + j]) - 2.0f * __uint_as_float(v[j]);
              tmin = fminf(tmin, t);
            }
          } else {
            const float thr = tmin + twoE;
#pragma unroll
            for (int g8 = 0; g8 < 4; ++g8) {
              bool hit = false;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float t = (xxi + cn[c0 + g8 * 8 + j]) - 2.0f * __uint_as_float(v[g8 * 8 + j]);
                hit = hit || (t <= thr);
              }
              if (hit && live) {
                const unsigned pos = atomicAdd(&a.pair_count[0], 1u);
                if (pos < a.cap) {
                  a.pair_group[pos] = (nb * TC_BN + c0) / 8 + g8;
                  a.pair_row[pos] = (int)(i - a.lo);
                }
              }
            }
            if (a.verify && live && ((i + c0) % 61) == 0) {   // sampled check of the bound against fp64
              const int j = (int)(i % 32);
              const int gc = nb * TC_BN + c0 + j;
              if (gc < a.L) {
                const float* xr = a.X + (size_t)i * TC_D;
                const float* cr = a.X + (size_t)a.centers[gc] * TC_D;
                double dot = 0.0;
                for (int kx = 0; kx < TC_D; ++kx) dot = fma((double)xr[kx], (double)cr[kx], dot);
                const double texact = xxi_d + a.xx[a.centers[gc]] - 2.0 * dot;
                float sv = 0.f;
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) sv = (jj == j) ? __uint_as_float(v[jj]) : sv;   // (keeps v[] in registers)
                const float t = (xxi + cn[c0 + j]) - 2.0f * sv;
                if (fabs((double)t - texact) > E) atomicAdd(&a.pair_count[1], 1u);
              }
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
        if (++acc == 2) {
          acc = 0;
          aph ^= 1u;
        }
      }
      if (a.tmin_out && live) a.tmin_out[i - a.lo] = tmin;
    }
  }
  // ---- teardown
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// gather the labelled rows into a contiguous (Lpad, 2048) fp32 matrix (TMA wants a dense tensor) + fp32 |c|^2
__global__ void __launch_bounds__(256) tc_gather_kernel(const float* __restrict__ X, const long long* __restrict__ centers, int L,
                                                        const double* __restrict__ xx, float* __restrict__ C,
                                                        float* __restrict__ cnorm2, unsigned long long* cmax2_bits) {
  const int c = blockIdx.x;
  if (c >= L) return;
  const long long p = centers[c];
  const float4* src = reinterpret_cast<const float4*>(X) + (size_t)p * (TC_D / 4);
  float4* dst = reinterpret_cast<float4*>(C) + (size_t)c * (TC_D / 4);
  for (int q = threadIdx.x; q < TC_D / 4; q += blockDim.x) dst[q] = __ldg(src + q);
  if (threadIdx.x == 0) {
    const double v = xx[p];
    cnorm2[c] = (float)v;
    atomicMax(cmax2_bits, (unsigned long long)__double_as_longlong(fmax(v, 0.0)));   // non-negative doubles order like integers
  }
}

// ---- exact re-scoring of the listed (centre group, row) pairs on the canonical fp64 tile (canonical.cuh) --------
// (the helpers the exact passes of coreset.cu use: 8 K-segments by 8 warps, four DMMA chains per segment, fixed
// combine tree, so the re-scored distances are theirs bit for bit)
// one CTA per centre group (8 labelled centres): its slice of the sorted pair list is found by binary search
__global__ void __launch_bounds__(kSeg * 32, 1)
tc_rescore_kernel(const float* __restrict__ X, long long lo, const long long* __restrict__ centers, int L,
                  const double* __restrict__ xx, const int* __restrict__ sorted_group, const int* __restrict__ sorted_row,
                  const unsigned int* __restrict__ pair_count, unsigned int cap, double* __restrict__ min_d) {
  __shared__ __align__(16) double s_part[kSeg][64];
  __shared__ double s_xxc[8];
  __shared__ int s_rng[2];
  const unsigned int npairs = min(pair_count[0], cap);
  const int grp = blockIdx.x;
  if (threadIdx.x == 0) {
    int b0 = 0, e0 = (int)npairs;                 // lower bound of grp
    while (b0 < e0) {
      const int mid = (b0 + e0) >> 1;
      if (sorted_group[mid] < grp) b0 = mid + 1; else e0 = mid;
    }
    int b1 = b0, e1 = (int)npairs;                // lower bound of grp + 1
    while (b1 < e1) {
      const int mid = (b1 + e1) >> 1;
      if (sorted_group[mid] < grp + 1) b1 = mid + 1; else e1 = mid;
    }
    s_rng[0] = b0;
    s_rng[1] = b1;
  }
  __syncthreads();
  const int beg = s_rng[0], end = s_rng[1];
  if (beg >= end) return;
  const int lane = threadIdx.x & 31, seg = threadIdx.x >> 5, g = lane >> 2, kk = lane & 3;
  const float4* X4 = reinterpret_cast<const float4*>(X);
  const int lane_off = seg * (kSteps * 4) + kk;
  const int nc = min(8, L - grp * 8);
  double breg[kSteps][4];
  centre_slice(X, TC_D / 4, centers[grp * 8 + min(g, nc - 1)], seg, kk, breg);
  if (threadIdx.x < 8) s_xxc[threadIdx.x] = xx[centers[grp * 8 + min((int)threadIdx.x, nc - 1)]];
  for (int t0 = beg; t0 < end; t0 += 8) {
    const long long row = lo + sorted_row[min(t0 + g, end - 1)];
    const float4* rp = X4 + (size_t)row * (TC_D / 4) + lane_off;
    float4 xr[kSteps];
#pragma unroll
    for (int s = 0; s < kSteps; ++s) xr[s] = __ldg(rp + 4 * s);
    double c[4][2];
#pragma unroll
    for (int e = 0; e < 4; ++e) c[e][0] = c[e][1] = 0.0;
#pragma unroll
    for (int s = 0; s < kSteps; ++s) seg_step(c, xr[s], breg[s]);
    __syncthreads();                               // (the previous tile's partials have been consumed)
    *reinterpret_cast<double2*>(&s_part[seg][lane * 2]) = seg_partial(c);
    __syncthreads();
    // warp w finishes row w of the tile: lane j < 8 holds centre j
    const int myrow = t0 + seg;
    if (myrow < end) {
      const long long ri = lo + sorted_row[myrow];
      double sq = INFINITY;
      // (padded centres repeat the last one: min is idempotent)
      if (lane < 8) sq = sq_from_dot(combine8(&s_part[0][seg * 8 + lane], 64), xx[ri], s_xxc[lane]);
#pragma unroll
      for (int o = 4; o; o >>= 1) sq = fmin(sq, __shfl_xor_sync(0xffffffffu, sq, o));
      if (lane == 0) {
        const double dist = sqrt(fmax(sq, 0.0));
        atomicMin(reinterpret_cast<unsigned long long*>(&min_d[ri]), (unsigned long long)__double_as_longlong(dist));
      }
    }
  }
}

// ---------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}
static int make_map(CUtensorMap* tm, const float* base, uint64_t rows, uint32_t box_rows) {
  EncodeTiledFn enc = encode_tiled();
  VQ_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  const cuuint64_t gdim[2] = {(cuuint64_t)TC_D, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)TC_D * 4};
  const cuuint32_t box[2] = {(cuuint32_t)TC_BK, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return VATLQ_EINVAL;
  }
  return 0;
}

struct TcLayout {
  size_t xx, C, cnorm, cmax, count, pg, pr, sg, sr, cub, tmin, total;
  size_t cub_bytes;
  unsigned int cap;
};
static TcLayout tc_layout(int64_t n, int64_t own, int64_t L) {
  TcLayout T{};
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t at = o;
    o += align_up(bytes, 1024);
    return at;
  };
  T.xx = take((size_t)n * 8);
  const size_t Lpad = align_up((size_t)std::max<int64_t>(L, 1), TC_BN);
  T.C = take(Lpad * TC_D * 4);
  T.cnorm = take(Lpad * 4);
  T.cmax = take(64);
  T.count = take(64);
  T.cap = (unsigned int)std::min<size_t>((size_t)own * 24 + (1u << 20), 0x7fffff00u);
  T.pg = take((size_t)T.cap * 4);
  T.pr = take((size_t)T.cap * 4);
  T.sg = take((size_t)T.cap * 4);
  T.sr = take((size_t)T.cap * 4);
  size_t cb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cb, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, (int)T.cap);
  T.cub_bytes = cb;
  T.cub = take(cb);
  T.tmin = take((size_t)own * 4);
  T.total = o;
  return T;
}

}  // namespace vatlq

using namespace vatlq;

extern "C" size_t vatlq_coreset_init_tc_workspace_bytes(int64_t n, int64_t n_owned, int64_t n_labeled) {
  if (n < 0 || n_owned < 0 || n_labeled < 0) return 0;
  return tc_layout(n, n_owned, n_labeled).total;
}

// stats4: {pairs listed, pair capacity, bound violations seen by the sampled check (flags & 1), centre groups}
extern "C" int vatlq_coreset_init_tc(const float* X, int64_t n, int d, int64_t row_lo, int64_t row_hi, const int64_t* labeled,
                                     int64_t n_labeled, double* min_d, void* ws, size_t ws_bytes, int flags,
                                     int64_t* host_stats4, float* tmin_out, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(X && labeled && min_d && ws, "null pointer");
  VQ_REQUIRE(d == TC_D, "the tensor-core initialisation is built for d = 2048");
  VQ_REQUIRE(0 <= row_lo && row_lo < row_hi && row_hi <= n && n_labeled > 0 && n_labeled < (1LL << 27), "bad sizes");
  VQ_REQUIRE(((uintptr_t)X & 15) == 0, "X must be 16-byte aligned");
  const int64_t own = row_hi - row_lo;
  const TcLayout T = tc_layout(n, own, n_labeled);
  VQ_REQUIRE(ws_bytes >= T.total, "workspace too small (vatlq_coreset_init_tc_workspace_bytes)");
  const int verify = flags & 1;
  char* w = (char*)ws;
  double* xx = (double*)(w + T.xx);
  if (int e = vq_launch_norms(X, n, d, xx, stream)) return e;
  float* C = (float*)(w + T.C);
  float* cnorm = (float*)(w + T.cnorm);
  unsigned long long* cmax_bits = (unsigned long long*)(w + T.cmax);
  unsigned int* count = (unsigned int*)(w + T.count);
  const int L = (int)n_labeled;
  const size_t Lpad = align_up((size_t)L, TC_BN);
  VQ_CUDA(cudaMemsetAsync(cmax_bits, 0, 64, stream));
  VQ_CUDA(cudaMemsetAsync(count, 0, 64, stream));
  if (Lpad > (size_t)L) VQ_CUDA(cudaMemsetAsync(C + (size_t)L * TC_D, 0, (Lpad - L) * TC_D * 4, stream));
  tc_gather_kernel<<<L, 256, 0, stream>>>(X, (const long long*)labeled, L, xx, C, cnorm, cmax_bits);
  VQ_LAUNCHED();
  double cmax2 = 0.0;
  VQ_CUDA(cudaMemcpyAsync(&cmax2, cmax_bits, 8, cudaMemcpyDeviceToHost, stream));
  VQ_CUDA(cudaStreamSynchronize(stream));       // (one scalar: the bound needs max|c| before the GEMM is launched)
  CUtensorMap tmA, tmB;
  if (int e = make_map(&tmA, X + (size_t)row_lo * TC_D, (uint64_t)own, TC_BM)) return e;
  if (int e = make_map(&tmB, C, (uint64_t)Lpad, TC_BN)) return e;
  static bool cfg = false;
  if (!cfg) {
    VQ_CUDA(cudaFuncSetAttribute(tc_prefilter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM));
    cfg = true;
  }
  TcArgs a{};
  a.xx = xx; a.centers = (const long long*)labeled; a.cnorm2 = cnorm; a.lo = row_lo; a.hi = row_hi; a.L = L;
  a.cmax = sqrt(cmax2);
  a.pair_group = (int*)(w + T.pg); a.pair_row = (int*)(w + T.pr); a.pair_count = count; a.cap = T.cap;
  a.verify = verify; a.X = X; a.tmin_out = tmin_out;
  const int num_m = (int)((own + TC_BM - 1) / TC_BM);
  const int grid = std::min(num_m, sm_count());
  tc_prefilter_kernel<<<grid, TC_THREADS, TC_SMEM, stream>>>(tmA, tmB, a);
  VQ_LAUNCHED();
  unsigned int h_count[2] = {0, 0};
  VQ_CUDA(cudaMemcpyAsync(h_count, count, 8, cudaMemcpyDeviceToHost, stream));
  VQ_CUDA(cudaStreamSynchronize(stream));
  if (host_stats4) {
    host_stats4[0] = h_count[0];
    host_stats4[1] = T.cap;
    host_stats4[2] = h_count[1];
    host_stats4[3] = (L + 7) / 8;
  }
  if (h_count[0] > T.cap) {
    snprintf(g_err, sizeof(g_err), "tensor-core initialisation: candidate list overflow (%u pairs, capacity %u)", h_count[0], T.cap);
    return VATLQ_ESTATE;      // the caller falls back to the exact passes (vatlq_coreset_init)
  }
  size_t cb = T.cub_bytes;
  VQ_CUDA(cub::DeviceRadixSort::SortPairs(w + T.cub, cb, (const int*)(w + T.pg), (int*)(w + T.sg), (const int*)(w + T.pr),
                                          (int*)(w + T.sr), (int)h_count[0], 0, 32, stream));
  g_launches.fetch_add(1);
  if (int e = fill_f64(min_d + row_lo, own, INFINITY, stream)) return e;
  tc_rescore_kernel<<<(L + 7) / 8, kSeg * 32, 0, stream>>>(X, row_lo, (const long long*)labeled, L, xx, (const int*)(w + T.sg),
                                                            (const int*)(w + T.sr), count, T.cap, min_d);
  VQ_LAUNCHED();
  return 0;
}
