// K-Means / weighted K-Means query filters (active_learning/ActiveLearning.py:553-580, 593-608): the reference
// clusters the candidate embeddings with sklearn.cluster.KMeans(n_clusters=query_size, random_state=318) and
// queries, per cluster, the member closest to its centre.  sklearn's algorithm (scikit-learn 1.7.1 pinned by the
// reference, sklearn/cluster/_kmeans.py, _k_means_lloyd.pyx, _k_means_common.pyx) restated for the device:
//   * k-means++ seeding (_kmeans_plusplus): per new centre 2 + int(log k) candidates drawn with probability
//     proportional to w * closest_dist_sq (searchsorted into its cumulative sum), squared distances of all rows to
//     the candidates, the candidate with the smallest potential wins.  The random numbers come from the host's
//     numpy RandomState(318) stream exactly as sklearn draws them; everything data-sized runs here, with no
//     host synchronisation between the k steps.
//   * Lloyd iterations (lloyd_iter_chunked_dense): labels = argmin_j (|c_j|^2 - 2 x.c_j) (first minimum), centre
//     sums in ascending row order, empty clusters relocated to the farthest rows, centres *= 1 / weight, centre
//     shifts; strict (labels unchanged) or tolerance convergence is decided by the host from a few scalars.
//   * selection: dis_i = |x_i - c_label(i)|^2, per cluster the row with the smallest dis (lowest index on ties).
// All arithmetic is fp64 over the fp32 embeddings (the reference clusters the same values held as float64); the
// two GEMM-shaped steps (rows x candidates, rows x centres) run on the fp64 tensor cores (mma.sync.m8n8k4.f64,
// DMMA) from a cp.async-staged shared-memory pipeline.
// Which bits matter: label decisions are robust to rounding, but "the member closest to its centre" is a structural
// TIE in every two-member cluster (both members are equally far from their mean), which the reference resolves by the
// rounding of its own arithmetic.  The M step and the final distances therefore follow sklearn / numpy operation by
// operation: X_mean = X.mean(axis=0) (sequential over rows), centre sums of (x - X_mean) * w in ascending row order
// (= sklearn with one OpenMP thread; any thread count for clusters of <= 2 members), * (1 / weight), + X_mean, and
// dis = ((X - centre) ** 2).sum(axis=1) in numpy's pairwise order.  DESIGN.md 4.7.
// Every kernel that reads X is a template on its element type T (float, __half, __nv_bfloat16): a 16-bit feature is
// widened exactly to fp32 where it is loaded and the fp64 instruction sequence after the load is the fp32 one, so a
// 16-bit X gives, bit for bit, every result of its fp32 upcast.
#include <cub/device/device_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

#include <algorithm>
#include <cmath>

#include "canonical.cuh"

namespace vatlq {

namespace km {

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  const unsigned sz = valid ? 16u : 0u;      // src-size 0: the 16 bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem)), "l"(gmem), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// four 16-bit features (8 bytes): the .ca form is the one that copies fewer than 16 bytes
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem, bool valid) {
  const unsigned sz = valid ? 8u : 0u;       // src-size 0: the 8 bytes are zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smem_u32(smem)), "l"(gmem), "r"(sz) : "memory");
}
// a chunk of four X features, copied in X's own type
template <typename T>
__device__ __forceinline__ void cp_async_quad(T* smem, const T* gmem, bool valid) {
  if constexpr (sizeof(T) == 4) cp_async16(smem, gmem, valid);
  else cp_async8(smem, gmem, valid);
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------
// Tile machine: S[i][j] = sum_k X[i][k] * C[j][k], X of type T (n x d, converted on the fly), C fp64 (m x d).
// CTA tile BM rows x BN centres, WM x WN warps, each warp (BM/WM) x (BN/WN) as 8x8 DMMA tiles.  A k-block is 32
// features = two sub-tiles of 16: lane (g = lane/4, q = lane%4) takes features 4q..4q+3 of a sub-tile for its
// row g (one LDS.128 of X, two of C) and feeds them to four DMMAs — the k order inside a DMMA is free as long as
// both operands agree.  Sub-tile rows: X 16 floats (64 B), C 16 + 2 doubles (144 B): both conflict-free.
// A 16-bit X is staged in its own type (16 features = 32 B per sub-tile row, 8-byte cp.async chunks, one LDS.64 per
// lane widened to a float4 in registers): lane (g, q) feeds the same four features to the same four DMMAs as in fp32,
// so the accumulators hold the same bits.
// MODE 0 (assign): running argmin_j (cn[j] - 2 S) over all centre chunks -> labels (+ count of changed labels)
// MODE 1 (dist)  : out[i*BN + j] = max(0, (-2 S + cc[j]) + xx[i])   (sklearn _euclidean_distances, squared)
// ------------------------------------------------------------------------------------
constexpr int kBK = 32;
constexpr int kStages = 3;
constexpr int kCS = 18;      // doubles per C sub-tile row

template <typename T, int BM, int BN>
struct GemmStage {
  static constexpr size_t kXBytes = (size_t)2 * BM * 16 * sizeof(T);
  static constexpr size_t kBytes = kXBytes + (size_t)2 * BN * kCS * 8;
};

struct GemmArgs {
  const void* X;         // n x d of the kernel's element type
  long long n;
  int d;
  const double* C;       // m x d
  long long m;
  const double* cn;      // MODE 0: |c_j|^2;  MODE 1: cc[j] (candidate norms)
  const double* xx;      // MODE 1: |x_i|^2
  int* labels;           // MODE 0
  const int* labels_old; // MODE 0, optional
  int* changed;          // MODE 0, optional: += rows whose label differs from labels_old
  double* out;           // MODE 1: n x BN
};

template <typename T, int BM, int BN, int WM, int WN, int MODE>
__global__ void __launch_bounds__(WM * WN * 32) km_gemm_kernel(GemmArgs a) {
  pdl_enter();
  using Stage = GemmStage<T, BM, BN>;
  const T* X = static_cast<const T*>(a.X);
  constexpr int kThreads = WM * WN * 32;
  constexpr int TM = BM / WM / 8, TN = BN / WN / 8;
  extern __shared__ __align__(16) unsigned char km_smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp / WN, wn = warp % WN;
  const int g = lane >> 2, q = lane & 3;
  const long long row0 = (long long)blockIdx.x * BM;
  const int KT = (a.d + kBK - 1) / kBK;
  const int chunks = (int)((a.m + BN - 1) / BN);
  const long long total = (long long)chunks * KT;

  auto stage_A = [&](int s, int u) { return reinterpret_cast<T*>(km_smem + (size_t)s * Stage::kBytes) + u * BM * 16; };
  auto stage_C = [&](int s, int u) {
    return reinterpret_cast<double*>(km_smem + (size_t)s * Stage::kBytes + Stage::kXBytes) + u * BN * kCS;
  };
  auto load_stage = [&](long long it) {
    const int s = (int)(it % kStages);
    const int jc = (int)(it / KT), kt = (int)(it - (long long)jc * KT);
    const int k0 = kt * kBK;
    // X: BM rows x 8 chunks of 4 features
    for (int c = tid; c < BM * 8; c += kThreads) {
      const int r = c >> 3, ch = c & 7;
      const long long row = min(row0 + r, a.n - 1);
      const int col = k0 + ch * 4;
      const bool ok = col < a.d;
      cp_async_quad(stage_A(s, ch >> 2) + r * 16 + (ch & 3) * 4, X + (size_t)row * a.d + (ok ? col : 0), ok);
    }
    // C: BN rows x 16 chunks of 2 doubles
    for (int c = tid; c < BN * 16; c += kThreads) {
      const int r = c >> 4, ch = c & 15;
      const long long cr = min((long long)jc * BN + r, a.m - 1);
      const int col = k0 + ch * 2;
      const bool ok = col < a.d;
      cp_async16(stage_C(s, ch >> 3) + r * kCS + (ch & 7) * 2, a.C + (size_t)cr * a.d + (ok ? col : 0), ok);
    }
  };

  double acc[TM][TN][2];
  double bestv[TM];
  int bestj[TM];
#pragma unroll
  for (int mi = 0; mi < TM; ++mi) {
    bestv[mi] = INFINITY;
    bestj[mi] = 0x7fffffff;
#pragma unroll
    for (int ni = 0; ni < TN; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
  }

  for (int s = 0; s < kStages - 1; ++s) {
    if (s < total) load_stage(s);
    cp_async_commit();
  }
  for (long long it = 0; it < total; ++it) {
    cp_async_wait<kStages - 2>();
    __syncthreads();
    if (it + kStages - 1 < total) load_stage(it + kStages - 1);
    cp_async_commit();
    const int s = (int)(it % kStages);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const T* As = stage_A(s, u);
      const double* Cs = stage_C(s, u);
      float4 xa[TM];
      double cb[TN][4];
#pragma unroll
      for (int mi = 0; mi < TM; ++mi) xa[mi] = load_quad(As + (wm * TM * 8 + mi * 8 + g) * 16 + 4 * q, 0);
#pragma unroll
      for (int ni = 0; ni < TN; ++ni) {
        const double2* p = reinterpret_cast<const double2*>(Cs + (wn * TN * 8 + ni * 8 + g) * kCS + 4 * q);
        const double2 v0 = p[0], v1 = p[1];
        cb[ni][0] = v0.x; cb[ni][1] = v0.y; cb[ni][2] = v1.x; cb[ni][3] = v1.y;
      }
#pragma unroll
      for (int mi = 0; mi < TM; ++mi) {
        const double x0 = (double)xa[mi].x, x1 = (double)xa[mi].y, x2 = (double)xa[mi].z, x3 = (double)xa[mi].w;
#pragma unroll
        for (int ni = 0; ni < TN; ++ni) {
          dmma(acc[mi][ni], x0, cb[ni][0]);
          dmma(acc[mi][ni], x1, cb[ni][1]);
          dmma(acc[mi][ni], x2, cb[ni][2]);
          dmma(acc[mi][ni], x3, cb[ni][3]);
        }
      }
    }
    const int jc = (int)(it / KT), kt = (int)(it - (long long)jc * KT);
    if (kt == KT - 1) {      // the chunk's dot products are complete: accumulator (row g, cols 2q, 2q+1) per 8x8 tile
#pragma unroll
      for (int mi = 0; mi < TM; ++mi) {
        const long long row = row0 + wm * TM * 8 + mi * 8 + g;
#pragma unroll
        for (int ni = 0; ni < TN; ++ni)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const long long j = (long long)jc * BN + wn * TN * 8 + ni * 8 + 2 * q + e;
            if (MODE == 0) {
              if (j < a.m) {
                const double v = __dadd_rn(__dmul_rn(-2.0, acc[mi][ni][e]), a.cn[j]);
                if (v < bestv[mi] || (v == bestv[mi] && (int)j < bestj[mi])) {
                  bestv[mi] = v;
                  bestj[mi] = (int)j;
                }
              }
            } else {
              if (row < a.n) {
                double v = 0.0;
                if (j < a.m) {
                  v = __dadd_rn(__dadd_rn(__dmul_rn(-2.0, acc[mi][ni][e]), a.cn[j]), a.xx[row]);
                  v = v > 0.0 ? v : 0.0;          // np.maximum(distances, 0)
                }
                a.out[(size_t)row * BN + (j - (long long)jc * BN)] = v;
              }
            }
            acc[mi][ni][e] = 0.0;
          }
      }
    }
  }
  cp_async_wait<0>();
  if (MODE == 0) {
    // first minimum over all centres: quad lanes, then the WN warps of a row
    __shared__ double s_v[WN][BM];
    __shared__ int s_j[WN][BM];
#pragma unroll
    for (int mi = 0; mi < TM; ++mi) {
#pragma unroll
      for (int o = 1; o <= 2; o <<= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, bestv[mi], o);
        const int j2 = __shfl_xor_sync(0xffffffffu, bestj[mi], o);
        if (v2 < bestv[mi] || (v2 == bestv[mi] && j2 < bestj[mi])) {
          bestv[mi] = v2;
          bestj[mi] = j2;
        }
      }
      if (q == 0) {
        s_v[wn][wm * TM * 8 + mi * 8 + g] = bestv[mi];
        s_j[wn][wm * TM * 8 + mi * 8 + g] = bestj[mi];
      }
    }
    __syncthreads();
    int nchanged = 0;
    for (int r = tid; r < BM; r += kThreads) {
      const long long row = row0 + r;
      if (row >= a.n) continue;
      double v = s_v[0][r];
      int j = s_j[0][r];
#pragma unroll
      for (int w2 = 1; w2 < WN; ++w2)
        if (s_v[w2][r] < v || (s_v[w2][r] == v && s_j[w2][r] < j)) {
          v = s_v[w2][r];
          j = s_j[w2][r];
        }
      if (j == 0x7fffffff) j = 0;                  // every value NaN / +inf: sklearn keeps label 0
      a.labels[row] = j;
      if (a.labels_old && a.labels_old[row] != j) ++nchanged;
    }
    if (a.changed) {
      nchanged = warp_sum(nchanged);
      if (lane == 0 && nchanged) atomicAdd(a.changed, nchanged);
    }
  }
}

// ------------------------------------------------------------------------------------ small kernels
// seeds: Cc[t] = X[ids[t]] - X_mean (sklearn's centres live in the centred frame), Cr[t] = Cc[t] + X_mean
template <typename T>
__global__ void __launch_bounds__(256) km_gather_kernel(const T* __restrict__ X, int d, const int* __restrict__ ids,
                                                        const double* __restrict__ mean, double* __restrict__ Cc, double* __restrict__ Cr) {
  const int t = blockIdx.x;
  const long long r = ids[t];
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const double v = __dsub_rn((double)to_f32(X[(size_t)r * d + c]), mean[c]);
    Cc[(size_t)t * d + c] = v;
    Cr[(size_t)t * d + c] = __dadd_rn(v, mean[c]);
  }
}

// |c_j|^2 of fp64 centres: one warp per centre
__global__ void __launch_bounds__(256) km_cnorm_kernel(const double* __restrict__ C, long long k, int d, double* __restrict__ cn) {
  const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= k) return;
  double s = 0.0;
  for (int c = lane; c < d; c += 32) {
    const double v = C[(size_t)j * d + c];
    s = fma(v, v, s);
  }
  s = warp_sum(s);
  if (lane == 0) cn[j] = s;
}

// k-means++ state on the device
struct PpState {
  double current_pot;
  int best;           // winning candidate slot of the last step
  int cand[16];
  double pot[16];
};

constexpr int kPotBlocks = 512;

// partial potentials: part[b][t] = sum over the block's rows of w_i * min(closest_i, D[i][t]), fixed order.
// BN = row stride of D = candidates computed per row (8 or 16)
template <int BN>
__global__ void __launch_bounds__(256) km_pot_partial_kernel(const double* __restrict__ D, const double* __restrict__ closest,
                                                             const double* __restrict__ w, long long n, double* __restrict__ part) {
  pdl_enter();
  __shared__ double s_p[8][BN];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double p[BN];
#pragma unroll
  for (int t = 0; t < BN; ++t) p[t] = 0.0;
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long lo = (long long)blockIdx.x * per, hi = min(n, lo + per);
  for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const double c = closest[i], wi = w ? w[i] : 1.0;
    const double2* dr = reinterpret_cast<const double2*>(D + (size_t)i * BN);
#pragma unroll
    for (int t2 = 0; t2 < BN / 2; ++t2) {
      const double2 v = dr[t2];
      p[2 * t2] = __dadd_rn(p[2 * t2], __dmul_rn(wi, fmin(c, v.x)));
      p[2 * t2 + 1] = __dadd_rn(p[2 * t2 + 1], __dmul_rn(wi, fmin(c, v.y)));
    }
  }
#pragma unroll
  for (int t = 0; t < BN; ++t) {
    p[t] = warp_sum(p[t]);
    if (lane == 0) s_p[warp][t] = p[t];
  }
  __syncthreads();
  if (threadIdx.x < BN) {
    double s = 0.0;
    for (int w2 = 0; w2 < 8; ++w2) s = __dadd_rn(s, s_p[w2][threadIdx.x]);
    part[(size_t)blockIdx.x * 16 + threadIdx.x] = s;
  }
}

// potentials of the candidates (warp t sums the partials of candidate t in a fixed order), best = first minimum
__global__ void __launch_bounds__(512) km_pot_final_kernel(const double* __restrict__ part, int blocks, int trials, PpState* st,
                                                           int* __restrict__ center_ids, int step) {
  pdl_enter();
  __shared__ double s_pot[16];
  const int t = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double s = 0.0;
  if (t < trials)
    for (int b = lane; b < blocks; b += 32) s = __dadd_rn(s, part[(size_t)b * 16 + t]);
  s = warp_sum(s);
  if (lane == 0) s_pot[t] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double bv = s_pot[0];
    int bt = 0;
    for (int u = 1; u < trials; ++u)
      if (s_pot[u] < bv) {            // np.argmin: first minimum
        bv = s_pot[u];
        bt = u;
      }
    for (int u = 0; u < 16; ++u) st->pot[u] = u < trials ? s_pot[u] : 0.0;
    st->best = bt;
    st->current_pot = bv;
    center_ids[step] = st->cand[bt];
  }
}

// inclusive prefix sum in a fixed order (the same bits on every run): tiles of 1024 values
constexpr int kScanTile = 1024;
// closest_i = min(closest_i, D[i][best]) and the tile sums of wc_i = w_i * closest_i (the vector whose cumulative sum
// the next step searches)
template <int BN>
__global__ void __launch_bounds__(256) km_commit_tiles_kernel(const double* __restrict__ D, const PpState* __restrict__ st,
                                                              const double* __restrict__ w, long long n, double* __restrict__ closest,
                                                              double* __restrict__ wc, double* __restrict__ tile_sum) {
  pdl_enter();
  using BS = cub::BlockScan<double, 256>;
  __shared__ typename BS::TempStorage tmp;
  const int best = st->best;
  const long long base = (long long)blockIdx.x * kScanTile + threadIdx.x * 4;
  double s = 0.0;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const long long i = base + e;
    if (i < n) {
      const double c = fmin(closest[i], D[(size_t)i * BN + best]);
      closest[i] = c;
      const double v = w ? __dmul_rn(w[i], c) : c;
      wc[i] = v;
      s = __dadd_rn(s, v);
    }
  }
  double incl, total;
  BS(tmp).InclusiveSum(s, incl, total);
  if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}
// exclusive scan of the tile sums: one block, chunks of 1024 tiles with a running carry
__global__ void __launch_bounds__(256) km_scan_offsets_kernel(double* __restrict__ tile_sum, int tiles) {
  pdl_enter();
  using BS = cub::BlockScan<double, 256>;
  __shared__ typename BS::TempStorage tmp;
  __shared__ double s_carry;
  if (threadIdx.x == 0) s_carry = 0.0;
  __syncthreads();
  for (int c0 = 0; c0 < tiles; c0 += 1024) {
    const int base = c0 + threadIdx.x * 4;
    double x[4], s = 0.0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      x[e] = base + e < tiles ? tile_sum[base + e] : 0.0;
      s = __dadd_rn(s, x[e]);
    }
    double excl, total;
    BS(tmp).ExclusiveSum(s, excl, total);
    double run = __dadd_rn(s_carry, excl);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (base + e < tiles) tile_sum[base + e] = run;
      run = __dadd_rn(run, x[e]);
    }
    __syncthreads();
    if (threadIdx.x == 0) s_carry = __dadd_rn(s_carry, total);
    __syncthreads();
  }
}
__global__ void __launch_bounds__(256) km_scan_apply_kernel(const double* __restrict__ v, long long n, const double* __restrict__ tile_off,
                                                            double* __restrict__ cum) {
  pdl_enter();
  using BS = cub::BlockScan<double, 256>;
  __shared__ typename BS::TempStorage tmp;
  const long long base = (long long)blockIdx.x * kScanTile + threadIdx.x * 4;
  double x[4], s = 0.0;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    x[e] = base + e < n ? v[base + e] : 0.0;
    s = __dadd_rn(s, x[e]);
  }
  double excl;
  BS(tmp).ExclusiveSum(s, excl);
  double run = __dadd_rn(tile_off[blockIdx.x], excl);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    run = __dadd_rn(run, x[e]);
    if (base + e < n) cum[base + e] = run;
  }
}
__global__ void km_pp_seed_kernel(PpState* st, int first) {
  st->current_pot = 0.0;
  st->best = 0;
  for (int t = 0; t < 16; ++t) {
    st->cand[t] = first;
    st->pot[t] = 0.0;
  }
}
// candidate t of the step: clip(searchsorted(cum, rand_t * current_pot), n - 1) (side='left': first cum >= value;
// rand_vals == NULL: the seed row already in the state), then its row as fp64 into the candidate tile + its norm
template <typename T>
__global__ void __launch_bounds__(256) km_candidates_kernel(const T* __restrict__ X, int d, long long n, const double* __restrict__ cum,
                                                            const double* __restrict__ rand_vals, PpState* st, int trials,
                                                            const double* __restrict__ xx, double* __restrict__ C, double* __restrict__ cc) {
  pdl_enter();
  __shared__ int s_row;
  const int t = blockIdx.x;
  const bool live = t < trials;
  if (threadIdx.x == 0) {
    int id = st->cand[0];
    if (live && rand_vals) {
      const double v = __dmul_rn(rand_vals[t], st->current_pot);
      long long lo = 0, hi = n;
      while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (cum[mid] < v) lo = mid + 1;
        else hi = mid;
      }
      id = (int)min(lo, n - 1);
    }
    s_row = id;
  }
  __syncthreads();
  const long long r = s_row;
  for (int c = threadIdx.x; c < d; c += blockDim.x) C[(size_t)t * d + c] = live ? (double)to_f32(X[(size_t)r * d + c]) : 0.0;
  if (threadIdx.x == 0) {
    cc[t] = live ? xx[r] : 0.0;
    if (rand_vals && live) st->cand[t] = (int)r;      // (dead blocks may see either cand[0]: they never use the row)
  }
}

// ---- M step
__global__ void __launch_bounds__(256) km_iota_kernel(const int* __restrict__ labels, long long n, int* __restrict__ keys, int* __restrict__ vals) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = labels[i];
  vals[i] = (int)i;
}
// starts[j] = first position of label >= j in the sorted keys (j = 0..k)
__global__ void __launch_bounds__(256) km_starts_kernel(const int* __restrict__ keys, long long n, long long k, int* __restrict__ starts) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j > k) return;
  long long lo = 0, hi = n;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (keys[mid] < j) lo = mid + 1;
    else hi = mid;
  }
  starts[j] = (int)lo;
}
// centre sums in ascending row order: sums[j][c] = sum_i (x_i[c] - X_mean[c]) * w_i, wsum[j] = sum_i w_i; one CTA per cluster
template <typename T>
__global__ void __launch_bounds__(256) km_sums_kernel(const T* __restrict__ X, int d, const double* __restrict__ w, const double* __restrict__ mean,
                                                      const int* __restrict__ order, const int* __restrict__ starts, long long k,
                                                      double* __restrict__ sums, double* __restrict__ wsum, int* __restrict__ n_empty) {
  const long long j = blockIdx.x;
  const int lo = starts[j], hi = starts[j + 1];
  for (int c0 = threadIdx.x * 4; c0 < d; c0 += blockDim.x * 4) {
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const double m0 = mean[c0], m1 = mean[c0 + 1], m2 = mean[c0 + 2], m3 = mean[c0 + 3];
    for (int p = lo; p < hi; ++p) {
      const int i = order[p];
      const double wi = w ? w[i] : 1.0;
      const float4 v = ldg_quad(X + (size_t)i * d + c0, 0);
      s0 = __dadd_rn(s0, __dmul_rn(__dsub_rn((double)v.x, m0), wi));
      s1 = __dadd_rn(s1, __dmul_rn(__dsub_rn((double)v.y, m1), wi));
      s2 = __dadd_rn(s2, __dmul_rn(__dsub_rn((double)v.z, m2), wi));
      s3 = __dadd_rn(s3, __dmul_rn(__dsub_rn((double)v.w, m3), wi));
    }
    double* o = sums + (size_t)j * d + c0;
    o[0] = s0; o[1] = s1; o[2] = s2; o[3] = s3;
  }
  if (threadIdx.x == 0) {
    double ws = 0.0;
    for (int p = lo; p < hi; ++p) ws = __dadd_rn(ws, w ? w[order[p]] : 1.0);
    wsum[j] = ws;
    if (ws == 0.0) atomicAdd(n_empty, 1);
  }
}
// _relocate_empty_clusters_dense: sequential over the empty clusters (a row's old cluster may repeat)
template <typename T>
__global__ void __launch_bounds__(256) km_relocate_kernel(const T* __restrict__ X, int d, const double* __restrict__ w,
                                                          const double* __restrict__ mean, const int* __restrict__ labels, const int* __restrict__ empty_ids,
                                                          const int* __restrict__ far_ids, int n_empty, double* __restrict__ sums,
                                                          double* __restrict__ wsum) {
  for (int e = 0; e < n_empty; ++e) {
    const int nw = empty_ids[e], far = far_ids[e], old = labels[far];
    const double wi = w ? w[far] : 1.0;
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      const double xv = __dmul_rn(__dsub_rn((double)to_f32(X[(size_t)far * d + c]), mean[c]), wi);
      sums[(size_t)old * d + c] = __dsub_rn(sums[(size_t)old * d + c], xv);
      sums[(size_t)nw * d + c] = xv;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      wsum[nw] = wi;
      wsum[old] = __dsub_rn(wsum[old], wi);
    }
    __syncthreads();
  }
}
// _average_centers + _center_shift in the centred frame, and the raw-frame copy (centre + X_mean) the E step and the
// final distances use (KMeans.fit: best_centers += X_mean); one CTA per cluster
__global__ void __launch_bounds__(256) km_average_kernel(const double* __restrict__ sums, const double* __restrict__ wsum, int d,
                                                         long long argmax_w, const double* __restrict__ mean,
                                                         const double* __restrict__ Cc_old, double* __restrict__ Cc_new,
                                                         double* __restrict__ Cr_new, double* __restrict__ shift) {
  __shared__ double s_red[8];
  const long long j = blockIdx.x;
  const double wj = wsum[j];
  long long src = j;
  double alpha = 1.0;
  bool scale = false;
  if (wj > 0.0) {
    alpha = __ddiv_rn(1.0, wj);
    scale = true;
  } else if (argmax_w >= 0) {        // empty cluster: the biggest cluster's row as it stands when row j is reached
    src = argmax_w;
    if (argmax_w < j) {
      alpha = __ddiv_rn(1.0, wsum[argmax_w]);
      scale = true;
    }
  }
  double s = 0.0;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const double raw = sums[(size_t)src * d + c];
    const double v = scale ? __dmul_rn(raw, alpha) : raw;
    Cc_new[(size_t)j * d + c] = v;
    Cr_new[(size_t)j * d + c] = __dadd_rn(v, mean[c]);
    const double df = __dsub_rn(v, Cc_old[(size_t)j * d + c]);
    s = fma(df, df, s);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w2 = 0; w2 < 8; ++w2) t = __dadd_rn(t, s_red[w2]);
    shift[j] = sqrt(t);             // _euclidean_dense_dense(..., squared=False)
  }
}
// dis_i = ((x_i - C[label_i]) ** 2).sum() in numpy's pairwise order (numpy/_core/src/umath/loops_utils.h.src,
// DOUBLE_pairwise_sum: < 8 sequential; <= 128: eight strided accumulators, fixed combine tree, sequential tail;
// else split at n/2 rounded down to a multiple of 8).  One thread per row.
template <typename T>
__device__ __forceinline__ double km_sq(const T* __restrict__ x, const double* __restrict__ c, int i) {
  const double t = __dsub_rn((double)to_f32(x[i]), c[i]);
  return __dmul_rn(t, t);
}
template <typename T>
__device__ __forceinline__ double km_pairwise_leaf(const T* __restrict__ x, const double* __restrict__ c, int n) {   // n <= 128
  if (n < 8) {
    double res = 0.0;
    for (int i = 0; i < n; ++i) res = __dadd_rn(res, km_sq(x, c, i));
    return res;
  }
  double r[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = km_sq(x, c, k);
  int i = 8;
  for (; i < n - (n % 8); i += 8)
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], km_sq(x, c, i + k));
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __dadd_rn(res, km_sq(x, c, i));
  return res;
}
// the recursion "pairwise(a, n2) + pairwise(a + n2, n - n2)" unrolled onto an explicit stack (depth <= log2(n / 128) + 1)
template <typename T>
__device__ double km_pairwise(const T* __restrict__ x, const double* __restrict__ c, int n) {
  constexpr int kDepth = 24;
  int off[kDepth], len[kDepth];
  double acc[kDepth];
  unsigned char stage[kDepth];      // 0: nothing done, 1: left child running, 2: right child running
  int sp = 0;
  off[0] = 0; len[0] = n; stage[0] = 0;
  while (true) {
    if (len[sp] > 128) {            // descend into the left child
      int n2 = len[sp] / 2;
      n2 -= n2 % 8;
      stage[sp] = 1;
      off[sp + 1] = off[sp]; len[sp + 1] = n2; stage[sp + 1] = 0;
      ++sp;
      continue;
    }
    double val = km_pairwise_leaf(x + off[sp], c + off[sp], len[sp]);
    --sp;
    while (sp >= 0 && stage[sp] == 2) {       // a right child returned: the parent is complete
      val = __dadd_rn(acc[sp], val);
      --sp;
    }
    if (sp < 0) return val;
    // a left child returned: keep its sum, run the right child
    acc[sp] = val;
    stage[sp] = 2;
    int n2 = len[sp] / 2;
    n2 -= n2 % 8;
    off[sp + 1] = off[sp] + n2; len[sp + 1] = len[sp] - n2; stage[sp + 1] = 0;
    ++sp;
  }
}
template <typename T>
__global__ void __launch_bounds__(128) km_rowdist_kernel(const T* __restrict__ X, long long n, int d, const double* __restrict__ C,
                                                         const int* __restrict__ labels, double* __restrict__ dis) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  dis[i] = km_pairwise(X + (size_t)i * d, C + (size_t)labels[i] * d, d);
}
// per cluster the member with the smallest dis (first minimum = lowest row index): one warp per cluster
__global__ void __launch_bounds__(256) km_pick_kernel(const double* __restrict__ dis, const int* __restrict__ order,
                                                      const int* __restrict__ starts, long long k, int* __restrict__ picks) {
  const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= k) return;
  const int lo = starts[j], hi = starts[j + 1];
  double bv = INFINITY;
  int bi = 0x7fffffff;
  for (int p = lo + lane; p < hi; p += 32) {
    const int i = order[p];
    const double v = dis[i];
    if (bi == 0x7fffffff || v < bv || (v == bv && i < bi)) {
      bv = v;
      bi = i;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const double v2 = __shfl_xor_sync(0xffffffffu, bv, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
    if (i2 != 0x7fffffff && (bi == 0x7fffffff || v2 < bv || (v2 == bv && i2 < bi))) {
      bv = v2;
      bi = i2;
    }
  }
  if (lane == 0) picks[j] = (bi == 0x7fffffff) ? -1 : bi;
}

// ---- X.mean(axis=0) exactly like numpy (out[c] += X[i][c] row after row, then / n): one thread per column,
// eight rows of loads in flight
template <typename T>
__global__ void __launch_bounds__(128) km_colmean_kernel(const T* __restrict__ X, long long n, int d, double* __restrict__ mean) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= d) return;
  double s = 0.0;
  long long i = 0;
  for (; i + 8 <= n; i += 8) {
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = ldg_f32(X + (size_t)(i + e) * d + c);
#pragma unroll
    for (int e = 0; e < 8; ++e) s = __dadd_rn(s, (double)v[e]);
  }
  for (; i < n; ++i) s = __dadd_rn(s, (double)ldg_f32(X + (size_t)i * d + c));
  mean[c] = __ddiv_rn(s, (double)n);
}
// ---- np.var(X, axis=0) (only feeds the convergence tolerance): fixed-order blocked sums of squared deviations
constexpr int kVarRowBlocks = 256;
template <typename T>
__global__ void __launch_bounds__(256) km_colvar_kernel(const T* __restrict__ X, long long n, int d, const double* __restrict__ mean,
                                                        double* __restrict__ part) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  const long long per = (n + gridDim.y - 1) / gridDim.y;
  const long long lo = (long long)blockIdx.y * per, hi = min(n, lo + per);
  if (c >= d) return;
  const double mu = mean[c];
  double s = 0.0;
  for (long long i = lo; i < hi; ++i) {
    const double df = __dsub_rn((double)to_f32(X[(size_t)i * d + c]), mu);
    s = fma(df, df, s);
  }
  part[(size_t)blockIdx.y * d + c] = s;
}
__global__ void __launch_bounds__(256) km_colfinal_kernel(const double* __restrict__ part, int blocks, int d, long long n,
                                                          double* __restrict__ out) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= d) return;
  double s = 0.0;
  for (int b = 0; b < blocks; ++b) s = __dadd_rn(s, part[(size_t)b * d + c]);
  out[c] = __ddiv_rn(s, (double)n);
}
__global__ void __launch_bounds__(256) km_mean_kernel(const double* __restrict__ v, int d, double* __restrict__ out) {
  __shared__ double s_red[8];
  double s = 0.0;
  for (int c = threadIdx.x; c < d; c += blockDim.x) s = __dadd_rn(s, v[c]);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w2 = 0; w2 < 8; ++w2) t = __dadd_rn(t, s_red[w2]);
    out[0] = __ddiv_rn(t, (double)d);
  }
}

template <typename T, int BM, int BN, int WM, int WN, int MODE>
static int launch_gemm(const GemmArgs& a, cudaStream_t stream, bool pdl = false) {
  const size_t smem = kStages * GemmStage<T, BM, BN>::kBytes;
  static bool configured = false;
  if (!configured) {
    VQ_CUDA(cudaFuncSetAttribute((km_gemm_kernel<T, BM, BN, WM, WN, MODE>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const unsigned grid = (unsigned)((a.n + BM - 1) / BM);
  VQ_CUDA(launch_pdl(km_gemm_kernel<T, BM, BN, WM, WN, MODE>, dim3(grid), dim3(WM * WN * 32), smem, stream, pdl, a));
  g_launches.fetch_add(1);
  return 0;
}

static size_t sort_bytes(long long n) {
  size_t cb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cb, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, (int)n);
  return cb;
}

}  // namespace km
}  // namespace vatlq

using namespace vatlq;
using namespace vatlq::km;

static bool km_shape_ok(int64_t n, int d) { return n > 0 && n < (1LL << 31) && d > 0 && d % 4 == 0; }

static size_t pp_ws_bytes(int64_t n, int d) {
  const size_t tiles = (size_t)((n + kScanTile - 1) / kScanTile);
  return align_up((size_t)16 * d * 8, 256) + align_up(16 * 8, 256) + align_up((size_t)n * 16 * 8, 256) +
         3 * align_up((size_t)n * 8, 256) + align_up((size_t)kPotBlocks * 16 * 8, 256) + align_up(sizeof(PpState), 256) +
         align_up(tiles * 8, 256);
}
static size_t update_ws_bytes(int64_t n) { return align_up(sort_bytes(n), 256) + 3 * align_up((size_t)n * 4, 256); }
static size_t var_ws_bytes(int d) { return (size_t)(kVarRowBlocks + 1) * d * 8; }

// X of a *_dt entry, checked in the entry itself (the message names it): a known dtype code, and a 16-bit X 8-byte
// aligned (its quad loads are 8 bytes wide).  An fp32 X keeps the checks its entry has always made.
#define KM_REQUIRE_DTYPE(X, dtype)                                                              \
  do {                                                                                          \
    VQ_REQUIRE(dtype_size(dtype) != 0, "dtype must be VATLQ_F32, VATLQ_F16 or VATLQ_BF16");     \
    VQ_REQUIRE((dtype) == VATLQ_F32 || quad_aligned(X, dtype), "a 16-bit X must be 8-byte aligned"); \
  } while (0)

// the element type of a with_dtype tag
template <typename P>
using km_elem_t = std::remove_const_t<std::remove_pointer_t<P>>;

/* one scratch size that serves every vatlq_kmeans_* call (they never run concurrently on one workspace) */
extern "C" size_t vatlq_kmeans_workspace_bytes(int64_t n, int d, int64_t k) {
  if (n <= 0 || d <= 0 || k <= 0) return 0;
  return std::max(std::max(pp_ws_bytes(n, d), update_ws_bytes(n)), std::max(var_ws_bytes(d), align_up((size_t)k * 8, 256)));
}

/* mean[d] = X.mean(axis=0) (numpy's order), out1[0] = np.mean(np.var(X, axis=0)) */
extern "C" int vatlq_kmeans_mean_var_dt(const void* X, int dtype, int64_t n, int d, double* mean, double* out1, void* ws,
                                        size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  KM_REQUIRE_DTYPE(X, dtype);
  VQ_REQUIRE(km_shape_ok(n, d) && X && mean && out1 && ws, "bad arguments");
  VQ_REQUIRE(ws_bytes >= var_ws_bytes(d), "workspace too small (vatlq_kmeans_workspace_bytes)");
  double* part = (double*)ws;
  double* var = part + (size_t)kVarRowBlocks * d;
  const int rb = (int)std::min<long long>(kVarRowBlocks, n);
  const int rc = with_dtype(dtype, [&](auto tag) {
    using T = km_elem_t<decltype(tag)>;
    km_colmean_kernel<T><<<(d + 127) / 128, 128, 0, stream>>>((const T*)X, n, d, mean);
    VQ_LAUNCHED();
    km_colvar_kernel<T><<<dim3((d + 255) / 256, rb), 256, 0, stream>>>((const T*)X, n, d, mean, part);
    VQ_LAUNCHED();
    return 0;
  });
  if (rc) return rc;
  km_colfinal_kernel<<<(d + 255) / 256, 256, 0, stream>>>(part, rb, d, n, var);
  VQ_LAUNCHED();
  km_mean_kernel<<<1, 256, 0, stream>>>(var, d, out1);
  VQ_LAUNCHED();
  return 0;
}
extern "C" int vatlq_kmeans_mean_var(const float* X, int64_t n, int d, double* mean, double* out1, void* ws, size_t ws_bytes,
                                     vatlq_stream_t stream) {
  return vatlq_kmeans_mean_var_dt(X, VATLQ_F32, n, d, mean, out1, ws, ws_bytes, stream);
}

// the k-means++ chain of element type T (arguments checked by the entry)
template <typename T>
static int kmeans_pp(const T* X, int64_t n, int d, const double* w, int64_t k, int64_t first_center, const double* rand_vals,
                     int trials, int32_t* center_ids, double* closest, void* ws, cudaStream_t stream) {
  char* p = (char*)ws;
  auto take = [&](size_t bytes) {
    char* r = p;
    p += align_up(bytes, 256);
    return r;
  };
  const int tiles = (int)((n + kScanTile - 1) / kScanTile);
  double* Cbuf = (double*)take((size_t)16 * d * 8);     // the step's candidate rows as fp64
  double* cc = (double*)take(16 * 8);                   // their squared norms
  double* D = (double*)take((size_t)n * 16 * 8);        // squared distances of every row to the candidates
  double* wc = (double*)take((size_t)n * 8);            // w * closest
  double* cum = (double*)take((size_t)n * 8);           // its cumulative sum
  double* xx = (double*)take((size_t)n * 8);            // |x_i|^2
  double* part = (double*)take((size_t)kPotBlocks * 16 * 8);
  PpState* st = (PpState*)take(sizeof(PpState));
  double* tile_off = (double*)take((size_t)tiles * 8);
  int rc = vq_launch_norms(X, n, d, xx, stream);
  if (rc) return rc;
  rc = fill_f64(closest, n, INFINITY, stream);
  if (rc) return rc;
  const int pot_blocks = (int)std::min<long long>(kPotBlocks, (n + 255) / 256);
  // candidates per step: 8 columns of fp64 tensor-core work when n_local_trials <= 8 (k < 403), else 16
  const bool narrow = trials <= 8;
  const int bn = narrow ? 8 : 16;
  GemmArgs g{};
  g.X = X; g.n = n; g.d = d; g.C = Cbuf; g.m = bn; g.cn = cc; g.xx = xx; g.out = D;
  km_pp_seed_kernel<<<1, 1, 0, stream>>>(st, (int)first_center);
  VQ_LAUNCHED();
  for (int64_t c = 0; c < k; ++c) {
    const int tr = c == 0 ? 1 : trials;       // step 0: the first centre alone (closest = its distances)
    // (with rand_vals == NULL the state's seed row is used and no block writes the state).  Every kernel of the chain
    // is a programmatic dependent of the one before it (pdl_enter() at kernel entry keeps the data flow in stream order)
    VQ_CUDA(launch_pdl(km_candidates_kernel<T>, dim3(bn), dim3(256), 0, stream, c > 0, X, d, (long long)n, (const double*)cum,
                       c == 0 ? (const double*)nullptr : rand_vals + (size_t)(c - 1) * trials, st, tr, (const double*)xx, Cbuf, cc));
    rc = narrow ? launch_gemm<T, 128, 8, 4, 1, 1>(g, stream, true) : launch_gemm<T, 128, 16, 4, 1, 1>(g, stream, true);
    if (rc) return rc;
    if (narrow)
      VQ_CUDA(launch_pdl(km_pot_partial_kernel<8>, dim3(pot_blocks), dim3(256), 0, stream, true, (const double*)D, (const double*)closest, w,
                         (long long)n, part));
    else
      VQ_CUDA(launch_pdl(km_pot_partial_kernel<16>, dim3(pot_blocks), dim3(256), 0, stream, true, (const double*)D, (const double*)closest, w,
                         (long long)n, part));
    VQ_CUDA(launch_pdl(km_pot_final_kernel, dim3(1), dim3(512), 0, stream, true, (const double*)part, pot_blocks, tr, st, center_ids, (int)c));
    if (narrow)
      VQ_CUDA(launch_pdl(km_commit_tiles_kernel<8>, dim3(tiles), dim3(256), 0, stream, true, (const double*)D, (const PpState*)st, w, (long long)n,
                         closest, wc, tile_off));
    else
      VQ_CUDA(launch_pdl(km_commit_tiles_kernel<16>, dim3(tiles), dim3(256), 0, stream, true, (const double*)D, (const PpState*)st, w, (long long)n,
                         closest, wc, tile_off));
    g_launches.fetch_add(4);
    if (c + 1 < k) {
      VQ_CUDA(launch_pdl(km_scan_offsets_kernel, dim3(1), dim3(256), 0, stream, true, tile_off, tiles));
      VQ_CUDA(launch_pdl(km_scan_apply_kernel, dim3(tiles), dim3(256), 0, stream, true, (const double*)wc, (long long)n, (const double*)tile_off, cum));
      g_launches.fetch_add(2);
    }
  }
  return 0;
}

extern "C" int vatlq_kmeans_pp_dt(const void* X, int dtype, int64_t n, int d, const double* w, int64_t k, int64_t first_center,
                                  const double* rand_vals, int trials, int32_t* center_ids, double* closest, void* ws,
                                  size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  KM_REQUIRE_DTYPE(X, dtype);
  VQ_REQUIRE(km_shape_ok(n, d) && k >= 1 && k <= n, "bad shape (1 <= k <= n < 2^31, d % 4 == 0)");
  VQ_REQUIRE(trials >= 1 && trials <= 16, "1 <= n_local_trials <= 16 (2 + int(log k) stays below 16 for k < 1.2e6)");
  VQ_REQUIRE(first_center >= 0 && first_center < n, "first centre out of range");
  VQ_REQUIRE(X && center_ids && closest && ws && (k == 1 || rand_vals), "null pointer");
  VQ_REQUIRE(dtype != VATLQ_F32 || (reinterpret_cast<uintptr_t>(X) & 15) == 0, "X must be 16-byte aligned");
  VQ_REQUIRE(ws_bytes >= pp_ws_bytes(n, d), "workspace too small (vatlq_kmeans_workspace_bytes)");
  return with_dtype(dtype, [&](auto tag) {
    using T = km_elem_t<decltype(tag)>;
    return kmeans_pp((const T*)X, n, d, w, k, first_center, rand_vals, trials, center_ids, closest, ws, stream);
  });
}
extern "C" int vatlq_kmeans_pp(const float* X, int64_t n, int d, const double* w, int64_t k, int64_t first_center,
                               const double* rand_vals, int trials, int32_t* center_ids, double* closest, void* ws,
                               size_t ws_bytes, vatlq_stream_t stream) {
  return vatlq_kmeans_pp_dt(X, VATLQ_F32, n, d, w, k, first_center, rand_vals, trials, center_ids, closest, ws, ws_bytes, stream);
}

extern "C" int vatlq_kmeans_gather_dt(const void* X, int dtype, int d, const int32_t* ids, int64_t k, const double* mean, double* Cc,
                                      double* Cr, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  KM_REQUIRE_DTYPE(X, dtype);
  VQ_REQUIRE(X && ids && mean && Cc && Cr && k >= 1 && d > 0, "bad arguments");
  return with_dtype(dtype, [&](auto tag) {
    using T = km_elem_t<decltype(tag)>;
    km_gather_kernel<T><<<(unsigned)k, 256, 0, stream>>>((const T*)X, d, ids, mean, Cc, Cr);
    VQ_LAUNCHED();
    return 0;
  });
}
extern "C" int vatlq_kmeans_gather(const float* X, int d, const int32_t* ids, int64_t k, const double* mean, double* Cc, double* Cr,
                                   vatlq_stream_t stream) {
  return vatlq_kmeans_gather_dt(X, VATLQ_F32, d, ids, k, mean, Cc, Cr, stream);
}

extern "C" int vatlq_kmeans_assign_dt(const void* X, int dtype, int64_t n, int d, const double* C, int64_t k, int32_t* labels,
                                      const int32_t* labels_old, int32_t* changed, void* ws, size_t ws_bytes,
                                      vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  KM_REQUIRE_DTYPE(X, dtype);
  VQ_REQUIRE(km_shape_ok(n, d) && k >= 1 && X && C && labels && ws, "bad arguments");
  VQ_REQUIRE((dtype != VATLQ_F32 || (reinterpret_cast<uintptr_t>(X) & 15) == 0) && (reinterpret_cast<uintptr_t>(C) & 15) == 0,
             "X and C must be 16-byte aligned");
  VQ_REQUIRE(ws_bytes >= align_up((size_t)k * 8, 256), "workspace too small (vatlq_kmeans_workspace_bytes)");
  double* cn = (double*)ws;
  km_cnorm_kernel<<<(unsigned)((k * 32 + 255) / 256), 256, 0, stream>>>(C, k, d, cn);
  VQ_LAUNCHED();
  if (changed) VQ_CUDA(cudaMemsetAsync(changed, 0, 4, stream));
  GemmArgs g{};
  g.X = X; g.n = n; g.d = d; g.C = C; g.m = k; g.cn = cn; g.labels = labels; g.labels_old = labels_old; g.changed = changed;
  return with_dtype(dtype, [&](auto tag) { return launch_gemm<km_elem_t<decltype(tag)>, 64, 64, 2, 2, 0>(g, stream); });
}
extern "C" int vatlq_kmeans_assign(const float* X, int64_t n, int d, const double* C, int64_t k, int32_t* labels,
                                   const int32_t* labels_old, int32_t* changed, void* ws, size_t ws_bytes,
                                   vatlq_stream_t stream) {
  return vatlq_kmeans_assign_dt(X, VATLQ_F32, n, d, C, k, labels, labels_old, changed, ws, ws_bytes, stream);
}

extern "C" int vatlq_kmeans_update_dt(const void* X, int dtype, int64_t n, int d, const double* w, const double* mean,
                                      const int32_t* labels, int64_t k, double* sums, double* wsum, int32_t* order, int32_t* starts,
                                      int32_t* n_empty, void* ws, size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  KM_REQUIRE_DTYPE(X, dtype);
  VQ_REQUIRE(km_shape_ok(n, d) && k >= 1 && X && mean && labels && sums && wsum && order && starts && n_empty && ws, "bad arguments");
  const size_t cb = sort_bytes(n);
  VQ_REQUIRE(ws_bytes >= update_ws_bytes(n), "workspace too small (vatlq_kmeans_workspace_bytes)");
  char* p = (char*)ws;
  void* tmp = p;
  p += align_up(cb, 256);
  int* keys_in = (int*)p;
  p += align_up((size_t)n * 4, 256);
  int* keys_out = (int*)p;
  p += align_up((size_t)n * 4, 256);
  int* vals_in = (int*)p;
  km_iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(labels, n, keys_in, vals_in);
  VQ_LAUNCHED();
  int bits = 1;
  while ((1LL << bits) < k && bits < 31) ++bits;
  size_t cb2 = cb;
  VQ_CUDA(cub::DeviceRadixSort::SortPairs(tmp, cb2, keys_in, keys_out, vals_in, order, (int)n, 0, bits, stream));
  g_launches.fetch_add(1);
  km_starts_kernel<<<(unsigned)((k + 1 + 255) / 256), 256, 0, stream>>>(keys_out, n, k, starts);
  VQ_LAUNCHED();
  VQ_CUDA(cudaMemsetAsync(n_empty, 0, 4, stream));
  return with_dtype(dtype, [&](auto tag) {
    using T = km_elem_t<decltype(tag)>;
    km_sums_kernel<T><<<(unsigned)k, 256, 0, stream>>>((const T*)X, d, w, mean, order, starts, k, sums, wsum, n_empty);
    VQ_LAUNCHED();
    return 0;
  });
}
extern "C" int vatlq_kmeans_update(const float* X, int64_t n, int d, const double* w, const double* mean, const int32_t* labels, int64_t k,
                                   double* sums, double* wsum, int32_t* order, int32_t* starts, int32_t* n_empty, void* ws,
                                   size_t ws_bytes, vatlq_stream_t stream) {
  return vatlq_kmeans_update_dt(X, VATLQ_F32, n, d, w, mean, labels, k, sums, wsum, order, starts, n_empty, ws, ws_bytes, stream);
}

extern "C" int vatlq_kmeans_relocate_dt(const void* X, int dtype, int d, const double* w, const double* mean, const int32_t* labels,
                                        const int32_t* empty_ids, const int32_t* far_ids, int n_empty, double* sums, double* wsum,
                                        vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  KM_REQUIRE_DTYPE(X, dtype);
  VQ_REQUIRE(X && mean && labels && empty_ids && far_ids && sums && wsum && n_empty >= 0 && d > 0, "bad arguments");
  if (n_empty == 0) return 0;
  return with_dtype(dtype, [&](auto tag) {
    using T = km_elem_t<decltype(tag)>;
    km_relocate_kernel<T><<<1, 256, 0, stream>>>((const T*)X, d, w, mean, labels, empty_ids, far_ids, n_empty, sums, wsum);
    VQ_LAUNCHED();
    return 0;
  });
}
extern "C" int vatlq_kmeans_relocate(const float* X, int d, const double* w, const double* mean, const int32_t* labels, const int32_t* empty_ids,
                                     const int32_t* far_ids, int n_empty, double* sums, double* wsum, vatlq_stream_t stream) {
  return vatlq_kmeans_relocate_dt(X, VATLQ_F32, d, w, mean, labels, empty_ids, far_ids, n_empty, sums, wsum, stream);
}

extern "C" int vatlq_kmeans_average(const double* sums, const double* wsum, int64_t k, int d, int64_t argmax_weight, const double* mean,
                                    const double* Cc_old, double* Cc_new, double* Cr_new, double* shift, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(sums && wsum && mean && Cc_old && Cc_new && Cr_new && shift && k >= 1 && d > 0 && argmax_weight < k, "bad arguments");
  km_average_kernel<<<(unsigned)k, 256, 0, stream>>>(sums, wsum, d, argmax_weight, mean, Cc_old, Cc_new, Cr_new, shift);
  VQ_LAUNCHED();
  return 0;
}

extern "C" int vatlq_kmeans_rowdist_dt(const void* X, int dtype, int64_t n, int d, const double* C, const int32_t* labels, double* dis,
                                       vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  KM_REQUIRE_DTYPE(X, dtype);
  VQ_REQUIRE(km_shape_ok(n, d) && X && C && labels && dis, "bad arguments");
  return with_dtype(dtype, [&](auto tag) {
    using T = km_elem_t<decltype(tag)>;
    km_rowdist_kernel<T><<<(unsigned)((n + 127) / 128), 128, 0, stream>>>((const T*)X, n, d, C, labels, dis);
    VQ_LAUNCHED();
    return 0;
  });
}
extern "C" int vatlq_kmeans_rowdist(const float* X, int64_t n, int d, const double* C, const int32_t* labels, double* dis,
                                    vatlq_stream_t stream) {
  return vatlq_kmeans_rowdist_dt(X, VATLQ_F32, n, d, C, labels, dis, stream);
}

extern "C" int vatlq_kmeans_pick(const double* dis, const int32_t* order, const int32_t* starts, int64_t k, int32_t* picks,
                                 vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VQ_REQUIRE(dis && order && starts && picks && k >= 1, "bad arguments");
  km_pick_kernel<<<(unsigned)((k * 32 + 255) / 256), 256, 0, stream>>>(dis, order, starts, k, picks);
  VQ_LAUNCHED();
  return 0;
}
