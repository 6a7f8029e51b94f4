// k-center greedy core-set selection (ActiveLearning.coreset_selection,
// active_learning/ActiveLearning.py:798-850) with fp64 distance arithmetic on fp32 features.
//
// One canonical distance d(i,c) is used everywhere (every kernel builds it from the shared tile of
// canonical.cuh, see "the fp64 tensor-core tile" there):
//   dot(i,c): fp64 tensor-core MMAs (mma.sync.m8n8k4.f64) over the features in a fixed order,
//             fp32 inputs widened exactly, fp64 accumulation;
//   d(i,c) = sqrt(max(0, (-2*dot + xx_i) + xx_c))   (sklearn _euclidean_distances order).
//
// Exact batching (DESIGN.md §coreset): scores only ever decrease, so the next greedy picks
// can be decided in advance on the candidate set {score >= theta}: as long as the best
// surviving candidate still scores >= theta it beats every non-candidate (all < theta), ties
// resolving to the lowest index exactly like np.argmax.  One pass over X then applies up to
// 16 picks at once, reading the rows it streams from HBM once instead of 16 times.
//
// A round (d = 2048, up to 16 picks) is: pairs_plan_kernel (candidate x candidate distances, symmetric
// tiles; its last CTA replays the greedy rule on the candidates, emits the picks and chooses the next
// theta from the score histogram) -> the segment filter (exact pruning flags of both centre groups: the
// FILTER mode of the pass kernel on the segment anchors) -> the paired pass (a cluster of two CTAs
// applies the round's 1..16 picks in one read of X; its epilogue lists the next candidates, the exact
// arg-max for the fallback and the next histogram, and pushes the rank's block to the peers' mailboxes).
// Selections that do not pair (batch < 16, or no clusters of two) and the labelled-set initialisation take
// the solo forms of the same kernel (filter, then pass, per 8 centres).  Other feature widths use the
// generic kernels (pairs / plan / pass).
#include <dlfcn.h>

#include <algorithm>
#include <vector>
#include <cstdlib>
#include <cstring>

#include "canonical.cuh"

namespace vatlq {

constexpr int kB = 8;        // centres applied per pass over X (the DMMA tile width)
constexpr int kMaxPicks = 16; // picks planned per round: applied by kMaxPicks / kB passes back to back
#ifndef VQ_PASS_THREADS
#define VQ_PASS_THREADS 512
#endif
constexpr int kPassThreads = VQ_PASS_THREADS;
constexpr int kCapL = 1024;  // candidate records per rank
constexpr int kCap = 1024;   // candidates the planner handles (one per thread)
constexpr int kNB = 1024;    // score-histogram bins
constexpr int kTarget = 256; // default wanted candidates per round (all ranks together); VATLQ_TARGET overrides
constexpr int kMaxRanks = 16;
constexpr int kMaxSmem = 220 * 1024;

struct RankBlock {  // the all-gather unit: one per rank per round
  long long count;  // rows with score >= theta (records beyond kCapL are dropped -> overflow)
  double theta;     // every owned row with score >= theta is listed below
  double smax;      // exact maximum score of the owned rows ...
  long long smax_idx;  // ... and its lowest index
  long long inwin;  // owned rows inside the histogram window
  long long mode;   // how theta was chosen: 0 no list requested, 1 from the histogram, 2 even the top bin overflows
  long long pad[2];
  long long idx[kCapL];
  double m[kCapL];
  double unc[kCapL];
  double score[kCapL];
};

struct Ctl {
  long long n_picked, k;
  long long picks[kMaxPicks];
  int nb;           // picks this round applies (pass p takes picks[8p .. 8p+7])
  int first_round;  // labelled set empty: score = unc, exactly one pick (ActiveLearning.py:816-818)
  int rule, world;
  int maxb, pad1;   // picks per pass allowed (1 = GEMV form: plain argmax every round)
  double wd, wu;    // score = wd*min_d + wu*unc
  double U, W;      // histogram window [U-W, U]; W <= 0: no window yet
  double theta_emit;   // the pass lists every owned row whose new score is >= theta_emit (+inf: none)
  int emit_mode, target; // RankBlock::mode of that list; wanted candidates per round
  unsigned int filter_ticket, pairs_ticket;
  long long stat_passes, stat_rounds, stat_fallback_empty, stat_fallback_overflow, stat_cand_sum;
  // where a round's planning time goes (ns, %globaltimer; summed over the rounds of a call)
  unsigned long long t_start, stat_ns_wait, stat_ns_tiles, stat_ns_plan;
  // phases of the (paired or solo) pass as seen by CTA 0 (ns, summed): prologue, tile loop, row finishing, publishing
  unsigned long long stat_ns_pass[4];
  // phases of the planner (ns, summed): theta + histogram clear, candidate records + distance rows staged, pick loop, tail
  unsigned long long stat_ns_planph[4];
};
__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

struct Best {
  double s;
  long long i;
};
__device__ __forceinline__ bool better(double s, long long i, double s2, long long i2) {
  return (s > s2) || (s == s2 && i < i2);  // np.argmax: first index of the maximum
}
__device__ __forceinline__ Best warp_best(Best b) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const double s2 = __shfl_xor_sync(0xffffffffu, b.s, o);
    const long long i2 = __shfl_xor_sync(0xffffffffu, b.i, o);
    if (better(s2, i2, b.s, b.i)) {
      b.s = s2;
      b.i = i2;
    }
  }
  return b;
}

// ---- candidate-block exchange over peer memory (NVLink) ------------------------------------
// Every rank owns a mailbox in its own HBM: two parities of kMaxRanks block slots plus one flag
// per source rank.  The CTA that finishes a rank's block header pushes the block (header + the
// listed records) straight into slot [parity][rank] of EVERY rank's mailbox with peer stores,
// fences system-wide and raises flag[rank] = sequence number in each mailbox; the kernel that
// consumes the blocks spins on its LOCAL flags.  No collective launch sits between the pass
// that produces the candidates and the planner that consumes them.
struct Mailbox {
  RankBlock slots[2][kMaxRanks];
  unsigned long long flags[kMaxRanks];
  unsigned long long error;      // set when a wait timed out
};
struct PushArgs {
  Mailbox* const* peers;         // device array [world]: every rank's mailbox (own one included)
  int rank, world;
  unsigned long long seq;        // sequence number of the block being produced (parity = seq & 1)
};

// called by every thread of ONE CTA after the block header in `send` is complete
__device__ void push_block(const PushArgs& p, const RankBlock* send) {
  const int tid = threadIdx.x, nthr = blockDim.x;
  const long long cnt = min(__ldcg(&send->count), (long long)kCapL);
  const int par = (int)(p.seq & 1ULL);
  for (int r = 0; r < p.world; ++r) {
    RankBlock* dst = &p.peers[r]->slots[par][p.rank];
    // header (64 bytes) then the first `cnt` entries of the four record arrays
    if (tid < 8) reinterpret_cast<long long*>(dst)[tid] = __ldcg(reinterpret_cast<const long long*>(send) + tid);
    for (long long q = tid; q < cnt; q += nthr) {
      dst->idx[q] = __ldcg(&send->idx[q]);
      dst->m[q] = __ldcg(&send->m[q]);
      dst->unc[q] = __ldcg(&send->unc[q]);
      dst->score[q] = __ldcg(&send->score[q]);
    }
  }
  // release: the barrier orders every thread's record stores before the flag writers' system-scope fence (fences are
  // cumulative), which orders them before the flag.  ONE fence per flag writer — a MEMBAR.SYS by all twelve warps
  // ahead of the barrier, as in round 1, only added its latency to every multi-GPU round.
  __syncthreads();
  if (tid < p.world) {
    __threadfence_system();
    *((volatile unsigned long long*)&p.peers[tid]->flags[p.rank]) = p.seq;
  }
}

// thread 0 of a CTA waits until every rank's block `seq` has landed in the local mailbox
__device__ long long g_mail_timeout_clk = 60000000000LL;   // ~30 s at 2 GHz (VATLQ_MAILBOX_TIMEOUT_S, set at comm attach)
__device__ __forceinline__ void wait_blocks(Mailbox* mine, int world, unsigned long long seq) {
  const long long t0 = clock64();
  const long long limit = g_mail_timeout_clk;
  for (int r = 0; r < world; ++r) {
    while (*((volatile unsigned long long*)&mine->flags[r]) < seq) {
      if (clock64() - t0 > limit) {   // a peer died (or was held up for longer than the limit): report instead of hanging the GPU
        mine->error = seq;
        return;
      }
    }
  }
  __threadfence_system();
}

__device__ __forceinline__ double score_of(int rule, double wd, double wu, double m, double u) {
  if (rule == 0) return __dadd_rn(__dmul_rn(wd, m), __dmul_rn(wu, u));  // :819
  if (rule == 1) return __dadd_rn(m, __dmul_rn(wu, u));                  // :826 (wu = lambda)
  return m;                                                              // :832
}

#ifndef VQ_DEPTH
#define VQ_DEPTH 8
#endif
constexpr int kDepth = VQ_DEPTH;     // super-steps of x in flight per lane (register ring)

// centers in shared memory: fp64, row stride S = dpad + 2 doubles (== 16 bytes mod 128, which
// makes the two 16-byte B loads of a quarter-warp conflict free), features >= d zero
template <typename T>
__device__ __forceinline__ void stage_center(const T* __restrict__ X, int d4, int dpad, int S, long long row, int j,
                                             double* s_c) {
  const quad_t<T>* src = reinterpret_cast<const quad_t<T>*>(X) + (size_t)row * d4;
  for (int q = threadIdx.x; q < dpad / 4; q += blockDim.x) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q < d4) v = ldg_q<T>(src + q);
    double2* dst = reinterpret_cast<double2*>(s_c + (size_t)j * S + 4 * q);
    dst[0] = make_double2((double)v.x, (double)v.y);
    dst[1] = make_double2((double)v.z, (double)v.w);
  }
}

// x[row][4q..4q+3]; GUARD only when d is not a multiple of 16 (the last super-step is ragged)
template <bool GUARD, typename T>
__device__ __forceinline__ float4 load_x(const quad_t<T>* p, int q, int d4) {
  if (GUARD && q >= d4) return make_float4(0.f, 0.f, 0.f, 0.f);
  return quad_f32(ldg_stream(p + q), (const T*)nullptr);
}

__device__ __forceinline__ void dmma_step(double (&c)[4][2], const float4& x, const double* bp) {
  const double2 b01 = *reinterpret_cast<const double2*>(bp);
  const double2 b23 = *reinterpret_cast<const double2*>(bp + 2);
  const double x0 = (double)x.x, x1 = (double)x.y, x2 = (double)x.z, x3 = (double)x.w;
  dmma(c[0], x0, b01.x);
  dmma(c[1], x1, b01.y);
  dmma(c[2], x2, b23.x);
  dmma(c[3], x3, b23.y);
}
__device__ __forceinline__ void dmma_step_self(double (&c)[4][2], const float4& x) {
  const double x0 = (double)x.x, x1 = (double)x.y, x2 = (double)x.z, x3 = (double)x.w;
  dmma(c[0], x0, x0);
  dmma(c[1], x1, x1);
  dmma(c[2], x2, x2);
  dmma(c[3], x3, x3);
}

// canonical dots of one 8-row block (this lane's row pointer `rowp`, never null) against the 8
// staged centers, all four segments by one warp (four independent chains): used by the small
// kernels.  self != 0: B = A (row norms, no shared memory).
template <bool GUARD, bool SELF, typename T>
__device__ __forceinline__ void dmma_block(const quad_t<T>* rowp, int d4, int nss, const double* __restrict__ s_c, int S,
                                           int lane, double (&out)[2]) {
  const int g = lane >> 2, kk = lane & 3;
  const int seglen = (nss + kSeg - 1) / kSeg;
  const double* bptr = SELF ? nullptr : s_c + (size_t)g * S + 4 * kk;
  double P[2][kSeg];
  // the segments are independent chains: run them four at a time (register budget)
#pragma unroll
  for (int grp = 0; grp < kSeg / 4; ++grp) {
    double c[4][4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int e = 0; e < 4; ++e) c[q][e][0] = c[q][e][1] = 0.0;
    for (int s = 0; s < seglen; ++s) {
      float4 x[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int ss = (grp * 4 + q) * seglen + s;
        x[q] = (ss < nss) ? load_x<GUARD, T>(rowp, 4 * ss + kk, d4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int ss = (grp * 4 + q) * seglen + s;
        if (ss < nss) {
          if (SELF) dmma_step_self(c[q], x[q]);
          else dmma_step(c[q], x[q], bptr + 16 * ss);
        }
      }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int q = 0; q < 4; ++q) P[h][grp * 4 + q] = combine4(c[q][0][h], c[q][1][h], c[q][2][h], c[q][3][h]);
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) out[h] = combine8(P[h], 1);
}

// ---------------------------------------------------------------- squared row norms
// xx_i = dot(x_i, x_i): in the diagonal 8x8 block the B operand of lane (g,kk) is its own A
// operand; the diagonal element (g,g) lives in lane (g, g>>1), slot g&1.
template <bool GUARD, typename T>
__global__ void __launch_bounds__(256) row_norms_kernel(const T* __restrict__ X, long long n, int d4, int nss,
                                                        double* __restrict__ xx) {
  const int lane = threadIdx.x & 31, g = lane >> 2, kk = lane & 3;
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r0 = w * 8; r0 < n; r0 += nw * 8) {
    const long long row = min(r0 + g, n - 1);
    double c[2];
    dmma_block<GUARD, true, T>(reinterpret_cast<const quad_t<T>*>(X) + (size_t)row * d4, d4, nss, nullptr, 0, lane, c);
    if (kk == (g >> 1) && r0 + g < n) xx[r0 + g] = (g & 1) ? c[1] : c[0];
  }
}

// ---------------------------------------------------------------- the pass over X
struct PassArgs {
  const void* X;             // [n][d] of the kernel's element type T
  long long n;
  int d4, nss, S;
  long long lo, hi;          // owned rows
  const double* xx;
  double* m;
  double* unc;               // null: distance-only pass (labelled-set initialisation)
  double* score;
  const long long* centers;  // device list of centers to apply
  const int* n_centers;      // device count of the whole list, or null -> n_centers_imm
  int n_centers_imm;
  int center_off;            // this pass applies centers[center_off .. center_off + kB); the pass that
                             // reaches the end of the list is the one that emits / publishes
  Ctl* ctl;                  // null for initialisation passes
  unsigned int* hist;        // null: no histogram
  RankBlock* send;           // null: do not list candidates / arg-max (initialisation passes)
  Best* partial;             // per-CTA arg-max scratch (gridDim entries)
  PushArgs push;             // push.peers != null: the published block is pushed to every rank's mailbox
  unsigned char* did_work;   // optional: set to 1 when this launch applied centres (pass timing bookkeeping)
  double* dots;              // fast path: [owned row][8 or 16] canonical dot products: epilogue warps -> row finishing
  // exact pruning (fast path only, see "pruning" below): tiles whose segments were all flagged by
  // the filter mode are not streamed; their rows keep min_d and only take part in the epilogue
  const int* seg_of_row;             // [owned row] -> segment id, or null
  size_t skip_stride;                // paired pass: the flags of centre group 1 start at seg_skip + skip_stride
  const unsigned char* seg_skip;     // [segment] 1: no row of the segment can get closer to this pass's centres
  // filter mode (pass_kernel_tma<.., FILTER = true>): the tiles are groups of 8 segment ANCHOR rows and the epilogue
  // writes the segments' skip flags instead of dot products
  const int* seg_start;              // [nseg + 1] first owned row of every segment
  const double* seg_r;               // [nseg] segment radius
  const int* nseg;                   // device count of segments
  unsigned char* seg_skip_out;       // flags written by the filter mode (paired: group 1's at + skip_stride)
  int prune_mode;                    // 0 off, 1 skip, 2 verify (stream everything, count rows that changed anyway)
  unsigned long long* prune_stats;   // [0] tiles seen, [1] tiles streamed, [2] verify violations
  // paired pass only, see "the screen" at pass_kernel_tma: 0 off, 1 DMMA only the rows the fp16 screen cannot
  // decide, 2 verify (DMMA every streamed row, count unlisted rows whose min_d moved anyway)
  int screen_mode;
  unsigned long long* screen_stats;  // [0] rows screened, [1] rows listed, [2] verify violations
  const __half* Xh;                  // screen_mode != 0: X[lo, hi) in 16 bits, row r - lo at Xh + (r - lo) * 2048: the
                                     // fp16 copy for an fp32 X, X itself for a 16-bit X (bf16 bits: only addressed)
};

// centres of THIS pass: count (<= 0: nothing to do) and whether it is the round's last pass
__device__ __forceinline__ int pass_centers(const PassArgs& a, bool& final_pass) {
  const int total = a.n_centers ? *a.n_centers : a.n_centers_imm;
  final_pass = a.center_off + kB >= total;
  return min(kB, total - a.center_off);
}

// ---- what the epilogue of a pass leaves behind for the next round -------------------------
// every owned row: running arg-max of the new scores; rows with score >= theta_emit are listed
__device__ __forceinline__ void emit_row(RankBlock* send, double theta_emit, long long i, double dmin, double u,
                                         double sc, Best& best) {
  if (better(sc, i, best.s, best.i)) {
    best.s = sc;
    best.i = i;
  }
  if (sc >= theta_emit) {
    const unsigned long long pos = atomicAdd((unsigned long long*)&send->count, 1ULL);
    if (pos < (unsigned long long)kCapL) {
      send->idx[pos] = i;
      send->m[pos] = dmin;
      send->unc[pos] = u;
      send->score[pos] = sc;
    }
  }
}

// reduce the arg-max over the CTA and let the last CTA of the grid finish the rank's block header `out`: the exact
// arg-max, theta, mode, the in-window count (*inwin, read once every CTA is done; null: 0) and, with reset_count,
// count = 0; then push it to the peers (every thread of the CTA calls this; nw: warps of the CTA)
__device__ void publish_header(int nw, Best best, Best* partial, Ctl* ctl, RankBlock* out, const PushArgs& push,
                               double theta, long long mode, const unsigned int* inwin, bool reset_count) {
  __shared__ Best s_best[32];
  __shared__ unsigned int s_last;
  const int tid = threadIdx.x;
  best = warp_best(best);
  if ((tid & 31) == 0) s_best[tid >> 5] = best;
  __syncthreads();
  if (tid == 0) {
    for (int k = 1; k < nw; ++k)
      if (better(s_best[k].s, s_best[k].i, best.s, best.i)) best = s_best[k];
    partial[blockIdx.x] = best;
    __threadfence();
    s_last = (atomicAdd(&ctl->filter_ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    Best b{-INFINITY, 0x7fffffffffffffffLL};
    for (int k = tid; k < (int)gridDim.x; k += blockDim.x) {
      Best q;
      q.s = ((volatile Best*)partial)[k].s;
      q.i = ((volatile Best*)partial)[k].i;
      if (better(q.s, q.i, b.s, b.i)) b = q;
    }
    b = warp_best(b);
    __syncthreads();
    if ((tid & 31) == 0) s_best[tid >> 5] = b;
    __syncthreads();
    if (tid == 0) {
      for (int k = 1; k < nw; ++k)
        if (better(s_best[k].s, s_best[k].i, b.s, b.i)) b = s_best[k];
      if (reset_count) out->count = 0;
      out->smax = b.s;
      out->smax_idx = b.i;
      out->theta = theta;
      out->mode = mode;
      out->inwin = inwin ? (long long)*(volatile const unsigned int*)inwin : 0;
      ctl->filter_ticket = 0;
      __threadfence();
    }
    if (push.peers != nullptr) {
      __syncthreads();
      push_block(push, out);
    }
  }
}

// flush the CTA's histogram; the round's last pass publishes the block header (every thread of the CTA calls this)
__device__ void publish_pass(const PassArgs& a, Best best, bool do_hist, const unsigned int* s_hist, bool final_pass) {
  if (do_hist) {
    for (int b = threadIdx.x; b < kNB + 1; b += blockDim.x)
      if (s_hist[b]) atomicAdd(&a.hist[b], s_hist[b]);
  }
  if (a.send == nullptr || !final_pass) return;
  publish_header((blockDim.x + 31) >> 5, best, a.partial, a.ctl, a.send, a.push, a.ctl->theta_emit, a.ctl->emit_mode,
                 do_hist ? a.hist + kNB : nullptr, false);
}

// what a pass reads from the control block to finish its rows
struct ApplyConst {
  double h_lo, h_inv, wd, wu, theta_emit;
  int rule;
  bool do_hist, emit;
};
__device__ __forceinline__ ApplyConst apply_const(const PassArgs& a, bool final_pass) {
  ApplyConst c{0.0, 0.0, 0.0, 0.0, INFINITY, 0, false, false};
  c.do_hist = a.hist != nullptr && a.ctl != nullptr && a.ctl->W > 0.0 && final_pass;
  c.emit = a.send != nullptr && final_pass;
  if (a.ctl) {
    c.rule = a.ctl->rule;
    c.wd = a.ctl->wd;
    c.wu = a.ctl->wu;
    c.theta_emit = a.ctl->theta_emit;
    if (c.do_hist) {
      c.h_lo = a.ctl->U - a.ctl->W;
      c.h_inv = (double)kNB / a.ctl->W;
    }
  }
  return c;
}
// the end of a row's finishing once its new min_d is known (and written): unc := 0 for a pick, the score, the
// candidate record and the arg-max.  Returns the histogram bin of the new score (-1: outside the window / no histogram)
__device__ __forceinline__ int finish_row(const PassArgs& a, const ApplyConst& c, long long i, double dmin, bool picked,
                                          Best& best) {
  if (a.unc) {
    double u = a.unc[i];
    if (picked) {
      u = 0.0;  // uncertainty[ind] = 0  (:848)
      a.unc[i] = 0.0;
    }
    const double sc = score_of(c.rule, c.wd, c.wu, dmin, u);
    a.score[i] = sc;
    if (c.emit) emit_row(a.send, c.theta_emit, i, dmin, u, sc, best);
    if (c.do_hist) {
      const double fb = (sc - c.h_lo) * c.h_inv;
      if (fb >= 0.0) return (int)fmin(fb, (double)(kNB - 1));
    }
  }
  return -1;
}

constexpr int kTeams = kPassThreads / 32 / kSeg;   // 2 teams of 8 warps

template <bool GUARD, typename T>
__global__ void __launch_bounds__(kPassThreads, 1) pass_kernel_generic(PassArgs a) {
  using Q = quad_t<T>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  bool final_pass;
  const int nb = pass_centers(a, final_pass);
  if (nb <= 0) return;
  const long long* centers = a.centers + a.center_off;
  double* s_c = reinterpret_cast<double*>(smem_raw);
  double* s_xxc = s_c + (size_t)kB * a.S;
  double* s_part = s_xxc + kB;                               // [team][buf][seg][64]
  long long* s_pick = reinterpret_cast<long long*>(s_part + kTeams * 2 * kSeg * 64);
  unsigned int* s_hist = reinterpret_cast<unsigned int*>(s_pick + kB);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, kk = lane & 3;
  const int team = warp / kSeg, seg = warp % kSeg;
  const int dpad = a.nss * 16;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (a.ctl) a.ctl->stat_passes += 1;
    if (a.did_work) *a.did_work = 1;
  }
  for (int j = 0; j < kB; ++j) {
    const long long p = centers[min(j, nb - 1)];  // pad with the last center: min() is idempotent
    stage_center(static_cast<const T*>(a.X), a.d4, dpad, a.S, p, j, s_c);
    if (threadIdx.x == 0) {
      s_xxc[j] = a.xx[p];
      s_pick[j] = p;
    }
  }
  const ApplyConst ac = apply_const(a, final_pass);
  Best best{-INFINITY, 0x7fffffffffffffffLL};
  if (ac.do_hist)
    for (int b = threadIdx.x; b < kNB + 1; b += blockDim.x) s_hist[b] = 0u;
  __syncthreads();

  const Q* X4 = reinterpret_cast<const Q*>(a.X);
  const long long ntiles = (a.hi - a.lo + 7) / 8;
  const long long t0 = (long long)blockIdx.x * kTeams + team, tstride = (long long)gridDim.x * kTeams;
  const long long nt = (t0 < ntiles) ? (ntiles - t0 + tstride - 1) / tstride : 0;
  const int seglen = (a.nss + kSeg - 1) / kSeg;
  const int seg_beg = min(a.nss, seg * seglen), seg_end = min(a.nss, seg_beg + seglen), mylen = seg_end - seg_beg;
  const double* bptr = s_c + (size_t)g * a.S + 4 * kk + 16 * seg_beg;
  double* my_part = s_part + ((size_t)(team * 2) * kSeg + seg) * 64 + lane * 2;   // + buf*kSeg*64
  const double* team_part = s_part + (size_t)(team * 2) * kSeg * 64 + lane * 2;

  auto row_ptr = [&](long long t) {
    const long long row = min(a.lo + t * 8 + g, a.hi - 1);   // rows past the end re-read the last row
    return X4 + (size_t)row * a.d4 + 4 * seg_beg + kk;
  };
  // tile epilogue: publish this segment's partial; the seg-0 warp of the team finishes the block
  int buf = 0;
  auto finish_tile = [&](long long t, double (&c)[4][2]) {
    double* dst = my_part + buf * (kSeg * 64);
    dst[0] = combine4(c[0][0], c[1][0], c[2][0], c[3][0]);
    dst[1] = combine4(c[0][1], c[1][1], c[2][1], c[3][1]);
    asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "r"(kSeg * 32) : "memory");
    if (seg == 0) {
      const double* src = team_part + buf * (kSeg * 64);
      const double d0 = combine8(src, 64);
      const double d1 = combine8(src + 1, 64);
      const long long i = a.lo + t * 8 + g;
      const bool live = i < a.hi;
      const double xxi = live ? a.xx[i] : 0.0;
      double dm = fmin(dist_from_dot(d0, xxi, s_xxc[2 * kk]), dist_from_dot(d1, xxi, s_xxc[2 * kk + 1]));
      dm = fmin(dm, __shfl_xor_sync(0xffffffffu, dm, 1));
      dm = fmin(dm, __shfl_xor_sync(0xffffffffu, dm, 2));
      if (live && kk == 0) {
        const double dmin = fmin(a.m[i], dm);
        a.m[i] = dmin;
        bool picked = false;
#pragma unroll
        for (int j = 0; j < kB; ++j) picked = picked || (s_pick[j] == i);
        const int b = finish_row(a, ac, i, dmin, picked, best);
        if (b >= 0) {
          atomicAdd(&s_hist[b], 1u);
          atomicAdd(&s_hist[kNB], 1u);
        }
      }
    }
    buf ^= 1;
#pragma unroll
    for (int e = 0; e < 4; ++e) c[e][0] = c[e][1] = 0.0;
  };

  double c[4][2];
#pragma unroll
  for (int e = 0; e < 4; ++e) c[e][0] = c[e][1] = 0.0;
  if (mylen == 0) {
    for (long long k = 0; k < nt; ++k) finish_tile(t0 + k * tstride, c);   // (tiny d: empty segment)
  } else {
    // flattened (tile, step) stream with an 8-deep register ring: the loads of the next tile are
    // already in flight while the current one is finished
    const long long F = nt * mylen;
    long long ct = t0;                 // tile being consumed
    int cs = 0;                        // step inside its segment
    long long lt = t0;                 // load cursor
    int ls = 0;
    const Q* lp = (nt > 0) ? row_ptr(lt) : X4;
    float4 ring[kDepth];
#pragma unroll
    for (int p = 0; p < kDepth; ++p) {
      ring[p] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p < F) {
        ring[p] = load_x<GUARD, T>(lp, 4 * ls, a.d4 - 4 * seg_beg - kk);
        if (++ls == mylen) {
          ls = 0;
          lt += tstride;
          if (lt < ntiles) lp = row_ptr(lt);
        }
      }
    }
    for (long long f0 = 0; f0 < F; f0 += kDepth) {
#pragma unroll
      for (int p = 0; p < kDepth; ++p) {
        const long long f = f0 + p;
        if (f < F) {
          const double2 b01 = *reinterpret_cast<const double2*>(bptr + 16 * cs);
          const double2 b23 = *reinterpret_cast<const double2*>(bptr + 16 * cs + 2);
          const double x0 = (double)ring[p].x, x1 = (double)ring[p].y, x2 = (double)ring[p].z, x3 = (double)ring[p].w;
          if (f + kDepth < F) {          // refill the slot that was just consumed
            ring[p] = load_x<GUARD, T>(lp, 4 * ls, a.d4 - 4 * seg_beg - kk);
            if (++ls == mylen) {
              ls = 0;
              lt += tstride;
              if (lt < ntiles) lp = row_ptr(lt);
            }
          }
          dmma(c[0], x0, b01.x);
          dmma(c[1], x1, b01.y);
          dmma(c[2], x2, b23.x);
          dmma(c[3], x3, b23.y);
          if (++cs == mylen) {
            finish_tile(ct, c);
            ct += tstride;
            cs = 0;
          }
        }
      }
    }
  }
  __syncthreads();
  publish_pass(a, best, ac.do_hist, s_hist, final_pass);
}

// second half of the fast-path pass: one thread per row turns the kB canonical dot products
// into the distance to the nearest new centre (min_j sqrt(max(t_j, 0)) == sqrt(max(min_j t_j, 0))
// bit for bit, sqrt being monotone and correctly rounded: one square root per row instead of kB),
// the running minimum, unc/score, the candidate list, the histogram and the arg-max
// tile_mode: 0 streamed, 1 pruned (no dot products were computed: min_d stays), 2 verify (streamed
// although the filter flagged it: count the rows whose min_d moved anyway — must stay 0), 3 screen verify
// (computed although the screen decided the row: the same count, into screen_stats[2])
// Returns the histogram bin of the row's new score (-1: outside the window / no histogram): the caller adds it
// warp-aggregated (rows of one track score alike, so per-row shared-memory atomics on one bin — and on the in-window
// counter — serialised the whole CTA: 145 us of a 1 M-row pass).
template <int NC = kB>
__device__ __forceinline__ int apply_row(const PassArgs& a, const ApplyConst& c, long long i, const double* s_xxc,
                                         const long long* s_pick, Best& best, int tile_mode = 0) {
  const double2* dp = reinterpret_cast<const double2*>(a.dots + (i - a.lo) * NC);
  const double xxi = a.xx[i];
  double tm = INFINITY;
  bool picked = false;
  if (tile_mode != 1) {
#pragma unroll
    for (int q = 0; q < NC / 2; ++q) {
      const double2 d2 = __ldcg(dp + q);
      tm = fmin(tm, sq_from_dot(d2.x, xxi, s_xxc[2 * q]));
      tm = fmin(tm, sq_from_dot(d2.y, xxi, s_xxc[2 * q + 1]));
      picked = picked || s_pick[2 * q] == i || s_pick[2 * q + 1] == i;
    }
  }
  const double m_old = a.m[i];
  const double dmin = fmin(m_old, sqrt(fmax(tm, 0.0)));
  if (tile_mode == 2 && (dmin != m_old || picked)) atomicAdd(&a.prune_stats[2], 1ULL);
  if (tile_mode == 3 && (dmin != m_old || picked)) atomicAdd(&a.screen_stats[2], 1ULL);
  if (tile_mode != 1) a.m[i] = dmin;
  return finish_row(a, c, i, dmin, picked, best);
}

// ---------------------------------------------------------------- the pass over X, fast path
// d == kFastD (2048).  Warp-specialised, one CTA per SM, 8-row tiles:
//   * PRODUCER (one warp): streams tiles into a ring of kStagesX shared-memory stages with 1-D TMA
//     bulk copies (one 8 KB cp.async.bulk per row, completion counted on the stage's mbarrier) and
//     refills a stage as soon as the 8 compute warps have released it, so two to three tiles
//     (128-192 KB per SM) are always in flight no matter how the math is scheduled.
//   * 8 COMPUTE warps = the 8 K-segments of a tile.  Warp w keeps ITS 1/8 of the 8 centres in
//     registers as fp64 B operands (kSteps x 4 doubles per lane); per super-step it reads one
//     float4 of A from the stage (row stride 8 KB + 64 B: conflict free), converts and issues four
//     DMMAs.  A tile ends with one 16-byte shared store of the segment's partial dots and a
//     non-blocking bar.arrive.
//   * 3 EPILOGUE warps, one per partial buffer (tile k -> warp k mod 3, a pair of named barriers
//     per buffer): split-K reduction in the canonical order, 8x8 dot products to global memory
//     (64 B per row, < 1 % of the traffic).
// After the tile loop the compute warps finish the CTA's own rows from those dot products
// (apply_row) and the last CTA of the grid publishes the rank's block header.
// setmaxnreg: compute warpgroups 216 registers, the producer/epilogue warpgroup 72.
constexpr int kStagesX = 3;
constexpr int kPartBufs = 3;
constexpr int kRowBytesX = kFastD * 4 + 64;                // stage row stride
constexpr int kStageBytesX = 8 * kRowBytesX;               // 66 048
// the screen's stages hold TWO tiles of fp16 rows (16 x 4 KB, the bytes of one fp32 tile).  Row stride = 32 mod 128
// bytes: the 8-byte loads of rows g = 0..3 (lanes 4g .. 4g+3, 32 contiguous bytes each) hit all 32 banks
constexpr int kRowBytesH = kFastD * 2 + 32;
static_assert(16 * kRowBytesH == kStageBytesX, "an fp16 stage of two tiles fills an fp32 stage exactly");

constexpr int kWsThreads = (kSeg + 4) * 32;                // 8 compute warps + producer + 3 epilogue warps
constexpr int kMaxTilesCta = 2048;                         // tiles per CTA the pruned-tile list can hold
constexpr size_t kWsSmem = (size_t)kStagesX * kStageBytesX + sizeof(double) * kPartBufs * kSeg * 64 + 2 * kStagesX * 8 +
                           2 * kB * 16 + (kNB + 1) * 4 + 128 + kMaxTilesCta * 2 + kMaxTilesCta / 8 + 16 +
                           kMaxTilesCta + 2 * kB * 8 + 16;   // the screen: listed-row mask per tile, centre norms

__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void named_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ float4 lds128(unsigned addr) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
  return r;
}
__device__ __forceinline__ uint2 lds64(unsigned addr) {
  uint2 r;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr));
  return r;
}
// quad of a staged row, widened to fp32 (16 bytes in fp32, 8 in 16 bits)
template <typename T>
__device__ __forceinline__ float4 lds_quad(unsigned addr) {
  if constexpr (sizeof(T) == 4) return lds128(addr);
  else return quad_f32(lds64(addr), (const T*)nullptr);
}

// PAIR = true ("paired pass"): the grid is launched as clusters of two CTAs (one TPC).  Both CTAs of a pair walk the
// SAME tile sequence, CTA r holding centre group r (picks 8r .. 8r+7) as its register-resident B operands, so a round
// of up to 16 picks reads X from HBM ONCE: the pair's two TMA requests for a tile arrive at the L2 together and
// are served by one DRAM fetch.  The cluster only provides co-scheduling and the barrier between the tile loop and the
// row finishing (each CTA finishes half of the pair's rows from both CTAs' dot products, 16 per row).
__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 32-bit word at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ unsigned ld_dsmem_u32(const void* p, unsigned rank) {
  unsigned remote, v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_addr(p)), "r"(rank));
  asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(remote) : "memory");
  return v;
}

// ---- the screen (paired pass, screen_mode != 0) ------------------------------------------------
// A round only needs to know which rows get closer to one of its <= 16 centres: min_d[i] changes iff
// d(i,c) < m_old = min_d[i] for some c.  Before the DMMA tile loop each CTA of a pair streams the tiles of ITS
// parity (the rows it finishes) through the same TMA ring, read from an fp16 copy of the owned rows (PassArgs::Xh,
// filled once per selection call by half_copy_kernel: half the bytes of the fp32 rows), and the compute warps
// evaluate S~ = x~.c~ for all 16 centres with mma.sync m16n8k16 f16 (A = 16 centres from registers, read from the
// fp32 X and rounded the same way, B = a tile's 8 rows, fp32 accumulation; warp w = K segment w as in the DMMA
// loop).  A row is DECIDED when for every centre
//     S~ finite  and  fl(t~ - 2E) > m_old^2 rounded up,   t~ = (|x|^2 + |c|^2) - 2 S~,
//     E = 2u |x||c| + 2^-20 (|x|^2 + |c|^2) + 2^-17 (|x| + |c|),  u = 2^-8,
// with m_old finite and the row not one of the picks.  Proof that a decided row keeps min_d bit for bit (S: the
// exact dot of the fp32 features, K = 2048).  cvt.rn to fp16 moves an element v by |dv| <= 2^-11 |v| in the normal
// range and by |dv| <= 2^-25 in the subnormal range (|v| < 2^-14), so |dv| <= 2^-11 |v| + 2^-25 and, 0 being
// representable, |dv| <= |v|.  Then x~c~ - xc = dx c + x dc + dx dc with |dx dc| <= (2^-11|x_k| + 2^-25)|dc| <=
// 2^-22 |x_k c_k| + 2^-36 |x_k| + 2^-25 |c_k|, so the exact dot of the fp16 operands is within
//     (2^-10 + 2^-22) sum|x_k c_k| + 2^-24 (|x|_1 + |c|_1)
// of S; with sum|x_k c_k| <= |x||c| (Cauchy-Schwarz) and |v|_1 <= sqrt(2048) |v|_2 this is
// <= (2^-10 + 2^-22) |x||c| + 2^-18.5 (|x| + |c|).  The products of two fp16 values are exact in fp32, and the fp32
// accumulation is ASSUMED to add at most 2048 * 2^-23 = 2^-12 relative to sum |x~_k c~_k| (not proven for the
// tensor core's internal order; the verify mode of tests/test_gpu_pass_screen*.py checks it): in all
//     |S~ - S| <= (2^-10 + 2^-12 + 2^-20) |x||c| + 2^-18.4 (|x| + |c|) <= u |x||c| + 2^-18 (|x| + |c|).
// The canonical fp64 value t = fl(fl(-2 dot + xx_i) + xx_c) is within 2^-48 (|x|^2 + |c|^2) of |x|^2 + |c|^2 - 2S,
// so t >= t~ - 2u|x||c| - 2^-17 (|x| + |c|) - 2^-48(..) = (t~ - 2E) + 2u|x||c| + 2^-19 (|x|^2 + |c|^2)
// + 2^-17 (|x| + |c|) - 2^-48 (..), which exceeds the computed fl(t~ - 2E) by more than that subtraction's own
// rounding (and that of |x|, |c|, which enter E only scaled by u or 2^-17): t > m_old^2.  sqrt is correctly rounded
// and monotone and m_old is a double, so d = sqrt(max(t, 0)) >= m_old and fmin(m_old, d) == m_old: the row's
// min_d, score and candidate record are exactly what the full pass writes.  Any NaN / Inf makes the test false
// (the row is listed); in particular an element with |v| >= 65520 becomes +-Inf in fp16, and S~ is then +-Inf or
// NaN (Inf x 0), never finite.  The undecided rows are then gathered 8 per tile (the per-row TMA copies of the fp32
// rows the producer always issues) and only those go through the canonical DMMA tile machine.
//
// 16-BIT X (fp16 or bf16): the screen streams X itself through the same stages (its rows are the copy's 4 KB), reads
// the 16 centres from X as they are, and issues mma.sync m16n8k16 in X's own type (f16 or bf16).  No operand is
// rounded: x~ = x and c~ = c, so the input terms above vanish.  A product of two fp16 (11 x 11 significant bits) or two
// bf16 values (8 x 8 bits) is exact in fp32, so S~ differs from S only by the fp32 accumulation, which is ASSUMED, as
// above, to add at most 2048 * 2^-23 = 2^-12 relative to sum |x_k c_k| <= |x||c| (checked by verify mode, not proven).
// bf16 has fp32's exponent range, so an input below 2^-126 may be flushed by the tensor core (moving the dot by
// < 2^-126 |c|_1 <= 2^-120.5 |c|, likewise for x), a product or a partial sum may fall below 2^-126 (at worst flushed:
// < 2^-114 over the 2048 products and additions), and a product or a sum may overflow to Inf / NaN.  Hence
//     |S~ - S| <= 2^-12 |x||c| + 2^-120 (|x| + |c|) + 2^-114,
//     E16 = 2 u16 |x||c| + 2^-20 (|x|^2 + |c|^2) + 2^-100 (1 + |x| + |c|),   u16 = 2^-12,
// and the proof above goes through with E16 for E: t >= t~ - 2|S~ - S| - 2^-48 (..) exceeds fl(t~ - 2 E16) by more than
// its rounding.  A row whose S~ overflowed is not finite and is listed, never decided.  (An fp16 dot product cannot
// overflow fp32: 2048 x 65504^2 < 2^44; its products are >= 2^-48 and never underflow.)
constexpr double kScreenU = 0.00390625;               // 2^-8
constexpr double kScreenAbs = 9.5367431640625e-07;    // 2^-20
constexpr double kScreenAbs1 = 7.62939453125e-06;     // 2^-17
constexpr double kScreenU16 = 0.000244140625;         // 2^-12
constexpr double kScreenAbs16 = 7.888609052210118e-31;  // 2^-100
template <typename T = __half>
__device__ __forceinline__ void mma_f16(float (&d)[4], const unsigned (&a)[4], uint2 b) {
  if constexpr (std::is_same<T, __nv_bfloat16>::value)
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
  else
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
}
__device__ __forceinline__ unsigned half2_bits(float lo, float hi) {   // cvt.rn.f16x2.f32: lo in the low half
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&h);
}
// the screen's fp16 copy of rows [lo, lo + n4 / 512) of X (d = 2048): one float4 -> four halves per thread and step
__global__ void __launch_bounds__(256) half_copy_kernel(const float4* __restrict__ X, long long lo, long long n4,
                                                        uint2* __restrict__ Xh) {
  const float4* src = X + lo * 512;
  for (long long q = (long long)blockIdx.x * 256 + threadIdx.x; q < n4; q += (long long)gridDim.x * 256) {
    const float4 v = ldg_stream(src + q);
    Xh[q] = make_uint2(half2_bits(v.x, v.y), half2_bits(v.z, v.w));
  }
}
// entry e of the list of undecided rows -> the walker's tile k and row r (s_pre: inclusive prefix of the listed
// rows per tile, nt entries; s_mask: the listed rows of every tile)
__device__ __forceinline__ int listed_row(const unsigned short* s_pre, const unsigned char* s_mask, int nt, int e) {
  int lo = 0, hi = nt - 1;   // smallest k with s_pre[k] > e
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((int)s_pre[mid] > e) hi = mid;
    else lo = mid + 1;
  }
  int skip = e - (lo ? (int)s_pre[lo - 1] : 0);
  const unsigned m = s_mask[lo];
  int r = 0;
#pragma unroll
  for (int b = 0; b < 8; ++b)
    if ((m >> b) & 1u) {
      if (skip == 0) r = b;
      --skip;
    }
  return lo * 8 + r;
}

template <bool PAIR, bool FILTER = false, typename T = float>
__global__ void __launch_bounds__(kWsThreads, 1) pass_kernel_tma(PassArgs a) {
  using Q = quad_t<T>;
  constexpr bool X16 = sizeof(T) == 2;            // 16-bit X: the screen reads X itself (see "the screen")
  // stage row stride of the DMMA tiles: a 16-bit X keeps its rows at the screen's stride (8-byte loads, conflict
  // free), one tile in the first half of a stage
  constexpr int kRowB = X16 ? kRowBytesH : kRowBytesX;
  constexpr unsigned kXRowBytes = kFastD * sizeof(T);
  constexpr int NC = PAIR ? 2 * kB : kB;          // dot products per row the finishing reads
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* stage0 = smem_raw;
  double (*s_part)[kSeg][64] = reinterpret_cast<double (*)[kSeg][64]>(smem_raw + (size_t)kStagesX * kStageBytesX);
  uint64_t* full = reinterpret_cast<uint64_t*>(s_part + kPartBufs);
  uint64_t* empty = full + kStagesX;
  double* s_xxc = reinterpret_cast<double*>(empty + kStagesX);
  long long* s_pick = reinterpret_cast<long long*>(s_xxc + 2 * kB);
  unsigned int* s_hist = reinterpret_cast<unsigned int*>(s_pick + 2 * kB);
  // pruning: the tiles this CTA streams (indices k into its own tile sequence), a bitmap of the
  // flagged ones, and the number of streamed tiles
  unsigned short* s_tiles = reinterpret_cast<unsigned short*>(s_hist + (kNB + 1) + 3);
  unsigned int* s_flagged = reinterpret_cast<unsigned int*>(s_tiles + kMaxTilesCta);
  int* s_na = reinterpret_cast<int*>(s_flagged + kMaxTilesCta / 32);   // [0] streamed tiles, [1] of them of this CTA's
                                                                        // parity, [2] rows the screen listed
  // the screen: listed (undecided) rows of every tile of the walker as a bit mask, |c| of the 16 centres
  unsigned char* s_mask = reinterpret_cast<unsigned char*>(s_na + 4);
  double* s_nc = reinterpret_cast<double*>(s_mask + kMaxTilesCta);

  pdl_enter();
  // this launch applies centres [center_off, center_off + NC) of the list, CTA r of a pair group r (the filter: the
  // flags of group r); a short group is padded with the last centre (min() is idempotent), so a paired pass applies
  // any round of 1..16 picks and a group without centres of its own only repeats the last one
  const int total = (a.n_centers ? *a.n_centers : a.n_centers_imm) - a.center_off;
  if (total <= 0) return;
  const bool final_pass = NC >= total;
  auto centre = [&](int j) { return (a.centers + a.center_off)[min(j, total - 1)]; };
  const int crank = PAIR ? (int)cluster_ctarank() : 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool clocked = !FILTER && a.ctl != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  unsigned long long tq0 = 0, tq1 = 0, tq2 = 0, tq3 = 0;
  if (clocked) tq0 = gtime_ns();
  const int ncl = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;       // independent tile walkers
  const int cid = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  if (!FILTER && blockIdx.x == 0 && threadIdx.x == 0) {
    if (a.ctl) a.ctl->stat_passes += 1;
    if (a.did_work) *a.did_work = 1;
  }
  if (threadIdx.x < NC) {
    const long long p = centre(threadIdx.x);   // every centre the finishing sees
    s_xxc[threadIdx.x] = a.xx[p];
    s_nc[threadIdx.x] = sqrt(a.xx[p]);
    s_pick[threadIdx.x] = p;
  }
  for (int b = threadIdx.x; b < kNB + 1; b += blockDim.x) s_hist[b] = 0u;
  if (threadIdx.x == 0) {
    for (int q = 0; q < kStagesX; ++q) {
      mbar_init(&full[q], 1);        // one expect_tx arrival + the bytes
      mbar_init(&empty[q], kSeg);    // one arrival per compute warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const int nseg = FILTER ? *a.nseg : 0;
  const long long ntiles = FILTER ? (nseg + 7) / 8 : (a.hi - a.lo + 7) / 8;
  const int nt = ((long long)cid < ntiles) ? (int)((ntiles - cid + ncl - 1) / ncl) : 0;
  // tile j of the streamed sequence is tile k = tile_of(j) of the walker (rows (cid + k*ncl)*8 ...)
  const bool use_list = !FILTER && a.seg_skip != nullptr && a.prune_mode != 0 && nt <= kMaxTilesCta;
  const int screen = (PAIR && !FILTER && nt <= kMaxTilesCta) ? a.screen_mode : 0;   // the same on both CTAs of a pair
  const unsigned own_par = crank ? 0xaaaaaaaau : 0x55555555u;   // tiles base + lane of this CTA's parity (base % 32 == 0)
  if (screen)
    for (int k = threadIdx.x; k < nt; k += blockDim.x) s_mask[k] = 0;
  // The list of streamed tiles is built by ALL warps (chunks of 32 tiles dealt round-robin: the two dependent loads per
  // tile — segment ids, then their flags — are one memory round trip per chunk instead of one per 32 tiles of the
  // whole CTA); the chunk counts are scanned by one warp and every warp then writes its chunks at their offsets.
  unsigned int* s_cnt = reinterpret_cast<unsigned int*>(s_part);   // [kMaxTilesCta / 32] chunk counts (the partial buffers are idle)
  constexpr int kWarps = kWsThreads / 32;
  unsigned my_sm[(kMaxTilesCta / 32 + kWarps - 1) / kWarps];
  if (use_list) {
    int ci = 0;
    for (int base = warp * 32; base < nt; base += kWarps * 32, ++ci) {
      const int k = base + lane;
      bool flagged = false;
      if (k < nt) {
        const long long r0 = ((long long)cid + (long long)k * ncl) * 8;   // relative to a.lo
        const long long r1 = min(r0 + 7, a.hi - a.lo - 1);
        const int s0 = a.seg_of_row[r0], s1 = a.seg_of_row[r1];
        flagged = true;
        for (int sg = s0; sg <= s1; ++sg) {
          flagged = flagged && (a.seg_skip[sg] != 0);
          if (PAIR) flagged = flagged && (a.seg_skip[a.skip_stride + sg] != 0);   // ... for BOTH centre groups
        }
      }
      const unsigned fm = __ballot_sync(0xffffffffu, flagged);
      const bool stream = (k < nt) && !(flagged && a.prune_mode == 1);
      const unsigned sm = __ballot_sync(0xffffffffu, stream);
      my_sm[ci] = sm;
      if (lane == 0) {
        s_flagged[base >> 5] = fm;
        s_cnt[base >> 5] = __popc(sm);
        s_cnt[kMaxTilesCta / 32 + (base >> 5)] = __popc(sm & own_par);
      }
    }
    __syncthreads();
    if (warp == 0) {                     // exclusive scan of the chunk counts (<= 64 chunks: two per lane)
      const int nch = (nt + 31) >> 5;
      const unsigned c0 = (2 * lane < nch) ? s_cnt[2 * lane] : 0u, c1 = (2 * lane + 1 < nch) ? s_cnt[2 * lane + 1] : 0u;
      const int n1 = warp_sum((int)((2 * lane < nch ? s_cnt[kMaxTilesCta / 32 + 2 * lane] : 0u) +
                                    (2 * lane + 1 < nch ? s_cnt[kMaxTilesCta / 32 + 2 * lane + 1] : 0u)));
      if (lane == 0) s_na[1] = n1;
      unsigned incl = c0 + c1;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const unsigned excl = incl - (c0 + c1);
      if (2 * lane < nch) s_cnt[2 * lane] = excl;
      if (2 * lane + 1 < nch) s_cnt[2 * lane + 1] = excl + c0;
      if (lane == 31) {
        *s_na = (int)incl;
        if (a.prune_stats && nt > 0 && crank == 0) {
          atomicAdd(&a.prune_stats[0], (unsigned long long)nt);
          atomicAdd(&a.prune_stats[1], (unsigned long long)incl);
        }
      }
    }
    __syncthreads();
    ci = 0;
    for (int base = warp * 32; base < nt; base += kWarps * 32, ++ci) {
      const unsigned sm = my_sm[ci];
      if ((sm >> lane) & 1u) s_tiles[s_cnt[base >> 5] + __popc(sm & ((1u << lane) - 1u))] = (unsigned short)(base + lane);
    }
  } else if (threadIdx.x == 0) {
    *s_na = nt;
    s_na[1] = (nt + 1 - crank) / 2;
    if (!FILTER && a.prune_stats && nt > 0 && crank == 0) {   // (the filter's anchor tiles are not rows streamed)
      atomicAdd(&a.prune_stats[0], (unsigned long long)nt);
      atomicAdd(&a.prune_stats[1], (unsigned long long)nt);
    }
  }
  __syncthreads();
  if (clocked) tq1 = gtime_ns();
  const int na = *s_na;
  auto tile_of = [&](int j) -> int { return use_list ? (int)s_tiles[j] : j; };
  // the screen's tiles are the streamed tiles of this CTA's parity (the rows it finishes): n1 of them
  const int n1 = s_na[1];
  // between the screen and the DMMA tiles (every thread of both CTAs): merge the partner's listed rows, so that
  // both CTAs of the pair walk the same list of undecided rows, and (list mode) count them per tile
  auto screen_join = [&]() {
    named_sync(7, kWsThreads);
    cluster_sync_all();
    for (int w = threadIdx.x; w < (nt + 3) / 4; w += blockDim.x)
      reinterpret_cast<unsigned*>(s_mask)[w] |= ld_dsmem_u32(s_mask + 4 * w, (unsigned)crank ^ 1u);
    named_sync(7, kWsThreads);
    if (screen == 1) {
      if (warp == kSeg) {   // inclusive prefix of the listed rows per tile (s_tiles is no longer read)
        const int k0 = lane * (kMaxTilesCta / 32), k1 = min(nt, k0 + kMaxTilesCta / 32);
        int sum = 0;
        for (int k = k0; k < k1; ++k) sum += __popc(s_mask[k]);
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += t;
        }
        int run = incl - sum;
        for (int k = k0; k < k1; ++k) {
          run += __popc(s_mask[k]);
          s_tiles[k] = (unsigned short)run;
        }
        if (lane == 31) s_na[2] = incl;
      }
      named_sync(7, kWsThreads);
    }
  };
  // row (relative to a.lo) of entry e of the listed rows
  auto list_row = [&](int e) -> long long {
    const int q = listed_row(s_tiles, s_mask, nt, e);
    return ((long long)cid + (long long)(q >> 3) * ncl) * 8 + (q & 7);
  };

  if (warp < kSeg) {
    // ------------------------------------------------------------------ compute warps
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    const int seg = warp, g = lane >> 2, kk = lane & 3;
    const unsigned a_off = smem_addr(stage0) + g * kRowB + seg * (kSteps * 4 * (int)sizeof(Q)) + kk * (int)sizeof(Q);
    int st = 0, pb = 0;
    unsigned phase = 0;
    if (screen) {
      // A operand of mma.m16n8k16: centres g and g + 8 of the round at the features this lane reads of a row, as
      // fp16 or X's 16-bit type (the k slots {2kk, 2kk+1} and {2kk+8, 2kk+9} of super-step s are features
      // 16s + 4kk + {0, 1} and {2, 3}: the same permutation of K for A and B)
      unsigned af[kSteps][4];
      {
        const long long p0 = centre(g), p1 = centre(g + kB);
        const Q* c0 = reinterpret_cast<const Q*>(a.X) + (size_t)p0 * a.d4 + seg * (kSteps * 4) + kk;
        const Q* c1 = reinterpret_cast<const Q*>(a.X) + (size_t)p1 * a.d4 + seg * (kSteps * 4) + kk;
#pragma unroll
        for (int s = 0; s < kSteps; ++s) {
          const Q v0 = __ldg(c0 + 4 * s), v1 = __ldg(c1 + 4 * s);
          if constexpr (X16) {   // the centres as they are (element 2j in the low half of word j)
            af[s][0] = v0.x;
            af[s][1] = v1.x;
            af[s][2] = v0.y;
            af[s][3] = v1.y;
          } else {
            af[s][0] = half2_bits(v0.x, v0.y);
            af[s][1] = half2_bits(v1.x, v1.y);
            af[s][2] = half2_bits(v0.z, v0.w);
            af[s][3] = half2_bits(v1.z, v1.w);
          }
        }
      }
      const unsigned h_off = smem_addr(stage0) + g * kRowBytesH + seg * (kSteps * 32) + kk * 8;
      const unsigned my_partf = smem_addr(&s_part[0][seg][0]) + lane * 16;
      // a stage holds tiles k and k + 1 (rows 0-7, 8-15); with n1 odd the last stage's second half repeats tile k
      for (int k = 0; k < n1; k += 2) {
        mbar_wait(&full[st], phase);
        const unsigned ap = h_off + st * kStageBytesX;
        float d[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
        for (int s = 0; s < kSteps; ++s) {
          mma_f16<T>(d[0], af[s], lds64(ap + s * 32));
          mma_f16<T>(d[1], af[s], lds64(ap + 8 * kRowBytesH + s * 32));
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);
        if (++st == kStagesX) {
          st = 0;
          phase ^= 1u;
        }
        // one partial buffer per tile, as the epilogue warps expect them
        for (int h = 0; h < 2 && k + h < n1; ++h) {
          if (k + h >= kPartBufs) named_sync(1 + kPartBufs + pb, kSeg * 32 + 32);
          // lane (g,kk): centre g at rows 2kk, 2kk+1, centre g+8 at rows 2kk, 2kk+1
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(my_partf + pb * (unsigned)(sizeof(double) * kSeg * 64)),
                       "f"(d[h][0]), "f"(d[h][1]), "f"(d[h][2]), "f"(d[h][3])
                       : "memory");
          asm volatile("fence.acq_rel.cta;" ::: "memory");
          named_arrive(1 + pb, kSeg * 32 + 32);
          if (++pb == kPartBufs) pb = 0;
        }
      }
      screen_join();
      pb = 0;
    }
    const int nd = screen == 1 ? (s_na[2] + 7) / 8 : na;   // DMMA tiles
    double breg[kSteps][4];
    centre_slice(static_cast<const T*>(a.X), a.d4, centre(kB * crank + g), seg, kk, breg);
    const unsigned my_part = smem_addr(&s_part[0][seg][lane * 2]);
    for (int k = 0; k < nd; ++k) {
      mbar_wait(&full[st], phase);
      const unsigned ap = a_off + st * kStageBytesX;
      double c[4][2];
#pragma unroll
      for (int e = 0; e < 4; ++e) c[e][0] = c[e][1] = 0.0;
#pragma unroll
      for (int s = 0; s < kSteps; ++s) seg_step(c, lds_quad<T>(ap + s * 4 * (unsigned)sizeof(Q)), breg[s]);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[st]);          // this warp has read its slice of the stage
      if (++st == kStagesX) {
        st = 0;
        phase ^= 1u;
      }
      if (k >= kPartBufs) named_sync(1 + kPartBufs + pb, kSeg * 32 + 32);   // buffer released by its epilogue warp
      // lane (g,kk) holds (row g, centres 2kk, 2kk+1)
      const double2 part = seg_partial(c);
      asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(my_part + pb * (unsigned)(sizeof(double) * kSeg * 64)),
                   "d"(part.x), "d"(part.y) : "memory");
      asm volatile("fence.acq_rel.cta;" ::: "memory");   // partials visible before the arrive is counted
      named_arrive(1 + pb, kSeg * 32 + 32);
      if (++pb == kPartBufs) pb = 0;
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == kSeg) {
      // ---------------------------------------------------------------- producer warp
      // lane r < 8 copies row r of every tile; rows past the end re-read the last row
      int st = 0, fills = 0;
      unsigned phase = 0;
      auto fill = [&](auto row_of_lane) {
        if (fills++ >= kStagesX) mbar_wait(&empty[st], phase ^ 1u);   // the stage's previous tile was released
        if (lane == 0) mbar_expect_tx(&full[st], 8u * kXRowBytes);
        __syncwarp();
        if (lane < 8) {
          const long long row = row_of_lane();
          tma_load_1d(stage0 + (size_t)st * kStageBytesX + lane * kRowB, static_cast<const T*>(a.X) + (size_t)row * kFastD,
                      kXRowBytes, &full[st]);
        }
        if (++st == kStagesX) {
          st = 0;
          phase ^= 1u;
        }
      };
      if (screen) {
        // two tiles of this CTA's parity per stage, 16-bit rows of 4 KB (the fp16 copy, or a 16-bit X itself): lane
        // r < 16 copies row r & 7 of the first (r < 8) or second tile; a lone last tile fills both halves
        auto fill_half = [&](int k0, int k1) {
          if (fills++ >= kStagesX) mbar_wait(&empty[st], phase ^ 1u);
          if (lane == 0) mbar_expect_tx(&full[st], 16u * 2048u * 2u);
          __syncwarp();
          if (lane < 16) {
            const int k = lane < 8 ? k0 : k1;
            const long long row = min(((long long)cid + (long long)k * ncl) * 8 + (lane & 7), a.hi - a.lo - 1);   // relative to a.lo
            tma_load_1d(stage0 + (size_t)st * kStageBytesX + lane * kRowBytesH, a.Xh + (size_t)row * 2048, 2048u * 2u, &full[st]);
          }
          if (++st == kStagesX) {
            st = 0;
            phase ^= 1u;
          }
        };
        int held = -1;
        for (int j = 0; j < na; ++j) {
          const int k = tile_of(j);
          if ((k & 1) != crank) continue;
          if (held < 0) {
            held = k;
          } else {
            fill_half(held, k);
            held = -1;
          }
        }
        if (held >= 0) fill_half(held, held);
        screen_join();
      }
      if (screen == 1) {
        const int nl = s_na[2];
        for (int j = 0; j < (nl + 7) / 8; ++j) fill([&]() { return a.lo + list_row(min(j * 8 + lane, nl - 1)); });
      } else {
        for (int j = 0; j < na; ++j) {
          const int k = tile_of(j);
          fill([&]() {
            if (FILTER) return a.lo + a.seg_start[min((int)(((long long)cid + (long long)k * ncl) * 8 + lane), nseg - 1)];   // anchor rows
            return min(a.lo + ((long long)cid + (long long)k * ncl) * 8 + lane, a.hi - 1);
          });
        }
      }
    } else {
      // ---------------------------------------------------------------- epilogue warps
      const int ew = warp - kSeg - 1;             // partial buffer of this warp: tiles k = ew, ew+3, ...
      const int r = lane >> 2;                    // lane (r,kk): row r, centres 2kk, 2kk+1 (the DMMA C layout)
      if (screen) {
        // lane (r, q): row r of the tile against centres q, q+4, q+8, q+12
        const int q = lane & 3;
        const float* sf = reinterpret_cast<const float*>(&s_part[ew][0][0]);
        unsigned long long n_rows = 0, n_listed = 0;
        for (int j = 0, jj = 0; j < na; ++j) {
          const int k = tile_of(j);
          if ((k & 1) != crank) continue;
          if (jj++ % kPartBufs != ew) continue;
          const long long i = a.lo + ((long long)cid + (long long)k * ncl) * 8 + r;
          const bool valid = i < a.hi;
          const long long ic = valid ? i : a.hi - 1;
          const double xxi = a.xx[ic], m_old = a.m[ic];
          named_sync(1 + ew, kSeg * 32 + 32);
          double S[4];
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const int c = q + 4 * c4;
            const int at = ((c & 7) * 4 + (r >> 1)) * 4 + ((c >> 3) << 1) + (r & 1);
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < kSeg; ++w) s += (double)sf[w * 128 + at];
            S[c4] = s;
          }
          if (jj - 1 + kPartBufs < n1) named_arrive(1 + kPartBufs + ew, kSeg * 32 + 32);
          const double nx = sqrt(xxi), m2 = __dmul_ru(m_old, m_old);
          bool und = !isfinite(m_old);
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const int c = q + 4 * c4;
            const double xs = xxi + s_xxc[c];
            const double t = xs - 2.0 * S[c4];
            const double E = X16 ? 2.0 * kScreenU16 * nx * s_nc[c] + kScreenAbs * xs + kScreenAbs16 * (1.0 + nx + s_nc[c])
                                 : 2.0 * kScreenU * nx * s_nc[c] + kScreenAbs * xs + kScreenAbs1 * (nx + s_nc[c]);
            und = und || !(isfinite(S[c4]) && t - 2.0 * E > m2) || s_pick[c] == i;
          }
          const unsigned ub = __ballot_sync(0xffffffffu, und && valid);
          unsigned byte = 0;
#pragma unroll
          for (int rr = 0; rr < 8; ++rr)
            if ((ub >> (4 * rr)) & 0xfu) byte |= 1u << rr;
          if (lane == 0) {
            s_mask[k] = (unsigned char)byte;
            n_rows += (unsigned long long)min(8LL, a.hi - (a.lo + ((long long)cid + (long long)k * ncl) * 8));
            n_listed += __popc(byte);
          }
        }
        if (lane == 0 && a.screen_stats && n_rows) {
          atomicAdd(&a.screen_stats[0], n_rows);
          atomicAdd(&a.screen_stats[1], n_listed);
        }
        screen_join();
      }
      const int nl = screen == 1 ? s_na[2] : 0;
      const int nd = screen == 1 ? (nl + 7) / 8 : na;
      for (int j = ew; j < nd; j += kPartBufs) {
        named_sync(1 + ew, kSeg * 32 + 32);
        const double dot0 = combine8(&s_part[ew][0][lane * 2], 64);
        const double dot1 = combine8(&s_part[ew][0][lane * 2 + 1], 64);
        if (j + kPartBufs < nd) named_arrive(1 + kPartBufs + ew, kSeg * 32 + 32);   // partials consumed
        if (screen == 1) {
          if (j * 8 + r < nl)
            *reinterpret_cast<double2*>(a.dots + list_row(j * 8 + r) * NC + crank * kB + (lane & 3) * 2) = make_double2(dot0, dot1);
          continue;
        }
        const int k = tile_of(j);
        const long long row = ((long long)cid + (long long)k * ncl) * 8 + r;   // relative to a.lo (FILTER: segment id)
        if (FILTER) {
          // segment `row`: nearest of this group's centres to its anchor, largest min_d of its rows, the test of
          // "pruning (exact)" below, on the pass's tile machine
          const int kk = lane & 3, sg = (int)min(row, (long long)nseg - 1);
          const int a0 = a.seg_start[sg], e0 = a.seg_start[sg + 1];
          const double xxa = a.xx[a.lo + a0];
          double sq = fmin(sq_from_dot(dot0, xxa, s_xxc[crank * kB + 2 * kk]), sq_from_dot(dot1, xxa, s_xxc[crank * kB + 2 * kk + 1]));
          double M = 0.0;
          for (int q = a0 + kk; q < e0; q += 4) M = fmax(M, a.m[a.lo + q]);
          sq = fmin(sq, __shfl_xor_sync(0xffffffffu, sq, 1));
          sq = fmin(sq, __shfl_xor_sync(0xffffffffu, sq, 2));
          M = fmax(M, __shfl_xor_sync(0xffffffffu, M, 1));
          M = fmax(M, __shfl_xor_sync(0xffffffffu, M, 2));
          if (kk == 0 && row < nseg) {
            double cn = 0.0;
#pragma unroll
            for (int jc = 0; jc < kB; ++jc) cn = fmax(cn, s_xxc[crank * kB + jc]);
            a.seg_skip_out[(size_t)crank * a.skip_stride + row] = segment_skip(sq, a.seg_r[row], M, xxa, cn) ? 1 : 0;
          }
        } else if (a.lo + row < a.hi) {
          *reinterpret_cast<double2*>(a.dots + row * NC + crank * kB + (lane & 3) * 2) = make_double2(dot0, dot1);
        }
      }
      if (PAIR && !FILTER) __threadfence();       // the partner CTA reads these dot products
    }
  }
  // ---- apply phase: the walker's own rows (their dot products were written by its own epilogue
  // warps, visible after the barrier), one row per compute-warpgroup thread at a time; a pair splits
  // its rows by tile parity after the cluster barrier that makes both CTAs' dot products visible
  __syncthreads();
  if (FILTER) return;                             // flags written; no rows to finish
  if (PAIR) cluster_sync_all();
  if (clocked) tq2 = gtime_ns();
  Best best{-INFINITY, 0x7fffffffffffffffLL};
  const ApplyConst ac = apply_const(a, final_pass);
  if (warp < kSeg) {
    // this CTA's tiles: every tile of the walker (solo) or the tiles of its parity (pair), rows dealt densely to the
    // lanes (a warp covers four whole tiles: 128 contiguous bytes of dot products per lane)
    const int own_tiles = PAIR ? (nt + 1 - crank) / 2 : nt;
    const int nrows = own_tiles * 8;
    int inwin = 0;
    for (int q0 = warp * 32; q0 < nrows; q0 += kSeg * 32) {      // (uniform trip count per warp)
      const int q = q0 + lane;
      int bin = -1;
      if (q < nrows) {
        const int k = PAIR ? 2 * (q >> 3) + crank : (q >> 3);
        const long long i = a.lo + ((long long)cid + (long long)k * ncl) * 8 + (q & 7);
        int tile_mode = (use_list && ((s_flagged[k >> 5] >> (k & 31)) & 1u)) ? a.prune_mode : 0;
        // a row the screen decided: no dot products (list mode) or a verify count
        if (screen && !((s_mask[k] >> (q & 7)) & 1u)) tile_mode = (screen == 1) ? 1 : (tile_mode ? tile_mode : 3);
        if (i < a.hi) bin = apply_row<NC>(a, ac, i, s_xxc, s_pick, best, tile_mode);
      }
      if (ac.do_hist) {                                            // one shared atomic per distinct bin per warp
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0) {
          if (lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], (unsigned)__popc(peers));
          inwin += 1;
        }
      }
    }
    if (ac.do_hist) {
      inwin = warp_sum(inwin);
      if (lane == 0 && inwin) atomicAdd(&s_hist[kNB], (unsigned)inwin);
    }
  }
  __syncthreads();
  if (clocked) tq3 = gtime_ns();
  publish_pass(a, best, ac.do_hist, s_hist, final_pass);
  if (clocked) {
    a.ctl->stat_ns_pass[0] += tq1 - tq0;
    a.ctl->stat_ns_pass[1] += tq2 - tq1;
    a.ctl->stat_ns_pass[2] += tq3 - tq2;
    a.ctl->stat_ns_pass[3] += gtime_ns() - tq3;
  }
}

// ---------------------------------------------------------------- pruning (exact)
// Pools are id-sorted video tracks, so consecutive rows of X are near each other.  The owned rows
// are cut into SEGMENTS (a new one wherever the distance between consecutive rows exceeds twice
// its mean, and at least every kSegMax rows); segment s has an anchor row a_s (its first) and a
// radius R_s = max_i d(a_s, i).  For a new centre c the triangle inequality gives, for every
// row i of the segment,  d(i,c) >= d(a_s,c) - R_s,  so when
//     min_j d(a_s, c_j) - R_s  >=  max_{i in s} min_d[i] + margin
// no row of the segment can get closer to any centre c_j of this pass: min(min_d, d) leaves every
// min_d untouched and the rows need not be streamed.  `margin` (1e-6 x the norms involved) is
// orders of magnitude above the rounding of the canonical fp64 distances (<= ~5e-7 at d -> 0), so
// the pruned pass writes exactly the bits the full pass would: the pick list cannot change.  A
// picked row is never pruned (its own segment has d(a_s,c) <= R_s).  VATLQ_PRUNE=verify streams
// everything and counts rows of flagged tiles whose min_d moved (tests assert 0).
// The flags come from the FILTER mode of pass_kernel_tma: its tiles are 8 anchor rows, and its epilogue takes the
// canonical distances of each anchor to the group's 8 centres, the largest min_d of the segment's rows and the test.
// Every group of a round is flagged before the round's first pass: the largest min_d a later group reads can only
// be larger than what its pass will see, so its flags stay exact.
constexpr int kSegMax = 64;   // longest segment (rows): bounds the min_d reads of the filter per segment
struct PruneCtl {
  double sum;                      // sum of the finite consecutive-row distances
  unsigned long long cnt;
  int nseg, pad;
  unsigned long long stats[3];     // tiles seen, tiles streamed, verify violations (PassArgs::prune_stats)
  unsigned long long screen[3];    // rows screened, rows listed, verify violations (PassArgs::screen_stats)
};

// squared distance of two rows as sum((x-y)^2) in fp64 (every lane returns the warp total)
template <typename T>
__device__ __forceinline__ double warp_sqdist(const quad_t<T>* __restrict__ x, const quad_t<T>* __restrict__ y, int d4, int lane) {
  double acc = 0.0;
  for (int c = lane; c < d4; c += 32) {
    const float4 u = ldg_q<T>(x + c), v = ldg_q<T>(y + c);
    const double a0 = (double)u.x - (double)v.x, a1 = (double)u.y - (double)v.y;
    const double a2 = (double)u.z - (double)v.z, a3 = (double)u.w - (double)v.w;
    acc = fma(a0, a0, acc);
    acc = fma(a1, a1, acc);
    acc = fma(a2, a2, acc);
    acc = fma(a3, a3, acc);
  }
  return warp_sum(acc);
}

// cd[r] = d(row lo+r-1, row lo+r) for r >= 1 (cd[0] = +inf), and their sum / count
template <typename T>
__global__ void __launch_bounds__(256) consec_kernel(const T* __restrict__ X, int d4, long long lo, long long hi,
                                                     double* __restrict__ cd, PruneCtl* pc) {
  const int lane = threadIdx.x & 31;
  const long long w0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const quad_t<T>* X4 = reinterpret_cast<const quad_t<T>*>(X);
  double local = 0.0;
  unsigned long long cnt = 0;
  for (long long r = w0; r < hi - lo; r += nwarps) {
    double dist = INFINITY;
    if (r > 0) {
      dist = sqrt(warp_sqdist<T>(X4 + (size_t)(lo + r) * d4, X4 + (size_t)(lo + r - 1) * d4, d4, lane));
      if (isfinite(dist)) {
        local += dist;
        cnt += 1;
      }
    }
    if (lane == 0) cd[r] = dist;
  }
  if (lane == 0 && cnt) {
    atomicAdd(&pc->sum, local);
    atomicAdd(&pc->cnt, cnt);
  }
}

// one CTA: segment ids from the cuts (cd > 2 x mean, or kSegMax rows since the last cut)
__global__ void __launch_bounds__(1024) segment_kernel(const double* __restrict__ cd, int n, PruneCtl* pc,
                                                       int* __restrict__ seg_of_row, int* __restrict__ seg_start) {
  __shared__ int s_a[1024], s_b[1024];
  const int t = threadIdx.x, T = blockDim.x;
  const int per = (n + T - 1) / T;
  const int r0 = min(n, t * per), r1 = min(n, r0 + per);
  const double tau = pc->cnt ? 2.0 * pc->sum / (double)pc->cnt : INFINITY;
  int last = -1;
  for (int i = r0; i < r1; ++i)
    if (i == 0 || cd[i] > tau) last = i;
  s_a[t] = last;
  __syncthreads();
  for (int off = 1; off < T; off <<= 1) {   // inclusive max-scan: last threshold cut at or before the chunk
    const int v = (t >= off) ? s_a[t - off] : -1;
    __syncthreads();
    s_a[t] = max(s_a[t], v);
    __syncthreads();
  }
  const int run_in = (t > 0) ? s_a[t - 1] : -1;
  int cnt = 0, rs = run_in;
  for (int i = r0; i < r1; ++i) {
    bool cut = (i == 0 || cd[i] > tau);
    if (cut) rs = i;
    else cut = ((i - rs) % kSegMax) == 0;
    cnt += cut ? 1 : 0;
  }
  s_b[t] = cnt;
  __syncthreads();
  for (int off = 1; off < T; off <<= 1) {   // inclusive sum-scan of the cut counts
    const int v = (t >= off) ? s_b[t - off] : 0;
    __syncthreads();
    s_b[t] += v;
    __syncthreads();
  }
  int id = ((t > 0) ? s_b[t - 1] : 0) - 1;
  rs = run_in;
  for (int i = r0; i < r1; ++i) {
    bool cut = (i == 0 || cd[i] > tau);
    if (cut) rs = i;
    else cut = ((i - rs) % kSegMax) == 0;
    if (cut) {
      ++id;
      seg_start[id] = i;
    }
    seg_of_row[i] = id;
  }
  if (t == T - 1) {
    pc->nseg = s_b[T - 1];
    seg_start[s_b[T - 1]] = n;
  }
}

// R_s = max_i d(anchor_s, i): one warp per segment
template <typename T>
__global__ void __launch_bounds__(256) seg_radius_kernel(const T* __restrict__ X, int d4, long long lo,
                                                         const int* __restrict__ seg_start, const PruneCtl* pc,
                                                         double* __restrict__ segR) {
  const int lane = threadIdx.x & 31;
  const int w0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const quad_t<T>* X4 = reinterpret_cast<const quad_t<T>*>(X);
  const int nseg = pc->nseg;
  for (int sg = w0; sg < nseg; sg += nwarps) {
    const int a = seg_start[sg], e = seg_start[sg + 1];
    double R = 0.0;
    for (int r = a + 1; r < e; ++r)
      R = fmax(R, sqrt(warp_sqdist<T>(X4 + (size_t)(lo + r) * d4, X4 + (size_t)(lo + a) * d4, d4, lane)));
    if (lane == 0) segR[sg] = R;
  }
}

static size_t pass_smem_bytes(int S) {
  return (size_t)kB * S * sizeof(double) + kB * sizeof(double) + (size_t)kTeams * 2 * kSeg * 64 * sizeof(double) +
         kB * sizeof(long long) + (kNB + 1) * sizeof(unsigned int);
}


// ---------------------------------------------------------------- initial scores
__global__ void __launch_bounds__(256) score_init_kernel(long long lo, long long hi, const double* __restrict__ m,
                                                         const double* __restrict__ unc, double* __restrict__ score,
                                                         const Ctl* ctl) {
  const long long i = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hi) return;
  score[i] = ctl->first_round ? unc[i] : score_of(ctl->rule, ctl->wd, ctl->wu, m[i], unc[i]);
}

// ---------------------------------------------------------------- bootstrap: arg-max of the initial scores
// Only before the first round: afterwards every pass leaves the block header behind itself.
__global__ void __launch_bounds__(256) bootstrap_kernel(long long lo, long long hi, const double* __restrict__ score,
                                                        Best* partial, RankBlock* out, Ctl* ctl, PushArgs push) {
  Best best{-INFINITY, 0x7fffffffffffffffLL};
  for (long long i = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (long long)gridDim.x * blockDim.x) {
    const double s = score[i];
    if (better(s, i, best.s, best.i)) {
      best.s = s;
      best.i = i;
    }
  }
  publish_header(8, best, partial, ctl, out, push, INFINITY, 0, nullptr, true);   // (256 threads) no list, exact arg-max
}

// ---------------------------------------------------------------- candidate bookkeeping
struct CandView {
  int total;        // candidates over all ranks (records actually stored)
  int fallback;     // 0 plan on candidates, 1 nothing listed, 2 overflow, 3 no list was requested
  double theta;     // max over ranks
  int start[kMaxRanks + 1];
};
__device__ __forceinline__ CandView view_of(const RankBlock* blocks, int world) {
  CandView v;
  v.total = 0;
  v.fallback = 0;
  v.theta = -INFINITY;
  bool overflow = false, unlisted = false;
  for (int r = 0; r < world; ++r) {
    v.start[r] = v.total;
    const long long c = blocks[r].count;
    if (c > kCapL || blocks[r].mode == 2) overflow = true;
    if (blocks[r].mode == 0) unlisted = true;
    v.total += (int)min(c, (long long)kCapL);
    v.theta = fmax(v.theta, blocks[r].theta);
  }
  v.start[world] = v.total;
  if (overflow || v.total > kCap) v.fallback = 2;
  else if (unlisted || isinf(v.theta)) v.fallback = 3;
  else if (v.total == 0) v.fallback = 1;
  return v;
}
__device__ __forceinline__ void locate(const CandView& v, int world, int pos, int& r, int& s) {
  r = 0;
  while (r + 1 < world && pos >= v.start[r + 1]) ++r;
  s = pos - v.start[r];
}

// ---------------------------------------------------------------- candidate x candidate distances
template <typename T>
__global__ void __launch_bounds__(256) pairs_kernel(const T* __restrict__ X, int d4, int nss, int S, int guard,
                                                    const double* __restrict__ xx, const RankBlock* blocks,
                                                    const Ctl* ctl, double* __restrict__ Dcc) {
  if (ctl->n_picked >= ctl->k) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double s_xxc[kB];
  const int world = ctl->world;
  const CandView v = view_of(blocks, world);
  if (v.fallback) return;
  const int col0 = blockIdx.x * kB;
  if (col0 >= v.total) return;
  double* s_c = reinterpret_cast<double*>(smem_raw);
  for (int j = 0; j < kB; ++j) {
    int r, s;
    locate(v, world, min(col0 + j, v.total - 1), r, s);
    const long long p = blocks[r].idx[s];
    stage_center(X, d4, nss * 16, S, p, j, s_c);
    if (threadIdx.x == 0) s_xxc[j] = xx[p];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5, g = lane >> 2, kk = lane & 3;
  const quad_t<T>* X4 = reinterpret_cast<const quad_t<T>*>(X);
  for (int r0 = (blockIdx.y * nwarp + warp) * 8; r0 < v.total; r0 += gridDim.y * nwarp * 8) {
    const int pos = min(r0 + g, v.total - 1);
    int rr, ss;
    locate(v, world, pos, rr, ss);
    const long long ridx = blocks[rr].idx[ss];
    double c[2];
    if (guard) dmma_block<true, false, T>(X4 + (size_t)ridx * d4, d4, nss, s_c, S, lane, c);
    else dmma_block<false, false, T>(X4 + (size_t)ridx * d4, d4, nss, s_c, S, lane, c);
    if (r0 + g < v.total) {
      const double xxi = xx[ridx];
#pragma unroll
      for (int e = 0; e < 2; ++e) {   // Dcc[w * kCap + c] = d(row c, centre w): stored by CENTRE so that the planner reads a row
        const int col = col0 + 2 * kk + e;
        if (col < v.total) Dcc[(size_t)col * kCap + (r0 + g)] = dist_from_dot(c[e], xxi, s_xxc[2 * kk + e]);
      }
    }
  }
}

__device__ void plan_body(const RankBlock* blocks, RankBlock* send, const double* Dcc, unsigned int* hist,
                          long long* out_idx, Ctl* ctl, double* s_D = nullptr, int s_D_cap = 0);

// Candidate x candidate distances, symmetric: only the tile pairs (column block cb <= row tile t) are computed and
// every 8 x 8 block is written twice (d is symmetric; both halves hold the SAME bits, so the planner may read rows).
// The pairs are dealt round-robin to the CTAs of the grid: with ~250 candidates that is 528 pairs over 148 CTAs
// (3-4 each, all loads of a pair in flight together) instead of 8 sequential tiles per CTA on a quarter of the SMs.
template <typename T>
__device__ __forceinline__ void pairs_tiles(const T* __restrict__ X, int d4, const double* __restrict__ xx,
                                            const RankBlock* blocks, const CandView& v, int world,
                                            double* __restrict__ Dcc, double (*s_part)[kSeg][64], double* s_xxc) {
  const int lane = threadIdx.x & 31, seg = threadIdx.x >> 5, g = lane >> 2, kk = lane & 3;
  const quad_t<T>* X4 = reinterpret_cast<const quad_t<T>*>(X);
  const int lane_off = seg * (kSteps * 4) + kk;
  auto cand_row = [&](int pos) {
    int r, q;
    locate(v, world, min(pos, v.total - 1), r, q);
    return blocks[r].idx[q];
  };
  const int nt = (v.total + 7) / 8;
  const int npairs = nt * (nt + 1) / 2;
  const int ncta = gridDim.x * gridDim.y, cta = blockIdx.y * gridDim.x + blockIdx.x;
  int buf = 0;
  for (int p = cta; p < npairs; p += ncta) {
    int cb = 0, q = p;                                   // p -> (cb, t), cb <= t
    while (q >= nt - cb) {
      q -= nt - cb;
      ++cb;
    }
    const int t = cb + q, col0 = cb * kB;
    // both operand tiles are requested back to back: one memory round trip per pair
    const long long crow = cand_row(col0 + g), arow = cand_row(t * 8 + g);
    const quad_t<T>* cp = X4 + (size_t)crow * d4 + lane_off;
    const quad_t<T>* ap = X4 + (size_t)arow * d4 + lane_off;
    float4 cb4[kSteps], ring[kSteps];
#pragma unroll
    for (int s = 0; s < kSteps; ++s) cb4[s] = ldg_q<T>(cp + 4 * s);
#pragma unroll
    for (int s = 0; s < kSteps; ++s) ring[s] = ldg_q<T>(ap + 4 * s);
    if (threadIdx.x < kB) s_xxc[buf * kB + threadIdx.x] = xx[cand_row(col0 + threadIdx.x)];
    const int myrow = t * 8 + seg;                       // the row this warp finishes
    const double xxi = (myrow < v.total) ? xx[cand_row(myrow)] : 0.0;
    double c[4][2];
#pragma unroll
    for (int e = 0; e < 4; ++e) c[e][0] = c[e][1] = 0.0;
#pragma unroll
    for (int s = 0; s < kSteps; ++s) seg_step(c, ring[s], cb4[s]);
    *reinterpret_cast<double2*>(&s_part[buf][seg][lane * 2]) = seg_partial(c);
    __syncthreads();
    if (myrow < v.total && lane < kB && col0 + lane < v.total) {
      // Dcc[w * kCap + c] = d(row c, centre w) with the pass's operand roles (sklearn: (-2 x.c + |x|^2) + |c|^2, the
      // two norms are NOT interchangeable in the last bit): the dot product is symmetric bit for bit (same products,
      // same order), so one tile yields both orientations exactly.  The planner reads row w = the picked centre.
      const double dot = combine8(&s_part[buf][0][seg * 8 + lane], 64);
      const double xxo = s_xxc[buf * kB + lane];
      Dcc[(size_t)(col0 + lane) * kCap + myrow] = dist_from_dot(dot, xxi, xxo);   // row = myrow,   centre = col
      Dcc[(size_t)myrow * kCap + col0 + lane] = dist_from_dot(dot, xxo, xxi);     // row = col,     centre = myrow
    }
    buf ^= 1;
  }
}

// fast path (d == kFastD): the pass kernel's tile machine on the gathered candidates.
// CTA (cb, y): the 8 candidates of column block cb are the centres (their 1/8 K-slices live in the
// registers of the 8 warps), row tiles y, y + gridDim.y, ... of the candidate list stream through
// a register ring (from L2 mostly: the rows were just touched by the pass).  After the split-K
// exchange warp w finishes row w of the tile: lane j writes d(row, centre j).
// The last CTA of the grid to finish runs the planner (plan_body) on the completed matrix, so a
// round needs no separate plan launch.
constexpr int kPlanSmem = 208 * 1024;    // dynamic shared memory of pairs_plan_kernel: the planner's staged distance rows
template <typename T>
__global__ void __launch_bounds__(kSeg * 32, 1) pairs_plan_kernel(const T* __restrict__ X, int d4,
                                                                  const double* __restrict__ xx, const RankBlock* blocks,
                                                                  RankBlock* send, unsigned int* hist, long long* out_idx,
                                                                  Ctl* ctl, double* __restrict__ Dcc, Mailbox* mail,
                                                                  unsigned long long seq, int plan_smem_doubles) {
  __shared__ __align__(16) double s_part[2][kSeg][64];
  __shared__ double s_xxc[2 * kB];
  __shared__ unsigned int s_last;
  pdl_enter();
  if (ctl->n_picked >= ctl->k) {       // (uniform over the grid: nobody takes a ticket)
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) ctl->nb = 0;
    return;
  }
  unsigned long long t0 = 0, t1 = 0;
  const bool clocked = blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0;
  if (clocked) t0 = gtime_ns();
  if (mail != nullptr) {               // peer-memory exchange: the blocks of this round land in the local mailbox
    if (threadIdx.x == 0) wait_blocks(mail, ctl->world, seq);
    __syncthreads();
  }
  if (clocked) {
    t1 = gtime_ns();
    ctl->t_start = t1;
    ctl->stat_ns_wait += t1 - t0;
  }
  {
    const int world = ctl->world;
    const CandView v = view_of(blocks, world);
    if (!v.fallback) pairs_tiles<T>(X, d4, xx, blocks, v, world, Dcc, s_part, s_xxc);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int total = gridDim.x * gridDim.y;
    s_last = (atomicAdd(&ctl->pairs_ticket, 1u) == total - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    unsigned long long t2 = 0;
    if (threadIdx.x == 0) {
      ctl->pairs_ticket = 0;
      t2 = gtime_ns();
      ctl->stat_ns_tiles += t2 - *((volatile unsigned long long*)&ctl->t_start);
    }
    extern __shared__ __align__(16) double s_plan_dyn[];
    plan_body(blocks, send, Dcc, hist, out_idx, ctl, s_plan_dyn, plan_smem_doubles);
    __syncthreads();
    if (threadIdx.x == 0) ctl->stat_ns_plan += gtime_ns() - t2;
  }
}

// exact global argmax from the per-rank headers: always the correct next greedy pick
__device__ void fallback_pick(const RankBlock* blocks, int world, int kind, RankBlock* send,
                              long long* __restrict__ out_idx, Ctl* ctl) {
  Best b{-INFINITY, 0x7fffffffffffffffLL};
  for (int r = 0; r < world; ++r) {
    if (better(blocks[r].smax, blocks[r].smax_idx, b.s, b.i)) {
      b.s = blocks[r].smax;
      b.i = blocks[r].smax_idx;
    }
  }
  ctl->picks[0] = b.i;
  ctl->nb = 1;
  out_idx[ctl->n_picked] = b.i;
  ctl->n_picked += 1;
  ctl->stat_rounds += 1;
  if (ctl->first_round) {
    // the score changes meaning after the first pick (unc -> distance mix): no bound yet
    ctl->first_round = 0;
    ctl->U = 0.0;
    ctl->W = -1.0;  // next round: plain argmax again, then U = smax
  } else if (ctl->maxb > 1) {
    double W = ctl->W;
    ctl->U = b.s;  // scores only decrease
    if (kind == 2) {
      ctl->stat_fallback_overflow += 1;
      W = (W > 0.0) ? W / 16.0 : b.s / 64.0;
    } else if (kind == 1) {
      ctl->stat_fallback_empty += 1;
      W = (W > 0.0) ? fmin(b.s, W * 4.0) : b.s / 64.0;
    } else if (!(W > 0.0)) {   // kind 3: no list was requested yet -> open the first window
      W = b.s / 64.0;
    }
    if (!(W > 0.0)) W = b.s;
    ctl->W = W;
  }
  send->count = 0;
}

// ---------------------------------------------------------------- the planner: exact greedy on candidates
// theta for the list the NEXT pass emits, from the histogram the PREVIOUS pass left behind
// (scores only decrease, so the real list can only be shorter than the histogram says): the
// highest bin edge whose suffix count reaches the target, raised until the list fits a block.
// Called by the first 256 threads of the CTA with block-wide barriers around it.
__device__ void choose_theta(const unsigned int* __restrict__ hist, double U, double W, int target, int tid,
                             double* s_theta, int* s_mode) {
  __shared__ unsigned int s_wtot[8];
  __shared__ int s_bstar[8], s_bfit[8];
  if (tid < 256) {
    const int lane = tid & 31, wp = tid >> 5;
    unsigned int h[4], tot = 0;
#pragma unroll
    for (int c = 3; c >= 0; --c) {
      tot += hist[tid * 4 + c];
      h[c] = tot;                    // bins c..3 of this thread's chunk
    }
    unsigned int v = tot;            // inclusive suffix over the lanes of this warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int t = __shfl_down_sync(0xffffffffu, v, o);
      if (lane + o < 32) v += t;
    }
    if (lane == 0) s_wtot[wp] = v;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    unsigned int run = v - tot;      // rows in bins of higher-indexed threads
    for (int w = wp + 1; w < 8; ++w) run += s_wtot[w];
    int bstar = -1;                  // highest bin whose suffix count reaches the target
    int bfit = kNB;                  // lowest bin whose suffix count still fits the record capacity
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const unsigned int cum = run + h[e];
      if (cum >= (unsigned)target) bstar = max(bstar, tid * 4 + e);
      if (cum <= (unsigned)kCapL) bfit = min(bfit, tid * 4 + e);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      bstar = max(bstar, __shfl_xor_sync(0xffffffffu, bstar, o));
      bfit = min(bfit, __shfl_xor_sync(0xffffffffu, bfit, o));
    }
    if (lane == 0) {
      s_bstar[wp] = bstar;
      s_bfit[wp] = bfit;
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (tid == 0) {
      for (int w = 1; w < 8; ++w) {
        bstar = max(bstar, s_bstar[w]);
        bfit = min(bfit, s_bfit[w]);
      }
      if (bstar < 0) bstar = 0;
      if (bfit == kNB) {             // even the top bin overflows: exact-argmax rounds until the window shrinks
        *s_theta = INFINITY;
        *s_mode = 2;
      } else {
        const int bb = max(bstar, bfit);
        *s_theta = (bb == 0) ? (U - W) : (U - W) + (double)bb * (W / (double)kNB);
        *s_mode = 1;
      }
    }
  }
}

constexpr int kPlanThreads = 256;
constexpr int kPerThread = kCap / kPlanThreads;   // candidates per planner thread (strided: c = tid + 256 j)

// order-preserving 64-bit key of a (non-NaN) score: key(a) > key(b) <=> a > b; -0.0 and +0.0 share a key
__device__ __forceinline__ unsigned long long score_key(double s) {
  if (s == 0.0) s = 0.0;
  const unsigned long long b = (unsigned long long)__double_as_longlong(s);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ double key_score(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k));
}
// warp arg-max of (key, idx, pos): largest key, lowest idx on equal keys; every lane ends with the winner.
// idx < 2^32 - 1 (0xffffffff marks "no candidate")
__device__ __forceinline__ void warp_argmax_key(unsigned long long& key, unsigned& idx, int& pos) {
  const unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
  const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
  const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
  const bool top = hi == mh && lo == ml;
  const unsigned mi = __reduce_min_sync(0xffffffffu, top ? idx : 0xffffffffu);
  const unsigned holders = __ballot_sync(0xffffffffu, top && idx == mi);
  pos = __shfl_sync(0xffffffffu, pos, __ffs(holders) - 1);
  key = ((unsigned long long)mh << 32) | ml;
  idx = mi;
}

// s_D (optional, s_D_cap doubles of shared memory): the candidate x candidate distances of as many centre rows as
// fit are staged there with cp.async while the list is read, so that a pick's row costs a shared-memory read instead
// of an L2 round trip on the sequential pick chain (a list of <= 163 candidates fits whole in 208 KB)
__device__ void plan_body(const RankBlock* blocks, RankBlock* send, const double* Dcc, unsigned int* hist,
                          long long* out_idx, Ctl* ctl, double* s_D, int s_D_cap) {
  __shared__ Best s_b[2][8];
  __shared__ int s_pos[2][8];
  __shared__ unsigned long long s_key[2][8];
  __shared__ unsigned int s_idx[2][8];
  __shared__ double s_theta;
  __shared__ int s_mode;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (ctl->n_picked >= ctl->k) {
    if (tid == 0) ctl->nb = 0;
    return;
  }
  const int world = ctl->world;
  const unsigned long long tp_begin = (tid == 0) ? gtime_ns() : 0ULL;
  // ---- theta of the list the coming pass emits (window the histogram was built with: the
  // U, W this kernel has not updated yet), then clear the histogram for that pass
  {
    const double U0 = ctl->U, W0 = ctl->W;
    const bool windowed = W0 > 0.0 && ctl->maxb > 1 && !ctl->first_round;
    if (tid == 0) {
      s_theta = INFINITY;
      s_mode = 0;
    }
    __syncthreads();
    if (windowed) choose_theta(hist, U0, W0, max(1, ctl->target / max(1, world)), tid, &s_theta, &s_mode);
    __syncthreads();
    for (int k = tid; k < kNB + 1; k += blockDim.x) hist[k] = 0u;
    if (tid == 0) {
      ctl->theta_emit = s_theta;
      ctl->emit_mode = s_mode;
    }
  }
  unsigned long long tp0 = 0, tp1 = 0, tp2 = 0, tp3 = 0;
  if (tid == 0) tp1 = gtime_ns();
  const CandView v = view_of(blocks, world);
  const int rule = ctl->rule;
  const double wd = ctl->wd, wu = ctl->wu;
  const long long picked0 = ctl->n_picked;      // (constant until the tail: read ONCE — a load per pick would stall warp 0,
  const long long remaining = ctl->k - picked0; //  and with it every barrier of the pick chain, for an L2 round trip)
  const int maxpicks = (int)min((long long)(ctl->first_round ? 1 : min(kMaxPicks, ctl->maxb)), remaining);
  __syncthreads();   // every thread has read the block headers / ctl before thread 0 may change them
  if (v.fallback) {
    if (tid == 0) fallback_pick(blocks, world, v.fallback, send, out_idx, ctl);
    return;
  }
  // stage the rows of centres [0, staged) of Dcc (columns [0, total)), 16 bytes per cp.async
  const int dstride = (v.total + 1) & ~1;
  const int staged = (s_D != nullptr && dstride > 0) ? min(v.total, s_D_cap / dstride) : 0;
  {
    const int per_row = dstride >> 1;
    for (int q = tid; q < staged * per_row; q += kPlanThreads) {
      const int r = q / per_row, c2 = q - r * per_row;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(s_D + (size_t)r * dstride + 2 * c2)),
                   "l"(Dcc + (size_t)r * kCap + 2 * c2)
                   : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  // candidates c = tid + 256 j live in registers
  long long idx[kPerThread];
  double m[kPerThread], u[kPerThread], sc[kPerThread];
#pragma unroll
  for (int j = 0; j < kPerThread; ++j) {
    const int c = tid + kPlanThreads * j;
    idx[j] = 0x7fffffffffffffffLL;
    m[j] = 0.0;
    u[j] = 0.0;
    sc[j] = -INFINITY;
    if (c < v.total) {
      int r, q;
      locate(v, world, c, r, q);
      idx[j] = blocks[r].idx[q];
      m[j] = blocks[r].m[q];
      u[j] = blocks[r].unc[q];
      sc[j] = blocks[r].score[q];
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  if (tid == 0) tp2 = gtime_ns();
  int nb = 0;
  for (int b = 0; b < maxpicks; ++b) {
    // block arg-max on order-preserving integer keys (largest score, lowest row index on ties = better()): thread-local,
    // three redux.sync per warp, ONE barrier, every warp reduces the 8 warp winners the same way.  (The butterfly over
    // (fp64 score, int64 index) pairs it replaces spent ~0.8 us per pick in dependent fp64 compares and 64-bit shuffles.)
    unsigned long long mk = score_key(sc[0]);
    unsigned mi = (unsigned)idx[0];
    int pos = tid;
#pragma unroll
    for (int j = 1; j < kPerThread; ++j) {
      const unsigned long long kj = score_key(sc[j]);
      const unsigned ij = (unsigned)idx[j];
      if (kj > mk || (kj == mk && ij < mi)) {
        mk = kj;
        mi = ij;
        pos = tid + kPlanThreads * j;
      }
    }
    warp_argmax_key(mk, mi, pos);
    if (lane == 0) {
      s_key[b & 1][warp] = mk;
      s_idx[b & 1][warp] = mi;
      s_pos[b & 1][warp] = pos;
    }
    __syncthreads();
    unsigned long long wk = lane < 8 ? s_key[b & 1][lane] : 0ULL;
    unsigned wi = lane < 8 ? s_idx[b & 1][lane] : 0xffffffffu;
    int wpos = lane < 8 ? s_pos[b & 1][lane] : 0;
    warp_argmax_key(wk, wi, wpos);
    Best win{key_score(wk), wi == 0xffffffffu ? 0x7fffffffffffffffLL : (long long)wi};
    if (!(win.s >= v.theta)) {  // a non-candidate (score < theta) could be ahead now
      if (b == 0) {             // (only possible when the rank that set theta listed nothing)
        if (tid == 0) fallback_pick(blocks, world, 1, send, out_idx, ctl);
        return;
      }
      break;
    }
    if (tid == 0) {
      ctl->picks[nb] = win.i;
      out_idx[picked0 + nb] = win.i;
    }
    nb += 1;
    const double* drow = Dcc + (size_t)wpos * kCap;   // drow[c] = d(row c, centre = the winner), coalesced
    const double* srow = s_D + (size_t)wpos * dstride;
    const bool in_smem = wpos < staged;
#pragma unroll
    for (int j = 0; j < kPerThread; ++j) {
      const int c = tid + kPlanThreads * j;
      if (c < v.total) {
        m[j] = fmin(m[j], in_smem ? srow[c] : __ldcg(drow + c));
        if (c == wpos) u[j] = 0.0;
        sc[j] = score_of(rule, wd, wu, m[j], u[j]);
      }
    }
  }
  if (tid == 0) tp3 = gtime_ns();
  // best surviving candidate score -> upper bound of every score after the pass
  Best me{sc[0], idx[0]};
#pragma unroll
  for (int j = 1; j < kPerThread; ++j)
    if (better(sc[j], idx[j], me.s, me.i)) {
      me.s = sc[j];
      me.i = idx[j];
    }
  me = warp_best(me);
  __syncthreads();
  if (lane == 0) s_b[0][warp] = me;
  __syncthreads();
  if (tid == 0) {
    Best bb = s_b[0][0];
    for (int k = 1; k < 8; ++k)
      if (better(s_b[0][k].s, s_b[0][k].i, bb.s, bb.i)) bb = s_b[0][k];
    long long inwin = 0;
    for (int r = 0; r < world; ++r) inwin += blocks[r].inwin;
    const double U = ctl->U;
    double W = ctl->W;
    const double frac = (U - v.theta) / W;
    if (inwin < ctl->target) W = fmin(U, W * 4.0);
    else if (frac < 1.0 / 16.0) W = W * 0.5;
    else if (frac > 0.5) W = fmin(U, W * 2.0);
    ctl->U = fmax(bb.s, v.theta);
    ctl->W = W;
    ctl->nb = nb;          // nb >= 1: the first winner is the global argmax (score >= theta)
    ctl->n_picked = picked0 + nb;
    ctl->stat_rounds += 1;
    ctl->stat_cand_sum += v.total;
    ctl->first_round = 0;
    send->count = 0;
    tp0 = gtime_ns();
    ctl->stat_ns_planph[0] += tp1 - tp_begin;
    ctl->stat_ns_planph[1] += tp2 - tp1;
    ctl->stat_ns_planph[2] += tp3 - tp2;
    ctl->stat_ns_planph[3] += tp0 - tp3;
  }
}

__global__ void __launch_bounds__(kPlanThreads) plan_kernel(const RankBlock* blocks, RankBlock* send, const double* Dcc,
                                                            unsigned int* hist, long long* out_idx, Ctl* ctl) {
  plan_body(blocks, send, Dcc, hist, out_idx, ctl);
}

// generic-shape rounds with the peer-memory exchange: one thread waits for the round's blocks
__global__ void wait_blocks_kernel(Mailbox* mail, const Ctl* ctl, unsigned long long seq) {
  if (ctl->n_picked >= ctl->k) return;
  wait_blocks(mail, ctl->world, seq);
}

// distances of every row to a list of centers, for the parity tests
template <typename T>
__global__ void __launch_bounds__(256) pairwise_kernel(const T* __restrict__ X, long long n, int d4, int nss, int S,
                                                       int guard, const double* __restrict__ xx, const long long* __restrict__ centers,
                                                       long long mcols, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double s_xxc[kB];
  double* s_c = reinterpret_cast<double*>(smem_raw);
  const long long col0 = (long long)blockIdx.x * kB;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5, g = lane >> 2, kk = lane & 3;
  const quad_t<T>* X4 = reinterpret_cast<const quad_t<T>*>(X);
  for (int j = 0; j < kB; ++j) {
    const long long p = centers[min(col0 + j, mcols - 1)];
    stage_center(X, d4, nss * 16, S, p, j, s_c);
    if (threadIdx.x == 0) s_xxc[j] = xx[p];
  }
  __syncthreads();
  for (long long r0 = ((long long)blockIdx.y * nwarp + warp) * 8; r0 < n; r0 += (long long)gridDim.y * nwarp * 8) {
    const long long i = min(r0 + g, n - 1);
    double c[2];
    if (guard) dmma_block<true, false, T>(X4 + (size_t)i * d4, d4, nss, s_c, S, lane, c);
    else dmma_block<false, false, T>(X4 + (size_t)i * d4, d4, nss, s_c, S, lane, c);
    if (r0 + g < n) {
      const double xxi = xx[i];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const long long col = col0 + 2 * kk + e;
        if (col < mcols) out[(size_t)i * mcols + col] = dist_from_dot(c[e], xxi, s_xxc[2 * kk + e]);
      }
    }
  }
}

// ---------------------------------------------------------------- NCCL through dlopen
struct Id128 {  // ncclUniqueId is a 128-byte struct passed by value
  char b[128];
};
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, Id128, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int load_nccl() {
  if (g_nccl.lib) return 0;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) {
    snprintf(g_err, sizeof(g_err), "NCCL not found: %s", dlerror());
    return VATLQ_ECOMM;
  }
  g_nccl.GetUniqueId = (int (*)(void*))dlsym(h, "ncclGetUniqueId");
  g_nccl.CommInitRank = (int (*)(void**, int, Id128, int))dlsym(h, "ncclCommInitRank");
  g_nccl.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
  g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(h, "ncclAllGather");
  g_nccl.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllGather) {
    snprintf(g_err, sizeof(g_err), "NCCL symbols missing");
    return VATLQ_ECOMM;
  }
  g_nccl.lib = h;
  return 0;
}
struct Comm {
  void* nccl;
  int rank, world;
  // peer-memory mailbox (vatlq_comm_mailbox_handle / vatlq_comm_attach); null -> NCCL all-gather
  Mailbox* mail = nullptr;           // this rank's mailbox (cudaMalloc)
  Mailbox** peers_dev = nullptr;     // device array of every rank's mailbox pointer
  void* opened[kMaxRanks] = {};      // cudaIpcOpenMemHandle results to close
  unsigned long long seq = 0;        // last sequence number used (monotonic over the communicator's life)
};

// ---------------------------------------------------------------- workspace layout
struct WsLayout {
  size_t xx, score, hist, partial, send, recv, dcc, ctl, dots, flags, total;
  size_t prune, seg_of_row, seg_start, seg_r, seg_skip, skip_stride;   // pruning state (cd aliases dots during set-up)
  size_t xh;   // the screen's fp16 copy of the owned rows, n * 4096 bytes from here (beyond `total`: only a
               // selection whose rounds take the paired pass needs it; sized by n, so a rank of an 8-way shard
               // uses an eighth of it)
};
// rounds of 16 picks, applied by the paired pass (and screened): d == 2048 and batch >= 16 (vatlq_coreset_select
// rounds batch down to a power of two)
static bool paired_rounds(int d, int batch) { return d == kFastD && batch >= 2 * kB; }
static WsLayout ws_layout(long long n, int world) {
  WsLayout L;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t at = o;
    o += align_up(bytes, 256);
    return at;
  };
  L.ctl = take(sizeof(Ctl));
  L.xx = take((size_t)n * 8);
  L.score = take((size_t)n * 8);
  L.hist = take((kNB + 1) * 4);
  L.partial = take(4096 * sizeof(Best));
  L.send = take(sizeof(RankBlock));
  L.recv = take(sizeof(RankBlock) * (size_t)kMaxRanks);
  L.dcc = take((size_t)kCap * kCap * 8);
  L.dots = take((size_t)n * 2 * kB * 8);   // up to 16 dot products per owned row (paired pass)
  L.flags = take(1024);
  L.prune = take(sizeof(PruneCtl));
  L.seg_of_row = take((size_t)n * 4);
  L.seg_start = take((size_t)(n + 1) * 4);
  L.seg_r = take((size_t)n * 8);
  L.seg_skip = take((size_t)n * (kMaxPicks / kB));   // one flag array per centre group of a round
  L.skip_stride = align_up((size_t)n, 256);
  L.total = o;
  L.xh = o;
  return L;
}

// ---------------------------------------------------------------- pass-kernel timing (bench.py roofline)
struct PassProfiler {
  bool on = false;
  std::vector<cudaEvent_t> ev;   // start/stop pairs
  size_t used = 0;
  double total_ms = 0.0;         // summed duration of real passes (nb > 0)
  long long timed = 0;           // how many real passes were timed
  long long picks = 0;           // picks those passes applied
};
static PassProfiler g_prof;
static long long g_prune[4] = {0, 0, 0, 0};   // tiles seen, tiles streamed, verify violations, segments (last call)
static int g_prune_mode_set = -1;              // vatlq_coreset_set_prune: -1 = take VATLQ_PRUNE
static long long g_prune_min_set = -1;         //                          -1 = take VATLQ_PRUNE_MIN_ROWS
static long long g_screen[3] = {0, 0, 0};      // rows screened, rows listed, verify violations (paired passes)
static int g_screen_mode_set = -1;             // vatlq_coreset_set_screen: -1 = take VATLQ_PASS_SCREEN

}  // namespace vatlq

using namespace vatlq;

extern "C" size_t vatlq_coreset_workspace_bytes_dt(int64_t n, int d, int batch, int dtype) {
  if (n < 0 || dtype_size(dtype) == 0) return 0;
  const WsLayout L = ws_layout(n, kMaxRanks);
  // the fp16 copy only for an fp32 X: the screen reads a 16-bit X itself
  return (dtype == VATLQ_F32 && paired_rounds(d, batch)) ? L.xh + (size_t)n * 4096 : L.total;
}
extern "C" size_t vatlq_coreset_workspace_bytes(int64_t n, int d, int batch) {
  return vatlq_coreset_workspace_bytes_dt(n, d, batch, VATLQ_F32);
}

struct Geom {
  int d4, nss, S, guard;
  size_t smem;
};
static Geom geom_of(int d) {
  Geom g;
  g.d4 = d / 4;
  g.nss = (d + 15) / 16;          // super-steps of 16 features (tail zero padded)
  g.S = g.nss * 16 + 2;           // center row stride in doubles: 16 bytes mod 128
  g.smem = (size_t)kB * g.S * sizeof(double);
  g.guard = (d % 16) != 0;   // ragged last super-step: guarded loads
  return g;
}

static int check_x(const void* X, int dtype, int64_t n, int d, int64_t lo, int64_t hi) {
  VQ_REQUIRE(dtype_size(dtype) != 0, "dtype must be VATLQ_F32, VATLQ_F16 or VATLQ_BF16");
  VQ_REQUIRE(X != nullptr && quad_aligned(X, dtype), "X must be a device pointer aligned to 16 bytes (fp32) or 8 bytes (16 bits)");
  VQ_REQUIRE(n > 0 && d > 0 && (d & 3) == 0, "d must be a positive multiple of 4");
  VQ_REQUIRE(n < 0xffffffffLL, "n must be below 2^32 - 1 (the planner reduces 32-bit row ids)");
  VQ_REQUIRE(0 <= lo && lo <= hi && hi <= n, "bad row range");
  VQ_REQUIRE(pass_smem_bytes(geom_of(d).S) <= (size_t)kMaxSmem, "d too large (centers must fit shared memory)");
  return 0;
}

template <typename T>
static int launch_norms(const T* X, int64_t n, int d, double* xx, cudaStream_t stream) {
  const Geom g = geom_of(d);
  const int grid = sm_count() * 8;
  if (g.guard) row_norms_kernel<true, T><<<grid, 256, 0, stream>>>(X, n, g.d4, g.nss, xx);
  else row_norms_kernel<false, T><<<grid, 256, 0, stream>>>(X, n, g.d4, g.nss, xx);
  VQ_LAUNCHED();
  return 0;
}

template <typename T>
static int configure_pass_of() {
  VQ_CUDA(cudaFuncSetAttribute(pass_kernel_generic<false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  VQ_CUDA(cudaFuncSetAttribute(pass_kernel_generic<true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  VQ_CUDA(cudaFuncSetAttribute(pass_kernel_tma<false, false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmem));
  VQ_CUDA(cudaFuncSetAttribute(pass_kernel_tma<false, true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmem));
  VQ_CUDA(cudaFuncSetAttribute(pass_kernel_tma<true, false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmem));
  VQ_CUDA(cudaFuncSetAttribute(pass_kernel_tma<true, true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmem));
  VQ_CUDA(cudaFuncSetAttribute(pairs_plan_kernel<T>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  VQ_CUDA(cudaFuncSetAttribute(pairs_plan_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPlanSmem));
  VQ_CUDA(cudaFuncSetAttribute(pairs_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  VQ_CUDA(cudaFuncSetAttribute(pairwise_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  return 0;
}
// the opt-in shared-memory sizes (and the planner's carve-out) of every kernel of every element type, once
static int configure_pass() {
  static bool configured = false;
  if (!configured) {
    if (int e = configure_pass_of<float>()) return e;
    if (int e = configure_pass_of<__half>()) return e;
    if (int e = configure_pass_of<__nv_bfloat16>()) return e;
    configured = true;
  }
  return 0;
}

// CTAs of the paired pass: the largest even count whose clusters of two are all co-resident (0: clusters unavailable)
static int pair_grid() {
  static int grid = -1;
  if (grid < 0) {
    grid = 0;
    if (configure_pass() != 0) return grid;   // (the occupancy query needs the opt-in shared-memory size)
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(sm_count() & ~1));
    cfg.blockDim = dim3(kWsThreads);
    cfg.dynamicSmemBytes = kWsSmem;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = 2;
    at.val.clusterDim.y = at.val.clusterDim.z = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    int ncl = 0;
    if (cudaOccupancyMaxActiveClusters(&ncl, pass_kernel_tma<true>, &cfg) == cudaSuccess && ncl > 0)
      grid = 2 * std::min(ncl, sm_count() / 2);
    cudaGetLastError();
  }
  return grid;
}

// pass_kernel_tma (d = 2048) in its four forms.  pair: clusters of two CTAs on pair_grid() CTAs, applying a round of up
// to 16 picks in one read of X; else one CTA per SM applying the 8 centres from center_off.  filter: the segment
// filter over the anchor rows, which writes the skip flags of those centres instead of applying them.
template <typename T>
static int launch_tma(const PassArgs& a, bool pair, bool filter, cudaStream_t stream, bool pdl, cudaEvent_t ev0 = nullptr,
                      cudaEvent_t ev1 = nullptr) {
  if (int e = configure_pass()) return e;
  void (*kernel)(PassArgs) = pair ? (filter ? pass_kernel_tma<true, true, T> : pass_kernel_tma<true, false, T>)
                                  : (filter ? pass_kernel_tma<false, true, T> : pass_kernel_tma<false, false, T>);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(pair ? pair_grid() : sm_count()));
  cfg.blockDim = dim3(kWsThreads);
  cfg.dynamicSmemBytes = kWsSmem;
  cfg.stream = stream;
  cudaLaunchAttribute at[2] = {};
  unsigned nat = 0;
  if (pair) {
    at[nat].id = cudaLaunchAttributeClusterDimension;
    at[nat].val.clusterDim.x = 2;
    at[nat].val.clusterDim.y = at[nat].val.clusterDim.z = 1;
    ++nat;
  }
  if (pdl) {
    at[nat].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[nat].val.programmaticStreamSerializationAllowed = 1;
    ++nat;
  }
  cfg.attrs = at;
  cfg.numAttrs = nat;
  if (ev0) cudaEventRecord(ev0, stream);
  VQ_CUDA(cudaLaunchKernelEx(&cfg, kernel, a));
  if (ev1) cudaEventRecord(ev1, stream);
  VQ_LAUNCHED();
  return 0;
}

// the solo pass: the TMA kernel at d = 2048, else the generic kernel
template <typename T>
static int launch_pass(PassArgs& a, cudaStream_t stream, cudaEvent_t ev0 = nullptr, cudaEvent_t ev1 = nullptr, bool pdl = false) {
  if (a.d4 == kFastD / 4 && a.dots != nullptr) return launch_tma<T>(a, false, false, stream, pdl, ev0, ev1);
  if (int e = configure_pass()) return e;
  if (ev0) cudaEventRecord(ev0, stream);
  if ((a.d4 & 3) != 0) pass_kernel_generic<true, T><<<sm_count(), kPassThreads, pass_smem_bytes(a.S), stream>>>(a);
  else pass_kernel_generic<false, T><<<sm_count(), kPassThreads, pass_smem_bytes(a.S), stream>>>(a);
  if (ev1) cudaEventRecord(ev1, stream);
  VQ_LAUNCHED();
  return 0;
}

// ---- exact pruning: mode resolution and per-call set-up shared by init and select
struct PruneState {
  int mode = 0;   // 0 off, 1 prune, 2 verify
  PruneCtl* pc = nullptr;
  int* seg_of_row = nullptr;
  int* seg_start = nullptr;
  double* seg_r = nullptr;
  unsigned char* seg_skip = nullptr;
  size_t skip_stride = 0;
  // the pruning fields of a pass (mode != 0): the pass reads the flags of its centre group at seg_skip (group g's at
  // + g * skip_stride), its filter launch writes them at seg_skip_out
  void fill(PassArgs& a) const {
    a.seg_of_row = seg_of_row; a.seg_skip = seg_skip; a.prune_mode = mode; a.prune_stats = pc->stats;
    a.seg_start = seg_start; a.seg_r = seg_r; a.nseg = &pc->nseg; a.seg_skip_out = seg_skip; a.skip_stride = skip_stride;
  }
};
template <typename T>
static int prune_setup(PruneState& P, const T* X, const Geom& G, int64_t row_lo, int64_t row_hi, char* w,
                       const WsLayout& L, cudaStream_t stream) {
  static const int prune_env = []() {
    const char* e = getenv("VATLQ_PRUNE");
    if (!e) return 1;
    if (!strcmp(e, "0") || !strcmp(e, "off")) return 0;
    return !strcmp(e, "verify") ? 2 : 1;
  }();
  static const long long prune_min_rows = []() {
    const char* e = getenv("VATLQ_PRUNE_MIN_ROWS");
    return e ? atoll(e) : 8192LL;
  }();
  const long long own = row_hi - row_lo;
  P.pc = (PruneCtl*)(w + L.prune);
  P.seg_of_row = (int*)(w + L.seg_of_row);
  P.seg_start = (int*)(w + L.seg_start);
  P.seg_r = (double*)(w + L.seg_r);
  P.seg_skip = (unsigned char*)(w + L.seg_skip);
  P.skip_stride = L.skip_stride;
  const long long prune_min = g_prune_min_set >= 0 ? g_prune_min_set : prune_min_rows;
  P.mode = (G.d4 == kFastD / 4 && own >= prune_min && own >= 8 && own < (1LL << 30))
               ? (g_prune_mode_set >= 0 ? g_prune_mode_set : prune_env) : 0;
  VQ_CUDA(cudaMemsetAsync(P.pc, 0, sizeof(PruneCtl), stream));
  if (P.mode) {
    double* cd = (double*)(w + L.dots);   // the dot-product scratch is idle until the first pass
    consec_kernel<T><<<sm_count() * 8, 256, 0, stream>>>(X, G.d4, row_lo, row_hi, cd, P.pc);
    VQ_LAUNCHED();
    segment_kernel<<<1, 1024, 0, stream>>>(cd, (int)own, P.pc, P.seg_of_row, P.seg_start);
    VQ_LAUNCHED();
    seg_radius_kernel<T><<<sm_count() * 8, 256, 0, stream>>>(X, G.d4, row_lo, P.seg_start, P.pc, P.seg_r);
    VQ_LAUNCHED();
  }
  return 0;
}
// accumulate the device-side tile statistics of a finished call (the caller has synchronised)
static void prune_collect(const PruneState& P) {
  PruneCtl hp{};
  if (cudaMemcpy(&hp, P.pc, sizeof(PruneCtl), cudaMemcpyDeviceToHost) == cudaSuccess) {
    g_prune[0] += (long long)hp.stats[0];
    g_prune[1] += (long long)hp.stats[1];
    g_prune[2] += (long long)hp.stats[2];
    g_prune[3] = hp.nseg;
    for (int q = 0; q < 3; ++q) g_screen[q] += (long long)hp.screen[q];
  }
}

namespace vatlq {
int vq_launch_norms(const float* X, int64_t n, int d, double* xx, cudaStream_t stream) { return launch_norms(X, n, d, xx, stream); }
int vq_launch_norms(const __half* X, int64_t n, int d, double* xx, cudaStream_t stream) { return launch_norms(X, n, d, xx, stream); }
int vq_launch_norms(const __nv_bfloat16* X, int64_t n, int d, double* xx, cudaStream_t stream) { return launch_norms(X, n, d, xx, stream); }
}  // namespace vatlq

// X of the core-set calls: check_x, plus 16-byte alignment when d = 2048 (the TMA passes copy whole rows with
// cp.async.bulk, which needs a 16-byte aligned source in every dtype)
static int check_coreset_x(const void* X, int dtype, int64_t n, int d, int64_t lo, int64_t hi) {
  if (int e = check_x(X, dtype, n, d, lo, hi)) return e;
  VQ_REQUIRE(d != kFastD || ((uintptr_t)X & 15) == 0, "X must be 16-byte aligned when d = 2048");
  return 0;
}

template <typename T>
static int coreset_init(const T* X, int64_t n, int d, int64_t row_lo, int64_t row_hi, const int64_t* labeled,
                        int64_t n_labeled, double* min_d, void* ws, size_t ws_bytes, cudaStream_t stream) {
  const WsLayout L = ws_layout(n, kMaxRanks);
  VQ_REQUIRE(ws != nullptr && ws_bytes >= L.total, "workspace too small");
  char* w = (char*)ws;
  double* xx = (double*)(w + L.xx);
  if (int e = fill_f64(min_d + row_lo, row_hi - row_lo, INFINITY, stream)) return e;
  if (n_labeled == 0) return 0;
  VQ_REQUIRE(labeled != nullptr, "labeled is null");
  if (int e = launch_norms(X, n, d, xx, stream)) return e;
  const Geom G = geom_of(d);
  // the labelled set is applied 8 centres per pass; as soon as a track holds a labelled row the
  // later passes stop streaming it (same exact pruning as the selection passes)
  PruneState P;
  if (int e = prune_setup(P, X, G, row_lo, row_hi, w, L, stream)) return e;
  for (int64_t c0 = 0; c0 < n_labeled; c0 += kB) {
    PassArgs a{};
    a.X = X; a.n = n; a.d4 = G.d4; a.nss = G.nss; a.S = G.S; a.lo = row_lo; a.hi = row_hi; a.xx = xx; a.m = min_d;
    a.dots = (double*)(w + L.dots);
    a.unc = nullptr; a.score = nullptr; a.centers = (const long long*)labeled + c0; a.n_centers = nullptr;
    a.n_centers_imm = (int)std::min<int64_t>(kB, n_labeled - c0); a.ctl = nullptr; a.hist = nullptr;
    if (P.mode) {
      P.fill(a);
      if (int e = launch_tma<T>(a, false, true, stream, false)) return e;   // the flags of this pass
    }
    if (int e = launch_pass<T>(a, stream)) return e;
  }
  if (P.mode == 2) {   // verify mode only: wait and collect the violation count of the initialisation passes
    VQ_CUDA(cudaStreamSynchronize(stream));
    prune_collect(P);
  }
  return 0;
}

extern "C" int vatlq_coreset_init_dt(const void* X, int dtype, int64_t n, int d, int64_t row_lo, int64_t row_hi,
                                     const int64_t* labeled, int64_t n_labeled, double* min_d, void* ws,
                                     size_t ws_bytes, vatlq_stream_t stream) {
  if (int e = check_coreset_x(X, dtype, n, d, row_lo, row_hi)) return e;
  VQ_REQUIRE(min_d != nullptr && n_labeled >= 0, "null min_d");
  return with_dtype(dtype, [&](auto t) {
    using T = std::remove_cv_t<std::remove_pointer_t<decltype(t)>>;
    return coreset_init<T>(static_cast<const T*>(X), n, d, row_lo, row_hi, labeled, n_labeled, min_d, ws, ws_bytes,
                           (cudaStream_t)stream);
  });
}
extern "C" int vatlq_coreset_init(const float* X, int64_t n, int d, int64_t row_lo, int64_t row_hi,
                                  const int64_t* labeled, int64_t n_labeled, double* min_d, void* ws,
                                  size_t ws_bytes, vatlq_stream_t stream) {
  return vatlq_coreset_init_dt(X, VATLQ_F32, n, d, row_lo, row_hi, labeled, n_labeled, min_d, ws, ws_bytes, stream);
}

template <typename T>
static int coreset_select(const T* X, int dtype, int64_t n, int d, int64_t row_lo, int64_t row_hi, double* min_d,
                          double* unc, int rule, double moks, double lambda, int64_t n_labeled, int64_t first_pick,
                          int64_t k, int batch, int64_t* out_idx, void* comm_, void* ws, size_t ws_bytes,
                          int64_t* host_stats, cudaStream_t stream) {
  VQ_REQUIRE(min_d && unc && out_idx, "null pointer");
  VQ_REQUIRE(rule >= 0 && rule <= 2, "rule must be 0, 1 or 2");
  VQ_REQUIRE(k >= 0 && k <= n, "k must be in [0, n]");
  VQ_REQUIRE(batch >= 1, "batch must be >= 1");
  Comm* comm = (Comm*)comm_;
  const int world = comm ? comm->world : 1;
  VQ_REQUIRE(world >= 1 && world <= kMaxRanks, "world size not supported");
  VQ_REQUIRE(world > 1 || (row_lo == 0 && row_hi == n), "single GPU must own every row");
  const WsLayout L = ws_layout(n, kMaxRanks);
  VQ_REQUIRE(ws != nullptr && ws_bytes >= vatlq_coreset_workspace_bytes_dt(n, d, batch, dtype),
             "workspace too small (vatlq_coreset_workspace_bytes_dt(n, d, batch, dtype))");
  if (k == 0) return 0;
  char* w = (char*)ws;
  Ctl* ctl = (Ctl*)(w + L.ctl);
  double* xx = (double*)(w + L.xx);
  double* score = (double*)(w + L.score);
  unsigned int* hist = (unsigned int*)(w + L.hist);
  Best* partial = (Best*)(w + L.partial);
  RankBlock* send = (RankBlock*)(w + L.send);
  RankBlock* recv = (world > 1) ? (RankBlock*)(w + L.recv) : send;
  const bool p2p = world > 1 && comm->peers_dev != nullptr;   // peer-memory mailbox instead of ncclAllGather
  const unsigned long long seq0 = p2p ? comm->seq : 0ULL;
  if (p2p) VQ_CUDA(cudaMemsetAsync(&comm->mail->error, 0, 8, stream));   // a past time-out must not fail this call
  auto push_of = [&](unsigned long long seq) {
    PushArgs pa{};
    if (p2p) {
      pa.peers = comm->peers_dev;
      pa.rank = comm->rank;
      pa.world = world;
      pa.seq = seq;
    }
    return pa;
  };
  double* Dcc = (double*)(w + L.dcc);
  unsigned char* flags = (unsigned char*)(w + L.flags);
  const Geom G = geom_of(d);
  int nbk = 1;   // picks per round: the power of two <= min(batch, kMaxPicks)
  while (nbk * 2 <= kMaxPicks && nbk * 2 <= batch) nbk *= 2;

  Ctl h{};
  h.n_picked = 0; h.k = k; h.nb = 0; h.rule = rule; h.world = world;
  h.first_round = (n_labeled == 0) ? 1 : 0;
  h.maxb = nbk;
  h.wd = (rule == 0) ? (1.0 - moks) : 1.0;
  h.wu = (rule == 0) ? (lambda * moks) : lambda;
  h.U = 0.0; h.W = -1.0;
  {
    static const int target = []() {
      const char* e = getenv("VATLQ_TARGET");
      const int t = e ? atoi(e) : 0;
      return (t >= 16 && t <= kCap) ? t : 0;
    }();
    // wanted candidates per round (all ranks together).  The candidate x candidate tiles and the planner cost grow with
    // the square of the list while a short list ends rounds early: measured on B200 (tools/round_cost.py, 16 picks per
    // round) 192 is best for 64 k .. 300 k rows per rank, 256 above, 384 for small pools.  n / world is the same on
    // every rank.
    const long long per_rank = n / std::max(1, world);
    const int t16 = n < 65536 ? kTarget + kTarget / 2 : (per_rank <= 300000 ? 192 : 256);
    h.target = target ? target : (nbk > kB ? t16 : kTarget);
  }
  if (n_labeled == 0 && rule == 2) {
    // _query (:828-833): the caller drew the random first pick
    VQ_REQUIRE(first_pick >= 0 && first_pick < n, "rule 2 with an empty labelled set needs first_pick");
  }
  VQ_CUDA(cudaMemcpyAsync(ctl, &h, sizeof(Ctl), cudaMemcpyHostToDevice, stream));
  VQ_CUDA(cudaMemsetAsync(hist, 0, (kNB + 1) * 4, stream));
  VQ_CUDA(cudaMemsetAsync(send, 0, 64, stream));
  if (int e = launch_norms(X, n, d, xx, stream)) return e;

  const int own = (int)std::min<int64_t>(row_hi - row_lo, 1LL << 30);
  // ---- exact pruning set-up (fast path only): segments of near-consecutive rows, anchors, radii
  PruneState P;
  if (int e = prune_setup(P, X, G, row_lo, row_hi, w, L, stream)) return e;
  const int prune_mode = P.mode;
  int fgrid = std::max(1, std::min(sm_count() * 4, (own + 255) / 256));
  VQ_REQUIRE(fgrid <= 4096 && sm_count() <= 4096, "grid too large for the arg-max scratch");
  const size_t pairs_smem = G.smem;
  const bool fast_d = (G.d4 == kFastD / 4);   // register-resident centres
  const bool use_pair = paired_rounds(d, batch) && pair_grid() >= 2;   // 16 picks per round in one read of X
  // the fp16 screen of the paired pass (see "the screen" at pass_kernel_tma): 0 off, 1 on, 2 verify
  static const int screen_env = []() {
    const char* e = getenv("VATLQ_PASS_SCREEN");
    if (!e) return 1;
    if (!strcmp(e, "0") || !strcmp(e, "off")) return 0;
    return !strcmp(e, "verify") ? 2 : 1;
  }();
  const int screen_mode = g_screen_mode_set >= 0 ? g_screen_mode_set : screen_env;
  // the screen reads the owned rows in 16 bits: an fp32 X from its fp16 copy at the end of the workspace, filled once
  // per call; a 16-bit X as it is
  const __half* Xh = nullptr;
  if (use_pair && screen_mode) {
    if constexpr (sizeof(T) == 2) {
      Xh = reinterpret_cast<const __half*>(X) + (size_t)row_lo * 2048;
    } else {
      Xh = (const __half*)(w + L.xh);
      if (row_hi > row_lo) {
        half_copy_kernel<<<sm_count() * 8, 256, 0, stream>>>((const float4*)X, row_lo, (row_hi - row_lo) * 512, (uint2*)(w + L.xh));
        VQ_LAUNCHED();
      }
    }
  }
  // (the same shared-memory carve-out for the planner as for the pass kernels on either side of it: no SM
  // reconfiguration between them)
  if (int e = configure_pass()) return e;
  auto fill_pass = [&](PassArgs& a) {
    a.X = X; a.n = n; a.d4 = G.d4; a.nss = G.nss; a.S = G.S; a.lo = row_lo; a.hi = row_hi; a.xx = xx; a.m = min_d;
    a.unc = unc; a.score = score; a.centers = ctl->picks; a.n_centers = &ctl->nb; a.n_centers_imm = 0; a.ctl = ctl;
    a.hist = (nbk > 1) ? hist : nullptr; a.send = send; a.partial = partial; a.dots = (double*)(w + L.dots);
    a.prune_stats = P.pc->stats;
    if (prune_mode) P.fill(a);
  };

  if (n_labeled == 0 && rule == 2) {
    // apply the given first pick directly (one pass), then continue with argmax(min_d)
    Ctl h2 = h;
    h2.first_round = 0; h2.n_picked = 1; h2.picks[0] = first_pick; h2.nb = 1;
    VQ_CUDA(cudaMemcpyAsync(ctl, &h2, sizeof(Ctl), cudaMemcpyHostToDevice, stream));
    VQ_CUDA(cudaMemcpyAsync(out_idx, &first_pick, 8, cudaMemcpyHostToDevice, stream));
    PassArgs a{};
    fill_pass(a);
    a.send = nullptr;   // the bootstrap below computes the arg-max of the scores this pass writes
    a.seg_skip = nullptr; a.prune_mode = 0;
    if (int e = launch_pass<T>(a, stream)) return e;
  } else {
    const long long cnt = row_hi - row_lo;
    if (cnt > 0) {
      score_init_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, stream>>>(row_lo, row_hi, min_d, unc, score, ctl);
      VQ_LAUNCHED();
    }
  }
  // block header of round 0 (no list, exact arg-max); later headers come from the passes
  bootstrap_kernel<<<fgrid, 256, 0, stream>>>(row_lo, row_hi, score, partial, send, ctl, push_of(seq0 + 1));
  VQ_LAUNCHED();

  // rounds: [all-gather] -> pairs -> plan -> pass.  The host only learns the pick count every
  // `chunk` rounds; kernels of surplus rounds exit on n_picked >= k.
  long long picked = (n_labeled == 0 && rule == 2) ? 1 : 0;
  long long rounds_done = 0;
  long long passes_seen = (n_labeled == 0 && rule == 2) ? 1 : 0;
  g_prof.used = 0;
  Ctl h_ctl{};                      // host copy of the control block, refreshed every chunk of rounds
  Ctl* h_picked = &h_ctl;
  int rc = 0;
  while (picked < k && rc == 0) {
    const long long remaining = k - picked;
    double per_round = (rounds_done > 8 && picked > 0) ? (double)picked / (double)rounds_done : (double)std::max(1, nbk / 2);
    long long chunk = (long long)((double)remaining / std::max(1.0, per_round)) + 2;
    chunk = std::max<long long>(4, std::min<long long>(chunk, 256));
    if (g_prof.on) VQ_CUDA(cudaMemsetAsync(flags, 0, 1024, stream));
    for (long long it = 0; it < chunk && rc == 0; ++it) {
      const unsigned long long round_no = (unsigned long long)(rounds_done + it) + 1;   // 1-based over the call
      const RankBlock* blocks = recv;
      Mailbox* mail = nullptr;
      if (p2p) {
        mail = comm->mail;
        blocks = &comm->mail->slots[(seq0 + round_no) & 1ULL][0];
      } else if (world > 1) {
        const int e = g_nccl.AllGather(send, recv, sizeof(RankBlock), /*ncclChar*/ 0, comm->nccl, stream);
        if (e != 0) {
          snprintf(g_err, sizeof(g_err), "ncclAllGather failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(e) : "?");
          rc = VATLQ_ECOMM;
          break;
        }
      }
      if (nbk > 1) {
        dim3 pg(kCap / kB, 4);
        if (fast_d) {
          const cudaError_t le = launch_pdl(pairs_plan_kernel<T>, dim3(sm_count()), dim3(kSeg * 32), kPlanSmem, stream, true, X, G.d4,
                                            (const double*)xx, blocks, send, hist, (long long*)out_idx, ctl, Dcc, mail,
                                            (unsigned long long)(seq0 + round_no), kPlanSmem / 8);
          if (le != cudaSuccess) {
            snprintf(g_err, sizeof(g_err), "pairs_plan launch failed: %s", cudaGetErrorString(le));
            rc = (int)le;
            break;
          }
        } else {
          if (p2p) wait_blocks_kernel<<<1, 1, 0, stream>>>(mail, ctl, seq0 + round_no);
          pairs_kernel<T><<<pg, 256, pairs_smem, stream>>>(X, G.d4, G.nss, G.S, G.guard, xx, blocks, ctl, Dcc);
        }
        g_launches.fetch_add(1);
      } else if (p2p) {
        wait_blocks_kernel<<<1, 1, 0, stream>>>(mail, ctl, seq0 + round_no);
      }
      if (nbk == 1 || !fast_d) {
        plan_kernel<<<1, kPlanThreads, 0, stream>>>(blocks, send, Dcc, hist, (long long*)out_idx, ctl);
        g_launches.fetch_add(1);
      }
      if (prune_mode) {   // the flags of every centre group of the round, before its first pass
        PassArgs a{};
        fill_pass(a);
        if (use_pair) rc = launch_tma<T>(a, true, true, stream, true);
        for (int off = 0; !use_pair && off < nbk && rc == 0; off += kB) {
          a.center_off = off;
          a.seg_skip_out = P.seg_skip + (size_t)(off / kB) * P.skip_stride;
          rc = launch_tma<T>(a, false, true, stream, true);
        }
      }
      auto timed_launch = [&](PassArgs& a, bool pair) {
        const bool timed = g_prof.on && g_prof.used + 2 <= g_prof.ev.size() && g_prof.used / 2 < 1024;
        if (timed) a.did_work = flags + g_prof.used / 2;
        cudaEvent_t e0 = timed ? g_prof.ev[g_prof.used] : nullptr, e1 = timed ? g_prof.ev[g_prof.used + 1] : nullptr;
        const int r = pair ? launch_tma<T>(a, true, false, stream, true, e0, e1) : launch_pass<T>(a, stream, e0, e1, true);
        if (timed) g_prof.used += 2;
        return r;
      };
      if (use_pair && rc == 0) {
        // every round, of 1 to 16 picks, is applied by ONE paired pass (X read once)
        PassArgs a{};
        fill_pass(a);
        a.push = push_of(seq0 + round_no + 1);   // the block this round's (only) pass publishes
        a.screen_mode = screen_mode;
        a.screen_stats = P.pc->screen;
        a.Xh = Xh;
        rc = timed_launch(a, true);
      } else {
        for (int off = 0; off < nbk && rc == 0; off += kB) {   // picks [off, off+8) of the round; the last pass emits
          PassArgs a{};
          fill_pass(a);
          a.center_off = off;
          if (prune_mode) a.seg_skip = P.seg_skip + (size_t)(off / kB) * P.skip_stride;
          a.push = push_of(seq0 + round_no + 1);   // the block this round's final pass publishes
          rc = timed_launch(a, false);
        }
      }
    }
    if (rc) break;
    rounds_done += chunk;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_picked, ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
      snprintf(g_err, sizeof(g_err), "coreset rounds failed: %s", cudaGetErrorString(e));
      rc = (int)e;
      break;
    }
    const Ctl* hc = (const Ctl*)h_picked;
    if (g_prof.on) {
      // launches of surplus rounds / of a round's unused second pass return at once: only the
      // launches that flagged work are timed
      unsigned char h_flags[1024];
      if (cudaMemcpy(h_flags, flags, 1024, cudaMemcpyDeviceToHost) == cudaSuccess) {
        for (size_t i = 0; i < g_prof.used / 2; ++i) {
          float ms = 0.f;
          if (h_flags[i] && cudaEventElapsedTime(&ms, g_prof.ev[2 * i], g_prof.ev[2 * i + 1]) == cudaSuccess) {
            g_prof.total_ms += ms;
            g_prof.timed += 1;
          }
        }
      }
      g_prof.picks += hc->n_picked - picked;
      g_prof.used = 0;
    }
    passes_seen = hc->stat_passes;
    if (hc->n_picked <= picked && hc->n_picked < k) {
      snprintf(g_err, sizeof(g_err), "coreset made no progress (picked %lld of %lld)", (long long)hc->n_picked, (long long)k);
      rc = VATLQ_ESTATE;
      break;
    }
    picked = hc->n_picked;
  }
  if (p2p) {
    comm->seq = seq0 + (unsigned long long)rounds_done + 2;
    unsigned long long err = 0;
    if (rc == 0 && cudaMemcpy(&err, &comm->mail->error, 8, cudaMemcpyDeviceToHost) == cudaSuccess && err != 0) {
      snprintf(g_err, sizeof(g_err), "peer-memory exchange timed out waiting for block %llu", err);
      rc = VATLQ_ECOMM;
    }
  }
  if (rc == 0) prune_collect(P);
  if (rc == 0 && host_stats) {
    const Ctl* hc = (const Ctl*)h_picked;
    host_stats[0] = hc->stat_passes;
    host_stats[1] = hc->n_picked;
    host_stats[2] = hc->stat_rounds;
    host_stats[3] = hc->stat_fallback_empty;
    host_stats[4] = hc->stat_fallback_overflow;
    host_stats[5] = hc->stat_cand_sum;
    host_stats[6] = rounds_done;
    host_stats[7] = nbk;
    host_stats[8] = (int64_t)hc->stat_ns_wait;
    host_stats[9] = (int64_t)hc->stat_ns_tiles;
    host_stats[10] = (int64_t)hc->stat_ns_plan;
    if (getenv("VATLQ_PASS_PHASES"))
      fprintf(stderr, "[vatlq] planner phases, us per round: theta %.1f, records + staging %.1f, pick loop %.1f, tail %.1f (%lld rounds)\n",
              hc->stat_ns_planph[0] / 1e3 / std::max<long long>(1, hc->stat_rounds), hc->stat_ns_planph[1] / 1e3 / std::max<long long>(1, hc->stat_rounds),
              hc->stat_ns_planph[2] / 1e3 / std::max<long long>(1, hc->stat_rounds), hc->stat_ns_planph[3] / 1e3 / std::max<long long>(1, hc->stat_rounds),
              (long long)hc->stat_rounds);
    if (getenv("VATLQ_PASS_PHASES"))
      fprintf(stderr, "[vatlq] pass phases as seen by CTA 0, us per launch: prologue %.1f, tiles %.1f, finishing %.1f, publish %.1f (%lld launches)\n",
              hc->stat_ns_pass[0] / 1e3 / std::max<long long>(1, hc->stat_passes), hc->stat_ns_pass[1] / 1e3 / std::max<long long>(1, hc->stat_passes),
              hc->stat_ns_pass[2] / 1e3 / std::max<long long>(1, hc->stat_passes), hc->stat_ns_pass[3] / 1e3 / std::max<long long>(1, hc->stat_passes),
              (long long)hc->stat_passes);
    PruneCtl hp{};     // this call's tiles seen / streamed / verify violations / segments (no process-wide state needed)
    if (cudaMemcpy(&hp, P.pc, sizeof(PruneCtl), cudaMemcpyDeviceToHost) == cudaSuccess) {
      host_stats[11] = (int64_t)hp.stats[0];
      host_stats[12] = (int64_t)hp.stats[1];
      host_stats[13] = (int64_t)hp.stats[2];
      host_stats[14] = hp.nseg;
    }
  }
  return rc;
}

extern "C" int vatlq_coreset_select_dt(const void* X, int dtype, int64_t n, int d, int64_t row_lo, int64_t row_hi,
                                       double* min_d, double* unc, int rule, double moks, double lambda,
                                       int64_t n_labeled, int64_t first_pick, int64_t k, int batch, int64_t* out_idx,
                                       void* comm, void* ws, size_t ws_bytes, int64_t* host_stats,
                                       vatlq_stream_t stream) {
  if (int e = check_coreset_x(X, dtype, n, d, row_lo, row_hi)) return e;
  return with_dtype(dtype, [&](auto t) {
    using T = std::remove_cv_t<std::remove_pointer_t<decltype(t)>>;
    return coreset_select<T>(static_cast<const T*>(X), dtype, n, d, row_lo, row_hi, min_d, unc, rule, moks, lambda,
                             n_labeled, first_pick, k, batch, out_idx, comm, ws, ws_bytes, host_stats, (cudaStream_t)stream);
  });
}
extern "C" int vatlq_coreset_select(const float* X, int64_t n, int d, int64_t row_lo, int64_t row_hi,
                                    double* min_d, double* unc, int rule, double moks, double lambda,
                                    int64_t n_labeled, int64_t first_pick, int64_t k, int batch,
                                    int64_t* out_idx, void* comm, void* ws, size_t ws_bytes,
                                    int64_t* host_stats, vatlq_stream_t stream) {
  return vatlq_coreset_select_dt(X, VATLQ_F32, n, d, row_lo, row_hi, min_d, unc, rule, moks, lambda, n_labeled,
                                 first_pick, k, batch, out_idx, comm, ws, ws_bytes, host_stats, stream);
}

extern "C" int vatlq_coreset_set_prune(int mode, int64_t min_rows) {
  VQ_REQUIRE(mode >= -1 && mode <= 2, "mode must be -1 (environment), 0 (off), 1 (prune) or 2 (verify)");
  g_prune_mode_set = mode;
  g_prune_min_set = min_rows < 0 ? -1 : (long long)min_rows;
  return 0;
}

extern "C" int vatlq_coreset_set_screen(int mode) {
  VQ_REQUIRE(mode >= -1 && mode <= 2, "mode must be -1 (environment), 0 (off), 1 (screen) or 2 (verify)");
  g_screen_mode_set = mode;
  return 0;
}

extern "C" int vatlq_coreset_screen_stats(int64_t* host_out3, int reset) {
  if (host_out3)
    for (int i = 0; i < 3; ++i) host_out3[i] = g_screen[i];
  if (reset) g_screen[0] = g_screen[1] = g_screen[2] = 0;
  return 0;
}

extern "C" int vatlq_coreset_prune_stats(int64_t* host_out4, int reset) {
  if (host_out4)
    for (int i = 0; i < 4; ++i) host_out4[i] = g_prune[i];
  if (reset) g_prune[0] = g_prune[1] = g_prune[2] = g_prune[3] = 0;
  return 0;
}

extern "C" int vatlq_pairwise_dist_dt(const void* X, int dtype, int64_t n, int d, const int64_t* centers, int64_t m,
                                      double* out, void* ws, size_t ws_bytes, vatlq_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (int e = check_x(X, dtype, n, d, 0, n)) return e;
  VQ_REQUIRE(centers && out && m > 0, "null pointer");
  VQ_REQUIRE(ws != nullptr && ws_bytes >= (size_t)n * sizeof(double), "workspace must hold n doubles");
  const long long colblocks = (m + kB - 1) / kB;
  VQ_REQUIRE(colblocks <= 2147483647LL, "too many centers");
  if (int e = configure_pass()) return e;
  const Geom G = geom_of(d);
  double* xx = (double*)ws;
  const int gy = (int)std::max<long long>(1, std::min<long long>(64, (n + 127) / 128));
  dim3 grid((unsigned)colblocks, (unsigned)gy);
  return with_dtype(dtype, [&](auto t) {
    using T = std::remove_cv_t<std::remove_pointer_t<decltype(t)>>;
    const T* XT = static_cast<const T*>(X);
    if (int e = launch_norms(XT, n, d, xx, stream)) return e;
    pairwise_kernel<T><<<grid, 256, G.smem, stream>>>(XT, n, G.d4, G.nss, G.S, G.guard, xx, (const long long*)centers, m, out);
    VQ_LAUNCHED();
    return 0;
  });
}
extern "C" int vatlq_pairwise_dist(const float* X, int64_t n, int d, const int64_t* centers, int64_t m,
                                   double* out, void* ws, size_t ws_bytes, vatlq_stream_t stream) {
  return vatlq_pairwise_dist_dt(X, VATLQ_F32, n, d, centers, m, out, ws, ws_bytes, stream);
}

// ---------------------------------------------------------------- communicator
extern "C" int vatlq_comm_unique_id(void* host_id128) {
  VQ_REQUIRE(host_id128 != nullptr, "null id buffer");
  if (int e = load_nccl()) return e;
  const int e = g_nccl.GetUniqueId(host_id128);
  if (e != 0) {
    snprintf(g_err, sizeof(g_err), "ncclGetUniqueId failed (%d)", e);
    return VATLQ_ECOMM;
  }
  return 0;
}

extern "C" int vatlq_comm_init(const void* host_id128, int rank, int world, void** comm_out) {
  VQ_REQUIRE(host_id128 && comm_out && world >= 1 && rank >= 0 && rank < world, "bad arguments");
  VQ_REQUIRE(world <= kMaxRanks, "world too large");
  if (int e = load_nccl()) return e;
  Id128 id;
  memcpy(id.b, host_id128, 128);
  void* c = nullptr;
  const int e = g_nccl.CommInitRank(&c, world, id, rank);
  if (e != 0) {
    snprintf(g_err, sizeof(g_err), "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(e) : "?");
    return VATLQ_ECOMM;
  }
  Comm* cm = new Comm();
  cm->nccl = c;
  cm->rank = rank;
  cm->world = world;
  *comm_out = cm;
  return 0;
}

// ---- peer-memory mailbox: each rank allocates one, exports its IPC handle, imports the others'
extern "C" int vatlq_comm_mailbox_handle(void* comm, void* host_handle64) {
  VQ_REQUIRE(comm && host_handle64, "null argument");
  Comm* cm = (Comm*)comm;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (!cm->mail) {
    VQ_CUDA(cudaMalloc((void**)&cm->mail, sizeof(Mailbox)));
    VQ_CUDA(cudaMemset(cm->mail, 0, sizeof(Mailbox)));
  }
  cudaIpcMemHandle_t h;
  VQ_CUDA(cudaIpcGetMemHandle(&h, cm->mail));
  memcpy(host_handle64, &h, 64);
  return 0;
}

extern "C" int vatlq_comm_attach(void* comm, const void* host_handles, int world) {
  VQ_REQUIRE(comm && host_handles, "null argument");
  Comm* cm = (Comm*)comm;
  VQ_REQUIRE(world == cm->world && cm->mail != nullptr, "attach after vatlq_comm_mailbox_handle, same world size");
  Mailbox* ptrs[kMaxRanks] = {};
  for (int r = 0; r < world; ++r) {
    if (r == cm->rank) {
      ptrs[r] = cm->mail;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)host_handles + 64 * r, 64);
    void* p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      snprintf(g_err, sizeof(g_err), "cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
      for (int q = 0; q < r; ++q)
        if (cm->opened[q]) {
          cudaIpcCloseMemHandle(cm->opened[q]);
          cm->opened[q] = nullptr;
        }
      return VATLQ_ECOMM;
    }
    cm->opened[r] = p;
    ptrs[r] = (Mailbox*)p;
  }
  if (const char* e = getenv("VATLQ_MAILBOX_TIMEOUT_S")) {
    const double sec = atof(e);
    if (sec > 0.0) {
      const long long clk = (long long)(sec * 2.0e9);
      VQ_CUDA(cudaMemcpyToSymbol(g_mail_timeout_clk, &clk, sizeof(clk)));
    }
  }
  VQ_CUDA(cudaMalloc((void**)&cm->peers_dev, sizeof(Mailbox*) * kMaxRanks));
  VQ_CUDA(cudaMemcpy(cm->peers_dev, ptrs, sizeof(Mailbox*) * kMaxRanks, cudaMemcpyHostToDevice));
  return 0;
}

extern "C" int vatlq_comm_destroy(void* comm) {
  if (!comm) return 0;
  Comm* cm = (Comm*)comm;
  cudaDeviceSynchronize();
  for (int r = 0; r < kMaxRanks; ++r)
    if (cm->opened[r]) cudaIpcCloseMemHandle(cm->opened[r]);
  if (cm->peers_dev) cudaFree(cm->peers_dev);
  if (cm->mail) cudaFree(cm->mail);
  if (g_nccl.CommDestroy && cm->nccl) g_nccl.CommDestroy(cm->nccl);
  delete cm;
  return 0;
}

// ---------------------------------------------------------------- profiling hooks
extern "C" int vatlq_profile_passes(int enable) {
  if (enable && g_prof.ev.empty()) {
    g_prof.ev.resize(2 * 8192);
    for (auto& e : g_prof.ev) VQ_CUDA(cudaEventCreate(&e));
  }
  g_prof.on = enable != 0;
  return 0;
}

extern "C" int vatlq_profile_read(double* total_ms, int64_t* launches, int64_t* picks, int reset) {
  if (total_ms) *total_ms = g_prof.total_ms;
  if (launches) *launches = g_prof.timed;
  if (picks) *picks = g_prof.picks;
  if (reset) {
    g_prof.total_ms = 0.0;
    g_prof.timed = 0;
    g_prof.picks = 0;
  }
  return 0;
}
