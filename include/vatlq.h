/*
 * vatlq.h — C ABI of libvatlq.so, the B200 (sm_100a) implementation of VATL4Pose's
 * active-learning query pass.
 *
 * The reference (ImIntheMiddle/VATL4Pose-WACV2024) has no FFI for this path: the boundary
 * is Python (`ActiveLearning.eval_and_query`, active_learning/ActiveLearning.py:253-649).
 * Each entry point below names the reference function whose arithmetic it replaces; the
 * Python host layer (vatl4pose-wacv2024_b200/) binds these with ctypes and mirrors the
 * reference's callables.  INTEGRATION.md shows the reference-side binding.
 *
 * Conventions
 *   - every pointer is a BORROWED device pointer (torch.Tensor.data_ptr()) unless the
 *     parameter name starts with `host_`; the library never frees caller memory.
 *   - scratch comes from the caller: query `*_workspace_bytes()` and pass `ws`.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), except the
 *     ones documented as synchronising.
 *   - return 0 on success, a cudaError_t (>0) or a negative VATLQ_E* code otherwise;
 *     `vatlq_last_error()` returns a thread-local message.
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef VATLQ_H
#define VATLQ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VATLQ_ABI_VERSION 1

#define VATLQ_EINVAL (-1)  /* bad argument (shape, alignment, null pointer)        */
#define VATLQ_ENOMEM (-2)  /* workspace too small                                  */
#define VATLQ_ECOMM (-3)   /* NCCL missing or a collective failed                  */
#define VATLQ_ESTATE (-4)  /* internal invariant violated (reported, never hidden) */

typedef void* vatlq_stream_t; /* cudaStream_t */

/* Heat-map element types of the *_dt entry points.  Every fp16 and bf16 value is exactly representable in fp32
 * and the kernels convert at the load, so for H in fp16 or bf16 every output of a *_dt call equals, bit for bit,
 * what the fp32 entry point returns for the exact upcast of H (NaN positions included).  Halos and prev / next
 * tensors must share H's dtype.  16-bit heat maps must be 8-byte aligned wherever the fp32 form needs 16 bytes
 * (the scan's H stays 16-byte aligned: its maps are fetched by TMA bulk copies).  An unknown dtype or a
 * misaligned pointer returns VATLQ_EINVAL before any device work. */
#define VATLQ_F32 0
#define VATLQ_F16 1
#define VATLQ_BF16 2

int vatlq_abi_version(void);
const char* vatlq_last_error(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
uint64_t vatlq_launch_count(void);

/* ------------------------------------------------------------------------------------
 * Heat-map scan: THC + local-peak statistics + argmax / quarter-pixel coordinates.
 * Replaces, for a whole id-sorted pool at once,
 *   ActiveLearning.compute_thc            active_learning/ActiveLearning.py:747-760
 *   its call-site logic (x2 rule)         active_learning/ActiveLearning.py:345-363
 *   localpeak_values / localpeak_mean     active_learning/local_peak.py:5-22
 *   heatmap_to_coord_simple/get_max_pred  alphapose/utils/transforms.py:550-583,710-727
 *   transform_preds/get_affine_transform  alphapose/utils/transforms.py:704-708,753-792
 *
 * H          (n,J,h,w) fp32 contiguous heat maps (vatlq_heatmap_scan_dt: fp16 / bf16 too); every frame is
 *            read from HBM once.
 * is_prev/is_next  u8[n] track-adjacency flags (alphapose/datasets/posetrack21.py:148-178);
 *            the t-1 / t+1 maps are H[t-1] / H[t+1] (SURVEY.md §7.3-7).
 * halo_prev/halo_next  optional (J,h,w) frames that precede H[0] / follow H[n-1] when the
 *            pool is a shard or a chunk of a longer pool (NULL: no such neighbour).
 * bbox_xyxy  optional fp32[n,4] crop boxes; required for kpts.
 * Outputs (any may be NULL to skip):
 *   thc[n]        fp32  temporal heat-map continuity
 *   peak_sum[n], peak_cnt[n], peak_mean[n]  kept-peak sum / count / mean (NaN when count 0)
 *   coords_hm[n,J,2]  fp32 heat-map-space (x,y) incl. the +-0.25 shift  (bit-exact)
 *   kpts[n,J,3]   fp32 image-space x, y and peak value == the reference's `keypoints` row
 *                 (ActiveLearning.py:306-307)
 * ------------------------------------------------------------------------------------ */
size_t vatlq_heatmap_scan_workspace_bytes(int64_t n, int J);
int vatlq_heatmap_scan(const float* H, const uint8_t* is_prev, const uint8_t* is_next,
                       int64_t n, int J, int h, int w,
                       const float* halo_prev, const float* halo_next,
                       const float* bbox_xyxy,
                       float* thc, float* peak_sum, int32_t* peak_cnt, float* peak_mean,
                       float* coords_hm, float* kpts,
                       void* ws, size_t ws_bytes, vatlq_stream_t stream);
/* The same scan of H in any VATLQ_* dtype (vatlq_heatmap_scan is this call with VATLQ_F32).  In 16 bits the scan
 * reads 104 448 B per 17 x 64 x 48 frame (half of fp32) and writes 212 B (thc, peak_sum / cnt / mean, coords_hm,
 * kpts); halo_prev / halo_next are (J,h,w) frames of H's dtype.  Workspace as vatlq_heatmap_scan_workspace_bytes. */
int vatlq_heatmap_scan_dt(const void* H, int dtype, const uint8_t* is_prev, const uint8_t* is_next,
                          int64_t n, int J, int h, int w,
                          const void* halo_prev, const void* halo_next,
                          const float* bbox_xyxy,
                          float* thc, float* peak_sum, int32_t* peak_cnt, float* peak_mean,
                          float* coords_hm, float* kpts,
                          void* ws, size_t ws_bytes, vatlq_stream_t stream);

/* Strict three-tensor THC (cur, prev, next separately forwarded as the reference does,
 * ActiveLearning.py:293-297,345-363).  prev/next may be NULL when no flag needs them. */
int vatlq_thc3(const float* cur, const float* prev, const float* next,
               const uint8_t* is_prev, const uint8_t* is_next,
               int64_t n, int J, int h, int w, float* thc, vatlq_stream_t stream);
/* vatlq_thc3 with cur / prev / next in one VATLQ_* dtype */
int vatlq_thc3_dt(const void* cur, const void* prev, const void* next, int dtype,
                  const uint8_t* is_prev, const uint8_t* is_next,
                  int64_t n, int J, int h, int w, float* thc, vatlq_stream_t stream);

/* ------------------------------------------------------------------------------------
 * WPU: hybrid feature + whole-body auto-encoder + reconstruction MSE.  Replaces
 *   bbox_xyxy_to_xywh    alphapose/utils/bbox.py:91-97
 *   compute_hybrid       active_learning/Whole_body_AE/hybrid_feature.py:14-58 (fp64)
 *   WholeBodyAE.forward  active_learning/Whole_body_AE/AutoEncoder.py:13-39   (fp32)
 *   MSELoss call sites   active_learning/ActiveLearning.py:364-370 (all dims) and
 *                        :371-386 (drop_ears: dims 3,4,20,21 removed)
 * kpts[n,17,3] fp32 (x,y,score), bbox_xyxy[n,4] fp32 crop boxes.
 * weights: the 8 Linear layers packed back to back, each W[out][in] row-major then b[out],
 *          dims in_dim->24->12->7->z_dim->7->12->24->in_dim (in_dim must be 42).
 * wpu[n] fp32; feat (optional) fp32[n,in_dim] = the `.float()` feature fed to the AE;
 * status[n] u8: 0 ok, 1 height<=0, 2 sum(scores)<=0 (the reference's AssertionErrors,
 * hybrid_feature.py:25,31); wpu is NaN for those rows.
 * ------------------------------------------------------------------------------------ */
size_t vatlq_wpu_weight_count(int in_dim, int z_dim);
int vatlq_wpu(const float* kpts, const float* bbox_xyxy, const float* weights,
              int in_dim, int z_dim, int drop_ears,
              float* wpu, float* feat, uint8_t* status, int64_t n, vatlq_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Score fusion (active_learning/ActiveLearning.py:490-516) in float64 on the device.
 * Three steps so that a multi-GPU caller can all-reduce the 4 / 2 statistics in between:
 *   stats1[4] = {min thc, -max thc, min wpu, -max wpu} over rows with unlabeled[i]!=0
 *   combine   : u_i = combine(minmax(thc_i), minmax(wpu_i)); stats2[2] = {min u, -max u}
 *   final     : unc_i = minmax(u_i) for unlabelled rows, 0 for labelled rows
 * (all statistics are stored "min of value / min of negated value" so one MIN all-reduce
 * serves).  mode: 0 const (a+b), 1 increase, 2 decrease, 3 single criterion (wpu ignored).
 * ------------------------------------------------------------------------------------ */
int vatlq_fuse_stats(const float* thc, const float* wpu, const uint8_t* unlabeled, int64_t n,
                     double* stats1, vatlq_stream_t stream);
int vatlq_fuse_combine(const float* thc, const float* wpu, const uint8_t* unlabeled, int64_t n,
                       const double* stats1, int mode, double labeled_ratio,
                       double* u, double* stats2, vatlq_stream_t stream);
int vatlq_fuse_final(const uint8_t* unlabeled, int64_t n, const double* stats2,
                     double* u_inout, vatlq_stream_t stream);

/* ------------------------------------------------------------------------------------
 * k-center greedy core-set (ActiveLearning.coreset_selection,
 * active_learning/ActiveLearning.py:798-850; sklearn euclidean pairwise_distances in fp64).
 *
 * X[n,d] fp32 row-major (the reference holds the same values as float64, :270,286); all
 * distance arithmetic accumulates in fp64.  d must be a multiple of 4, X 16-byte aligned.
 * The handle owns nothing but small control blocks inside `ws`.
 *
 * Multi-GPU: X is replicated, rows [row_lo,row_hi) are owned by this rank; min_d / unc are
 * full-length arrays of which only the owned slice is maintained.  comm is a handle from
 * vatlq_comm_init (NULL for one GPU).
 *
 *   rule: 0 w_unc       argmax((1-moks)*min_d + (lambda*moks)*unc)   (:815-821)
 *         1 fixed       argmax(min_d + lambda*unc)                   (:822-827)
 *         2 dist        argmax(min_d); first pick given by caller    (:828-833)
 *   n_labeled == 0: the first pick is argmax(unc) (rule 0/1) or `first_pick` (rule 2).
 *   batch: 1 = one pick per round (GEMV form: plain arg-max, one pass over X per pick);
 *          >1 = up to `batch` (<= 16) picks per round, decided exactly in advance on a candidate
 *          set and applied 8 per pass over X (DESIGN.md §4.4).
 * out_idx[k] int64 picks in order (device).  min_d[n] fp64 in/out (initialised by
 * vatlq_coreset_init), unc[n] fp64 in/out (picked entries zeroed like :848).
 * host_stats (optional, 16 x int64, host memory, written at the end — the call synchronises
 * anyway): [0] passes over X, [1] picks, [2] rounds planned, [3] fallback rounds (nothing listed),
 * [4] fallback rounds (list overflow), [5] sum of candidates, [6] rounds launched, [7] picks per
 * round, [8..10] ns spent waiting for the peers' candidate blocks / in the candidate x candidate
 * tiles / in the planner (summed over the rounds), [11..14] this call's pruning statistics: tiles seen,
 * tiles streamed, verify violations, segments; [15] reserved.
 * ------------------------------------------------------------------------------------ */
size_t vatlq_coreset_workspace_bytes(int64_t n, int d, int batch);
int vatlq_coreset_init(const float* X, int64_t n, int d, int64_t row_lo, int64_t row_hi,
                       const int64_t* labeled, int64_t n_labeled,
                       double* min_d, void* ws, size_t ws_bytes, vatlq_stream_t stream);
int vatlq_coreset_select(const float* X, int64_t n, int d, int64_t row_lo, int64_t row_hi,
                         double* min_d, double* unc,
                         int rule, double moks, double lambda, int64_t n_labeled,
                         int64_t first_pick, int64_t k, int batch,
                         int64_t* out_idx, void* comm,
                         void* ws, size_t ws_bytes, int64_t* host_stats, vatlq_stream_t stream);

/* Labelled-set initialisation on the 5th-generation tensor cores (d == 2048): same result as
 * vatlq_coreset_init — min_d[i] = min over the labelled rows of the canonical fp64 distance, bit for bit —
 * but the N x L contraction runs as a TF32 tcgen05.mma GEMM (2-D TMA loads, fp32 accumulators in TMEM) whose
 * result, with a proved error bound, only decides WHICH (row, centre) pairs can be the minimum; those are
 * re-scored with the canonical fp64 arithmetic (csrc/tc_dist.cu).  Replaces sklearn's N x L distance matrix
 * of ActiveLearning.py:802-814,841.  ws from vatlq_coreset_init_tc_workspace_bytes(n, row_hi-row_lo, n_labeled).
 * flags & 1: also check a sample of the TF32 values against the bound (host_stats4[2] must stay 0).
 * host_stats4 = {pairs listed, pair capacity, bound violations, centre groups}; tmin_out (optional, fp32
 * [row_hi-row_lo]): the approximate minimum squared distance per row.  Returns VATLQ_ESTATE when the
 * candidate list overflows (call vatlq_coreset_init instead).  The call synchronises the stream. */
size_t vatlq_coreset_init_tc_workspace_bytes(int64_t n, int64_t n_owned, int64_t n_labeled);
int vatlq_coreset_init_tc(const float* X, int64_t n, int d, int64_t row_lo, int64_t row_hi,
                          const int64_t* labeled, int64_t n_labeled, double* min_d,
                          void* ws, size_t ws_bytes, int flags, int64_t* host_stats4, float* tmin_out,
                          vatlq_stream_t stream);

/* Exact pruning of the passes over X (d == 2048, >= VATLQ_PRUNE_MIN_ROWS owned rows, default 8192):
 * consecutive rows of an id-sorted pool are near each other, so the owned rows are cut into segments
 * with an anchor row and a radius, and a pass does not stream the 8-row tiles whose segments
 * provably (triangle inequality, with a margin far above the fp64 rounding) cannot get closer to
 * any of the pass's centres.  The pick list is unchanged.  Environment: VATLQ_PRUNE=0 disables,
 * VATLQ_PRUNE=verify streams everything and counts rows of flagged tiles whose min_d moved.
 * host_out4 = {tiles seen, tiles streamed, verify violations (must be 0), segments of the last
 * call}, accumulated over the vatlq_coreset_select calls since the last reset. */
int vatlq_coreset_prune_stats(int64_t* host_out4, int reset);
/* process-wide override of the two environment settings: mode -1 environment, 0 off, 1 prune,
 * 2 verify; min_rows < 0: environment */
int vatlq_coreset_set_prune(int mode, int64_t min_rows);

/* The TF32 screen of the 16-pick rounds (d == 2048): before a round's fp64 pass each streamed row is
 * compared with the round's centres on the tensor cores, and only the rows that an error bound cannot
 * prove unchanged (min_d[i] <= d(i,c) for every centre) go through the exact fp64 arithmetic.  The pick
 * list and min_d are unchanged bit for bit.  Environment: VATLQ_PASS_SCREEN=0 disables,
 * VATLQ_PASS_SCREEN=verify computes every streamed row exactly and counts the rows the screen did not
 * list whose min_d moved.  host_out3 = {rows screened, rows listed, verify violations (must be 0)},
 * accumulated over the vatlq_coreset_select calls since the last reset. */
int vatlq_coreset_screen_stats(int64_t* host_out3, int reset);
/* process-wide override of VATLQ_PASS_SCREEN: -1 environment, 0 off, 1 screen, 2 verify */
int vatlq_coreset_set_screen(int mode);

/* One pairwise-distance column block, exposed for parity tests of the distance arithmetic:
 * out[i*m + j] = d(X[i], X[centers[j]]) in fp64 (sklearn _euclidean_distances order). */
int vatlq_pairwise_dist(const float* X, int64_t n, int d, const int64_t* centers, int64_t m,
                        double* out, void* ws /* >= n*8 bytes */, size_t ws_bytes, vatlq_stream_t stream);

/* ------------------------------------------------------------------------------------
 * SURVEY.md 8f "next" rows: the other per-item uncertainties and the representativeness step.
 *
 * vatlq_pose_unc — pose-level uncertainties from the scan's outputs (no second pass over H):
 *   hp[n]  fp32  HP  = float(-np.sum(pose_scores))            ActiveLearning.py:329-330
 *   tpc[n] fp32  TPC = #joints that moved more than 0.01*sqrt(box area) between frame t and
 *                t-1 / t+1, the neighbour decoded with frame t's crop box, doubled when only
 *                one neighbour exists                          ActiveLearning.py:333-344,736-745
 *   coords_hm[n,J,2] / kpts[n,J,3] as written by vatlq_heatmap_scan; halo_*_xy: optional
 *   (J,2) heat-map-space coordinates of the frames next to the range (shards / chunks).
 * vatlq_heatmap_entropy — Entropy = sum_j scipy.stats.entropy(H[t,j].flatten()), fp32
 *   (ActiveLearning.py:790-796; -inf when a map holds negative values, NaN when it sums to 0);
 *   one streaming pass, ws >= n*J*4 bytes.
 * ------------------------------------------------------------------------------------ */
int vatlq_pose_unc(const float* coords_hm, const float* kpts, const float* bbox_xyxy,
                   const uint8_t* is_prev, const uint8_t* is_next, int64_t n, int J, int h, int w,
                   const float* halo_prev_xy, const float* halo_next_xy, float* hp, float* tpc,
                   vatlq_stream_t stream);
int vatlq_heatmap_entropy(const float* H, int64_t n, int J, int h, int w, float* entropy,
                          void* ws, size_t ws_bytes, vatlq_stream_t stream);
/* vatlq_heatmap_entropy of H in any VATLQ_* dtype */
int vatlq_heatmap_entropy_dt(const void* H, int dtype, int64_t n, int J, int h, int w, float* entropy,
                             void* ws, size_t ws_bytes, vatlq_stream_t stream);

/* Influence (ActiveLearning.py:467-477) and Diversity (:581-590): row sums of the cosine-distance
 * matrix that KNeighborsTransformer(mode='distance', metric='cosine', n_neighbors=m-1) builds
 * over the rows X[rows[0..m)] (rows == NULL: all n rows, m == n), via
 *   sum_j (1 - xh_i . xh_j) = m_total - xh_i . S,   S = sum_j xh_j,  xh = x / |x|   (fp64)
 * Two calls so that a multi-GPU caller can all-reduce S (SUM) in between:
 *   colsum: S[d] over this rank's rows;  rowsum: out[m] = m_total - (x_i . S) / |x_i|.
 * d must be a multiple of 4 and <= 2048; ws from vatlq_cosine_workspace_bytes(d). */
size_t vatlq_cosine_workspace_bytes(int d);
int vatlq_cosine_colsum(const float* X, int64_t n, int d, const int64_t* rows, int64_t m,
                        double* S, void* ws, size_t ws_bytes, vatlq_stream_t stream);
int vatlq_cosine_rowsum(const float* X, int64_t n, int d, const int64_t* rows, int64_t m,
                        const double* S, double m_total, double* out, vatlq_stream_t stream);

/* stats2[2] = {min v, -max v} over rows with mask != 0 (mask NULL: all rows): the statistics
 * vatlq_fuse_final consumes, for fp64 score vectors (influence normalisation, :477). */
int vatlq_minmax_stats_f64(const double* v, const uint8_t* mask, int64_t n, double* stats2,
                           vatlq_stream_t stream);
/* out_i = cw*unc_i + (1-cw)*infl_i on rows with mask != 0, else 0 (ActiveLearning.py:519). */
int vatlq_fuse_blend(const double* unc, const double* infl, const uint8_t* mask, int64_t n,
                     double combine_weight, double* out, vatlq_stream_t stream);

/* MPE and Margin uncertainties (ActiveLearning.py:762-788): per joint map the <= 5 peaks of
 * skimage.feature.peak_local_max(map, min_distance=5, num_peaks=5) — 11x11 maximum filter with edge
 * replication, pixel > map minimum, 5-pixel border excluded, greedy spacing in descending value —
 * MPE = sum_j entropy(softmax(peaks_j)), Margin = sum_j |peak_0 - peak_1| (fp32).  Either output may be NULL.
 * ws >= vatlq_peak_workspace_bytes(n, J, h, w).  64 x 48 maps take a register / warp-shuffle fast path; maps whose
 * peak-candidate list overflows (plateaus) are redone by the generic routine — same result either way.
 * (scikit-image is absent from the build container: parity with the library itself is
 * pinned only against a restatement of its published algorithm, oracle/vatl_oracle.py.) */
size_t vatlq_peak_workspace_bytes(int64_t n, int J, int h, int w);
int vatlq_peak_unc(const float* H, int64_t n, int J, int h, int w, float* mpe, float* margin,
                   void* ws, size_t ws_bytes, vatlq_stream_t stream);
/* vatlq_peak_unc of H in any VATLQ_* dtype (same workspace) */
int vatlq_peak_unc_dt(const void* H, int dtype, int64_t n, int J, int h, int w, float* mpe, float* margin,
                      void* ws, size_t ws_bytes, vatlq_stream_t stream);

/* Candidate ordering on the device (ActiveLearning.py:527-538, 587-589): out_idx[n] = row ids with mask != 0
 * (mask NULL: all) by descending (descending != 0) or ascending score, equal scores in ascending id order —
 * the order Python's stable sorted(..., reverse=True) yields; masked-out rows follow at the end. */
size_t vatlq_rank_workspace_bytes(int64_t n);
int vatlq_rank_scores(const double* score, const uint8_t* mask, int64_t n, int descending, int64_t* out_idx,
                      void* ws, size_t ws_bytes, vatlq_stream_t stream);

/* OKS of every item against its ground-truth pose (active_learning/al_metric.py:42-69, call site
 * ActiveLearning.py:309): kpts / gt_kpts [n,17,3] fp32 (x, y, score | visibility), bbox_ann_xyxy [n,4]
 * (converted like alphapose/utils/bbox.py:91-97), oks[n] fp64.  The controller derives moks_queried
 * (:858, the core-set's score weights :815-821) and the stopping criteria (:707-725) from it. */
int vatlq_oks(const float* kpts, const float* gt_kpts, const float* bbox_ann_xyxy, int64_t n, double* oks,
              vatlq_stream_t stream);

/* ------------------------------------------------------------------------------------
 * K-Means / weighted K-Means query filters (ActiveLearning.py:593-608 and :553-580): the device side of
 * sklearn.cluster.KMeans(n_clusters=query_size, random_state=318).fit_predict(embeddings[, sample_weight]) followed
 * by "per cluster, the member closest to its centre".  sklearn's algorithm (1.7.1 pinned by the reference:
 * _kmeans.py _kmeans_plusplus / _kmeans_single_lloyd, _k_means_lloyd.pyx, _k_means_common.pyx) in fp64 over the
 * fp32 embeddings; both GEMM-shaped steps run on the fp64 tensor cores.  The host layer (kmeans.py) draws the random
 * numbers from numpy's RandomState exactly as sklearn does and decides convergence from a few scalars.
 * X (n,d) fp32 row-major, 16-byte aligned, d % 4 == 0, n < 2^31; w fp64[n] sample weights or NULL (all 1).
 * One workspace of vatlq_kmeans_workspace_bytes(n,d,k) serves every call (they never overlap).
 *
 * Which bits matter: label decisions are robust to rounding, but the closest member of a TWO-member cluster is a
 * structural tie that the reference resolves by the rounding of its own arithmetic; the M step and the final
 * distances therefore follow sklearn / numpy operation by operation in the centred frame (see csrc/kmeans.cu).
 *
 * _mean_var   mean[d] = X.mean(axis=0) (numpy's sequential order), out1[0] = np.mean(np.var(X, axis=0)) (_tolerance)
 * _pp         k-means++ seeding: center_ids[k] (row ids), closest[n] = squared distance to the nearest seed.
 *             first_center = random_state.choice(n, p=w/sum(w)); rand_vals[(k-1)*trials] = the uniform draws of the
 *             k-1 later steps in order, trials = 2 + int(log(k)) <= 16.  No host synchronisation inside.
 * _gather     Cc[k][d] = X[ids[j]] - mean (centred frame, where sklearn keeps its centres), Cr = Cc + mean
 * _assign     labels[i] = first argmin_j (|c_j|^2 - 2 x_i.c_j) over the raw-frame centres C; *changed = #rows with
 *             labels[i] != labels_old[i] (labels_old / changed may be NULL)
 * _update     M step: order[n] = rows sorted by (label, row), starts[k+1], sums[k][d] = sum (x_i - mean) w_i in
 *             ascending row order, wsum[k], *n_empty = #clusters with zero weight
 * _relocate   _relocate_empty_clusters_dense for the (empty cluster, far row) pairs the host chose
 * _average    Cc_new = sums * (1 / wsum) (argmax_weight >= 0: clusters that stayed empty copy that cluster's row the
 *             way _average_centers does), Cr_new = Cc_new + mean, shift[j] = |Cc_new[j] - Cc_old[j]|
 * _rowdist    dis[i] = ((x_i - C[labels[i]]) ** 2).sum() in numpy's pairwise summation order     (:601-602)
 * _pick       picks[j] = member of cluster j with the smallest dis, lowest row on ties; -1 for an empty cluster (:603)
 * ------------------------------------------------------------------------------------ */
size_t vatlq_kmeans_workspace_bytes(int64_t n, int d, int64_t k);
int vatlq_kmeans_mean_var(const float* X, int64_t n, int d, double* mean, double* out1, void* ws, size_t ws_bytes,
                          vatlq_stream_t stream);
int vatlq_kmeans_pp(const float* X, int64_t n, int d, const double* w, int64_t k, int64_t first_center,
                    const double* rand_vals, int trials, int32_t* center_ids, double* closest, void* ws, size_t ws_bytes,
                    vatlq_stream_t stream);
int vatlq_kmeans_gather(const float* X, int d, const int32_t* ids, int64_t k, const double* mean, double* Cc, double* Cr,
                        vatlq_stream_t stream);
int vatlq_kmeans_assign(const float* X, int64_t n, int d, const double* C, int64_t k, int32_t* labels,
                        const int32_t* labels_old, int32_t* changed, void* ws, size_t ws_bytes, vatlq_stream_t stream);
int vatlq_kmeans_update(const float* X, int64_t n, int d, const double* w, const double* mean, const int32_t* labels,
                        int64_t k, double* sums, double* wsum, int32_t* order, int32_t* starts, int32_t* n_empty, void* ws,
                        size_t ws_bytes, vatlq_stream_t stream);
int vatlq_kmeans_relocate(const float* X, int d, const double* w, const double* mean, const int32_t* labels,
                          const int32_t* empty_ids, const int32_t* far_ids, int n_empty, double* sums, double* wsum,
                          vatlq_stream_t stream);
int vatlq_kmeans_average(const double* sums, const double* wsum, int64_t k, int d, int64_t argmax_weight,
                         const double* mean, const double* Cc_old, double* Cc_new, double* Cr_new, double* shift,
                         vatlq_stream_t stream);
int vatlq_kmeans_rowdist(const float* X, int64_t n, int d, const double* C, const int32_t* labels, double* dis,
                         vatlq_stream_t stream);
int vatlq_kmeans_pick(const double* dis, const int32_t* order, const int32_t* starts, int64_t k, int32_t* picks,
                      vatlq_stream_t stream);

/* fp64 tensor-core (mma.sync.m8n8k4.f64, DMMA) peak of the current device in FMA/s, measured with a saturating
 * register-only kernel (about 10 ms): the roofline denominator of the paired core-set pass, which is bound by the
 * DMMA pipe rather than by HBM.  ws >= 4 * SMs * 256 * 8 bytes. */
int vatlq_measure_fp64_mma(double* host_fma_per_s, void* ws, size_t ws_bytes, vatlq_stream_t stream);

/* Timing of the dominant kernel (the pass over X) for bench.py's roofline: when enabled,
 * vatlq_coreset_select brackets every pass launch with CUDA events on `stream`; read returns
 * the summed duration of the passes that applied picks, their number and the picks applied.
 * The picks counter only covers chunks of rounds that were timed from their first launch. */
int vatlq_profile_passes(int enable);
int vatlq_profile_read(double* host_total_ms, int64_t* host_launches, int64_t* host_picks, int reset);

/* ------------------------------------------------------------------------------------
 * NCCL plumbing for the multi-GPU argmax exchange (one process per GPU).  NCCL is
 * dlopen()ed (libnccl.so.2, the copy torch already loaded); absent -> VATLQ_ECOMM.
 * ------------------------------------------------------------------------------------ */
int vatlq_comm_unique_id(void* host_id128);                 /* rank 0: 128-byte id       */
int vatlq_comm_init(const void* host_id128, int rank, int world, void** comm_out);
/* Optional peer-memory candidate exchange (replaces the per-round ncclAllGather with NVLink peer
 * stores + flags issued by the kernels themselves): every rank calls _mailbox_handle (64-byte
 * cudaIpcMemHandle_t of its mailbox), the handles are exchanged out of band (rank order) and
 * every rank calls _attach with all of them.  Without _attach the NCCL path is used. */
int vatlq_comm_mailbox_handle(void* comm, void* host_handle64);
int vatlq_comm_attach(void* comm, const void* host_handles /* world x 64 bytes */, int world);
int vatlq_comm_destroy(void* comm);

#ifdef __cplusplus
}
#endif
#endif /* VATLQ_H */
