/*
 * pcdist.h -- C ABI of libpcdist.so, the B200 (sm_100a) point-set distance library.
 *
 * Drop-in boundary for the point-set distance hot path of LI-Yiquan/3DPointCloudAttack.
 * The reference has no FFI for this path -- it is stock PyTorch (ATen) called from Python --
 * so each entry point below names the reference Python symbols (file:line, relative to the
 * reference root) whose arithmetic it replaces.  Bindings: ctypes (see INTEGRATION.md and
 * 3dpointcloudattack_b200/_lib.py).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer on the current CUDA
 *     device unless stated otherwise; `stream` is a cudaStream_t passed as void*.
 *   - stream-ordered, re-entrant, allocation-free: the caller owns every input, output and
 *     workspace buffer and keeps it alive until the stream work has completed.
 *   - return value: 0 on success, otherwise a PCD_ERR_* code; pcd_last_error() gives a
 *     thread-local message.  Nothing throws or exits across the ABI.
 *   - there is NO CPU fallback.  Without a CUDA device every compute entry point returns
 *     PCD_ERR_CUDA.
 *   - clouds are fp32 with explicit element strides (batch, point, channel), so both the
 *     [B,N,3] point-major and the [B,3,N] channel-first layouts of the reference are
 *     accepted without a copy.  Indices are int32 on this side (N <= 2^31-1); the Python
 *     shim widens to int64 where the reference returns LongTensors.
 *
 * Arithmetic contract (bit-faithful to the reference's expansion-form evaluation):
 *     t(i,j) = -2 * fma(r_z,c_z, fma(r_y,c_y, r_x*c_x))           (GEMM, k ascending)
 *     PCD_FORM_ROW_COL    d = (t + nrow[i]) + ncol[j]
 *     PCD_FORM_COL_ROW    d = (t + ncol[j]) + nrow[i]
 *     PCD_FORM_SUM_FIRST  d = (nrow[i] + ncol[j]) + t
 * with every operation rounded to fp32 (no contraction beyond the stated FMAs).
 * Ties: the lowest index wins (torch.min(dim) semantics).
 */
#ifndef PCDIST_H_
#define PCDIST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCD_VERSION 203

enum pcd_status {
    PCD_OK = 0,
    PCD_ERR_ARG = 1,        /* bad shape / stride / enum / NULL pointer            */
    PCD_ERR_WORKSPACE = 2,  /* workspace smaller than pcd_*_workspace_bytes()      */
    PCD_ERR_CUDA = 3,       /* CUDA runtime error (launch, no device, ...)         */
    PCD_ERR_UNSUPPORTED = 4 /* e.g. K > PCD_KNN_MAX_K, C > PCD_KNN_MAX_C           */
};

enum pcd_form { PCD_FORM_ROW_COL = 0, PCD_FORM_COL_ROW = 1, PCD_FORM_SUM_FIRST = 2 };

/* How |p|^2 is rounded. MULSUM: ((x*x + y*y) + z*z) as torch.sum(p**2, dim);
 * FMA: fma(z,z, fma(y,y, x*x)) as the diagonal of torch.bmm(p, p^T). */
enum pcd_norm { PCD_NORM_MULSUM = 0, PCD_NORM_FMA = 1 };

/* Value transform applied to the minima before they are stored / reduced.
 * SQRT_CLAMP = sqrt(max(d, 0)): torch.cdist's clamp_min_(0).sqrt_(). */
enum pcd_transform { PCD_VALUE_SQUARED = 0, PCD_VALUE_SQRT_CLAMP = 1 };

#define PCD_KNN_MAX_K 64
#define PCD_KNN_MAX_C 128

/* pcd_knn_forward `strategy` for 3-channel clouds (identical results; tests and tuning pick the pipeline explicitly,
 * the library reads no environment): the default four-pass pipeline, the chunk-minima bound followed by the
 * warp-per-row select, or the warp-per-row select alone. */
enum pcd_knn_strategy { PCD_KNN_AUTO = 0, PCD_KNN_BOUND_SELECT = 1, PCD_KNN_SELECT_ONLY = 2 };
/* pcd_nn1_forward / pcd_nn1_workspace_bytes `sweep_mode`: kept for ABI compatibility.  Every value runs the same exact
 * sweep, with the same results, speed and workspace size. */
enum pcd_sweep_mode { PCD_SWEEP_AUTO = 0, PCD_SWEEP_EXACT = 1, PCD_SWEEP_APPROX = 2 };

int pcd_version(void);
const char *pcd_last_error(void);

/* ------------------------------------------------------------------------------------
 * NN-1 sweep: one pass over the N x M pair matrix of every sample that yields the row
 * minima (over j) AND the column minima (over i) with their lowest-index argmins, plus the
 * per-sample sum / max / first-argmax of both -- everything Chamfer and Hausdorff need.
 * The [B,N,M] matrix is never materialised.
 *
 * Replaces (forward):
 *   utils/dis_utils_torch.py:8-28            pairwise_distances+chamfer/sgd_/bid_hausdorff_dis
 *       form ROW_COL, norm MULSUM, transform SQRT_CLAMP, rows = a^T, cols = b^T
 *   attack/CW/CW_utils/distance.py:15-70     batch_pairwise_dist + Chamfer/HausdorffDistance
 *       form SUM_FIRST, norm FMA, rows = gts, cols = preds   (also Gen3DAdv, SIadv copies)
 *   attack/GeoA3/knn_utils.py:10-55 (K = 1)  knn_points / apply_knn
 *       form COL_ROW, norm MULSUM, swap_norms = 1, rows = p1, cols = p2
 *
 * rows  : [B,N,3] via strides (r_sb, r_sp, r_sc) in elements; cols likewise [B,M,3].
 * swap_norms != 0 (requires N == M): nrow[i] = |cols_i|^2 and ncol[j] = |rows_j|^2 -- the
 *   broadcast of attack/GeoA3/knn_utils.py:13-15.
 * Outputs (none may be NULL):
 *   row_min[B,N] row_arg[B,N] col_min[B,M] col_arg[B,M]   (values after `transform`)
 *   stats_f[4,B] = {row_sum_scale * sum_i row_min, max_i row_min,
 *                   col_sum_scale * sum_j col_min, max_j col_min}   (each row contiguous over B)
 *   stats_i[2,B] = {first argmax_i row_min, first argmax_j col_min}
 * row_sum_scale / col_sum_scale fold the reference's divisors into the kernel (1/N2 and 1/N1
 * for distance.py's means, 1/3 for dis_utils_torch.chamfer's quirk, 1 for plain sums); the sums
 * are accumulated in a fixed order (run-to-run deterministic).
 * NaN / inf coordinates never fault: a point without any finite distance gets arg 0 and the
 * value NaN (columns) or +inf (rows); NaN distances are skipped by the minima (the reference
 * propagates them).
 *
 * Launches: three kernels chained by programmatic dependent launch (reset of the workspace
 * keys -> sweep -> exact argmin + per-sample statistics).  Dense clouds -- point-major [.,N,3]
 * (sp = 3, sc = 1) or channel-major [.,3,N] (sp = 1), base 16-byte aligned, N % 4 == 0,
 * sb % 4 == 0 -- are streamed where they lie; any other layout and swap_norms are packed into
 * the workspace first (same results).
 * zero0 / zero1 (optional, NULL or 16-byte aligned, float counts multiples of 4): buffers the
 * last kernel clears on the way -- pass the gradient buffers of the coming pcd_nn1_backward
 * and call it with grads_prezeroed = 1.
 * rows_per_lane / col_tile: 0 = the built-in tile-shape heuristic; 2, 4, 8, 16 / a power of two in
 * 32..256 force the sweep's register blocking / TMA stage width (tests, tuning sweeps; results
 * are identical for every tiling).
 * sweep_mode (pcd_sweep_mode): kept for ABI compatibility.  0, 1 and 2 are accepted, and any other value is rejected with
 * PCD_ERR_ARG.  No accepted value changes the results, the speed or the workspace size: every one runs the exact sweep,
 * which ranks the pairs with the reference's own instruction sequence.
 * sweep_start_event / sweep_stop_event (optional cudaEvent_t): recorded on `stream` immediately
 * before / after the sweep kernel launch so a caller can time the dominant kernel live with
 * CUDA events (bench.py's roofline); per call, no global state.
 * ---------------------------------------------------------------------------------- */
size_t pcd_nn1_workspace_bytes(int B, int N, int M, int sweep_mode);

/* The tile shape the heuristic of pcd_nn1_forward picks for this problem on the current device
 * (HOST out-pointers): rows per lane R (2, 4, 8, 16) and the TMA stage width.  For reports. */
int pcd_nn1_query_tiling(int B, int N, int M, int *rows_per_lane, int *col_tile);

int pcd_nn1_forward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                    const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                    int B, int N, int M,
                    int form, int norm_kind, int swap_norms, int transform,
                    float row_sum_scale, float col_sum_scale,
                    float *row_min, int32_t *row_arg, float *col_min, int32_t *col_arg,
                    float *stats_f, int32_t *stats_i,
                    float *zero0, size_t zero0_floats, float *zero1, size_t zero1_floats,
                    void *workspace, size_t workspace_bytes, int rows_per_lane, int col_tile, int sweep_mode,
                    void *sweep_start_event, void *sweep_stop_event, void *stream);

/* Backward of everything derived from the NN-1 minima, through the saved argmins
 * (autograd of torch.min(dim) / torch.max / mean / cdist in the reference).
 * The upstream gradient of row minimum (b,i) is
 *     g_row[b,i] + row_sum_scale * w_row_all[b] + (i == row_argmax[b] ? w_row_max[b] : 0)
 * (each term optional: NULL = 0), the same for columns; w_*_all / w_*_max are the upstream
 * gradients of the four stats_f rows.  So Chamfer (scaled sum of minima: w_*_all), Hausdorff (max of minima: w_*_max) and knn_points(K=1).dists (g_row) are
 * all one call.  For PCD_VALUE_SQRT_CLAMP row_min/col_min (the stored post-sqrt values) must
 * be given: d/dp sqrt(d2) = (p - q)/sqrt(d2), 0 where it is 0 (cdist backward).
 * grad_rows / grad_cols are written in full (no need to zero them) with the caller's strides;
 * either may be NULL when that cloud needs no gradient.  grads_prezeroed != 0: the caller
 * guarantees both buffers are zero (pcd_nn1_forward's zero fill) -- one kernel launch, atomics only.
 * swap_norms: gradients of the swapped-norm surrogate exactly as autograd produces them
 * (norm terms land on the *other* index, attack/GeoA3/knn_utils.py:13-15).  Under PCD_VALUE_SQRT_CLAMP each
 * term, those norm terms included, is scaled by g / v of the minimum it belongs to.
 * ---------------------------------------------------------------------------------- */
int pcd_nn1_backward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                     const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                     int B, int N, int M, int swap_norms, int transform,
                     const int32_t *row_arg, const int32_t *col_arg,
                     const float *row_min, const float *col_min,
                     const float *g_row, const float *g_col,
                     const float *w_row_all, const float *w_row_max, const int32_t *row_argmax,
                     const float *w_col_all, const float *w_col_max, const int32_t *col_argmax,
                     const int64_t *w_strides /* HOST ptr to 4 element strides of the w arrays, NULL = {1,1,1,1};
                                                 0 = one broadcast value (autograd's expanded gradients) */,
                     float row_sum_scale, float col_sum_scale,
                     float *grad_rows, int64_t gr_sb, int64_t gr_sp, int64_t gr_sc,
                     float *grad_cols, int64_t gc_sb, int64_t gc_sp, int64_t gc_sc,
                     int grads_prezeroed, void *stream);

/* ------------------------------------------------------------------------------------
 * k-NN select sweep: the K smallest d(i,j) of every row, ascending by (distance, index).
 *
 * Replaces:
 *   attack/GeoA3/knn_utils.py:10-55 (K > 1)             form COL_ROW, swap_norms = 1
 *   attack/CW/CW_utils/dist_utils.py:133-143 (KNNDist)  form COL_ROW, rows = cols = pc
 *   model/dgcnn.py:194-200, model/curvenet_util.py:10-26, attack/AOF/TAOF_attack.py:13-28
 *       form COL_ROW on C-channel features (the reference's negated matrix + topk largest)
 *   model/pointnet2_utils.py:293-300 (3-NN of feature propagation)  form ROW_COL
 *
 * rows [B,N,C], cols [B,M,C] via strides; 1 <= C <= PCD_KNN_MAX_C, 1 <= K <= min(M,
 * PCD_KNN_MAX_K).  dists[B,N,K] fp32 (may be NULL), idx[B,N,K] int32.
 * ---------------------------------------------------------------------------------- */
size_t pcd_knn_workspace_bytes(int B, int N, int M, int C, int K);

int pcd_knn_forward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                    const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                    int B, int N, int M, int C, int K,
                    int form, int norm_kind, int swap_norms,
                    float *dists, int32_t *idx,
                    void *workspace, size_t workspace_bytes, int strategy, void *stream);

/* Backward of dists[B,N,K] w.r.t. both clouds through idx (3-channel clouds).
 * g_dists[B,N,K] upstream.  grad_* are written in full. */
int pcd_knn_backward(const float *rows, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                     const float *cols, int64_t c_sb, int64_t c_sp, int64_t c_sc,
                     int B, int N, int M, int K, int swap_norms,
                     const int32_t *idx, const float *g_dists,
                     float *grad_rows, int64_t gr_sb, int64_t gr_sp, int64_t gr_sc,
                     float *grad_cols, int64_t gc_sb, int64_t gc_sp, int64_t gc_sc,
                     void *stream);

/* ------------------------------------------------------------------------------------
 * Ordered ball query.  Replaces model/pointnet2_utils.py:84-104 (query_ball_point; copies in
 * pointnet/pointnet2_utils.py, model/curvenet_util.py:38-113, DUP_Net/pu_utils.py):
 * the first `nsample` indices j (ascending) with NOT(d(i,j) > radius2), d in form ROW_COL
 * with MULSUM norms (square_distance, :35-37), padded with the first hit; a row without any
 * hit is filled with N.  new_xyz [B,S,3] are the rows, xyz [B,N,3] the columns.
 * ---------------------------------------------------------------------------------- */
int pcd_ball_query(const float *xyz, int64_t x_sb, int64_t x_sp, int64_t x_sc,
                   const float *new_xyz, int64_t q_sb, int64_t q_sp, int64_t q_sc,
                   int B, int N, int S, float radius2, int nsample,
                   int32_t *idx, void *stream);

/* ------------------------------------------------------------------------------------
 * Edge features of a k-NN graph (the step after the k-NN select in the DGCNN / CurveNet victims).
 * Replaces the gather + subtract + cat + permute(0,3,1,2).contiguous() chains of
 *   model/dgcnn.py:203-227          get_graph_feature   ops = {DIFF, CENTER}           -> [B,2C,N,k]
 *   model/curvenet_util.py:206-236  LPFA.group_feature  ops = {CENTER, NEIGHBOR, DIFF} (xyz, 9 ch)
 *                                                        ops = {DIFF}                   (features)
 * x [B,C,N] contiguous fp32 (channel-first, as the victims hold it), idx [B,N,k] int32 with
 * entries in [0,N) (others are clamped), out [B, nblocks*C, N, k] contiguous:
 *   out[b, q*C + c, n, j] = ops[q](centre = x[b,c,n], neighbour = x[b,c,idx[b,n,j]])
 * `ops` is a HOST array of nblocks (1..4) pcd_edge_op values.  The backward accumulates
 * gx[b,c,n] from g [B, nblocks*C, N, k] (own terms plus the scatter through idx); gx is
 * written in full; N <= 51200; g and idx 16-byte aligned.
 * Backward workspace: with `workspace_bytes >= pcd_edge_feature_backward_workspace(B, N, k, nblocks)` (> 0 for
 * N <= 4096, 4 | N*k and stages that fit shared memory) the call inverts the graph once per sample and GATHERS:
 * no floating-point atomics, fixed summation order (bit-reproducible), ~0.8 of the HBM peak.  With workspace NULL
 * (or a shape the gather form does not cover: the query returns 0) it scatters with shared-memory atomics
 * (summation order not fixed, as in the reference's index backward).
 * ---------------------------------------------------------------------------------- */
enum pcd_edge_op { PCD_EDGE_CENTER = 0, PCD_EDGE_NEIGHBOR = 1, PCD_EDGE_DIFF = 2 };

int pcd_edge_feature_forward(const float *x, const int32_t *idx, int B, int C, int N, int k,
                             int nblocks, const int *ops, float *out, void *stream);
size_t pcd_edge_feature_backward_workspace(int B, int N, int k, int nblocks);
int pcd_edge_feature_backward(const float *g, const int32_t *idx, int B, int C, int N, int k,
                              int nblocks, const int *ops, float *gx, void *workspace, size_t workspace_bytes,
                              void *stream);

/* ------------------------------------------------------------------------------------
 * Farthest point sampling.  Replaces the npoint-iteration Python loop of
 *   model/pointnet2_utils.py:59-81 (random start, :71), model/curvenet_util.py:69-90 (start 0)
 * with one persistent CTA per sample.  Same arithmetic and tie rule: dist = ((dx*dx + dy*dy) +
 * dz*dz), distance = min(distance, dist) from 1e10, next = FIRST index of the maximum.
 * xyz [B,N,3] via strides; start [B] int32 (device; NULL = start at 0, out-of-range entries
 * = 0); out [B,npoint] int32 with out[b,0] = start[b].  N <= 51200.
 * ---------------------------------------------------------------------------------- */
int pcd_fps(const float *xyz, int64_t sb, int64_t sp, int64_t sc, int B, int N, int npoint,
            const int32_t *start, int32_t *out, void *stream);

/* ------------------------------------------------------------------------------------
 * Fused epilogue of the k-NN outlier / smoothing loss.  Replaces the nine-launch torch chain of
 *   attack/CW/CW_utils/dist_utils.py:143-153 (KNNDist; copies in Gen3DAdv, SIadv)
 *   attack/GeoA3/loss_utils.py:148-157 (kNN_smoothing_loss)
 * on the dists [B,N,K1] / idx [B,N,K1] of pcd_knn_forward(cloud, cloud, K1 = k + 1):
 *   value[b,i] = mean_j dists[b,i,j] (column 0 dropped when skip_first), threshold[b] = mean_i value +
 *   alpha * std_i value (unbiased), mask = value > threshold, loss[b] = mean_i value * mask.
 * forward: one kernel, one CTA per sample, fixed reduction order; outputs value, mask [B,N] (0/1
 *   floats), loss [B], threshold [B] (optional).
 * backward: d(sum_b g_loss[b] loss[b]) / d cloud through idx (the comparison is non-differentiable in
 *   both reference variants); g_loss read with element stride g_stride (0 = one broadcast value);
 *   grad_pc [B,N,3] contiguous, written in full; ONE kernel when the buffer was cleared by the forward
 *   (zero_grad / grad_prezeroed), else one memset + one kernel; only masked points do any work.
 * ---------------------------------------------------------------------------------- */
int pcd_knn_outlier_forward(const float *dists, int B, int N, int K1, int skip_first, float alpha,
                            float *value, float *mask, float *loss, float *threshold,
                            float *zero_grad /* optional [B,N,3]: cleared on the way for the backward */, void *stream);
int pcd_knn_outlier_backward(const float *pc, int64_t sb, int64_t sp, int64_t sc, const int32_t *idx,
                             const float *mask, const float *g_loss, int64_t g_stride,
                             int B, int N, int K1, int skip_first, float *grad_pc,
                             int grad_prezeroed /* grad_pc was handed to the forward's zero_grad */, void *stream);

/* ------------------------------------------------------------------------------------
 * Local geometry on a k-NN graph (the consumers of the k-NN select in GeoA3 / AOF), each ONE pass
 * over the index tensor -- the [B,N,K,3] neighbour gather of the reference never reaches HBM.
 * idx [B,N,K1] int32 is the output of pcd_knn_forward on the cloud itself; skip_first != 0 drops
 * column 0 (the point itself), as the reference's `[..., 1:]` slices do.
 *
 * pcd_local_frames   attack/GeoA3/utility.py:43-92 (estimate_normal) and :119-152
 *   (estimate_perpendicular): covariance of the k = K1 - skip neighbours formed in fp32 exactly as the
 *   reference forms it (mean, centring, bmm, 1/(k-1)), eigen-frame by a cyclic Jacobi iteration in
 *   fp64 (the reference's torch.symeig no longer exists).  Outputs, each optional (NULL):
 *     normal [B,N,3] via strides: eigenvector of the smallest eigenvalue times
 *            -sign(<n, sum of the centred neighbours>) (utility.py:67-69; that sum is rounding noise
 *            around zero, so the sign is as arbitrary as the reference's -- every consumer is sign-free)
 *     evecs [B,N,3,3] contiguous: rows = eigenvectors by ascending eigenvalue; evals [B,N,3].
 * pcd_kappa_forward / _backward   attack/GeoA3/loss_utils.py:60-70 (_get_kappa_ori), :72-90
 *   (_get_kappa_adv), :116-125 (corresponding_normal_loss):
 *     kappa[b,i] = mean_j |< (q_j - p_i) / max(|q_j - p_i|, 1e-12), n >|,  n = normal[b, nidx ? nidx[b,i] : i]
 *   (nidx = the adv->ori nearest-neighbour index of _get_kappa_adv, NULL for the point's own normal).
 *   The backward writes grad_pc [B,N,3] contiguous in full (own term + scatter through idx); the
 *   normals are constants, as in the reference (gathered from the detached ori normals).
 * pcd_graph_laplacian   attack/AOF/TAOF_attack.py:31-52 (get_Laplace_from_pc) up to the eigensolver:
 *   L [B,N,N] = D - A with A_ij = exp(-((dx^2 + dy^2) + dz^2)) on the symmetrised k-NN graph (idx [B,N,K],
 *   self column included).  Dense by design: the reference hands it to a dense eigendecomposition.
 * ---------------------------------------------------------------------------------- */
int pcd_local_frames(const float *pc, int64_t sb, int64_t sp, int64_t sc, const int32_t *idx,
                     int B, int N, int K1, int skip_first,
                     float *normal, int64_t n_sb, int64_t n_sp, int64_t n_sc,
                     float *evecs, float *evals, void *stream);
int pcd_kappa_forward(const float *pc, int64_t sb, int64_t sp, int64_t sc,
                      const float *normal, int64_t n_sb, int64_t n_sp, int64_t n_sc,
                      const int32_t *nidx, const int32_t *idx, int B, int N, int K1, int skip_first,
                      float *kappa, void *stream);
int pcd_kappa_backward(const float *pc, int64_t sb, int64_t sp, int64_t sc,
                       const float *normal, int64_t n_sb, int64_t n_sp, int64_t n_sc,
                       const int32_t *nidx, const int32_t *idx, int B, int N, int K1, int skip_first,
                       const float *g_kappa, float *grad_pc, void *stream);
int pcd_graph_laplacian(const float *pc, int64_t sb, int64_t sp, int64_t sc, const int32_t *idx,
                        int B, int N, int K, float *L, void *stream);

/* ------------------------------------------------------------------------------------
 * Projection / clipping epilogues of the attack loops (SURVEY.md section 8f row 1), one launch each instead of the
 * reference's chains of 8-25 elementwise torch ops; same fp32 operations in the same order.  All tensors are
 * channel-first contiguous [B,3,K] fp32 (as the attack loops hold them).
 * pcd_clip_points   in place on pc:
 *     PCD_CLIP_LINF          attack/CW/CW_utils/clip_utils.py:32-56   ClipPointsLinf: every point's offset from ori is
 *                            scaled by min(budget / (|offset| + 1e-9), 1)                        (bit-identical to torch)
 *     PCD_CLIP_PROJECT_LINF  clip_utils.py:59-136  ProjectInnerClipLinf: points with offset . normal < 0 are projected
 *                            (ProjectInnerPoints, normal [B,3,K] required), then PCD_CLIP_LINF
 *     PCD_CLIP_L2            clip_utils.py:5-29    ClipPointsL2: one scale per sample from the norm of the whole
 *                            perturbation (the 3K-term sum is in a fixed tree order: ~1e-7 from torch's, not bit-equal)
 * pcd_lp_clip       attack/GeoA3/GeoA3_attack.py:92-101: offsets longer than cc_linf are rescaled to cc_linf.
 * pcd_offset_proj   GeoA3_attack.py:62-81 after its knn_points(offset, ori_pc, K=1): idx [B,K] int32 = nearest original
 *                   point; out = the offset's component along that point's normalised normal (ori_normal [B,3,M]).
 * pcd_find_offset   GeoA3_attack.py:83-89 after its knn_points(adv_pc, ori_pc, K=1): out = adv - ori[:, :, idx].
 * Indices outside [0,M) are clamped.  out may alias the first input.
 * ---------------------------------------------------------------------------------- */
enum pcd_clip_mode { PCD_CLIP_LINF = 0, PCD_CLIP_PROJECT_LINF = 1, PCD_CLIP_L2 = 2 };

int pcd_clip_points(float *pc, const float *ori, const float *normal, int B, int K, int mode, float budget,
                    void *stream);
int pcd_lp_clip(const float *offset, int B, int K, float cc_linf, float *out, void *stream);
int pcd_offset_proj(const float *offset, const float *ori_normal, const int32_t *idx, int B, int K, int M,
                    float *out, void *stream);
int pcd_find_offset(const float *adv, const float *ori, const int32_t *idx, int B, int K, int M, float *out,
                    void *stream);

/* ------------------------------------------------------------------------------------
 * Statistical outlier removal (SOR), the standard point-cloud defence, evaluated in float64.
 * Replaces attack/SIadv/baselines/defense/drop_points/SOR.py:24-54 (outlier_removal): its two
 * [B,N,N] float64 matrices and topk(k + 1) are never materialised.
 *
 * pc [B,N,3] fp32 via element strides (sb, sp, sc): point-major and transposed channel-first
 * views both work.  For each sample b, in float64 on the exactly converted coordinates:
 *     xx[i]     = (x_i*x_i + y_i*y_i) + z_i*z_i
 *     dot(i,j)  = (x_i*x_j + y_i*y_j) + z_i*z_j                 (channels ascending)
 *     d(i,j)    = (xx[j] + (-2 * dot(i,j))) + xx[i]             (dist = xx + inner + xx^T)
 *     value[i]  = (s_1 + s_2 + ... + s_k) / k                   s_0 <= s_1 <= ... <= s_k are the k + 1 smallest
 *                                                               d(i,.) over ALL j, self included; s_0 is dropped;
 *                                                               the sum runs left to right
 *     mean      = mean_i value[i],  std = unbiased std_i value[i]   (a fixed order that depends on N only)
 *     threshold = mean + alpha * std
 *     keep[i]   = value[i] <= threshold
 * Only distance values enter, so tie order and which entry is "self" cannot change the result; d(i,i)
 * is exactly 0.  Results for sample b are bit-identical whatever B is, whatever else is in the batch
 * and whatever the input layout.
 * Outputs (all required, contiguous, written in full): value [B,N], threshold [B], keep [B,N] (0/1),
 * kept_idx [B,N] (the kept indices ascending, then -1), lengths [B] (the number of kept points).
 * Constraints: B >= 1, 1 <= k <= PCD_SOR_MAX_K, N >= k + 1, alpha finite; anything else returns
 * PCD_ERR_ARG before any CUDA call.  Non-finite coordinates never fault: a sample that holds one may
 * end with any lengths[b] in [0, N], and the other samples are unaffected.
 * Launches: two kernels (the pair sweep, then one CTA per sample for the statistics and the
 * compaction); no workspace.
 * ---------------------------------------------------------------------------------- */
#define PCD_SOR_MAX_K 15

int pcd_sor_forward(const float *pc, int64_t sb, int64_t sp, int64_t sc, int B, int N, int k, double alpha,
                    double *value /*[B,N]*/, double *threshold /*[B]*/, uint8_t *keep /*[B,N] 0/1*/,
                    int32_t *kept_idx /*[B,N]: kept indices ascending, then -1*/, int32_t *lengths /*[B]*/,
                    void *stream);

/* SOR on the first len[b] points of every sample (ragged or padded batches), with the columns of a
 * sample optionally split over several CTAs (small batches).
 * len: int32 [B] on the device, or NULL for "all N".  Each length is clamped to [0, N] on the
 * device (no host synchronisation); n = len[b] below, and sample b is pc[b, :n].  Nothing past n
 * is read into a result, so NaN or inf padding changes no output.
 *   n >= k + 1: value[b, :n], threshold[b], keep[b, :n], kept_idx[b, :] and lengths[b] are
 *     bit-identical to pcd_sor_forward on pc[b:b+1, :n] alone (kept_idx padded with -1 to N),
 *     whatever the rest of the batch, the layout or col_split: the reductions of the epilogue run
 *     in an order that depends on n only, and the k + 1 smallest values are one multiset at any
 *     split.  Rows i >= n get value NaN, keep 0 (and kept_idx holds -1 past lengths[b]).
 *   n < k + 1 (n = 0 included): no statistic.  value is NaN on every row, threshold NaN, keep all 0,
 *     kept_idx all -1, lengths[b] = 0 (value <= NaN is false).  Nothing faults.
 * col_split: 0 picks the number of column ranges per row tile from (B, N, k): more while B * row
 * tiles is small, never a range below one 64-column tile (so small inputs get one range).  Any
 * value > 0 forces it (testing and tuning; results do not change).
 * Workspace: at least pcd_sor_workspace_bytes(B, N, k, col_split) bytes, else PCD_ERR_WORKSPACE.
 * That size is 0 exactly when the split resolves to one range (workspace may then be NULL).
 * Constraints: B >= 1, N >= 1 (N may be below k + 1), 1 <= k <= PCD_SOR_MAX_K, alpha finite,
 * col_split >= 0, no NULL pointer (len aside); anything else returns PCD_ERR_ARG before any CUDA
 * call.  Non-finite coordinates inside the valid range never fault, as above.
 * Launches: two kernels (the sweep, then one CTA per sample) with one column range; three with
 * more (the sweep writes each range's sorted k + 1 smallest values to the workspace, and a
 * per-row merge over many CTAs forms the values before the epilogue).
 * ---------------------------------------------------------------------------------- */
size_t pcd_sor_workspace_bytes(int B, int N, int k, int col_split);
int pcd_sor_forward_len(const float *pc, int64_t sb, int64_t sp, int64_t sc, int B, int N, int k, double alpha,
                        const int32_t *len /*[B] device, or NULL*/, int col_split, double *value /*[B,N]*/,
                        double *threshold /*[B]*/, uint8_t *keep /*[B,N]*/, int32_t *kept_idx /*[B,N]*/,
                        int32_t *lengths /*[B]*/, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------
 * Exact float64 nearest-neighbour distances between two clouds, both directions, with the
 * per-sample Chamfer and Hausdorff reductions, for batches of clouds of unequal valid sizes.
 * The arithmetic of utils/dis_utils_numpy.py:13-38 (scipy distance_matrix in float64) without
 * the N x M matrix.
 *
 * a [B,N,3] and b [B,M,3] fp32 via element strides; a_len / b_len: int32 [B] on the device, or
 * NULL for "all N" / "all M".  Each length is clamped to [0, N] / [0, M] on the device (no host
 * synchronisation); n = a_len[b], m = b_len[b] below.  For each sample, in float64 on the
 * exactly converted coordinates, with every operation correctly rounded and none contracted:
 *     dx = b_x[j] - a_x[i]   (likewise dy, dz)
 *     s(i,j) = ((dx*dx) + (dy*dy)) + (dz*dz)
 * so sqrt_rn(s) is scipy's cdist(a, b, 'euclidean') / distance_matrix bit for bit.  s is
 * symmetric: (-d)*(-d) == d*d, so the b-side rows evaluate the same s.
 *   a_min[b,i] = min_{j<m} s(i,j), a_arg[b,i] = its index          (i < n)
 *   b_min[b,j] = min_{i<n} s(i,j), b_arg[b,j] = its index          (j < m)
 * with numpy's min / argmin semantics: the lowest index among equal minima; a NaN entry wins
 * and arg is the first NaN index.  Rows past their length, and every row when the other side
 * has length 0, get NaN and -1.  The ranking is on s, not on sqrt(s): where two different s
 * round to the same square root, an argmin over scipy's Euclidean matrix may pick another
 * index than a_arg / b_arg.
 * Per sample and direction (d = 0: the a rows, d = 1: the b rows), over the valid rows only,
 * numpy's reductions of the per-point minima v (a_min[b,:n] or b_min[b,:m]):
 *   stats[d,b,0] = mean(v)          stats[d,b,1] = mean(sqrt_rn(v))
 *   stats[d,b,2] = max(v)           stats[d,b,3] = sqrt_rn(max(v))      argmax[d,b] = argmax(v)
 * NaN propagates as in numpy (argmax = the first NaN index); no valid row gives NaN and -1.
 * The sums run in a fixed order that depends only on the number of valid rows, so every
 * output of a sample is bit-identical whatever B, the rest of the batch, the strides or
 * col_split; the means are within the recursive-summation bound (n-1)*2^-53*sum|v| (plus the
 * rounding of the division) of the exact mean.
 * col_split: 0 picks the number of column ranges per row tile from B, N and M (more when
 * B * row tiles is small); any value > 0 forces it (testing and tuning only; the results do
 * not depend on it).
 * Outputs (all required, contiguous, written in full): a_min [B,N], a_arg [B,N], b_min [B,M],
 * b_arg [B,M], stats [2,B,4], argmax [2,B].  Workspace: at least
 * pcd_nn_dist64_workspace_bytes(B, N, M, col_split) bytes, else PCD_ERR_WORKSPACE.
 * Constraints: B >= 1, N >= 1, M >= 1, col_split >= 0, no NULL pointer (a_len / b_len aside);
 * anything else returns PCD_ERR_ARG before any CUDA call.  Non-finite coordinates never fault.
 * Launches: two kernels (the sweep of both directions, then one CTA per sample and direction
 * that merges the column ranges and reduces); no host synchronisation.
 * ---------------------------------------------------------------------------------- */
size_t pcd_nn_dist64_workspace_bytes(int B, int N, int M, int col_split);
int pcd_nn_dist64_forward(const float *a, int64_t sab, int64_t sap, int64_t sac, const float *b, int64_t sbb,
                          int64_t sbp, int64_t sbc, int B, int N, int M, const int32_t *a_len, const int32_t *b_len,
                          int col_split, double *a_min /*[B,N]*/, int32_t *a_arg /*[B,N]*/, double *b_min /*[B,M]*/,
                          int32_t *b_arg /*[B,M]*/, double *stats /*[2,B,4]*/, int32_t *argmax /*[2,B]*/,
                          void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------
 * Uniform draws of points without replacement, per sample: the resampling of the SOR defence
 * (SORDefense.process_data's np.random.choice calls) and the simple random sampling (SRS)
 * defence, as one device-side, graph-capturable sampler.
 *
 * For every sample b, n = len[b] clamped to [0, N] on the device (len: int32 [B], or NULL for
 * "all N").  Draw counter c = counter[0] as it is when the call runs; global sample id
 * g = first_sample + b (its low 32 bits enter the counter block).  Key of point i < n:
 *     (w0, w1, w2, w3) = Philox4x32-10(counter = (i, g, c_lo, c_hi), key = (seed_lo, seed_hi))
 *                        (Random123 / curand round constants and Weyl increments)
 *     r      = (w0 << 32) | w1
 *     key[i] = (r & ~0x3FFF) | i                 distinct, totally ordered (unsigned 64-bit)
 * The points ranked by ascending key form a uniformly random permutation P of 0 .. n-1 (up to
 * the 2^-50 chance of equal random bits, which the index resolves).  out_idx[b, j], j < npoint:
 *     n >  npoint  P[j]                            np.random.choice(n, npoint, replace=False)
 *     n <  npoint  j < (npoint / n) * n: j % n;    the cloud npoint / n times, then
 *                  then P[j - (npoint / n) * n]    npoint % n of its points, distinct
 *     n == npoint  j                               the cloud as is (no draw)
 *     n == 0       -1                              (no host-side error without a synchronisation)
 * The draws follow np.random.choice in distribution, not its bits.  With a table (int32, row
 * b at table + b * table_stride, SOR's kept_idx), every value v >= 0 above becomes table[b][v]:
 * out_idx then indexes the original cloud.  A sample's draws depend only on (seed, g, c, n,
 * npoint): not on B, its batch position, N or the rest of the batch.
 * counter: int64 [2] on the device.  counter[0] is the draw counter; the call leaves it one
 * higher, in stream order (the last CTA to have read it advances it), so a captured graph draws
 * afresh on every replay.  counter[1] is the CTAs' arrival count: 0 between calls (the call
 * leaves it 0); calls that share a counter must be stream-ordered.
 * Constraints: B >= 1, 1 <= N, npoint >= 1, first_sample >= 0, table_stride >= N when a table
 * is given, counter and out_idx not NULL; anything else returns PCD_ERR_ARG before any CUDA
 * call.  N > PCD_SAMPLE_MAX_N returns PCD_ERR_UNSUPPORTED.
 * Launches: one kernel, one CTA per sample (a block radix sort of the keys in shared memory);
 * no workspace, no host synchronisation.  out_idx is int64 so that it feeds torch.gather as is.
 * ---------------------------------------------------------------------------------- */
#define PCD_SAMPLE_MAX_N 16384

int pcd_sample_points(int B, int N, int npoint, const int32_t *len /*[B] device, or NULL*/,
                      const int32_t *table /*[B, table_stride] device, or NULL*/, int64_t table_stride,
                      uint64_t seed, int64_t first_sample, int64_t *counter /*[2] device*/,
                      int64_t *out_idx /*[B, npoint]*/, void *stream);

/* ------------------------------------------------------------------------------------
 * One step of the SI-Adv shape-invariant attack, in place on pc: the tangent-plane gradient step and
 * the clip of attack/SIadv/SIadv_attack.py (PointCloudAttack.shape_invariant_ifgm, with
 * get_spin_axis_matrix, get_transformed_point_cloud and get_original_point_cloud) as one launch.
 *
 * pc, ori, normal, grad [B,N,3] fp32 via element strides (grad = dL/d pc).  All arithmetic is fp32
 * with every operation rounded on its own, none contracted.  Per sample b and point i, with
 * (x, y, z) = normal and p = the point:
 *   1. c = (px*x + py*y) + pz*z;  t = (c*x, c*y, c*z);  q = p + t
 *   2. spin-axis rows, den = sqrt(1 - z*z):  u0 = (y/den, -x/den, 0),
 *      u1 = ((x*z)/den, (y*z)/den, -den),  u2 = (x, y, z);  where |z*z - 1| < 1e-4 instead
 *      u0 = (r, -r, 0), u1 = (z/s2, z/s2, 0), u2 = (0, 0, z), r = fp32(1/sqrt 2), s2 = fp32(sqrt 2)
 *   3. p' = U q, g' = U grad, each component (u_r0*a0 + u_r1*a1) + u_r2*a2; then g'_2 = 0
 *      (dL/dP' = U dL/dP: the gradient restricted to the tangent plane, in the frame)
 *   4. norm_b = sqrt(S), S = the tree sum over the points of g'_0*g'_0 + g'_1*g'_1
 *   5. a = fp32(step_size * step_scale) (product in double); p''_r = p'_r - (a*g'_r) / (norm_b + 1e-9f)
 *   6. p_new_r = ((u_0r*p''_0 + u_1r*p''_1) + u_2r*p''_2) - t_r      (the explicit inverse transform)
 *   7. the clip: d = p_new - ori; per axis c, n_c = sqrt(tree sum over i of d_ic*d_ic);
 *      s_c = min(eps / (n_c + 1e-9f), 1);  pc = ori + d*s_c
 *      (ClipPointsLinf applied to [B,N,3] clouds, as the attack does: its "per-point" norm runs over
 *      the N points of each axis; the per-point clip is pcd_clip_points)
 *   8. gnorm [B] (optional, NULL when not wanted) = norm_b.
 * Tree sum: a node covering the aligned block [k*2^l, min((k+1)*2^l, N)) is left + right, or left when
 * the right half is empty; the leaves are the points in order.  A zero gradient gives a zero step; the
 * point then moves only by the rounding of the round trip through its frame.
 * A sample's outputs depend only on its own inputs and N: not on B, split or the strides.  A sample
 * with a non-finite gradient or normal goes non-finite alone.
 * split: 0 picks how many CTAs (a thread-block cluster, up to 8, 16 where the device schedules it)
 * share a sample from B, N and the SM count; a power of two <= 16 forces it (testing; results do not
 * change).  A split that leaves more than 2048 points per CTA returns PCD_ERR_ARG; 16 on a device
 * that cannot schedule it PCD_ERR_UNSUPPORTED.
 * Constraints: B >= 0 (0 is a no-op), N >= 1, eps >= 0, no NULL cloud; anything else returns
 * PCD_ERR_ARG before any CUDA call.  N > PCD_SI_MAX_N returns PCD_ERR_UNSUPPORTED.
 * Launches: one kernel; no workspace, no host synchronisation.  pc must not alias the inputs.
 * ---------------------------------------------------------------------------------- */
#define PCD_SI_MAX_N 16384

int pcd_si_step(float *pc, int64_t sb, int64_t sp, int64_t sc, const float *ori, int64_t o_sb, int64_t o_sp,
                int64_t o_sc, const float *normal, int64_t n_sb, int64_t n_sp, int64_t n_sc, const float *grad,
                int64_t g_sb, int64_t g_sp, int64_t g_sc, int B, int N, double step_size, double step_scale,
                float eps, int split, float *gnorm /*[B] or NULL*/, void *stream);

/* ------------------------------------------------------------------------------------
 * SI-Adv's query-based attack (attack/SIadv/SIadv_attack.py, shape_invariant_query_attack), restated
 * from the published algorithm: a sensitivity map from a surrogate's gradient in every point's tangent
 * plane, then SimBA-style trials of -step and +step at the most sensitive points, each scored by one
 * query of the black box.  Frames, rounding and the clip are those of pcd_si_step.
 *
 * pcd_si_sensitivity: grad (the surrogate's dL/d ori), normal [B,N,3] fp32 via element strides.  Per
 * point, with U the spin-axis rows of pcd_si_step step 2:  g'x, g'y = rows 0 and 1 of U grad (step 3's
 * rows product);  s = sqrt(g'x*g'x + g'y*g'y);  dir = (g'x / (s + 1e-16f), g'y / (s + 1e-16f)).
 * A NaN s is stored as -1 with dir (0, 0): such points rank last and move nothing.
 * s [B,N] and dir [B,N,2] are contiguous outputs.  One launch.  B >= 0 (0 is a no-op), N >= 1, no
 * NULL pointer, else PCD_ERR_ARG before any CUDA call.  The caller ranks the points by descending s,
 * ties by the lower index (a stable sort).
 *
 * pcd_si_query_round: one query round of every sample, after the black box has scored the trials.
 *   logits [B,C] fp32 via element strides (C >= 2), target [B] int64, ori / normal [B,N,3] (any
 *   strides), order [B,N] int32 and dir [B,N,2] contiguous (pcd_si_sensitivity's ranking); in/out:
 *   cloud (the current cloud P) and trial [B,N,3] (any strides, not the same memory), state [B,4]
 *   int32 contiguous = (sigma, cursor, queries, status), best [B] fp32.  status: 0 active, 1 success,
 *   2 failed.  The caller starts every sample at cloud = trial = ori, state = (-1, 0, 0, 0).
 *   Scoring a row: other = max(max over j != y of logits_j, -10000) (the max of (1 - onehot)*logits -
 *   onehot*10000), real = logits_y;  margin = real - other, or other - real when targeted;  the first
 *   arg-max decides success (!= y, or == y when targeted).  A row with a NaN, a non-finite margin or
 *   y outside [0, C) is neither a success nor an improvement.
 *   An active sample (others are left alone): q = queries + 1, then
 *     q == 1 (round 0, the trial is the cloud):  best = margin;  success -> status 1
 *     success                                   -> cloud = trial, status 1
 *     margin < best                             -> cloud = trial, best = margin, cursor += 1, sigma = -1
 *     sigma == -1                               -> sigma = +1 (the same point again)
 *     otherwise                                 -> cursor += 1, sigma = -1
 *   and q >= max_query leaves an active sample failed (status 2).  A sample that ends in this round gets
 *   trial = cloud.  One that goes on gets its next trial: point i = order[cursor mod N] of the cloud moved
 *   by the step's transform (pcd_si_step steps 1-3), pp_0 += (sigma*a)*dir_x, pp_1 += (sigma*a)*dir_y,
 *   a = step_size, and the inverse transform (step 6); every other point copied; then the whole cloud
 *   clipped as in pcd_si_step step 7 (per-axis norms of trial - ori over the fixed tree, eps).  An order
 *   entry outside [0, N) moves no point.
 *   active (optional, NULL when not wanted): every sample that leaves the active status in this round
 *   subtracts 1 from *active, so a caller that sets it to B before the first round reads the number of
 *   active samples there.
 *   A sample's bits depend only on its own inputs and N: not on B, C, strides or the launch geometry.
 *   Constraints: B >= 0 (0 is a no-op), N >= 1, C >= 2, finite step_size, eps >= 0, max_query >= 1,
 *   targeted 0 or 1, no NULL pointer but active, cloud != trial; anything else returns PCD_ERR_ARG before
 *   any CUDA call.  N > PCD_SI_MAX_N returns PCD_ERR_UNSUPPORTED.
 *   Launches: one kernel (one CTA per sample); no workspace, no host synchronisation.
 * ---------------------------------------------------------------------------------- */
int pcd_si_sensitivity(const float *grad, int64_t g_sb, int64_t g_sp, int64_t g_sc, const float *normal,
                       int64_t n_sb, int64_t n_sp, int64_t n_sc, int B, int N, float *s /*[B,N]*/,
                       float *dir /*[B,N,2]*/, void *stream);

int pcd_si_query_round(const float *logits, int64_t l_sb, int64_t l_sc, int C, const int64_t *target,
                       const float *ori, int64_t o_sb, int64_t o_sp, int64_t o_sc, const float *normal,
                       int64_t n_sb, int64_t n_sp, int64_t n_sc, const int32_t *order, const float *dir,
                       float *cloud, int64_t c_sb, int64_t c_sp, int64_t c_sc, float *trial, int64_t t_sb,
                       int64_t t_sp, int64_t t_sc, int32_t *state, float *best, int B, int N, float step_size,
                       float eps, int max_query, int targeted, int32_t *active /*or NULL*/, void *stream);

/* ------------------------------------------------------------------------------------
 * pcd_low_pass: the low-frequency component of AOF (attack on frequency, attack/AOF/TAOF_attack.py),
 * restated from the published method: y = V^T (V x) per sample and per channel, where the rows of
 * V [Kl,N] are the eigenvectors of the Kl smallest eigenvalues of the cloud's graph Laplacian
 * (pcd_graph_laplacian, then an eigensolver).  With orthonormal rows P = V^T V is a symmetric projector,
 * so the same call also gives the backward (y = P g).
 *   basis: V of sample b at basis + b*b_sb, row k at + k*N, contiguous along N (b_sb = 0 shares one
 *   basis over the batch).  x, y [B,N,3] fp32 via element strides (both the [B,N,3] and the [B,3,N]
 *   layouts); y must not overlap x.
 *   1. c[k][ch] = sum over n of V[k,n]*x[n][ch]: lane l of 32 sums the products of n = l (mod 32) in
 *      ascending n, starting from +0; then the 32 lane sums by an xor butterfly, s += s(lane ^ o) for
 *      o = 16, 8, 4, 2, 1 (every lane ends with the same value)
 *   2. y[n][ch] = sum over k ascending of V[k,n]*c[k][ch], starting from +0
 *   Every multiply and add is rounded to fp32 on its own.
 * split: 0 picks how many CTAs (a thread-block cluster, up to 8, 16 where the device schedules it)
 * share a sample from B, N, Kl and the SM count; a power of two <= 16 forces it (testing; the results
 * do not change).  16 on a device that cannot schedule it returns PCD_ERR_UNSUPPORTED.
 * A sample's outputs depend only on its own inputs: not on B, split or the strides.
 * Constraints: B >= 0 (0 is a no-op), N >= 1, 1 <= Kl <= N, b_sb >= 0, no NULL pointer; anything else
 * returns PCD_ERR_ARG before any CUDA call.  N > PCD_LP_MAX_N returns PCD_ERR_UNSUPPORTED.
 * Launches: one kernel; no workspace, no host synchronisation.
 * ---------------------------------------------------------------------------------- */
#define PCD_LP_MAX_N 16384

int pcd_low_pass(const float *basis, int64_t b_sb, int Kl, const float *x, int64_t x_sb, int64_t x_sp,
                 int64_t x_sc, int B, int N, float *y, int64_t y_sb, int64_t y_sp, int64_t y_sc, int split,
                 void *stream);

/* ------------------------------------------------------------------------------------
 * Measurement helper (bench.py): launches ONE FFMA-only probe kernel on `stream` (variant 0 =
 * scalar FFMA, 1 = packed FFMA2) and stores the number of FLOPs that launch performs in
 * *flop_count (HOST pointer).  The caller times it with its own CUDA events: achieved FLOP/s =
 * *flop_count / elapsed.  This is the measured roofline denominator for the sweep kernels (the
 * FP32 FMA peak is not in MEASURED_PEAKS.json).  scratch: >= 4 bytes of device memory (never
 * written in practice).  Stream-ordered, allocation-free, no synchronisation.
 * ---------------------------------------------------------------------------------- */
int pcd_fp32_probe_launch(int variant, int iters, float *scratch, double *flop_count, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PCDIST_H_ */
