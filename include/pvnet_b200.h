/*
 * pvnet_b200.h -- C ABI of libpvnet_b200.so: the B200 (sm_100a) implementation of
 * PVNet's per-image inference hot path (voting layer + Resnet18_8s backbone).
 *
 * Boundary rules (SURVEY.md §8b):
 *   - plain C types only: device pointers, sizes, strides; no torch/ATen types;
 *   - the CALLER owns every buffer, including the workspace; the library allocates
 *     nothing on the hot path and launches only on the given stream (CUDA-graph
 *     capturable); it never synchronises and never calls exit();
 *   - every function returns 0 on success, a negative PVNET_E_* code on failure;
 *     pvnet_last_error() returns a thread-local message for the last failure;
 *   - all pointers are DEVICE pointers on the current CUDA device unless a
 *     parameter says "host".
 *
 * Reference interfaces these entry points stand in for (paths relative to the
 * zju3dv/pvnet tree):
 *   lib/ransac_voting_gpu_layer/src/ransac_voting.cpp:20-31,103   generate_hypothesis
 *   lib/ransac_voting_gpu_layer/src/ransac_voting.cpp:41-55,104   voting_for_hypothesis
 *   lib/ransac_voting_gpu_layer/ransac_voting_gpu.py:514-598      ransac_voting_layer_v3
 *   lib/ransac_voting_gpu_layer/ransac_voting_gpu.py:333-406      estimate_voting_distribution_with_mean
 *   lib/ransac_voting_gpu_layer/ransac_voting_gpu.py:763-858      ransac_voting_layer_v5
 *   lib/ransac_voting_gpu_layer/ransac_voting_gpu.py:983-1034     generate_hypothesis (python level)
 *   lib/ransac_voting_gpu_layer/ransac_voting_gpu.py:99-216       ransac_voting_layer_v2 (refinement rounds)
 *   lib/ransac_voting_gpu_layer/src/ransac_voting.cpp:61-99       the vanishing-point kernel pair
 *   tools/train_linemod.py:119-130                                UncertaintyEvalWrapper.forward (v3 + with_mean)
 *   lib/utils/extend_utils/extend_utils.py:63-114                 uncertainty_pnp (+ evaluation_utils.py:165-201)
 *   lib/networks/model_repository.py:64-80                        Resnet18_8s.forward
 *   lib/utils/extend_utils/src/nearest_neighborhood.cu:48-163     findNearestPointIdxLauncher
 *   lib/utils/evaluation_utils.py:54-141                          Evaluator's metric methods
 * INTEGRATION.md shows the ctypes binding the reference's Python wrapper uses.
 */
#ifndef PVNET_B200_H_
#define PVNET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define PVNET_API __attribute__((visibility("default")))
#else
#define PVNET_API
#endif

/* opaque: a cudaStream_t passed as void* (torch: torch.cuda.current_stream().cuda_stream) */
typedef void *pvnet_stream_t;

enum {
    PVNET_OK = 0,
    PVNET_E_INVALID = -1,   /* bad argument (shape, stride, null pointer, size) */
    PVNET_E_WORKSPACE = -2, /* workspace too small */
    PVNET_E_CUDA = -3,      /* a CUDA runtime / driver call failed */
    PVNET_E_STATE = -4      /* object used before it was initialised */
};

/* How a mask element becomes "foreground". */
enum {
    PVNET_MASK_NONZERO_BYTE = 0, /* v3: `.byte()` then nonzero  (ransac_voting_gpu.py:527) */
    PVNET_MASK_EQUALS_ONE = 1    /* with_mean: `mask == 1`      (ransac_voting_gpu.py:339) */
};

PVNET_API const char *pvnet_last_error(void);
PVNET_API int pvnet_version(void);

/* ------------------------------------------------------------------ voting layer */

/* Bytes of workspace the fused voting entry points need for a batch of `b` images
 * of h*w pixels, `vn` keypoints and `hn_total` hypotheses per keypoint. */
PVNET_API int pvnet_vote_workspace_bytes(int b, int h, int w, int vn, int hn_total, size_t *bytes);

/* Per-image foreground counts (before any subsampling): fg_out[b] int32.
 * mask: [b,h,w] contiguous, elements of mask_elem_size bytes (1,2,4,8; integer or bool).
 * The host reads fg_out to replay the reference's torch RNG calls in the reference's
 * order (ransac_voting_gpu.py:531-547); nothing else in the layer needs the host. */
PVNET_API int pvnet_mask_foreground_count(const void *mask, int mask_elem_size, int mask_mode,
                                          int b, int h, int w, int32_t *fg_out,
                                          void *workspace, size_t workspace_bytes, pvnet_stream_t stream);

/* ransac_voting_layer_v3 (ransac_voting_gpu.py:514-598), whole batch, no host sync.
 *
 *   mask       [b,h,w] contiguous, foreground = low byte nonzero
 *   vertex     f32, logical shape [b,h,w,vn,2], addressed through vertex_strides[5]
 *              (in ELEMENTS).  The reference passes a permuted view of an NCHW tensor
 *              (tools/demo.py:48-50): strides {C*H*W, W, 1, 2*H*W, H*W}; it is read
 *              in place, never copied.
 *   idxs       int32 [b,hn,vn,2]: the pixel-pair samples (ransac_voting_gpu.py:547).
 *              Each value is reduced modulo the image's pixel count tn (identity for
 *              values already in [0,tn)).
 *   selection  f32 [b,h,w] or NULL: the uniform field of ransac_voting_gpu.py:538.
 *              Read only for images whose foreground count exceeds max_num; NULL means
 *              "never subsample" (all foreground pixels take part).
 *   out_pts    f32 [b,vn,2]  voted + least-squares-refitted keypoints (x,y);
 *              zeros for images with fewer than min_num foreground pixels (:531-534).
 *   out_counts int32 [b,hn,vn] or NULL: inlier count of every hypothesis (:561).
 *   out_hyp    f32 [b,hn,vn,2] or NULL: the hypotheses (:554).
 *   out_tn     int32 [b] or NULL: pixels that took part per image (after subsampling).
 *
 * The reference's `while True` (:552-576) re-scores the same idxs each round, so its
 * output does not depend on confidence/max_iter; one scoring pass is performed.
 */
PVNET_API int pvnet_ransac_voting_v3(const void *mask, int mask_elem_size,
                                     const float *vertex, const int64_t vertex_strides[5],
                                     const int32_t *idxs, const float *selection,
                                     int b, int h, int w, int vn, int hn,
                                     float inlier_thresh, int min_num, int max_num,
                                     float *out_pts, int32_t *out_counts, float *out_hyp, int32_t *out_tn,
                                     void *workspace, size_t workspace_bytes, pvnet_stream_t stream);

/* One refinement round of ransac_voting_layer_v2 (ransac_voting_gpu.py:178-204) for a whole batch: the
 * pixels (mask low byte nonzero, subsampled like v3) that are inliers of points [b,vn,2] re-estimate
 * them as the least-squares intersection of their lines -> out_pts [b,vn,2].  The reference's
 * pinverse(A) b equals this normal-equation solution for full-rank A.  Workspace:
 * pvnet_vote_workspace_bytes(b, h, w, vn, 1). */
PVNET_API int pvnet_refit_at_points(const void *mask, int mask_elem_size,
                                    const float *vertex, const int64_t vertex_strides[5],
                                    const float *selection, const float *points,
                                    int b, int h, int w, int vn, float inlier_thresh, int min_num, int max_num,
                                    float *out_pts, void *workspace, size_t workspace_bytes, pvnet_stream_t stream);

/* ransac_voting_layer_v5 (ransac_voting_gpu.py:763-858): v3 plus a per-keypoint confidence
 * out_conf [b,vn] = (inliers of the refitted point at conf_thresh, 0.999 in the reference :850)
 * / tn; zeros for skipped images (:788-793).  Same arguments as pvnet_ransac_voting_v3 otherwise. */
PVNET_API int pvnet_ransac_voting_v5(const void *mask, int mask_elem_size,
                                     const float *vertex, const int64_t vertex_strides[5],
                                     const int32_t *idxs, const float *selection,
                                     int b, int h, int w, int vn, int hn,
                                     float inlier_thresh, float conf_thresh, int min_num, int max_num,
                                     float *out_pts, float *out_conf, int32_t *out_counts, float *out_hyp,
                                     int32_t *out_tn, void *workspace, size_t workspace_bytes,
                                     pvnet_stream_t stream);

/* ransac_voting_layer_v4 (ransac_voting_gpu.py:669-760): v3 plus the residual variance of the
 * refit, out_var [b,vn] = sum over the winner's inliers of (n.p - n.c)^2 / #inliers with
 * n = (d_y,-d_x) and p the refitted point (:750-752; 0/0 = NaN as in torch); a skipped image
 * gives zeros and var = 1 (:685-689).  Same arguments as pvnet_ransac_voting_v3 otherwise. */
PVNET_API int pvnet_ransac_voting_v4(const void *mask, int mask_elem_size,
                                     const float *vertex, const int64_t vertex_strides[5],
                                     const int32_t *idxs, const float *selection,
                                     int b, int h, int w, int vn, int hn,
                                     float inlier_thresh, int min_num, int max_num,
                                     float *out_pts, float *out_var, int32_t *out_counts, float *out_hyp,
                                     int32_t *out_tn, void *workspace, size_t workspace_bytes,
                                     pvnet_stream_t stream);

/* ransac_motion_voting (ransac_voting_gpu.py:960-981; tools/train_linemod.py:117
 * `MotionEvalWrapper`): out_pts [b,vn,2] = mean over the foreground pixels (low byte nonzero, as
 * `.byte()`) of vertex + (x, y); zeros for an empty mask (:971-973).  Workspace:
 * pvnet_vote_workspace_bytes(b, h, w, vn, 1). */
PVNET_API int pvnet_ransac_motion_voting(const void *mask, int mask_elem_size,
                                         const float *vertex, const int64_t vertex_strides[5],
                                         int b, int h, int w, int vn, float *out_pts,
                                         void *workspace, size_t workspace_bytes, pvnet_stream_t stream);

/* estimate_voting_distribution_with_mean (ransac_voting_gpu.py:333-406).
 *
 *   mask       foreground = element == 1
 *   idxs       int32 [b,rounds*hn,vn,2], rounds = ceil(min_hyp_num/hn) (fresh draw per
 *              round, :367; the rounds are simply concatenated, :381-384)
 *   mean       f32 [b,vn,2] (from v3)
 *   out_cov    f32 [b,vn,2,2]: sum_h w_h d_h d_h^T / (sum_h w_h + 1e-3), d_h = hyp_h - mean,
 *              w_h = count_h/tn, zeroed where below (max_h w_h - 0.1)   (:394-401)
 *   Images with fewer than min_num foreground pixels use min_hyp_num hypotheses at
 *   (0,0) with weight 1 (:343-348).
 */
PVNET_API int pvnet_vote_cov_with_mean(const void *mask, int mask_elem_size,
                                       const float *vertex, const int64_t vertex_strides[5],
                                       const int32_t *idxs, const float *selection, const float *mean,
                                       int b, int h, int w, int vn, int hn, int rounds, int min_hyp_num,
                                       float inlier_thresh, int min_num, int max_num,
                                       float *out_cov, int32_t *out_counts, float *out_hyp, int32_t *out_tn,
                                       void *workspace, size_t workspace_bytes, pvnet_stream_t stream);

/* The uncertainty pipeline of tools/train_linemod.py:119-130 (`UncertaintyEvalWrapper.forward`):
 *     mean      = ransac_voting_layer_v3(mask, vertex, hn, inlier_thresh)            (ransac_voting_gpu.py:514-598)
 *     mean, cov = estimate_voting_distribution_with_mean(mask, vertex, mean, ...)     (ransac_voting_gpu.py:333-406)
 * as ONE launch sequence: the mask is compacted and the vector field gathered once for both
 * layers, and when both thresholds agree one kernel scores the v3 and the covariance hypotheses
 * together.  out_cov == NULL runs the v3 part alone.
 *
 *   mask_mode  how BOTH layers read the mask.  The reference's v3 takes nonzero (:527) and
 *              with_mean takes == 1 (:339); for the binary argmax mask of a 2-class network the
 *              two agree and either mode gives the reference's result.  (Callers with other
 *              masks use the two separate entry points.)
 *   idxs       int32 [b,hn,vn,2] or NULL; cov_idxs int32 [b,cov_rounds*cov_hn,vn,2] or NULL;
 *              selection f32 [b,h,w] or NULL (one field for both layers)
 *   rng_state  DEVICE pointer to {uint64 seed, uint64 offset} or NULL.  Whatever sample set is
 *              NULL is drawn on the device (Philox4x32-10; idxs = 32 random bits modulo tn like
 *              torch's random_, selection = 24 bits * 2^-24 like uniform_); the call then advances
 *              the offset, so a captured CUDA graph draws fresh samples on every replay.
 *              With rng_state == NULL a NULL selection means "never subsample".
 *   out_pts    f32 [b,vn,2]; out_cov f32 [b,vn,2,2] or NULL
 *   out_counts/out_hyp [b,hn,vn(,2)], out_cov_counts/out_cov_hyp [b,cov_rounds*cov_hn,vn(,2)],
 *   out_tn [b]: optional debug outputs.
 *   Workspace: pvnet_vote_workspace_bytes(b, h, w, vn, hn + cov_rounds*cov_hn). */
PVNET_API int pvnet_ransac_voting_pipeline(const void *mask, int mask_elem_size, int mask_mode,
                                           const float *vertex, const int64_t vertex_strides[5],
                                           const int32_t *idxs, const int32_t *cov_idxs, const float *selection,
                                           const unsigned long long *rng_state,
                                           int b, int h, int w, int vn, int hn, float inlier_thresh,
                                           int cov_hn, int cov_rounds, int cov_min_hyp_num, float cov_inlier_thresh,
                                           int min_num, int max_num, float *out_pts, float *out_cov,
                                           int32_t *out_counts, float *out_hyp,
                                           int32_t *out_cov_counts, float *out_cov_hyp, int32_t *out_tn,
                                           void *workspace, size_t workspace_bytes, pvnet_stream_t stream);

/* 1:1 stand-ins for the reference extension's two functions, same layouts:
 * direct [tn,vn,2] f32, coords [tn,2] f32 (x,y), idxs [hn,vn,2] i32, hypo [hn,vn,2] f32.
 * pvnet_generate_hypothesis writes every element of hypo (degenerate pairs -> (0,0),
 * ransac_voting_kernel.cu:42-43,75).  pvnet_voting_for_hypothesis only SETS inliers
 * [hn,vn,tn] u8 to 1 where the test passes (caller zero-fills, ransac_voting_gpu.py:557).
 * pvnet_vote_counts returns sum_t inliers as int32 [hn,vn] without the u8 tensor. */
PVNET_API int pvnet_generate_hypothesis(const float *direct, const float *coords, const int32_t *idxs,
                                        float *hypo, int tn, int vn, int hn, pvnet_stream_t stream);
PVNET_API int pvnet_voting_for_hypothesis(const float *direct, const float *coords, const float *hypo,
                                          uint8_t *inliers, int tn, int vn, int hn, float inlier_thresh,
                                          pvnet_stream_t stream);
PVNET_API int pvnet_vote_counts(const float *direct, const float *coords, const float *hypo,
                                int32_t *counts, int tn, int vn, int hn, float inlier_thresh,
                                pvnet_stream_t stream);

/* ------------------------------------------------------------------ uncertainty-driven PnP
 * The consumer of the keypoints + covariances above (SURVEY.md section 8 f-1); reference, per image on the
 * host: lib/utils/evaluation_utils.py:165-201 (`Evaluator.evaluate_uncertainty`) ->
 * lib/utils/extend_utils/extend_utils.py:63-114 (`uncertainty_pnp`) ->
 * lib/utils/extend_utils/src/uncertainty_pnp.cpp:61-92 (Ceres LM over 2 pn residuals x 6 parameters).
 *
 * pvnet_covariance_to_weights: cov f32 [n,2,2] -> weights f32 [n,3] = (wxx, wxy, wyy) of inv(sqrtm(cov)),
 *   zeros where cov[0,0] < 1e-6 or any element is NaN (evaluation_utils.py:170-181) or the matrix is not
 *   positive definite (where scipy's sqrtm + inv would fail).
 * pvnet_uncertainty_pnp: batched form of extend_utils.py:63 `uncertainty_pnp(points_2d, weights_2d,
 *   points_3d, camera_matrix)`: points_2d f32 [b,pn,2]; EITHER weights_2d f32 [b,pn,3] OR cov f32
 *   [b,pn,2,2] (converted as above; pass NULL for the other); points_3d f32 [pn,3] (one object);
 *   camera_matrix: HOST array of 9 doubles (row-major K).  4 <= pn <= 32.  One warp per image, fp64:
 *   P3P (Grunert) on the first three of the four points with the largest wxx + wxy (extend_utils.py:84;
 *   the fourth disambiguates, as OpenCV's SOLVEPNP_P3P), then Levenberg-Marquardt on
 *   sum_i |W_i (proj(R X_i + t) - x_i)|^2 (uncertainty_pnp.cpp:20-37) to the stationary point (pn == 4
 *   returns the P3P pose, :90-94).
 *   out_pose f64 [b,3,4] = (R | t) like the reference's return value; out_info int32 [b,2] or NULL =
 *   (status bits: 1 = P3P found no solution and the identity start was used, 2 = iteration cap hit;
 *   LM iterations). */
PVNET_API int pvnet_covariance_to_weights(const float *cov, int n, float *weights, pvnet_stream_t stream);
PVNET_API int pvnet_uncertainty_pnp(const float *points_2d, const float *cov, const float *weights_2d,
                                    const float *points_3d, const double camera_matrix[9], int b, int pn,
                                    double *out_pose, int32_t *out_info, pvnet_stream_t stream);

/* The vanishing-point pair of the reference extension (ransac_voting.cpp:61-99 ->
 * ransac_voting_kernel.cu:170-260, :263-351; used by ransac_voting_vanish_point_layer,
 * ransac_voting_gpu.py:408-501): hypotheses are homogeneous points hypo [hn,vn,3]; the vote sets
 * inliers [hn,vn,tn] u8 (caller zero-fills; may be NULL) and/or writes the row sums counts [hn,vn]. */
PVNET_API int pvnet_generate_hypothesis_vanishing_point(const float *direct, const float *coords, const int32_t *idxs,
                                                        float *hypo, int tn, int vn, int hn, pvnet_stream_t stream);
PVNET_API int pvnet_voting_for_hypothesis_vanishing_point(const float *direct, const float *coords, const float *hypo,
                                                          uint8_t *inliers, int32_t *counts, int tn, int vn, int hn,
                                                          float inlier_thresh, pvnet_stream_t stream);

/* ------------------------------------------------------------------ pose-accuracy metrics
 *
 * pvnet_find_nearest_point_idx: batched form of extend_utils.py:39-60 `find_nearest_point_idx(ref_pts,
 *   que_pts)`, the index the reference kernel findNearestPoint{2D,3D}IdxKernel (nearest_neighborhood.cu:48-117)
 *   returns, bit for bit:
 *     ref   f32 [b,pn1,dim]  the points searched
 *     que   f32 [b,pn2,dim]  one answer per query point
 *     idxs  int32 [b,pn2]    out: for que[bi,j], the i minimising |ref[bi,i] - que[bi,j]|^2
 *     dim   2 or 3;  exclude_self != 0 skips i == j (the launcher's last argument, :123-163)
 *   The distance is the reference's rounding sequence (d = ref - que; 2-D fma(dx,dx,dy*dy), 3-D
 *   fma(dz,dz,fma(dx,dx,dy*dy)), DESIGN.md §2); the selection starts at (FLT_MAX, 0) and replaces only on a
 *   strict `<` in increasing index: the lowest index wins a tie, NaN and +inf are never chosen, a query with
 *   no finite distance gets 0.  Offsets are 64-bit.  b <= 65535.  No workspace. */
PVNET_API int pvnet_find_nearest_point_idx(const float *ref, const float *que, int32_t *idxs, int b, int pn1, int pn2,
                                           int dim, int exclude_self, pvnet_stream_t stream);

/* Flags of pvnet_pose_metrics. */
enum {
    PVNET_METRICS_SYM_ADD = 1,  /* ADD-S: add_metric_sym (evaluation_utils.py:119-130) instead of add_metric */
    PVNET_METRICS_SYM_PROJ = 2, /* projection_2d_sym (:83-89) instead of projection_2d (:75-81) */
    PVNET_METRICS_PRED_F32 = 4, /* pose_pred holds float32 values: its cloud is float32, as numpy makes it */
    PVNET_METRICS_GT_F32 = 8    /* pose_gt holds float32 values (the data loader's dtype): likewise */
};

/* pvnet_pose_metrics: the metric methods of the reference's Evaluator (evaluation_utils.py:64-141) for a batch
 * of b images of one object, fp64, deterministic (fixed-order sums):
 *   pose_pred, pose_gt  f64 [b,3,4] (R | t)
 *   model_points        f32 [pn,3] (the object model, metres)
 *   camera_matrix       HOST array of 9 doubles, one K for all images; OR
 *   camera_matrices     f64 [b,3,3] on the device, one K per image (`use_camera_intrinsic`); pass NULL for the other
 *   flags               PVNET_METRICS_* above
 *   values              out f64 [b,4]:
 *     [0] add_dist        mean_X |(R_p X + t_p) - (R_g X + t_g)|                        add_metric      :91-117
 *                         with SYM_ADD: mean over target points of the distance to the nearest predicted point,
 *                         the index searched on both clouds rounded to f32 (find_nearest_point_distance :54-62)
 *     [1] proj_mean_diff  mean 2-D distance of the two projections (Projector.project_K)  projection_2d   :75-81
 *                         with SYM_PROJ: the same nearest-point rule in 2-D              projection_2d_sym :83-89
 *     [2] trans_cm        |t_p - t_g| * 100                                              cm_degree_5_metric :132-141
 *     [3] rot_deg         degrees(arccos((min(tr(R_p R_g^T), 3) - 1) / 2)); no lower clamp (NaN below -1)
 *   ok                  out u8 [b,3]: add_dist < add_threshold (the reference's percentage * diameter),
 *                       proj_mean_diff < proj_threshold (5), trans_cm < cm_threshold && rot_deg < deg_threshold (5, 5)
 *   workspace           pvnet_pose_metrics_workspace_bytes(b, pn, flags) bytes (0 without a SYM flag: may be NULL)
 * One launch, plus one cloud launch and one pvnet_find_nearest_point_idx launch per SYM flag. */
PVNET_API int pvnet_pose_metrics_workspace_bytes(int b, int pn, int flags, size_t *bytes);
PVNET_API int pvnet_pose_metrics(const double *pose_pred, const double *pose_gt, const float *model_points,
                                 const double camera_matrix[9], const double *camera_matrices, int b, int pn, int flags,
                                 double add_threshold, double proj_threshold, double cm_threshold,
                                 double deg_threshold, double *values, uint8_t *ok, void *workspace,
                                 size_t workspace_bytes, pvnet_stream_t stream);

/* Number of kernels this library has launched on the calling thread since the last
 * reset (bench.py's "gpu_launches"). */
PVNET_API long long pvnet_launch_count(void);
PVNET_API void pvnet_launch_count_reset(void);

/* -------------------------------------------------------------------- backbone */

/* One NHWC convolution on the tcgen05 tensor cores (TF32 inputs, fp32 accumulate), the
 * building block of Resnet18_8s (lib/networks/resnet.py:28-35,54-70; model_repository.py:22-58):
 *
 *   out[n,y,x,out_co+co] = act( bias[co] + res[n,y,x,res_co+co]
 *                               + sum_{kh,kw,ci} w[co][kh][kw][ci] * in[n, y*stride+(kh-c)*dil, x*stride+(kw-c)*dil, in_co+ci] )
 *
 *   in        NHWC buffer [b,H,W,in_cs]; the conv reads channels [in_co, in_co+Cin)
 *   w_packed  [Cout][ksize*ksize][cin_pad] fp32 (BatchNorm already folded in; cin_pad = Cin rounded up
 *             to a multiple of 32, zero padded; 16 stays 16), bias [Cout]
 *   res       NHWC [b,H/stride,W/stride,res_cs] read at res_co, or NULL
 *   out       NHWC [b,H/stride,W/stride,out_cs] written at channel offset out_co
 *             (writing into a slice of a wider buffer replaces torch.cat)
 *   ksize 1|3, stride 1|2 (2 needs even H,W, dilation 1), padding = dilation*(ksize-1)/2
 *   act 0 none, 1 ReLU, 2 LeakyReLU(0.1); round_out != 0 rounds the stored values to TF32
 *   Cin multiple of 4, Cout multiple of 32; strides/offsets multiples of 4 floats.
 */
PVNET_API int pvnet_conv2d_nhwc(const float *in, int in_cs, int in_co, int Cin,
                                const float *w_packed, const float *bias,
                                const float *res, int res_cs, int res_co,
                                float *out, int out_cs, int out_co, int Cout,
                                int b, int H, int W, int ksize, int stride, int dilation,
                                int act, int round_out, pvnet_stream_t stream);

/* Test hook: which convolution kernel pvnet_conv2d_nhwc / the backbone use for layers both can
 * run.  0 = automatic (persistent weights-resident column kernel for 3x3 stride-1 layers with
 * Cout <= 64 whose weights fit in shared memory, per-tap kernel otherwise), 1 = per-tap kernel
 * only, 2 = column kernel (error if the layer is not eligible). */
PVNET_API int pvnet_conv_set_mode(int mode);
/* Test hook: how the per-tap kernel runs 256-channel weight tiles.  0 (default) = single CTAs;
 * 1 = 2-CTA clusters with TMA multicast of the weight tile; 2 = 2-CTA clusters issuing
 * tcgen05.mma.cta_group::2 (each CTA holds half of the weight tile). */
PVNET_API int pvnet_conv_set_multicast(int on);
/* Test hook: 1 (default) runs single-CTA tiles of the per-tap kernel on its persistent variant
 * (continuous TMA ring, two TMEM accumulator stages); 0 = one tile per CTA. */
PVNET_API int pvnet_conv_set_persistent(int on);
/* Test hook / tuning knob: epilogue warp sets of the fused-head column kernel (convraw.0) in plans built
 * afterwards.  1 = one set of four warps (default), 2 = two sets alternating tiles (measured no faster: the
 * launch is tensor-pipe bound), 0 = default (environment variable PVNET_HEAD_EPI, else 1). */
PVNET_API int pvnet_conv_set_head_epilogue_sets(int sets);

/* Resnet18_8s.forward (lib/networks/model_repository.py:64-80), eval mode, whole batch.
 *
 * The handle is a host-side table of per-convolution weight pointers plus cached tensor
 * maps; it owns no device memory.  Weights are DEVICE pointers owned by the caller and
 * must stay valid while the handle is used:
 *   slot 0               stem conv1+bn1, packed [7*7][3][64] (tap, cin, cout), bias [64]
 *   slots 1..24          the 3x3 / 1x1 convs in execution order (layer1.0.conv1, layer1.0.conv2,
 *                        layer1.1.conv1, layer1.1.conv2, layer2.0.conv1, layer2.0.downsample,
 *                        layer2.0.conv2, layer2.1.conv1, layer2.1.conv2, layer3.* and layer4.* in the
 *                        same pattern, fc.0, conv8s.0, conv4s.0, conv2s.0, convraw.0), each packed
 *                        [Cout][kh*kw][cin_pad] with its BatchNorm folded in, bias [Cout].  convraw.0 reads
 *                        s2dim+8 buffer channels (s2dim upsampled, 3 image, 5 zeros); cin_pad rounds up to 32.
 *   slot 25              convraw.3 (1x1, with bias): [seg_dim+ver_dim][32], bias [seg_dim+ver_dim]
 *   slot 26              the stem once more for the tensor-core path: the 7x7 stride-2 conv written as
 *                        a 4x4 stride-1 conv over the 2x2 space-to-depth image, packed [64][4][4][16]
 *                        (tap (ty,tx), channel (py*2+px)*3+c holds w[c][2ty+py-1][2tx+px-1]; rest 0)
 * pvnet_backbone_forward:
 *   image_nchw  f32 [b,3,h,w] (h,w multiples of 8)
 *   out_nchw    f32 [b,seg_dim+ver_dim,h,w]: seg logits are channels [0,seg_dim), the vertex
 *               field the rest (model_repository.py:77-78)
 *   mask_out    optional [b,h,w] argmax over the seg channels (first maximum), int64
 *               (mask_elem_size 8, what torch.argmax returns) or uint8 (1); NULL to skip
 */
typedef struct pvnet_backbone pvnet_backbone_t;
PVNET_API int pvnet_backbone_create(int ver_dim, int seg_dim, int fcdim, int s8dim, int s4dim, int s2dim,
                                    int raw_dim, pvnet_backbone_t **out);
PVNET_API void pvnet_backbone_destroy(pvnet_backbone_t *m);
PVNET_API int pvnet_backbone_num_convs(void);
PVNET_API int pvnet_backbone_set_conv(pvnet_backbone_t *m, int slot, const float *w_packed, const float *bias);
/* Output layout of the following forward calls on this handle: 0 (default) = out [b,C,h,w], the
 * reference's NCHW tensor whose channel slices are seg_pred / ver_pred (model_repository.py:77-78);
 * 1 = pixel-major out [b,h,w,C]: the same values as one contiguous record per pixel, which is the
 * vertex layout [b,h,w,K,2] the voting layer's gather reads without sector waste (the contiguous
 * form of the permuted view of tools/demo.py:48-50). */
PVNET_API int pvnet_backbone_set_output_layout(pvnet_backbone_t *m, int pixel_major);
/* The last decoder upsampling, F.interpolate(x2s_up, scale_factor=2, mode='bilinear', align_corners=True)
 * (model_repository.py:75), can run inside convraw.0's operand loader: the full-resolution
 * [b,h,w,s2dim] tensor is then never written, the output is bit-identical.  on = 1 selects the fused
 * form with the interpolation on convraw.0's epilogue warps (two CTAs per SM), 2 the form with eight
 * dedicated interpolation warps (one CTA per SM, four-tile operand ring), 0 the separate upsampling
 * launch, -1 = default (environment variable PVNET_FUSE_UP; see DESIGN.md section 5 for the measurements). */
PVNET_API int pvnet_backbone_set_fused_upsample(pvnet_backbone_t *m, int on);
PVNET_API int pvnet_backbone_workspace_bytes(const pvnet_backbone_t *m, int b, int h, int w, size_t *bytes);
PVNET_API int pvnet_backbone_forward(pvnet_backbone_t *m, const float *image_nchw, int b, int h, int w,
                                     float *out_nchw, void *mask_out, int mask_elem_size,
                                     void *workspace, size_t workspace_bytes, pvnet_stream_t stream);
/* Same forward pass from a RAW image batch: image_hwc uint8 [b,h,w,3] (what an image decoder yields),
 * normalised on the device inside the packing kernel with torchvision's ToTensor + Normalize
 * arithmetic, (float(v)/255 - mean[c]) / std[c] in fp32 (tools/demo.py:89-95,
 * lib/datasets/linemod_dataset.py:191-195): bit-identical to pvnet_backbone_forward on the
 * torch-normalised float tensor, a quarter of the input bytes.  mean/std are HOST arrays. */
PVNET_API int pvnet_backbone_forward_u8(pvnet_backbone_t *m, const uint8_t *image_hwc, const float mean[3],
                                        const float std[3], int b, int h, int w,
                                        float *out_nchw, void *mask_out, int mask_elem_size,
                                        void *workspace, size_t workspace_bytes, pvnet_stream_t stream);
/* JPEG bytes -> the uint8 [b,h,w,3] RGB batch pvnet_backbone_forward_u8 takes, decoded on the device by
 * NVIDIA's nvJPEG (library code; dlopen'ed on first use -- pvnet_jpeg_available() says whether it was found).
 * Replaces the host-side `Image.open` of lib/datasets/linemod_dataset.py:180-195 / tools/demo.py:89.
 * jpeg_data / lengths: HOST arrays of b host pointers / sizes; every image must be h x w.  The decoder object
 * owns nvJPEG's internal buffers (the one place this library lets a dependency allocate).  Different decoder
 * than the reference's libjpeg: +-1 level from the IDCT, more at colour edges of chroma-subsampled files. */
typedef struct pvnet_jpeg_decoder pvnet_jpeg_decoder_t;
PVNET_API int pvnet_jpeg_available(void);
PVNET_API int pvnet_jpeg_decoder_create(pvnet_jpeg_decoder_t **out);
PVNET_API void pvnet_jpeg_decoder_destroy(pvnet_jpeg_decoder_t *d);
PVNET_API int pvnet_jpeg_decode_batch(pvnet_jpeg_decoder_t *d, const uint8_t *const *jpeg_data, const size_t *lengths,
                                      int b, int h, int w, uint8_t *out_hwc, pvnet_stream_t stream);

/* The forward pass is an ordered list of single-kernel stages; these run/describe one of
 * them with the same arguments (per-layer timing in bench.py, layer-wise parity tests). */
PVNET_API int pvnet_backbone_num_stages(void);
PVNET_API const char *pvnet_backbone_stage_name(int stage);
PVNET_API int pvnet_backbone_run_stage(pvnet_backbone_t *m, int stage, const float *image_nchw, int b, int h, int w,
                                       float *out_nchw, void *mask_out, int mask_elem_size,
                                       void *workspace, size_t workspace_bytes, pvnet_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PVNET_B200_H_ */
