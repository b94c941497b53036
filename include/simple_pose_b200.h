/*
 * simple_pose_b200 -- C ABI of the B200 (sm_100a) heatmap hot path.
 *
 * The reference (liangheming/simple_pose) is 100 % Python: it has no plugin, operator or FFI
 * layer. Its "interface" for this path is a set of Python call signatures; each entry point
 * below names the reference function it replaces (paths relative to the reference root).
 * The Python mirror of those signatures lives in simple_pose_b200/{commons,metrics,datasets,
 * processors}/ and reaches this library through ctypes (simple_pose_b200/_abi.py).
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every buffer is allocated and owned by the caller;
 *     the library never allocates or frees persistent device memory;
 *   - pointers are DEVICE pointers on the current CUDA device unless stated otherwise;
 *     tensors are dense, row-major ("C-contiguous"), base addresses 16-byte aligned;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); work is
 *     enqueued on it and the call returns without synchronising;
 *   - return value: 0 on success, a cudaError_t (> 0) for CUDA failures, or one of the
 *     SP_ERR_* codes (< 0) for argument errors; sp_error_string() names any of them.
 *     No exception crosses the boundary;
 *   - stateless and re-entrant; the only per-call scratch is the workspace the caller hands
 *     to the entry points that take one.
 */
#ifndef SIMPLE_POSE_B200_H
#define SIMPLE_POSE_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SP_ABI_VERSION 2

#define SP_ERR_BAD_ARGUMENT  (-1)   /* null pointer, non-positive size, unsupported value  */
#define SP_ERR_BAD_ALIGNMENT (-2)   /* a base pointer is not 16-byte aligned                */
#define SP_ERR_WORKSPACE     (-3)   /* workspace too small                                  */
#define SP_ERR_UNSUPPORTED   (-4)   /* shape outside what the kernels handle                */

/* decode modes of sp_decode_f32 */
#define SP_DECODE_GAUSS_TAYLOR 0    /* GaussTaylorKeyPointDecoder.__call__                  */
#define SP_DECODE_ARGMAX       1    /* BasicKeyPointDecoder.heat_map_to_axis (no affine)    */
#define SP_DECODE_BASIC        2    /* BasicKeyPointDecoder.__call__ (quarter-pixel shift)  */
#define SP_DECODE_DARK_ORIGINAL 3   /* DarkPoseOriginalKeyPointDecoder.__call__ (no clamp)  */

/* flags of sp_mse_fwd_bwd_f32 */
#define SP_MSE_SKIP_MASKED 1        /* do not read pred/target of joints whose mask is 0    */

int sp_abi_version(void);
const char* sp_error_string(int code);
/* SM count and compute capability of the current device (host-side query). */
int sp_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* The SP_* tuning variables (DESIGN.md "Tuning knobs") are read from the environment once per process,
 * at the first call into the library -- a launch never calls getenv. This re-reads them (tests and
 * parameter sweeps change a variable and reload). None of them changes results. */
int sp_reload_tuning(void);

/* ------------------------------------------------------------------------------------------
 * A1  RefineSimpleTransform.get_heat_map(joints, sigma=2.0, shape=(48, 64))
 *     commons/transforms.py:167-191, batched as MSCOCO.collate_fn does (datasets/coco.py:138-146).
 *
 * joints  [B,K,3] f32  (x, y, vis) in heatmap pixels
 * targets [B,K,H,W] f32 out; weights [B,K] f32 out
 * A joint is culled (weight 0, zero map) when int(x-3s) >= W or int(y-3s) >= H or
 * int(x+3s+1) < 0 or int(y+3s+1) < 0 (float32 arithmetic, truncation toward zero); a kept
 * joint with vis > 0.5 gets exp(-((px-x)^2+(py-y)^2)/(2 s^2)) over the whole map, evaluated
 * in float64 and rounded once to float32; otherwise a zero map. `sigma` is a double because
 * the reference uses a Python float.
 */
int sp_encode_f32(const float* joints, float* targets, float* weights,
                  int B, int K, int H, int W, double sigma, void* stream);

/* A1' BasicSimpleTransform.get_heat_map(joints, sigma=2.0, shape=(48, 64), stride=4)
 *     commons/transforms.py:80-116 (SURVEY section 8f rank 4). joints [B,K,3] f32 in INPUT pixels;
 *     the centre is quantised to int(x/stride + 0.5) and a side x side window of `table` is pasted
 *     (clipped to the map). table [side*side] f32 = the reference's float32 Gaussian patch
 *     exp(-((x-x0)^2+(y-y0)^2)/(2 s^2)), side = len(arange(0, 6s+1)), computed on the host with
 *     NumPy exactly as the reference does, so pasted values are bit-identical by construction.
 */
int sp_encode_basic_f32(const float* joints, const float* table, float* targets, float* weights,
                        int B, int K, int H, int W, double sigma, int stride, int side, void* stream);

/* ------------------------------------------------------------------------------------------
 * A2  0.5 * nn.MSELoss()(pred.mul(mask[..., None, None]), target.mul(mask[..., None, None]))
 *     and its backward; processors/dp_pose_hrnet_solver.py:86,106-107 (same expression in
 *     dp_pose_resnet_solver.py:107 and ddp_pose_resnet_solver.py:117).
 *
 * pred, target [B,K,HW] f32; mask [B,K] f32; grad [B,K,HW] f32 out (NULL = forward only);
 * loss: 1 f32 out = 0.5/(B*K*HW) * sum((m*p - m*t)^2);
 * grad = grad_scale * m * (m*p - m*t) / (B*K*HW)   (d loss / d pred).
 * One pass over pred/target; deterministic two-stage reduction in float64.
 * workspace: sp_mse_workspace_bytes() bytes, 16-byte aligned, ZERO-FILLED ONCE by the caller
 * before first use (the kernel restores the zero state before it finishes, so the same
 * buffer can be reused by later calls on the same stream without re-zeroing). It holds the
 * block partials, a completion ticket and -- for sp_encode_mse_fwd_bwd_f32 -- the grid-wide work
 * counter, so calls that may run CONCURRENTLY (different streams) need separate workspaces.
 */
size_t sp_mse_workspace_bytes(void);
int sp_mse_fwd_bwd_f32(const float* pred, const float* target, const float* mask,
                       float* grad, float* loss, void* workspace, size_t workspace_bytes,
                       int B, int K, int HW, float grad_scale, int flags, void* stream);

/* A2 under torch.cuda.amp (processors/dp_pose_hrnet_solver.py:111-120): `pred` in the autocast dtype, gradient in
 * the same dtype, arithmetic in float32 exactly as autocast runs the expression (the fp16 * fp32 product promotes
 * to float32, mse_loss is on autocast's float32 list, d loss / d pred is cast to pred's dtype once, after the
 * upstream gradient has been applied in float32).
 *   pred_dtype       SP_DTYPE_F32 / SP_DTYPE_F16 / SP_DTYPE_BF16; grad (nullable) has the same dtype
 *   loss             nullable: NULL = backward only (no reduction, workspace unused)
 *   grad_scale_dev   nullable device scalar (f32): the upstream gradient d L / d loss, e.g. GradScaler's scale,
 *                    multiplied with grad_scale on the device -- autograd's backward never has to read it
 *                    on the host. At least one of loss / grad must be given.
 * SP_DTYPE_F32 with loss != NULL and grad_scale_dev == NULL is sp_mse_fwd_bwd_f32 itself. */
#define SP_DTYPE_F32  0
#define SP_DTYPE_F16  1
#define SP_DTYPE_BF16 2
int sp_mse_fwd_bwd(const void* pred, int pred_dtype, const float* target, const float* mask,
                   void* grad, float* loss, void* workspace, size_t workspace_bytes,
                   int B, int K, int HW, float grad_scale, const float* grad_scale_dev, int flags, void* stream);

/* A2 + HeatMapAcc on the targets the loader ships, in the loss kernel's one pass -- what every solver computes per
 * batch from the same predicts / targets / mask (processors/dp_pose_hrnet_solver.py:106-107 and 123-124 in train(),
 * :156-157 in val(); the ResNet solvers alike):
 *   loss = 0.5 * MSELoss(predicts * mask, targets * mask)   (+ backward when grad is given)
 *   acc = HeatMapAcc()(predicts.mul(mask), targets.mul(mask))                  metrics/pose_metrics.py:212-245
 * i.e. sp_mse_fwd_bwd + the two masked copies + two sp_decode_f32(SP_DECODE_ARGMAX) + sp_heatmap_acc_f32.
 *   pred, target [B,K,H,W] (pred_dtype, grad, grad_scale_dev and flags as sp_mse_fwd_bwd; float16 / bfloat16 pred is
 *   multiplied by the mask in float32, as autocast's pred.mul(mask)); mask [B,K] f32; loss (1 f32) and acc (1 f32)
 *   are required (forward calls only: the backward-only call stays sp_mse_fwd_bwd with loss == NULL);
 *   pred_xy / label_xy [B,K,2] f32: heat_map_to_axis of the two masked maps (both NULL = kept in the workspace);
 *   distance_thresh, norm_frac: HeatMapAcc's constructor arguments (0.5, 10). H and W are separate because the
 *   coordinates and the thresholds are in (W, H) units. K <= 4096.
 * workspace: sp_mse_acc_workspace_bytes(B, K) bytes (0 = invalid sizes), 16-byte aligned, ZERO-FILLED ONCE by the
 * caller: the reduction workspace, the per-map argmax keys and room for the axes; every launch returns it to the
 * zero state, so it can be reused (and a captured graph replayed) on the same stream.
 * loss and grad are bit-identical to sp_mse_fwd_bwd, pred_xy / label_xy / acc to the composed calls. */
size_t sp_mse_acc_workspace_bytes(int B, int K);
int sp_mse_acc_fwd_bwd(const void* pred, int pred_dtype, const float* target, const float* mask, void* grad,
                       float* loss, float* acc, float* pred_xy, float* label_xy, void* workspace, size_t workspace_bytes,
                       int B, int K, int H, int W, float grad_scale, const float* grad_scale_dev,
                       float distance_thresh, float norm_frac, int flags, void* stream);

/* A1+A2(+HeatMapAcc) fused -- SURVEY section 8f ranks 1 and 2: targets are encoded on the fly and never
 * written (unless `targets` is given), so one pass reads pred and writes grad.
 *   targets, mask = get_heat_map(joints)                        commons/transforms.py:167-191
 *   loss = 0.5 * MSELoss(pred*mask, target*mask); backward       processors/dp_pose_hrnet_solver.py:106-107
 *   HeatMapAcc inputs: argmax of pred*mask and target*mask      metrics/pose_metrics.py:223-224
 * joints [B,K,3] f32 heatmap px; pred [B,K,H,W] f32; outputs: grad [B,K,H,W] (NULL = forward only),
 * targets [B,K,H,W] (NULL = do not materialise), weights [B,K] (NULL ok), loss (1 f32),
 * pred_xy / label_xy [B,K,2] f32 = heat_map_to_axis of the two masked maps (both NULL = skip).
 * Requires W % 4 == 0 (else SP_ERR_UNSUPPORTED: compose the two separate calls). Workspace as above.
 */
int sp_encode_mse_fwd_bwd_f32(const float* joints, const float* pred, float* grad, float* targets,
                              float* weights, float* loss, float* pred_xy, float* label_xy,
                              void* workspace, size_t workspace_bytes,
                              int B, int K, int H, int W, double sigma, float grad_scale, void* stream);

/* The same with `pred` / `grad` in the autocast dtype and the upstream gradient read on the device
 * (see sp_mse_fwd_bwd for pred_dtype, loss == NULL and grad_scale_dev). float16 / bfloat16 inputs, backward-only
 * calls and device-side scales run the plain-load kernel; SP_DTYPE_F32 with loss and without grad_scale_dev is
 * sp_encode_mse_fwd_bwd_f32 itself. */
int sp_encode_mse_fwd_bwd(const float* joints, const void* pred, int pred_dtype, void* grad, float* targets,
                          float* weights, float* loss, float* pred_xy, float* label_xy,
                          void* workspace, size_t workspace_bytes,
                          int B, int K, int H, int W, double sigma, float grad_scale, const float* grad_scale_dev,
                          void* stream);

/* The whole per-batch path over a predicted map in ONE launch: A1 + A2 (+ HeatMapAcc argmaxes) + A3/A4/A5, i.e.
 * sp_encode_f32 + sp_mse_fwd_bwd_f32 + sp_decode_f32(SP_DECODE_GAUSS_TAYLOR) (+ the two heat_map_to_axis passes of
 * HeatMapAcc) on the same `pred` -- the body of the solvers' val() loop (processors/dp_pose_hrnet_solver.py:150-161:
 * loss, acc, decoder on one `predicts`) and, with grad, BASELINE configs 1 + 2 together. Every map is staged in
 * shared memory once and read from HBM once.
 *   joints [B,K,3] f32 heatmap px; pred [B,K,H,W] f32; trans_inv [B,2,3] f32 (NULL = heatmap-space coords);
 *   blur_w [121] f32 (ksize must be 11); outputs: targets [B,K,H,W] (NULL = not materialised), weights [B,K]
 *   (NULL ok), grad [B,K,H,W] (NULL = no backward), loss (1 f32), coords [B,K,2], maxval [B,K] (both NULL = no decode pass),
 *   pred_xy / label_xy [B,K,2] (both NULL = skip). Workspace as sp_mse_fwd_bwd_f32.
 * coords / maxval / targets / weights / grad / pred_xy / label_xy are bit-identical to the stand-alone entry points,
 * the loss up to the float64 summation order. W % 4 != 0, ksize != 11 or maps too large for shared memory:
 * SP_ERR_UNSUPPORTED (compose the stand-alone calls). */
int sp_step_f32(const float* joints, const float* pred, const float* trans_inv, const float* blur_w,
                float* targets, float* weights, float* grad, float* loss, float* coords, float* maxval,
                float* pred_xy, float* label_xy, void* workspace, size_t workspace_bytes,
                int B, int K, int H, int W, double sigma, int ksize, float grad_scale, void* stream);

/* One validation batch in ONE launch: the body of every solver's val() -- processors/dp_pose_hrnet_solver.py:156-161,
 * dp_pose_resnet_solver.py and ddp_pose_resnet_solver.py alike:
 *   loss = 0.5 * MSELoss(predicts * mask, targets * mask)       (:156; forward only, val() runs under no_grad)
 *   acc = HeatMapAcc()(predicts * mask, targets * mask)          (:157)
 *   pred_kps, scores = decoder(predicts, tran_inv)               (:160; GaussTaylor or Basic KeyPointDecoder)
 *   kps_to_dict_(pred_kps, scores, img_ids, kps_dict_list)       (:161; as the sp_person_rows_f32 table)
 * i.e. sp_encode_mse_fwd_bwd_f32 (no grad, argmaxes) + sp_decode_ws_f32(mode) + sp_heatmap_acc_f32 + sp_person_rows_f32.
 *   joints [B,K,3] f32 heatmap px; pred [B,K,H,W] f32; trans_inv [B,2,3] f32 (NULL = heatmap-space coords);
 *   mode SP_DECODE_GAUSS_TAYLOR (blur_w [121] f32, ksize must be 11) or SP_DECODE_BASIC (blur_w and ksize unused);
 *   any other mode: SP_ERR_BAD_ARGUMENT.
 *   outputs: weights [B,K] (NULL ok), loss (1 f32), acc (1 f32), rows [B, 3K+1] f32 = (x, y, conf) * K then the person
 *   score mean(conf) + max(conf); coords [B,K,2] / maxval [B,K] (both NULL = rows only); pred_xy / label_xy [B,K,2]
 *   (the HeatMapAcc argmaxes; both NULL = kept in the workspace).
 *   distance_thresh, norm_frac: HeatMapAcc's constructor arguments (0.5, 10).
 * workspace: sp_val_step_workspace_bytes(B, K) bytes, 16-byte aligned, ZERO-FILLED ONCE by the caller. It holds the
 * reduction workspace, the per-person completion counters and room for the argmax axes; every launch returns the
 * counters to zero, so it can be reused (and a captured graph replayed) on the same stream.
 * rows, weights, coords, maxval, pred_xy, label_xy and acc are bit-identical to the composed entry points, the loss up to
 * the float64 summation order. W % 4 != 0, GaussTaylor with ksize != 11 or maps too large for shared memory:
 * SP_ERR_UNSUPPORTED (compose the stand-alone calls). */
size_t sp_val_step_workspace_bytes(int B, int K);
int sp_val_step_f32(const float* joints, const float* pred, const float* trans_inv, const float* blur_w, int mode,
                    float* weights, float* loss, float* acc, float* rows, float* coords, float* maxval,
                    float* pred_xy, float* label_xy, void* workspace, size_t workspace_bytes,
                    int B, int K, int H, int W, double sigma, int ksize, float distance_thresh, float norm_frac,
                    void* stream);

/* HeatMapAcc.__call__ epilogue, metrics/pose_metrics.py:225-245: per-joint fraction of persons whose
 * predicted argmax lies within distance_thresh (in units of (W,H)/norm_frac) of the target argmax, over
 * persons whose target argmax has x > 1 and y > 1, averaged over joints that have any. pred_xy, label_xy
 * [B,K,2] f32 (heat_map_to_axis outputs); acc: 1 f32 out. */
int sp_heatmap_acc_f32(const float* pred_xy, const float* label_xy, float* acc,
                       int B, int K, int H, int W, float distance_thresh, float norm_frac, void* stream);

/* grad[i] *= *scale_dev, skipped entirely (no memory traffic) when *scale_dev == 1.0f.
 * Used by the autograd wrapper when the upstream gradient is not 1 (e.g. GradScaler). */
int sp_scale_inplace_f32(float* data, long long n, const float* scale_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * A3/A4/A5/A6  decoders of metrics/pose_metrics.py.
 *   mode SP_DECODE_GAUSS_TAYLOR: GaussTaylorKeyPointDecoder.__call__ (:62-107)
 *   mode SP_DECODE_ARGMAX:       BasicKeyPointDecoder.heat_map_to_axis (:11-24); trans_inv unused
 *   mode SP_DECODE_BASIC:        BasicKeyPointDecoder.__call__ (:26-52)
 *   mode SP_DECODE_DARK_ORIGINAL: DarkPoseOriginalKeyPointDecoder.__call__ (:110-169), the reference's
 *                                NumPy/OpenCV per-joint decoder: same blur / log / Taylor step, the refined
 *                                coordinates are NOT clamped at 0; blur_w/ksize as for GAUSS_TAYLOR
 *
 * hm        [B,K,H,W] f32 (not modified)
 * hm_flip   NULL, or [B,K,H,W] f32: the network output for the horizontally mirrored image.
 *           Then the decoded map is 0.5*(hm[b,k,y,x] + hm_flip[b,perm[k],y,W-1-x]) -- the
 *           flip-test average composed from flip_joints (commons/joint_utils.py:102-112) and
 *           joint_pairs (datasets/coco.py:26); perm [K] i32 is required in that case.
 * trans_inv [B,2,3] f32 (NULL = identity, i.e. heatmap-space output)
 * blur_w    [ksize*ksize] f32 = float32(k k^T), k = cv.getGaussianKernel(ksize, 0)
 *           (:57-60); only read in GAUSS_TAYLOR mode; ksize odd, 3 <= ksize <= 15
 * coords    [B,K,2] f32 out (x, y); maxval [B,K] f32 out (un-blurred peak value)
 * argmax    NULL or [B,K] i32 out: flat index of the peak (first maximal index, NaN wins)
 */
int sp_decode_f32(const float* hm, const float* hm_flip, const int* perm,
                  const float* trans_inv, const float* blur_w,
                  float* coords, float* maxval, int* argmax,
                  int B, int K, int H, int W, int ksize, int mode, void* stream);

/* Same decoders, same results, with a scratch word the kernel deals its maps from GRID-WIDE (fast SMs
 * take more maps than slow ones; sp_decode_f32 gives every SM an equal range instead). workspace:
 * sp_decode_workspace_bytes() bytes, 16-byte aligned, ZERO-FILLED ONCE by the caller; every call
 * returns it to the zero state, so it can be reused by later calls ON THE SAME STREAM (calls that may
 * run concurrently need separate workspaces). */
size_t sp_decode_workspace_bytes(void);
int sp_decode_ws_f32(const float* hm, const float* hm_flip, const int* perm,
                     const float* trans_inv, const float* blur_w,
                     float* coords, float* maxval, int* argmax,
                     int B, int K, int H, int W, int ksize, int mode,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Decoder writing straight into the eval result table (eval.py:138-149 without the per-person
 * tolist()/JSON round trip): rows[b * row_stride + 3*k + {0,1,2}] = (x, y, peak value) of joint k of
 * person b; row_stride >= 3K floats (sp_eval_rows_nms_f32 wants >= 3K+3 and fills the remaining three).
 * coords / maxval (layouts as above) may be given as well or be NULL. Workspace as sp_decode_ws_f32. */
int sp_decode_rows_f32(const float* hm, const float* hm_flip, const int* perm,
                       const float* trans_inv, const float* blur_w,
                       float* rows, int row_stride, float* coords, float* maxval,
                       int B, int K, int H, int W, int ksize, int mode,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * A7  oks_iou(pick_kps, candi_kps, pick_area, candi_area, sigmas=None, in_vis_thresh=None)
 *     datasets/naive_data.py:120-150.  All float64.
 * pick_kps [K,3]; cand_kps [n,K,3]; pick_area: 1 f64 (device); cand_area [n]; sigmas [K]
 * (NULL = COCO 17-joint table, requires K == 17); use_vis_thresh 0 -> in_vis_thresh=None.
 */
int sp_oks_iou_f64(const double* pick_kps, const double* cand_kps, const double* pick_area,
                   const double* cand_area, const double* sigmas, double* out,
                   int n, int K, int use_vis_thresh, double vis_thresh, void* stream);

/* A8  oks_nms(kps, scores, areas, thresh, sigmas=None, in_vis_thresh=None)
 *     datasets/naive_data.py:153-173, segmented: one independent greedy NMS per image.
 * kps [N,K,3] f64; scores [N]; areas [N]; seg [I+1] i32 offsets (seg[0]=0, seg[I]=N);
 * keep [N] u8 out (1 = kept); rank [N] i32 out: position of each person in its image's
 * descending-score visiting order (ties: higher index first, as argsort()[::-1] of a stable
 * sort) so that the reference's pick-order list can be rebuilt without sorting again.
 * max_seg >= the largest seg[i+1]-seg[i] (sizes the per-image scratch in shared memory;
 * the caller builds seg on the host and knows it). Scores must not be NaN.
 */
int sp_oks_nms_f64(const double* kps, const double* scores, const double* areas, const int* seg,
                   const double* sigmas, unsigned char* keep, int* rank,
                   int N, int I, int K, int max_seg, double thresh,
                   int use_vis_thresh, double vis_thresh, void* stream);

/* A9  rescoring of eval.py:168-175: scores[i] = box_scores[i] * mean(conf[conf > thr]) (0 if none). */
int sp_rescore_f64(const double* kps, const double* box_scores, double* scores,
                   int N, int K, double in_vis_thre, void* stream);

/* Packs decoder output for the NMS stage without a host round trip: out_kps[n,k,:] =
 * (coords[n,k,0], coords[n,k,1], maxval[n,k]) widened to float64 (the JSON round trip of
 * eval.py:138-160 yields exactly these doubles). */
int sp_pack_kps_f64(const float* coords, const float* maxval, double* out_kps,
                    int N, int K, void* stream);

/* Result table of the sharded evaluation (eval.py:186-196 as one array instead of per-person dicts):
 * rows [N, 3K+2] f32 = (x, y, conf) * K from coords [N,K,2] / maxval [N,K], then the keep flag
 * (keep [N] u8, NULL = 0) and the rescored score (scores [N] f64, NULL = 0). */
int sp_pack_rows_f32(const float* coords, const float* maxval, const unsigned char* keep, const double* scores,
                     float* rows, int N, int K, void* stream);

/* A9 + A8 + result packing in ONE launch, the whole of eval.py:153-197 after the decoder: rows [N, row_stride]
 * f32 hold (x, y, conf) * K per person (sp_decode_rows_f32); per image (seg [I+1] i32) every person is
 * rescored (box_scores [N] f64 * mean(conf > in_vis_thre)), the greedy OKS-NMS of datasets/naive_data.py:153-173
 * runs on those scores with the float32 keypoints widened to float64 (exactly the doubles the reference
 * reads back from its JSON file), and the rows are completed in place:
 *   rows[i, 3K] = 1.0f if kept else 0.0f;  rows[i, 3K+1], rows[i, 3K+2] = low, high 32 bits of the float64
 *   score (reinterpret the two floats as one little-endian double: the score is NOT narrowed to float32).
 * areas: float64 [N] (areas_f64) or float32 [N] (areas_f32, what sp_box_affine_f64 writes); one non-NULL.
 * rank [N] i32 out (nullable) as in sp_oks_nms_f64. max_seg >= largest image. in_vis_thresh=None semantics. */
int sp_eval_rows_nms_f32(float* rows, int row_stride, const double* box_scores, const double* areas_f64,
                         const float* areas_f32, const int* seg, const double* sigmas, int* rank,
                         int N, int I, int K, int max_seg, double in_vis_thre, double oks_thre, void* stream);

/* The same kernel doing the multi-GPU all-gather of the result rows itself (one process per GPU; the reference
 * evaluates on one device, processors/ddp_pose_resnet_solver.py:155-156): `rows` is this rank's slot inside a
 * SYMMETRIC gather buffer that every rank has mapped (cuMem peer mappings over NVLink, e.g. torch's
 * torch.distributed._symmetric_memory), at float offset `slot_offset_floats` from the buffer's base. As soon as an
 * image's rows are complete the CTA that owns the image stores them into the same place of every rank's buffer:
 * through `multicast_base` (the NVLS multicast mapping of the buffer: one multimem.st is replicated to all ranks by
 * the NVSwitch) when it is non-NULL, else through `peer_bases` (DEVICE array [world] of the buffer's base address as
 * mapped for each rank) one peer at a time. No collective follows; the caller only needs a cross-rank barrier after
 * the kernel before any rank reads other ranks' rows. row_stride and slot_offset_floats must be even. */
int sp_eval_rows_nms_fanout_f32(float* rows, int row_stride, const double* box_scores, const double* areas_f64,
                                const float* areas_f32, const int* seg, const double* sigmas, int* rank,
                                int N, int I, int K, int max_seg, double in_vis_thre, double oks_thre,
                                void* multicast_base, const void* const* peer_bases, int world, int my_rank,
                                long long slot_offset_floats, void* stream);

/* A10 kps_to_dict_ (metrics/pose_metrics.py:172-179) as one table for a single device->host copy:
 * rows [N, 3K+1] f32 = (x, y, conf) * K from coords [N,K,2] / maxval [N,K], then the person score
 * mean(conf) + max(conf) (mean accumulated in float64, rounded once; NaN propagates). */
int sp_person_rows_f32(const float* coords, const float* maxval, float* rows, int N, int K, void* stream);

/* ------------------------------------------------------------------------------------------
 * A11 COCO keypoint AP: pycocotools' COCOeval(cocoGt, cocoDt, 'keypoints') with the keypoint defaults,
 *     catIds = [1] and maxDets = [20] -- evaluate(), accumulate() and the ten statistics of summarize()
 *     (eval.py:13-27, metrics/pose_metrics.py:182-209), without the result JSON file.
 *
 * Detections (N):
 *   det_rows   [N, det_stride] f32: x of joint k at 3k, y at 3k+1 (the eval table, stride 3K+3, and the
 *              kps_to_dict_ table, stride 3K+1, both fit); det_stride >= 3K
 *   det_scores [N] f64; det_img [N] i32: position of the detection's image in the evaluated image list;
 *              a detection with a position outside [0, I) is not evaluated; det_keep [N] u8 (NULL = all; 0 = not
 *              evaluated). Within an image the input order decides equal scores, as the results-list order does.
 * Ground truth (G persons, I evaluated images in params.imgIds order, parsed on the host once):
 *   gt_seg [I+1] i32 offsets (image i owns GT gt_seg[i]..gt_seg[i+1]-1, in annotation-file order);
 *   gt_kps [G, 3K] f64 (x, y, v); gt_area [G] f64; gt_bbox [G, 4] f64 (x, y, w, h);
 *   gt_flags [G] u8: bit 0 = ignore (iscrowd or num_keypoints == 0), bit 1 = iscrowd.
 * Parameters, computed on the host with NumPy exactly as Params.setKpParams does: iou_thrs [T] f64,
 *   rec_thrs [R] f64, area_rng [A, 2] f64. Anything but K = 17, T = 10, R = 101, A = 3, max_dets = 20:
 *   SP_ERR_UNSUPPORTED.
 * Outputs (f64, device): precision [T, R, A] and recall [T, A] (COCOeval's eval['precision'][:, :, 0, :, 0] and
 *   eval['recall'][:, 0, :, 0]; -1 where an area range has no non-ignored GT), stats [10] (summarize()).
 * Optional diagnostics (NULL = not written): oks_out [20 * G] f64: image i's [D_i, G_i] OKS matrix (detections
 *   ranked by score and cut to 20, GT in file order) row-major from oks_out + 20 * gt_seg[i]; det_flags_out
 *   [I * 20] u64 and det_order_out [I * 20] i32 per slot i * 20 + rank: bit (a * T + t) of the low word = matched
 *   at area range a and threshold t, of the high word = ignored; the detection's index (-1 = empty slot).
 * workspace: sp_coco_eval_workspace_bytes(N, I, G) bytes (0 = invalid sizes or no CUDA device), 16-byte aligned.
 *   Its contents on entry do not matter (every call writes what it reads), so it need not be zeroed; calls that
 *   may run concurrently need separate workspaces. No host synchronisation. */
size_t sp_coco_eval_workspace_bytes(int num_dets, int num_images, int num_gts);
int sp_coco_eval_kps_f32(const float* det_rows, int det_stride, const double* det_scores, const int* det_img,
                         const unsigned char* det_keep, int num_dets,
                         const double* gt_kps, const double* gt_area, const double* gt_bbox,
                         const unsigned char* gt_flags, const int* gt_seg, int num_images, int num_gts,
                         const double* iou_thrs, const double* rec_thrs, const double* area_rng,
                         int K, int T, int R, int A, int max_dets,
                         double* precision, double* recall, double* stats,
                         double* oks_out, unsigned long long* det_flags_out, int* det_order_out,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Eval-side caller of the decoder (SURVEY 8, "next": the data either side of the path):
 * BasicTransform.__call__ without the image warp, datasets/naive_data.py:44-56 =
 * box_to_center_scale (commons/joint_utils.py:39-56) + get_affine_transform(center, scale, 0,
 * output_shape) (commons/joint_utils.py:115-152, cv.getAffineTransform = 6x6 LU in float64).
 *
 * boxes         [P,4] f64  detection boxes, (x1, y1, x2, y2) as stored by :84-95 (SP_BOX_XYXY)
 *               or (x, y, w, h) as box_to_center_scale takes them (SP_BOX_XYWH)
 * center, scale [P,2] f32 out (nullable); area [P] f32 out = scale_w * scale_h (nullable)
 * trans_inv     [P,2,3] f32 out = what collate_fn ships (.float(), :114-116) (nullable)
 * trans_inv_f64 [P,2,3] f64 out = the unrounded cv result, heatmap -> image (nullable)
 * trans_f64     [P,2,3] f64 out = the forward (image -> heatmap) matrix, first return value of
 *               get_affine_transform (nullable)
 * w_h_ratio = input_w / input_h; (out_w, out_h) = heatmap size; scale_mult = 1.25.
 * Bit-identical to the reference (same roundings, same LU pivoting and operation order).
 */
#define SP_BOX_XYXY 0
#define SP_BOX_XYWH 1
int sp_box_affine_f64(const double* boxes, int box_format, float* center, float* scale, float* area,
                      float* trans_inv, double* trans_inv_f64, double* trans_f64, int P,
                      double w_h_ratio, int out_w, int out_h, float scale_mult, void* stream);

/* get_affine_transform(center, scale, rot = 0, (out_w, out_h)) (commons/joint_utils.py:115-152) for
 * P (center [P,2] f32, scale [P,2] f32) pairs; outputs as above (at least one non-null). */
int sp_center_scale_affine_f64(const float* center, const float* scale, float* trans_inv,
                               double* trans_inv_f64, double* trans_f64, int P, int out_w, int out_h,
                               void* stream);

/* get_affine_transform(center, scale, rot, (out_w, out_h)) with a rotation (commons/joint_utils.py:115-152;
 * the train-side call, commons/transforms.py:212-213). rot_deg [P] f64 degrees (NULL = all zero). */
int sp_center_scale_rot_affine_f64(const float* center, const float* scale, const double* rot_deg,
                                   float* trans_inv, double* trans_inv_f64, double* trans_f64, int P,
                                   int out_w, int out_h, void* stream);

/* ------------------------------------------------------------------------------------------
 * Train-side caller of the encoder: RefineSimpleTransform.__call__ (commons/transforms.py:193-223)
 * without the image work (cv.warpAffine, np.fliplr), its random draws passed in:
 *   box_to_center_scale (:200-201) -> scale * scale_ratio (:202-203, float32) -> flip_joints +
 *   centre mirror (:207-210; commons/joint_utils.py:102-112) -> get_affine_transform for the input
 *   and heatmap sizes (:212-213) -> affine_transform_batch (:217-218; joint_utils.py:88-99).
 * The result joints_hm feeds sp_encode_f32 / sp_encode_mse_fwd_bwd_f32 (:219).
 *
 * boxes        [P,4] f64  (x1, y1, x2, y2) AFTER box_crop
 * img_w        [P] i32    image widths (needed when flip != NULL)
 * joints       [P,K,3] f32 (x, y, vis) in image pixels
 * scale_ratio  [P] f64    draw of :202 (NULL = 1); rot_deg [P] f64 draw of :204 (NULL = 0)
 * flip         [P] u8     draw of :208 (NULL = never); perm [K] i32 with flipped[k] = original[perm[k]]
 * joints_hm    [P,K,3] f32 out  heatmap-pixel joints (rows with vis <= 0 are not mapped, as in the reference)
 * joints_input [P,K,3] f32 out  joint_info.joints, network-input pixels (nullable)
 * trans_inv    [P,2,3] f32 out  joint_info.trans_inv as collate_fn ships it (nullable)
 * trans_inv_f64, img_trans_f64 [P,2,3] f64 out: unrounded trans_inv; the image-warp matrix (nullable)
 * center, scale [P,2] f32 out after augmentation (center_scale_to_box of :220 follows from them) (nullable)
 * Same roundings as NumPy >= 2 / OpenCV; the only non-identical step is sin/cos of the rotation
 * (CUDA vs NumPy may differ in the last float64 bit, which the float32 rounding of the triangle
 * points absorbs except with probability ~1e-8).
 */
int sp_train_geometry_f32(const double* boxes, const int* img_w, const float* joints,
                          const double* scale_ratio, const double* rot_deg, const unsigned char* flip,
                          const int* perm, float* joints_hm, float* joints_input, float* trans_inv,
                          double* trans_inv_f64, double* img_trans_f64, float* center, float* scale, int P,
                          int K, int in_w, int in_h, int out_w, int out_h, float scale_mult, void* stream);

/* flip_joints (joint half, commons/joint_utils.py:102-112) and/or affine_transform_batch (:88-99) on
 * [P,K,3] f32 joints: flip [P] u8 + img_w [P] i32 + perm [K] i32 (all NULL = no flip), then
 * trans [P,2,3] f64 (NULL = no affine) applied to rows with vis > 0. out != joints. */
int sp_transform_joints_f32(const float* joints, const double* trans, const unsigned char* flip,
                            const int* img_w, const int* perm, float* out, int P, int K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SIMPLE_POSE_B200_H */
