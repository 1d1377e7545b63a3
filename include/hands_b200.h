/*
 * hands_b200.h -- C ABI of libhands_b200.so: the geometry hot path of ap229997/hands
 * (MANO layer + LBS + camera/projection + Perspective Crop Layer), forward and backward,
 * as hand-written CUDA for sm_100a.
 *
 * The reference has no FFI of its own: its seam is a set of Python call signatures
 * (SURVEY.md section 8(b)).  Each entry point below names the reference code it replaces.
 * Python (hands_b200/) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every function returns int: 0 = OK, <0 = argument error (HB_E_*), >0 = cudaError_t.
 *     hb_last_error_string() gives the text of the last failure on the calling thread.
 *   - all tensors are fp32, contiguous, row-major (except the bf16 crop planes of the *_bf16 crop-layer
 *     entry points); pointers are DEVICE pointers unless the parameter name ends in _host.  Float buffers
 *     must be 8-byte aligned.
 *   - the caller allocates and owns every buffer, including the workspace; the library never
 *     allocates per call and never frees caller memory.
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous on it.
 *   - nullable pointers are marked "or NULL"; a NULL output is simply not written, a NULL
 *     upstream gradient counts as zero.
 */
#ifndef HANDS_B200_H
#define HANDS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define HB_E_ARG (-1)      /* NULL / negative size / bad flag            */
#define HB_E_ALIGN (-2)    /* a float buffer is not 8-byte aligned       */
#define HB_E_WORKSPACE (-3)/* workspace too small                        */
#define HB_E_UNSUPPORTED (-4)

#define HB_NUM_VERTS 778
#define HB_NUM_JOINTS 16
#define HB_NUM_OUT_JOINTS 21
#define HB_NUM_BETAS 10

typedef struct hb_mano hb_mano; /* opaque: MANO constants of one hand side on one device */

/* pose input formats of hb_mano_head_fwd/bwd */
#define HB_POSE_AXIS_ANGLE 0
#define HB_POSE_ROTMAT 1
#define HB_POSE_ROT6D 2 /* + hb_rot6d_layout */
/* The reference's three 6D -> rotation-matrix conversions (Gram-Schmidt, F.normalize eps 1e-12) differ in layout: */
#define HB_ROT6D_ROWS 0        /* pytorch3d rotation_6d_to_matrix (src/nets/hand_heads/hand_hmr.py:85-87): a1=x[0:3], a2=x[3:6], b1,b2,b3 are ROWS */
#define HB_ROT6D_COLS 1        /* src/models/hamer_light/geometry.py:47-62, src/models/handoccnet_light/mano_head.py:132-141: a1=x[0:3], a2=x[3:6], COLUMNS */
#define HB_ROT6D_COLS_PAIRED 2 /* common/rot.py:367-381: a1=x[0,2,4], a2=x[1,3,5], COLUMNS */

#define HB_VERSION 206 /* hb_version() of a matching binary */
const char* hb_last_error_string(void);
int hb_version(void);

/* ---- MANO constants --------------------------------------------------------------------
 * Replaces: common/body_models.py:92-99 build_mano_aa -> smplx.MANO(...) buffer registration.
 * All inputs are HOST pointers in the smplx buffer layouts:
 *   v_template (778,3)  shapedirs (778,3,10)  posedirs (135,2334) [column 3v+k]
 *   J_regressor (16,778)  lbs_weights (778,16)  parents (16)  pose_mean (48)  tip_ids (5)
 * Copies them to `device` once, re-laid-out for the kernels (joint regression folded into
 * J_template/J_shapedirs in fp64). */
int hb_mano_create(const float* v_template_host, const float* shapedirs_host, const float* posedirs_host,
                   const float* J_regressor_host, const float* lbs_weights_host, const int32_t* parents_host,
                   const float* pose_mean_host, const int32_t* tip_ids_host, int device, hb_mano** out);
int hb_mano_destroy(hb_mano* h);

/* Bytes of scratch the fwd / bwd calls need for a batch of B hands. */
size_t hb_mano_workspace_bytes(int B, int backward);

/* ---- MANO layer + head, forward ----------------------------------------------------------
 * Replaces: src/nets/hand_heads/mano_head.py:21-65 MANOHead.forward (pose_format=1, cam and K
 * given) and smplx.MANO.forward as called at mano_head.py:34-38, process_arctic.py:16-34,
 * src/arctic/processing.py:175-188 (pose_format=0, cam=K=NULL, optional transl).
 *   pose      pose_format HB_POSE_AXIS_ANGLE: (B,48) axis-angle
 *             pose_format HB_POSE_ROTMAT:     (B,16,3,3) rotation matrices
 *             pose_format HB_POSE_ROT6D + L:  (B,16,6) 6D rotations in layout L (hb_rot6d_layout below): the
 *               6D -> matrix conversion the reference runs before the head (hand_hmr.py:85-87,
 *               hamer_light/mano_head.py:98-105, handoccnet_light/mano_head.py:194) fused in front of the log map
 *   pre_rot   (B,3,3) or NULL: left-multiplied onto joint 0 before the log map
 *             (src/models/hands_light/model.py:330-334, the PCL orientation fix-up)
 *   betas (B,10)   cam (B,3)=[s,tx,ty] or NULL   K (B,3,3) or NULL   transl (B,3) or NULL
 * Outputs (each or NULL): vertices (B,778,3), v3d_cam (B,778,3), joints3d (B,21,3),
 *   j3d_cam (B,21,3), j2d_norm (B,21,2), cam_t (B,3).  Camera outputs need cam and K.
 * Workspace: >= hb_mano_workspace_bytes(B, 0).  The forward's intermediates fill the start of the workspace in the
 *   layout the backward reads, so a backward-sized workspace can be handed on to hb_mano_head_bwd_reuse(). */
int hb_mano_head_fwd(const hb_mano* h, const float* pose, int pose_format, const float* pre_rot,
                     const float* betas, const float* cam, const float* K, const float* transl, int B,
                     float img_res, float min_s, float* vertices, float* v3d_cam, float* joints3d,
                     float* j3d_cam, float* j2d_norm, float* cam_t, void* workspace, size_t workspace_bytes,
                     void* stream);

/* ---- backward ----------------------------------------------------------------------------
 * Same inputs (saved by the caller; everything else is recomputed), upstream gradients of the
 * six outputs (each or NULL), and gradients w.r.t. pose (same shape as pose), betas, cam
 * (or NULL), transl (or NULL), pre_rot (or NULL).  K gets no gradient (data in the reference). */
int hb_mano_head_bwd(const hb_mano* h, const float* pose, int pose_format, const float* pre_rot,
                     const float* betas, const float* cam, const float* K, const float* transl, int B,
                     float img_res, float min_s, const float* g_vertices, const float* g_v3d_cam,
                     const float* g_joints3d, const float* g_j3d_cam, const float* g_j2d_norm,
                     const float* g_cam_t, float* g_pose, float* g_betas, float* g_cam, float* g_transl,
                     float* g_pre_rot, void* workspace, size_t workspace_bytes, void* stream);

/* Same backward when `workspace` is the very buffer a preceding hb_mano_head_fwd call on the SAME inputs was given, with
 * nothing written to it in between.  Like any backward it needs workspace_bytes >= hb_mano_workspace_bytes(B, 1).  The
 * forward's skinning transforms, feature slabs and v_posed (11.6 KB/hand) are picked up instead of recomputed (two launches
 * and the blendshape contraction less).  Results are bit-identical to hb_mano_head_bwd. */
int hb_mano_head_bwd_reuse(const hb_mano* h, const float* pose, int pose_format, const float* pre_rot,
                           const float* betas, const float* cam, const float* K, const float* transl, int B,
                           float img_res, float min_s, const float* g_vertices, const float* g_v3d_cam,
                           const float* g_joints3d, const float* g_j3d_cam, const float* g_j2d_norm,
                           const float* g_cam_t, float* g_pose, float* g_betas, float* g_cam, float* g_transl,
                           float* g_pre_rot, void* workspace, size_t workspace_bytes, void* stream);

/* ---- free functions of the path ------------------------------------------------------------
 * common/rot.py:180-193 matrix_to_axis_angle, forward and backward; N matrices. */
int hb_matrix_to_axis_angle_fwd(const float* R, int N, float* aa, void* stream);
int hb_matrix_to_axis_angle_bwd(const float* R, const float* g_aa, int N, float* g_R, void* stream);
/* 6D rotation representation -> rotation matrix, x6 (N,6) -> R (N,3,3), in one of the reference's three layouts
 * (HB_ROT6D_* above); backward w.r.t. x6. */
int hb_rot6d_to_rotmat_fwd(const float* x6, int N, int layout, float* R, void* stream);
int hb_rot6d_to_rotmat_bwd(const float* x6, const float* g_R, int N, int layout, float* g_x6, void* stream);
/* common/transforms.py:316-329 project2d_batch (+ optional data_utils.py:361-365 normalize_kp2d when
 * img_res > 0): K (B,3,3), pts (B,N,3) -> out (B,N,2); backward w.r.t. pts. */
int hb_project2d_fwd(const float* K, const float* pts, int B, int N, float img_res, float* out, void* stream);
int hb_project2d_bwd(const float* K, const float* pts, const float* g_out, int B, int N, float img_res,
                     float* g_pts, void* stream);
/* common/camera.py:456-474 weak_perspective_to_perspective_torch and :10-29 its inverse.
 * focal (B,).  backward of the first w.r.t. cam. */
int hb_weak_to_persp_fwd(const float* cam, const float* focal, int B, float img_res, float min_s, float* cam_t,
                         void* stream);
int hb_weak_to_persp_bwd(const float* cam, const float* focal, const float* g_cam_t, int B, float img_res,
                         float min_s, float* g_cam, void* stream);
int hb_persp_to_weak_fwd(const float* cam_t, const float* focal, int B, float img_res, float* cam_wp, void* stream);
/* src/models/hands_light/model.py:330-334: out[b] = (transpose_R ? R[b]^T : R[b]) @ M[b]; N 3x3 pairs. */
int hb_rot_apply(const float* R, const float* M, int N, int transpose_R, float* out, void* stream);

/* ---- key-point losses and metric partial sums on the head's outputs -------------------------------
 * One hand side per call.  Replaces, for the terms that read the path's outputs:
 *   src/callbacks/loss/loss_arctic_sf.py:70-92,131-136 (hand_kp3d_loss / joints_loss of src/utils/loss_modules.py:62-73,
 *   88-125 with MSE, masked by joints_valid (B,21), gated per sample by is_j3d_loss / is_j2d_loss (B) or NULL, .mean());
 *   common/metrics.py:23-45 via src/utils/eval_modules.py:95-118,407-421 (root-relative MPJPE per hand, pixel error per
 *   joint after data_utils.unormalize_kp2d) and common/metrics.py:47-55 (MRRPE).
 * sums (HB_KP_SUMS floats, device):
 *   [0] sum of masked/gated squared root-relative 3D errors     -> loss_kp3d = sums[0] / (B*21*3)
 *   [1] sum of masked/gated squared normalised 2D errors        -> loss_kp2d = sums[1] / (B*21*2)
 *   [2] sum over valid hands of mean_j ||root-relative error||,  [3] number of valid hands      (MPJPE-RA = [2]/[3])
 *   [4] sum over valid joints of pixel L2,                       [5] number of valid joints     (pix_err  = [4]/[5])
 * partial: (B, HB_KP_SUMS) floats of scratch.  The reduction order is fixed: bit-reproducible sums that can go straight
 * into a packed all-reduce buffer.  hand_valid (B) or NULL (= all valid) only affects the metric sums. */
#define HB_KP_SUMS 8
int hb_kp_loss_fwd(const float* j3d_cam, const float* j2d_norm, const float* gt_j3d_cam, const float* gt_j2d_norm,
                   const float* joints_valid, const float* hand_valid, const float* gate_j3d, const float* gate_j2d, int B,
                   float img_res, float* partial, float* sums, void* stream);
/* Gradients of (loss_kp3d, loss_kp2d) w.r.t. j3d_cam (B,21,3) and j2d_norm (B,21,2), scaled by the upstream gradients
 * g_loss_kp3d / g_loss_kp2d (device scalars, NULL = 0); either output may be NULL. */
int hb_kp_loss_bwd(const float* j3d_cam, const float* j2d_norm, const float* gt_j3d_cam, const float* gt_j2d_norm,
                   const float* joints_valid, const float* gate_j3d, const float* gate_j2d, int B, const float* g_loss_kp3d,
                   const float* g_loss_kp2d, float* g_j3d_cam, float* g_j2d_norm, void* stream);
/* Masked vector MSE terms of compute_loss_light (src/callbacks/loss/loss_arctic_sf.py:52-69 pose/beta via mano_loss, :94-129
 * cam_t.wp (+ cam_t.wp.init) and the relative translation l - r, gated at :134-145, .mean() at :146-158; vector_loss =
 * src/utils/loss_modules.py:99-113 with MSE, return_mean=False):
 *   d[b][e] = (pred - pred_minus)[b][e] - (gt - gt_minus)[b][e]                       (pred_minus, gt_minus or NULL)
 *   *sum    = sum_b valid[b] * valid2[b] * gate[b] * ( sum_e d^2 + sum_e (pred2 - (gt - gt_minus))^2 )   (pred2 or NULL)
 *   loss    = *sum / (B * D)
 * All arrays (B, D) fp32 on the device; valid, valid2, gate (B) or NULL (= 1).  partial: B floats of scratch.  Fixed
 * reduction order (bit-reproducible).  Uses: cam_t.wp.{r,l} with pred2 = cam_t.wp.init (D = 3); transl/l with
 * pred = cam_t.wp.l, pred_minus = cam_t.wp.r, valid2 = left_valid (D = 3); pose (D = 144) and beta (D = 10). */
int hb_vec_loss_fwd(const float* pred, const float* pred_minus, const float* gt, const float* gt_minus, const float* pred2,
                    const float* valid, const float* valid2, const float* gate, int B, int D, float* partial, float* sum,
                    void* stream);
/* Gradients of loss = *sum / (B*D), scaled by the device scalar g_loss, w.r.t. pred, pred_minus, pred2 (each or NULL). */
int hb_vec_loss_bwd(const float* pred, const float* pred_minus, const float* gt, const float* gt_minus, const float* pred2,
                    const float* valid, const float* valid2, const float* gate, int B, int D, const float* g_loss,
                    float* g_pred, float* g_pred_minus, float* g_pred2, void* stream);
/* pytorch3d axis_angle_to_matrix as applied to the GT pose at loss_arctic_sf.py:48-49 (= common/rot.py:754-784 then :86-115):
 * aa (N,3) -> R (N,3,3).  GT side, no gradient. */
int hb_axis_angle_to_matrix(const float* aa, int N, float* R, void* stream);
/* MRRPE partial sums: sums[0] = sum over valid samples of ||(root_l - root_r)_pred - (root_l - root_r)_gt||, sums[1] = count;
 * roots are joint 0 of the (B,21,3) arrays; valid (B) or NULL. */
int hb_mrrpe(const float* j3d_cam_r, const float* j3d_cam_l, const float* gt_j3d_cam_r, const float* gt_j3d_cam_l,
             const float* valid, int B, float* partial, float* sums, void* stream);
/* Procrustes-aligned and root-relative point errors (PA-MPJPE / PA-MPVPE, MPJPE-RA / root-relative MPVPE): the similarity
 * fit of the HMR / ARCTIC compute_similarity_transform (src/utils/eval_modules.py:136-219, numpy SVD per sample there).
 * For hand b with p_i = pred[b,i], q_i = gt[b,i], i < N:
 *   mu_p, mu_q = means;  X_i = p_i - mu_p;  Y_i = q_i - mu_q;  var = sum |X_i|^2;  C = sum X_i Y_i^T
 *   U, S, V^T = svd(C);  Z = diag(1, 1, sign(det(U V^T)));  R = V Z U^T;  s = trace(R C) / var;  t = mu_q - s R mu_p
 *   PA = (1/N) sum_i |s R p_i + t - q_i|        RA = (1/N) sum_i |(p_i - r_p) - (q_i - r_q)|
 * A hand whose var is exactly 0 (e.g. all predicted points equal, or N = 1) is degenerate.
 * pred, gt (B,N,3), N >= 1; root_pred, root_gt (B,3) or NULL (= point 0); hand_valid (B) or NULL (0 = invalid, else valid).
 * per_hand (B,2) or NULL: [PA, RA] per hand, NaN where hand_valid == 0, PA NaN where degenerate.
 * aligned (B,N,3) or NULL: s R p + t for every hand, NaN where degenerate.   partial: (B, HB_KP_SUMS) scratch.
 * sums: [0] sum of PA over valid non-degenerate hands, [1] their count,
 *       [2] sum of RA over valid hands, [3] their count, [4] valid hands excluded as degenerate, [5..7] 0.
 * Fixed reduction order: bit-reproducible, ready for a packed all-reduce.  No gradient. */
int hb_procrustes_metrics(const float* pred, const float* gt, int B, int N, const float* root_pred,
                          const float* root_gt, const float* hand_valid, float* per_hand, float* aligned,
                          float* partial, float* sums, void* stream);
/* GT-side glue of process_data_light (src/callbacks/process/process_arctic.py:42-65), one hand side, after the no-grad MANO
 * forward of the ground-truth parameters (hb_mano_head_fwd with HB_POSE_AXIS_ANGLE, cam = K = NULL):
 *   Tr0 = mean_j (j3d_full - joints3d);  v3d_cam = vertices + Tr0;  cam_t = j3d_full[:,0] - joints3d[:,0];
 *   cam_t_wp = perspective_to_weak_perspective_torch(cam_t, (K00+K11)/2, img_res)  (common/camera.py:10-29).
 * joints3d, j3d_full (B,21,3); vertices, v3d_cam (B,778,3); K (B,3,3); cam_t, cam_t_wp (B,3).  Outputs may be NULL. */
int hb_gt_process(const float* joints3d, const float* vertices, const float* j3d_full, const float* K, int B, float img_res,
                  float* v3d_cam, float* cam_t, float* cam_t_wp, void* stream);
/* KPE features of the crop boxes (src/datasets/hands_light_dataset.py:259-279, per sample on the CPU in the reference) and
 * their sinusoidal encodings (src/models/hands_light/model.py:444-460): bbox (n,4) int32 xyxy, K (n,3,3) ->
 * center_angle (n,2), corner_angle (n,8) [corners (x0,y0),(x0,y1),(x1,y0),(x1,y1)], center_enc (n, n_freq*2*2),
 * corner_enc (n, n_freq*8*2) laid out [freq][angle][sin,cos].  Outputs may be NULL. */
int hb_kpe_features(const int32_t* bbox, const float* K, int n, int n_freq, float* center_angle, float* corner_angle,
                    float* center_enc, float* corner_enc, void* stream);

/* ---- Perspective Crop Layer ------------------------------------------------------------------
 * Replaces: src/datasets/hands_light_dataset.py:354-467 (per-sample CPU closure in the data loader).
 * n_crops crops; crop c samples image c / crops_per_img of `img` (n_crops/crops_per_img, C, R, R).
 *   bbox (n_crops,4) int32 [x0,y0,x1,y1]; K (n_crops,3,3) fp32.
 * Step 1 (lines 357-386, 425-454): homography in float64 on the device -> params (n_crops records of
 *   HB_PCL_PARAM_FLOATS floats, caller-allocated) and R_virt2orig (n_crops,3,3) or NULL. */
#define HB_PCL_PARAM_FLOATS 32
int hb_pcl_setup(const int32_t* bbox, const float* K, int n_crops, int img_res, float* params,
                 float* R_virt2orig, void* stream);
/* Same arithmetic on the host (float64), one crop: P (9), R (9), s. */
int hb_pcl_homography_host(const int32_t* bbox_host, const float* K_host, int img_res, float* P_host,
                           float* R_host, int32_t* s_host);
/* Step 2 (lines 388-423, 457-462): grid_sample(bilinear, zeros, align_corners=False) to s x s then
 *   interpolate(bilinear, align_corners=True) to R x R, fused. out (n_crops, C, R, R). */
int hb_pcl_fwd(const float* img, const float* params, int n_crops, int crops_per_img, int C, int img_res,
               float* out, void* stream);
/* Forward arithmetic mode: 0 (default) = same sample positions as the reference's fp32 chain, resize evaluated separably
 *   (differs from torch's kernel by a few ulp of the output); 1 = torch's CPU operation order reproduced exactly
 *   (bit-identical on > 99.9 % of the pixels, ~1.3x the instructions).  Environment HB_PCL_EXACT sets the initial value.
 *   Returns the previous setting.  Process-wide. */
int hb_pcl_set_exact(int on);
/* Same crop from the data loader's 8-bit image (n_crops/crops_per_img, C, R, R) uint8: x = (u/255 - mean[c]) / std[c]
 *   (torchvision Normalize as the reference applies it to the full image, src/datasets/hands_light_dataset.py:177-184)
 *   is fused into the gather, so the result equals hb_pcl_fwd on the normalised fp32 image while a quarter of the bytes
 *   cross PCIe / HBM.  mean_host, std_host: C floats on the HOST.  hb_pcl_bwd is unchanged (gradient w.r.t. the normalised
 *   image). */
int hb_pcl_fwd_u8(const uint8_t* img, const float* mean_host, const float* std_host, const float* params, int n_crops,
                  int crops_per_img, int C, int img_res, float* out, void* stream);
/* Backward w.r.t. img (the grid is data).  Domain: boxes no larger than the image (s <= img_res), which the reference
 * guarantees by clipping boxes to the image (common/data_utils.py:508); a larger crop contributes no gradient here and
 * the Python wrapper rejects it up front.  g_out (n_crops,C,R,R) -> g_img (n_crops/crops_per_img,C,R,R),
 *   written exactly once (no float atomics, deterministic).  The backward runs in chunks of images sized by the
 *   workspace given: hb_pcl_bwd_workspace_bytes() is the recommended size, any size >= one image's worth works. */
size_t hb_pcl_bwd_workspace_bytes(int n_crops, int crops_per_img, int C, int img_res);
int hb_pcl_bwd(const float* g_out, const float* params, int n_crops, int crops_per_img, int C, int img_res,
               float* g_img, void* workspace, size_t workspace_bytes, void* stream);

/* The two stages of the backward separately (profiling / benchmarking): stages bit 0 = offset scan + transposed
 * resize (g_out -> workspace), bit 1 = transposed gather (workspace -> g_img).  hb_pcl_bwd == stages 3.  Only
 * meaningful stage by stage when the whole batch fits one chunk of the workspace. */
int hb_pcl_bwd_stages(const float* g_out, const float* params, int n_crops, int crops_per_img, int C, int img_res,
                      float* g_img, void* workspace, size_t workspace_bytes, int stages, void* stream);

/* bf16 crop planes, for backbones trained under bf16 autocast: the crop is written in the dtype its consumer reads and
 * its gradient is read in the dtype the consumer's backward produces, so no cast kernel runs on either side.
 * bf16 buffers hold bfloat16 bit patterns (uint16_t), round-to-nearest-even; they need only 2-byte alignment (better
 * alignment selects the vector paths, never a different result than stated below).  The source image and g_img stay fp32.
 *   hb_pcl_fwd_bf16 / hb_pcl_fwd_u8_bf16: `out` (n_crops,C,R,R) bf16 is bit-identical to the RNE bf16 rounding of what
 *     hb_pcl_fwd / hb_pcl_fwd_u8 write for the same inputs in the same arithmetic mode (hb_pcl_set_exact), i.e.
 *     crop_fp32.to(torch.bfloat16).  All internal arithmetic is fp32; only the final store rounds.
 *   hb_pcl_bwd_bf16: `g_img` (fp32) is bit-identical to hb_pcl_bwd on the exactly widened gradient g_out.float(), for the
 *     same workspace size (hence the same chunking) and g_out buffers aligned alike in elements.  Widening is exact, so
 *     the arithmetic and its order are those of hb_pcl_bwd.  hb_pcl_bwd_workspace_bytes serves both.
 * Argument errors are those of the fp32 twins (HB_E_ARG, HB_E_WORKSPACE, HB_E_ALIGN), with messages naming the function. */
int hb_pcl_fwd_bf16(const float* img, const float* params, int n_crops, int crops_per_img, int C, int img_res,
                    uint16_t* out, void* stream);
int hb_pcl_fwd_u8_bf16(const uint8_t* img, const float* mean_host, const float* std_host, const float* params,
                       int n_crops, int crops_per_img, int C, int img_res, uint16_t* out, void* stream);
int hb_pcl_bwd_bf16(const uint16_t* g_out, const float* params, int n_crops, int crops_per_img, int C, int img_res,
                    float* g_img, void* workspace, size_t workspace_bytes, void* stream);

/* ---- soft silhouette of the hand mesh -----------------------------------------------------------
 * Replaces: src/models/hands_light/renderer.py:124-199 (pytorch3d MeshRasterizer + SoftSilhouetteShader as configured at
 *   :128-139, cameras built at :187-191, flip_transpose_canvas :201-209) — the consumer of mano.v3d.cam.{r,l} behind
 *   `use_render_seg_loss` (src/models/hands_light/model.py:413-420, src/callbacks/loss/loss_arctic_sf.py:172-183).
 * mask[b,0,r,c] = 1 - prod_k (1 - sigmoid(-d_k / sigma)) over the HB_SIL_FACES_PER_PIXEL candidate faces of smallest
 *   (clipped-barycentric) depth at the pixel centre (c+0.5, r+0.5) of the K-projected image; d_k = squared NDC distance to
 *   the face's nearest edge, negative inside; candidates = inside, or closer than blur_radius.
 * The handle owns the face table (host int32 (n_faces,3) at creation) and a vertex->corner adjacency for the backward. */
typedef struct hb_sil hb_sil;
#define HB_SIL_FACES_PER_PIXEL 10
#define HB_SIL_MAX_FACES 12000
int hb_sil_create(const int32_t* faces_host, int n_faces, int n_verts, int device, hb_sil** out);
int hb_sil_destroy(hb_sil* h);
/* Caller-owned scratch shared by forward and backward: face records (80 B/face), (alpha, depth threshold) per pixel,
 *   per-face corner gradients.  hb_sil_bwd must see the workspace exactly as hb_sil_fwd of the same inputs left it. */
size_t hb_sil_workspace_bytes(const hb_sil* h, int n_meshes, int img_res);
/* verts_cam (n_meshes, n_verts, 3) camera space; K (n_meshes,3,3) pixel intrinsics; mask (n_meshes,1,img_res,img_res).
 *   At most 65535 meshes per call (HB_E_UNSUPPORTED beyond; split the batch), img_res <= 4096. */
int hb_sil_fwd(const hb_sil* h, const float* verts_cam, const float* K, int n_meshes, int img_res, float sigma,
               float blur_radius, float* mask, void* workspace, size_t workspace_bytes, void* stream);
/* g_mask (n_meshes,1,img_res,img_res) -> g_verts (n_meshes,n_verts,3), every element written once (no atomics). */
int hb_sil_bwd(const hb_sil* h, const float* verts_cam, const float* K, const float* g_mask, int n_meshes, int img_res,
               float sigma, float blur_radius, void* workspace, size_t workspace_bytes, float* g_verts, void* stream);
/* render_loss (src/utils/loss_modules.py:146-152) gated as in loss_arctic_sf.py:177-183: loss = mean over (B, n) of
 *   |pred - gt| * valid[b] * gate[b] (valid / gate may be NULL = 1).  partial (B) scratch; fixed-order reductions. */
int hb_mask_l1_loss_fwd(const float* pred, const float* gt, const float* valid, const float* gate, int B, int n,
                        float* partial, float* loss, void* stream);
int hb_mask_l1_loss_bwd(const float* pred, const float* gt, const float* valid, const float* gate, const float* g_loss,
                        int B, int n, float* g_pred, void* stream);

/* ---- counters ---------------------------------------------------------------------------------
 * Number of kernels this library has launched since load (all threads). bench.py reports the delta. */
uint64_t hb_launch_count(void);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* HANDS_B200_H */
