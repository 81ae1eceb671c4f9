/* libdanet_b200.so -- C ABI of the B200-native DaNet inference hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  Every entry point replaces one piece of the
 * reference's Python/ATen path (file:line of the reference cited per function).  Conventions:
 *   - all data pointers are DEVICE pointers (fp32 / int32 / uint8, contiguous, caller-owned)
 *     unless the name says `host`; no torch types cross this boundary;
 *   - every call takes a `cudaStream_t` (passed as void*) and is asynchronous on it;
 *   - return value: 0 = ok, <0 = error; `danet_last_error()` returns a thread-local message;
 *   - no allocation inside hot calls: handles own their constants, callers own activations and
 *     workspaces (sizes from the `*_workspace_bytes` helpers);
 *   - handles are not thread-safe: one handle per stream / rank.
 *
 * Activations of the network half are fp32 NHWC ("pixels x channels"); tensors that the
 * reference returns to its callers in NCHW are written in NCHW by the kernel that produces them.
 */
#ifndef DANET_B200_H
#define DANET_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef void* danet_stream_t;                 /* cudaStream_t */
typedef struct danet_smpl*   danet_smpl_t;
typedef struct danet_raster* danet_raster_t;

const char* danet_last_error(void);
int danet_version(void);                      /* ABI version, bumped on any signature change */
int danet_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * SMPL layer.  Replaces models/smpl.py:15-46 (SMPL.__init__/forward) and the third-party
 * smplx.lbs it calls (lbs, batch_rodrigues, batch_rigid_transform, vertices2joints,
 * VertexJointSelector), plus utils/geometry.py:9-61 (batch_rodrigues, rot6d_to_rotmat) as
 * pose front-ends and eval.py:78,186,202 (J_regressor_h36m matmul).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t num_verts;                 /* 6890 */
    int32_t num_joints;                /* 24 */
    int32_t num_betas;                 /* 10 */
    const float* v_template;           /* HOST [V,3] */
    const float* shapedirs;            /* HOST [V,3,num_betas] */
    const float* posedirs;             /* HOST [(J-1)*9, V*3]  (smplx layout) */
    const float* J_regressor;          /* HOST [J,V] */
    const float* lbs_weights;          /* HOST [V,J] */
    const int32_t* parents;            /* HOST [J], parents[0] = -1 */
    int32_t num_selected;              /* 21 vertices appended by VertexJointSelector */
    const int32_t* selected_verts;     /* HOST [num_selected] */
    int32_t num_extra;                 /* 9 rows of J_regressor_extra (models/smpl.py:21-22) */
    const float* J_regressor_extra;    /* HOST [num_extra,V] */
    int32_t num_h36m;                  /* 17 rows of J_regressor_h36m (eval.py:78) or 0 */
    const float* J_regressor_h36m;     /* HOST [num_h36m,V] or NULL */
    int32_t num_out_joints;            /* 49 */
    const int32_t* joint_map;          /* HOST [num_out_joints] into cat(J posed, selected, extra) */
} danet_smpl_desc;

enum { DANET_POSE_ROTMAT = 0,          /* pose [B,24,3,3]   (pose2rot=False)                       */
       DANET_POSE_AXIS_ANGLE = 1,      /* pose [B,24,3]     smplx Rodrigues (pose2rot=True)         */
       DANET_POSE_ROT6D = 2 };         /* pose [B,24,6]     utils/geometry.py:47-61                 */

int danet_smpl_create(const danet_smpl_desc* desc, danet_smpl_t* out);
int danet_smpl_destroy(danet_smpl_t h);
/* bytes of scratch `danet_smpl_forward` needs for a batch of B bodies */
int64_t danet_smpl_workspace_bytes(danet_smpl_t h, int32_t B);
/* outputs may be NULL to skip: verts [B,V,3]; joints [B,num_out_joints,3];
 * smpl_joints [B,J,3]; joints_h36m [B,num_h36m,3]; rotmats [B,J,3,3].
 * `bodies_per_cta` 0 = auto (tuning knob: 1,2,4,8,16). */
int danet_smpl_forward(danet_smpl_t h, int32_t B, const float* betas, const float* pose,
                       int32_t pose_kind, float* verts, float* joints, float* smpl_joints,
                       float* joints_h36m, float* rotmats, void* workspace,
                       int32_t bodies_per_cta, danet_stream_t stream);

/* Backward of the SMPL layer -- the first piece of the training step (train/trainer.py:148-215 back-propagates
 * vertex / joint losses through models/smpl.py:27-46 into the regressed betas and rotation matrices,
 * models/danet/smpl_regressor.py:131-221).  rotmats [B,24,3,3] are the matrices the forward consumed (pose2rot=False,
 * treated as free 3x3 inputs); grad_verts [B,V,3]; grad_smpl_joints [B,24,3] or NULL (gradients w.r.t. the regressed
 * joints are folded into grad_verts by the caller: J_regressor^T g); outputs grad_betas [B,num_betas],
 * grad_rotmats [B,24,3,3].  Recomputes the forward intermediates; fp32. */
int64_t danet_smpl_backward_workspace_bytes(danet_smpl_t h, int32_t B);
int danet_smpl_backward(danet_smpl_t h, int32_t B, const float* betas, const float* rotmats,
                        const float* grad_verts, const float* grad_smpl_joints, float* grad_betas,
                        float* grad_rotmats, void* workspace, danet_stream_t stream);

/* utils/geometry.py:47-61 rot6d_to_rotmat: x [n,6] (viewed [n,3,2]) -> R [n,3,3] */
int danet_rot6d_to_rotmat(int32_t n, const float* x, float* R, danet_stream_t stream);
/* utils/geometry.py:9-45 batch_rodrigues (quaternion route): aa [n,3] -> R [n,3,3];
 * flavor 1 = smplx.lbs.batch_rodrigues (matrix exponential form) */
int danet_batch_rodrigues(int32_t n, const float* aa, float* R, int32_t flavor, danet_stream_t stream);
/* utils/geometry.py:63-91 perspective_projection: points [B,N,3], rotation [B,3,3],
 * translation [B,3], focal [B] , center [B,2] -> out [B,N,2] */
int danet_perspective_projection(int32_t B, int32_t N, const float* points, const float* rotation,
                                 const float* translation, const float* focal, const float* center,
                                 float* out, danet_stream_t stream);
/* eval.py:202-212: pred_j17 [B,17,3] (J_regressor_h36m joints), gt_j14 [B,14,3] (already
 * pelvis-centred + H36M_TO_J14-selected) -> mpjpe [B] */
int danet_mpjpe_h36m(int32_t B, const float* pred_j17, const float* gt_j14, float* mpjpe,
                     danet_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Dense IUV losses of the training step (SURVEY section 8f-2), forward and backward in one pass.
 * Replaces models/danet/iuv_estimator.py:304-341 (IUV_Estimator.body_uv_losses) and the autograd
 * graph torch records for it.  Predictions u/v/index [N,C,HW] and targets U/V/I [N,C,HW] (fp32,
 * channel stride HW, image strides `pred_stride` / `map_stride` in elements, 0 = dense C*HW), optional
 * annotation logits / targets [N,Cann,HW] (dense, both NULL to skip), optional has_iuv [N] (uint8, NULL =
 * every image).  losses[4] = { point_weight/batch_size * sum smooth_l1(u - U | I > 0), the same for v,
 * mean cross-entropy(index, argmax I), mean cross-entropy(ann, argmax Ann) } over the images with
 * has_iuv (all zero when none has).  grad_* (NULL to skip; laid out like the predictions) receive
 * d losses[k] / d prediction.  The 24 per-part calls of iuv_estimator.py:232-255 are one call over the
 * (batch, part)-flattened axis: N = 24 B, batch_size = 24 B, strides 3*7*HW, has_iuv repeated per part.
 * Deterministic (fixed summation order). */
int64_t danet_body_uv_losses_workspace_bytes(int32_t N, int32_t HW);
int danet_body_uv_losses(int32_t N, int32_t C, int32_t Cann, int32_t HW, int64_t pred_stride, int64_t map_stride,
                         const float* u_pred, const float* v_pred, const float* index_pred, const float* ann_pred,
                         const float* Umap, const float* Vmap, const float* Imap, const float* Annmap,
                         const uint8_t* has_iuv, float batch_size, float point_weight, float* losses,
                         float* grad_u, float* grad_v, float* grad_index, float* grad_ann, void* workspace,
                         danet_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * DensePose-point losses of the training step (SURVEY section 8f-2), forward and backward in one
 * pass.  Replaces models/danet/iuv_estimator.py:343-419 (IUV_Estimator.dp_uvia_losses), the has_dp
 * selection of iuv_estimator.py:106-121 and the autograd graph torch records for them.
 * Predictions u/v/index [B,C,S,S], ann [B,Cann,S,S]; points X/Y/I [B,P] (pixel coordinates, part
 * label); U/V/point_weights [B,C*P] (channel c of point p at c*P + p); ann_labels [B,S*S] (pixel
 * h*S + w); labels are truncated like .to(int64); all fp32.  has_dp [B] uint8 or NULL (every sample).
 * The maps are sampled bilinearly (zero padding) at grid (X - S/2) * 2/S, (Y - S/2) * 2/S with
 * grid_sample's align_corners = `align_corners`.  losses[4] = { point_weight * sum w smooth_l1(w (u^ - U)),
 * the same for v, part_weight * mean cross-entropy(index^, I) over the selected samples' B_sel*P points,
 * index_weight * mean cross-entropy(ann, ann_labels) over their B_sel*S*S pixels } (all zero when no
 * sample is selected; a label outside [0, C) / [0, Cann) makes its loss NaN).  grad_* (NULL to skip)
 * receive d losses[k] / d prediction.  Deterministic (fixed summation order, no float atomics). */
int64_t danet_dp_uvia_losses_workspace_bytes(int32_t B, int32_t C, int32_t S, int32_t P);
int danet_dp_uvia_losses(int32_t B, int32_t C, int32_t Cann, int32_t S, int32_t P, const float* u_pred,
                         const float* v_pred, const float* index_pred, const float* ann_pred, const float* X_points,
                         const float* Y_points, const float* I_points, const float* U_points, const float* V_points,
                         const float* point_weights, const float* ann_labels, const uint8_t* has_dp,
                         int32_t align_corners, float index_weight, float part_weight, float point_weight,
                         float* losses, float* grad_u, float* grad_v, float* grad_index, float* grad_ann,
                         void* workspace, danet_stream_t stream);

/* STN key-point loss (loss_roi) through the soft-argmax.  Replaces iuv_estimator.py:137-140 (centres:
 * softmax_integral_tensor of 10 * map, utils/keypoints.py:334-394, / (S/2) - 1) and :159-171.  hm
 * [B,J,S,S], kps_gt [B,J,3] (x, y in [-1, 1], weight).  loss[1] = weight * sum over joints with
 * w != 0 of w * sum_xy smooth_l1(c - gt) / B; centers [B,J,2] (x from columns, y from rows);
 * grad_hm (NULL to skip) = d loss / d hm.  Deterministic. */
int64_t danet_stn_kps_losses_workspace_bytes(int32_t B, int32_t J);
int danet_stn_kps_losses(int32_t B, int32_t J, int32_t S, const float* hm, const float* kps_gt, float weight,
                         float* loss, float* centers, float* grad_hm, void* workspace, danet_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * IUV rasteriser.  Replaces utils/renderer.py:207-298 (IUV_Renderer) and the third-party
 * neural_renderer forward pass it calls; optionally fuses utils/iuvmap.py:103-151 (iuv_img2map).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t num_smpl_verts;            /* 6890 */
    int32_t num_mesh_verts;            /* 7829 */
    const int32_t* vert_mapping;       /* HOST [num_mesh_verts], 0-based into SMPL vertices */
    int32_t num_faces;                 /* 13774 */
    const int32_t* faces;              /* HOST [num_faces,3] into mesh verts */
    const float* textures;             /* HOST [num_faces,3]  (I/24, mean U, mean V) */
    int32_t orig_size;                 /* 224 */
    int32_t out_size;                  /* 56 */
    float focal_length;                /* 5000 (already scaled by orig_size/224 like renderer.py:222-227) */
    float near_plane, far_plane;       /* 0.1, 100 */
    int32_t tex_mode;                  /* 0 = face texture exactly; 1 = neural_renderer texture_size==1 blend */
} danet_raster_desc;

int danet_raster_create(const danet_raster_desc* desc, danet_raster_t* out);
int danet_raster_destroy(danet_raster_t h);
int64_t danet_raster_workspace_bytes(danet_raster_t h, int32_t B);
/* verts [B,V,3], cam [B,3] (s,tx,ty) -> img [B,3,S,S].  Optional (NULL to skip):
 * face_idx [B,S,S] int32 (-1 background), maps_u/v/i [B,25,S,S], maps_ann [B,15,S,S]. */
int danet_raster_iuv(danet_raster_t h, int32_t B, const float* verts, const float* cam, float* img,
                     int32_t* face_idx, float* maps_u, float* maps_v, float* maps_i, float* maps_ann,
                     void* workspace, danet_stream_t stream);
/* utils/iuvmap.py:103-151 on an arbitrary IUV image [B,3,S,S] */
int danet_iuv_img2map(int32_t B, int32_t S, const float* img, float* maps_u, float* maps_v,
                      float* maps_i, float* maps_ann, danet_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Network half (models/danet/, models/module/).  NHWC activations as danet_act views (fp32 and/or
 * split-fp16 planes): every glue kernel below reads the fp32 view when present, else hi(+lo), and writes
 * every view that is present.
 * ------------------------------------------------------------------------------------------ */
enum { DANET_CONV_SIMT = 0,            /* fp32 FMA implicit GEMM (independent fp32 check path)      */
       DANET_CONV_TC = 1 };            /* tcgen05 tensor-core implicit GEMM (danet_conv_tc_group)   */

typedef struct {
    int32_t N, H, W, Cin;              /* input  [N,H,W,Cin]                                      */
    int32_t Cout, ksize, stride, pad;  /* output [N,Ho,Wo,Cout], Ho = (H+2*pad-ksize)/stride+1     */
    int32_t wsets;                     /* weight sets: image n uses set n % wsets (grouped convs of
                                          res_module.py:335-342,500-535 become wsets=24 over the
                                          (batch,part)-flattened image axis)                       */
    int32_t relu;                      /* apply ReLU last                                         */
    int32_t flags;                     /* tensor-core path: DANET_CONV_EXACT                      */
} danet_conv_desc;
/* tensor-core path, exact mode: three MMAs per K step on split-fp16 operands (hi*hi + hi*lo + lo*hi,
 * fp32 accumulation): fp32-grade results (the reference computes these layers in fp32).  Without the flag
 * only hi*hi is issued (fp16-operand precision, ~1e-3 on the network output). */
#define DANET_CONV_EXACT 4

/* An activation tensor of the network half, NHWC.  Any subset of the three views may be present:
 *   f32      fp32 [N,H,W,C]
 *   hi / lo  SPLIT-FP16 planes, each IEEE fp16 [N,H,W,C], C % 8 == 0, 16-byte aligned:
 *            value = float(hi) + float(lo), hi = rn(value), lo = rn(value - hi)  (22 significant bits);
 *            lo == NULL means "hi only" (fast mode).
 * Tensor-core convolutions read hi/lo through TMA tensor maps and write any of the views. */
typedef struct { float* f32; void* hi; void* lo; } danet_act;

/* Weight packing for the SIMT path: w [wsets][ksize*ksize*Cin][Cout] (tap-major, then cin),
 * bias [wsets][Cout] (BN folded by the caller).  residual (or NULL) has the output's shape and is
 * added before the ReLU (res_module.py:40-56,77-97).  fp32 tensors only. */
int danet_conv2d(const danet_conv_desc* d, int32_t algo, const void* x, const float* w,
                 const float* bias, const float* residual, void* y, danet_stream_t stream);

/* Tensor-core path.  One launch runs up to 6 independent convolutions (e.g. the parallel branches of an
 * HRNet stage, hr_module.py:165-166) over one persistent grid.  w_packed comes from danet_conv_tc_pack with
 * the SAME descriptor (flags included).  x needs hi (+ lo in exact mode); res: f32, or hi(+lo), or all NULL;
 * y: f32 and/or hi(+lo).  Cin % 8 == 0, Cout % 8 == 0 (pad channels carry zero weights / zero data). */
typedef struct {
    danet_conv_desc d;
    danet_act x, res, y;
    const void* w_packed;
    const float* bias;                 /* [wsets][Cout] or NULL */
} danet_conv_problem;
int danet_conv_tc_group(int32_t n, const danet_conv_problem* problems, danet_stream_t stream);
/* The launch configuration a group of n problems would get: sub-tiles per pipeline step (1 or 2) of every problem and
 * the depth of the shared activation / weight rings (stages[0], stages[1]).  The rings are sized for the largest
 * member, so a host may use this to keep a dominant problem from losing its sub-tile pair to a small companion. */
int danet_conv_tc_config(int32_t n, const danet_conv_desc* descs, int32_t* subtiles, int32_t* stages);
/* bytes / packing helper: converts the SIMT layout above into the swizzled shared-memory image blocks of
 * split-fp16 weights the tcgen05 kernel bulk-copies (device -> device, once at load). */
int64_t danet_conv_tc_packed_bytes(const danet_conv_desc* d);
int danet_conv_tc_pack(const danet_conv_desc* d, const float* w_simt, void* w_packed, danet_stream_t stream);
int danet_conv_tc_supported(const danet_conv_desc* d);
/* bring-up instrumentation: 16 x int64 device buffer receiving per-role cycle counters of CTA 0 of
 * every following tensor-core launch (NULL = off; layout in csrc/conv_tc.cu) */
int danet_conv_tc_set_profile_buffer(void* dev_buf);
/* fp32 -> split-fp16 planes (lo may be NULL) and back (lo may be NULL); n elements */
int danet_act_split(int64_t n, const float* x, void* hi, void* lo, danet_stream_t stream);
int danet_act_merge(int64_t n, const void* hi, const void* lo, float* y, danet_stream_t stream);

/* input boundary: x NCHW [N,C,HW] -> y NHWC [N,HW,Cp] with Cp >= C zero-padded channels
 * (images arrive NCHW: demo.py:106, eval.py:147) */
int danet_nchw_to_nhwc(int32_t N, int32_t C, int32_t HW, int32_t Cp, const float* x, const danet_act* y,
                       danet_stream_t stream);

/* hr_module.py:161-179 fuse: y = relu(sum_j up_{f_j}(t_j)); t_j [N,H/f_j,W/f_j,C] nearest-upsampled
 * by f_j in {1,2,4,8}; nterms <= 4; summed in argument order */
int danet_fuse_sum(int32_t N, int32_t H, int32_t W, int32_t C, int32_t nterms,
                   const danet_act* terms /*[nterms]*/, const int32_t* factors, int32_t relu, const danet_act* y,
                   danet_stream_t stream);
/* nn.MaxPool2d(3,2,1) (res_module.py:409) NHWC */
int danet_maxpool3x3s2(int32_t N, int32_t H, int32_t W, int32_t C, const danet_act* x, const danet_act* y,
                       danet_stream_t stream);
/* nn.AdaptiveAvgPool2d(1) NHWC [N,H,W,C] -> [N,C] */
int danet_global_avgpool(int32_t N, int32_t HW, int32_t C, const danet_act* x, float* y, danet_stream_t stream);
/* y[n,o] = sum_i x[n,i] w[o,i] + b[o] (+ add[o])  (SmplResNet.final_layer + mean_cam_shape) */
int danet_linear(int32_t N, int32_t In, int32_t Out, const float* x, const float* w, const float* b,
                 const float* add, float* y, danet_stream_t stream);

/* utils/iuvmap.py:6-38 iuvmap_clean on the global prediction heads.
 * heads [B,HW,Chead] NHWC with channel blocks (U 25 | V 25 | Index 25 | Ann 15) at offsets
 * off_u/off_v/off_i/off_a.  Writes body_iuv [B,HW,Cbody>=75] NHWC (cat[U,V,I] of danet.py:85,
 * pad channels zeroed) and the
 * uint8 argmax map [B,HW]; optional NCHW outputs u/v/i [B,25,HW], ann [B,15,HW] (danet.py:81). */
int danet_iuv_clean_global(int32_t B, int32_t HW, int32_t Chead, int32_t off_u, int32_t off_v,
                           int32_t off_i, int32_t off_a, int32_t Cbody, const float* heads,
                           const danet_act* body_iuv, uint8_t* index_argmax, float* u_nchw, float* v_nchw,
                           float* i_nchw, float* ann_nchw, danet_stream_t stream);
/* utils/iuvmap.py:6-38 with the reference's own signature: NCHW maps U,V,Index [B,C,HW] and
 * optional AnnIndex [B,Ca,HW] (NULL to skip) -> cleaned maps of the same shapes */
int danet_iuvmap_clean_nchw(int32_t B, int32_t C, int32_t Ca, int32_t HW, const float* U, const float* V,
                            const float* I, const float* A, float* oU, float* oV, float* oI, float* oA,
                            danet_stream_t stream);
/* danet.py:93-98: 24 per-part iuvmap_clean calls.  x [N,HW,Cx] NHWC with (U 7|V 7|I 7) in the
 * first 21 channels (N = batch*24) -> y [N,HW,Cy>=21] cleaned (pad channels zeroed); optional raw
 * copy in the reference's
 * layout part_iuv_pred [N,21,HW] (iuv_estimator.py:208-211). */
int danet_iuv_clean_parts(int32_t N, int32_t HW, int32_t Cx, int32_t Cy, const float* x, const danet_act* y,
                          float* raw_nchw, danet_stream_t stream);
/* iuv_estimator.py:137-140,176-184,262-301: soft-argmax centres of 10*hm, part visibility,
 * affine thetas.  hm [B,HW,Chm] (24 heatmap channels first), index_argmax [B,HW] ->
 * centers [B,24,2] (x,y in [-1,1]), theta [B,24,3] = (scale, cx, cy).
 * smpl2dp/parents/children tables are the reference's (utils/smpl_utlis.py) and compiled in.
 * align_corners: 0 = torch>=1.3 default semantics, 1 = torch 1.1 semantics. */
int danet_stn_params(int32_t B, int32_t S, int32_t Chm, const float* hm, const uint8_t* index_argmax,
                     const float* learned_ratio, const float* learned_offset, float vis_thresh,
                     int32_t align_corners, float* centers, float* theta, danet_stream_t stream);
/* iuv_estimator.py:193-204: 24x affine_grid + grid_sample (bilinear, zeros) of xd [B,S,S,C]
 * -> crops [B*24,S,S,C] (image index b*24+part) */
int danet_stn_sample(int32_t B, int32_t S, int32_t C, const danet_act* xd, const float* theta,
                     int32_t align_corners, const danet_act* crops, danet_stream_t stream);

/* smpl_regressor.py:858-895 + GCN.py:29-92 + geometry.py:47-61: r2p_gcn -> refine_gcn(+res) ->
 * p2r_gcn -> grouped 1x1 pose head + mean_pose -> rot6d_to_rotmat; also concatenates
 * global_para (cam,shape) -> para [B,229].  All matrices are device pointers prepared once:
 *   adj [3][24*24]   (r2p_A, normalised refine adjacency, p2r_A)
 *   per GCN layer l (5 layers: r2p, refine0..2, p2r): W_l [in,out], b_l [out], bn scale/shift [24]
 *   head_w [24][6][128], head_b [24*6], mean_pose [144]. */
typedef struct {
    const float* adj;
    const float* W[5]; const float* b[5]; const float* bn_scale[5]; const float* bn_shift[5];
    int32_t dim_in[5]; int32_t dim_out[5];
    const float* head_w; const float* head_b; const float* mean_pose;
} danet_gcn_params;
int danet_gcn_pose_head(int32_t B, const danet_gcn_params* p, const float* rot_feats /*[B,24,128]*/,
                        const float* global_para /*[B,13]*/, float* para /*[B,229]*/,
                        danet_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Whole-network entry (csrc/net.cu).  Replaces the network half of DaNet.infer_net
 * (models/danet/danet.py:78-98: img2iuv -> iuvmap_clean -> iuv2smpl, up to `para`) for hosts without Python.
 * A "network program" is what danet_b200.plan.Plan.export() writes for ONE batch size: the launch steps (each one of
 * the entries above, with its arguments), the activation buffer table and the BN-folded, packed weights.  Loading
 * allocates everything on the CURRENT device; infer replays the steps (optionally as one CUDA graph, captured on the
 * first call).  A danet_net_t owns its buffers: one infer at a time per handle (load one handle per host thread / stream
 * that runs concurrently).  Outputs stay in the program's buffers until the next infer:
 *   "para" [B,229] f32 (cam 3 | shape 10 | 24 rotation matrices, danet.py:118), "centers" [B,24,2] (stn_kps_pred),
 *   "theta", "global_para", "rot_feats", "heads", "hm", "body_iuv", "amax" (u8 [B,S,S]) and, when the plan kept the
 *   visualisation maps, "vis_u" / "vis_v" / "vis_i" [B,25,S,S], "vis_a" [B,15,S,S], "part_iuv_raw" [B*24,21,S,S].
 * ------------------------------------------------------------------------------------------ */
typedef struct danet_net* danet_net_t;
#define DANET_NET_GRAPH 1              /* flags: replay as a CUDA graph (a NULL stream is served by an internal blocking stream) */
int danet_net_load(const void* program, uint64_t bytes, danet_net_t* out);         /* program: HOST memory */
int danet_net_load_file(const char* path, danet_net_t* out);
int danet_net_destroy(danet_net_t net);
/* batch size, input [C,H,W], number of outputs, number of launch steps (any pointer may be NULL) */
int danet_net_info(danet_net_t net, int32_t* batch, int32_t* chw, int32_t* n_outputs, int32_t* n_steps);
const char* danet_net_output_name(danet_net_t net, int32_t index);                  /* NULL past the end */
/* device pointer / byte size / dims[4] / element size of a named output */
int danet_net_output(danet_net_t net, const char* name, void** dev_ptr, uint64_t* bytes, int32_t* dims,
                     int32_t* elem_bytes);
/* images: fp32 NCHW [B,C,H,W], device (or pinned host) memory; asynchronous on `stream` */
int danet_net_infer(danet_net_t net, const float* images, int32_t flags, danet_stream_t stream);
/* convenience for hosts that do not touch CUDA: pageable host images -> H2D -> steps -> synchronise (own stream) */
int danet_net_infer_host(danet_net_t net, const float* images_host, int32_t flags);
/* synchronous device -> host copy of a named output; `bytes` must equal the output's size */
int danet_net_read_output(danet_net_t net, const char* name, void* host_dst, uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif
