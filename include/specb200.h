/* libspecb200 -- C ABI of the B200-native SPEC inference hot path.
 *
 * The reference (mkocabas/SPEC) is pure Python: there is no FFI to mirror.  This header is the
 * boundary a maintainer binds (ctypes, see INTEGRATION.md) underneath the two reference modules
 *
 *   CameraRegressorNetwork.forward   /root/reference/camcalib/model.py:72-81
 *   HMR.forward                      /root/reference/spec/models/hmr.py:82-122
 *
 * Conventions (SURVEY.md section 8b):
 *   - plain C, raw pointers + sizes + a cudaStream_t passed as void*; no torch types;
 *   - every function returns 0 on success, non-zero on failure; specb200_last_error() returns the
 *     message of the last failure on the calling thread;
 *   - "dev" pointers are device memory on the current CUDA device, "host" pointers are host memory;
 *   - forward functions only enqueue kernels on the caller's stream: no allocation, no
 *     synchronisation (CUDA-graph capturable after one warm-up call); workspaces are allocated by
 *     the caller, sized by the *_workspace_bytes() queries;
 *   - packed weights are copied at create/set time and owned by the handle until *_destroy();
 *   - one handle per (device, model); a handle is not thread-safe;
 *   - there is NO CPU path: every entry point that computes requires an sm_100 device.
 */
#ifndef SPECB200_H
#define SPECB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPECB200_ABI_VERSION 1

/* arithmetic / storage type of the backbone activations */
#define SPECB200_PREC_F32 0   /* fp32 storage, FFMA  (parity mode: north-star fp32 tolerances)  */
#define SPECB200_PREC_BF16 1  /* bf16 storage, tcgen05 tensor cores, fp32 accumulate            */
#define SPECB200_PREC_F16 2   /* fp16 storage, tcgen05 tensor cores, fp32 accumulate            */

/* trunk program op codes */
#define SPECB200_OP_CONV 1      /* dst[:, coff:coff+cout] = act(conv(src) + bias [+ src2])        */
#define SPECB200_OP_MAXPOOL 2   /* 3x3 stride 2 pad 1                                             */
#define SPECB200_OP_UPADD 3     /* dst += nearest_upsample(src, 2^shift) ; optional ReLU          */
#define SPECB200_OP_BILINEAR 4  /* dst[:, coff:] = bilinear(src -> spatial size of buffer src2)   */
#define SPECB200_OP_COPY 5      /* dst[:, coff:coff+C] = src                                      */

typedef struct specb200_op {
    int32_t type;
    int32_t src, src2, dst; /* activation buffer ids; src2 = residual / size reference, -1 if none */
    int32_t cin, cout;      /* conv: channels as stored (cin includes zero padding of the image)   */
    int32_t kh, kw, stride, pad;
    int32_t relu;
    int32_t dst_coff; /* channel offset inside dst (concat)                                  */
    int32_t shift;    /* UPADD: log2 of the upsampling factor                                */
    int32_t wslot;    /* conv: weight slot                                                   */
    int32_t pair;     /* conv 3x3/1 with cin=cout=32: run on the pixel-pair view [H][W/2][64] (see DESIGN.md) */
} specb200_op_t;

typedef struct specb200_trunk specb200_trunk_t;
typedef struct specb200_camtail specb200_camtail_t;
typedef struct specb200_hmrtail specb200_hmrtail_t;
typedef struct specb200_body specb200_body_t;

const char* specb200_last_error(void);
int specb200_abi_version(void);
/* 0 iff the current device is an sm_100 (B200) GPU; the product refuses to run anywhere else. */
int specb200_device_check(void);

/* ---- backbone trunk: replaces pare.models.backbone.{resnet,hrnet} called at
 *      /root/reference/camcalib/model.py:73 and /root/reference/spec/models/hmr.py:92 ------------ */
/* buf_channels[i] = channel stride of activation buffer i; buffer 0 is the NHWC image with 4 channels
 * (RGB + one zero channel). out_buf = buffer holding the final map. */
int specb200_trunk_create(specb200_trunk_t** out, const specb200_op_t* ops, int32_t n_ops,
                          const int32_t* buf_channels, int32_t n_bufs, int32_t n_wslots, int32_t out_buf,
                          int32_t precision);
/* w_oihw_host: [cout][cin][kh][kw] fp32 with BatchNorm already folded in; bias_host: [cout]. */
int specb200_trunk_set_conv(specb200_trunk_t* t, int32_t wslot, const float* w_oihw_host, const float* bias_host,
                            int32_t cout, int32_t cin, int32_t kh, int32_t kw);
/* images are processed `chunk` at a time so that layer-to-layer activations stay in L2 (0 = whole batch) */
int specb200_trunk_set_chunk(specb200_trunk_t* t, int32_t chunk);
int specb200_trunk_out_shape(specb200_trunk_t* t, int32_t h, int32_t w, int32_t* c_out, int32_t* h_out, int32_t* w_out);
int64_t specb200_trunk_workspace_bytes(specb200_trunk_t* t, int32_t batch, int32_t h, int32_t w);
/* images_nchw_dev: fp32 [batch][3][h][w].  pooled_out_dev: fp32, row stride pooled_ld floats, receives the
 * global average pool of the final map (AdaptiveAvgPool2d(1)+flatten, model.py:74-75).  feat_nchw_out_dev:
 * optional fp32 [batch][C][h/32][w/32] copy of the final map (the value `self.backbone(images)` returns). */
int specb200_trunk_forward(specb200_trunk_t* t, const float* images_nchw_dev, int32_t batch, int32_t h, int32_t w,
                           void* workspace_dev, int64_t workspace_bytes, float* pooled_out_dev, int32_t pooled_ld,
                           float* feat_nchw_out_dev, void* stream);
/* Diagnostic: runs ops 0..stop_op of the program and writes the destination buffer of op stop_op -- the activation as the
 * NEXT op would read it -- as fp32 NCHW [batch][*c_out][*h_out][*w_out] to act_out_dev (NULL: only report the shape).
 * Lets a test compare every intermediate tensor with the oracle's (tests/test_gpu_parity.py::test_hrnet_layerwise_lowp). */
int specb200_trunk_forward_until(specb200_trunk_t* t, const float* images_nchw_dev, int32_t batch, int32_t h, int32_t w,
                                 void* workspace_dev, int64_t workspace_bytes, int32_t stop_op, int32_t* c_out, int32_t* h_out,
                                 int32_t* w_out, float* act_out_dev, void* stream);
/* number of kernels the last forward enqueued (bench.py's gpu_launches) */
int64_t specb200_trunk_last_launches(specb200_trunk_t* t);
int32_t specb200_trunk_num_ops(specb200_trunk_t* t);
/* number of [downsample] conv1x1-conv3x3-conv1x1 bottleneck groups of the program that run as ONE fused launch
 * (64 mid channels, 256 outputs, stride 1: ResNet-50 / HRNet layer1; 16-bit modes only) */
int32_t specb200_trunk_num_fused_bottlenecks(specb200_trunk_t* t);
/* index of the first op of the fused group program op `op` belongs to, -1 if it runs on its own */
int32_t specb200_trunk_fused_group_first_op(specb200_trunk_t* t, int32_t op);
/* Diagnostic variant of specb200_trunk_forward: brackets every op with CUDA events on `stream`, SYNCHRONISES, and
 * writes per-op device milliseconds to op_ms_host[0 .. n_ops+1] (0 = image NCHW->NHWC conversion, 1..n_ops = ops in
 * program order, n_ops+1 = average pool), summed over batch chunks.  Used by bench.py for the live roofline. */
int specb200_trunk_profile(specb200_trunk_t* t, const float* images_nchw_dev, int32_t batch, int32_t h, int32_t w,
                           void* workspace_dev, int64_t workspace_bytes, float* pooled_out_dev, int32_t pooled_ld,
                           float* op_ms_host, void* stream);
void specb200_trunk_destroy(specb200_trunk_t* t);

/* ---- CamCalib tail: fc_vfov/fc_pitch/fc_roll (model.py:77-81) + convert_preds_to_angles
 *      (cam_utils.py:121-145) + f_pix (camcalib_demo.py:129) + read_cam_params (cam_params.py:24-50) */
int specb200_camtail_create(specb200_camtail_t** out, int32_t in_features, int32_t num_out);
/* append one Linear(in,out) to head `which` (0 vfov, 1 pitch, 2 roll); w_host [out][in], b_host [out] */
int specb200_camtail_add_linear(specb200_camtail_t* t, int32_t which, const float* w_host, const float* b_host,
                                int32_t out_features, int32_t in_features);
int specb200_camtail_finalize(specb200_camtail_t* t);
int64_t specb200_camtail_workspace_bytes(specb200_camtail_t* t, int32_t batch);
/* logits_out_dev: fp32 [batch][3*num_out] = [vfov | pitch | roll] logits.  workspace_dev (>= specb200_camtail_workspace_bytes)
 * is always required: hidden activations of multi-layer heads, or the split-K partial sums of the fused single-layer GEMM.
 * Calls on ONE handle must be stream-ordered with each other (the split-K arrival counters belong to the handle). */
int specb200_camtail_forward(specb200_camtail_t* t, const float* pooled_dev, int32_t pooled_ld, int32_t batch,
                             void* workspace_dev, int64_t workspace_bytes, float* logits_out_dev, void* stream);
/* logits -> angles_out_dev [batch][3] (vfov,pitch,roll radians).  If rotmat_out_dev != NULL also writes
 * cam_rotmat [batch][9], cam_intrinsics [batch][9] (K[2][2]=0) and f_pix [batch] (may be NULL) from
 * img_h_dev / img_w_dev (fp32 [batch]). */
int specb200_camcalib_decode(const float* logits_dev, int32_t logits_ld, int32_t num_out, int32_t batch,
                             const float* img_h_dev, const float* img_w_dev, float* angles_out_dev,
                             float* rotmat_out_dev, float* intrinsics_out_dev, float* fpix_out_dev, void* stream);
void specb200_camtail_destroy(specb200_camtail_t* t);

/* ---- HMR tail: HMRHead + SMPLCamHead/SMPLHead (hmr.py:94-113) ---------------------------------- */
typedef struct specb200_hmr_params {
    int32_t in_features;   /* backbone channels C                                                  */
    int32_t use_cam_feats; /* hmr.py:94-98                                                         */
    int32_t use_cam;       /* 1: SMPLCamHead (hmr.py:100-113), 0: SMPLHead (hmr.py:114-121)        */
    float focal_length, img_res;
    /* HMRHead (host, nn.Linear layout [out][in]) */
    const float *fc1_w, *fc1_b, *fc2_w, *fc2_b, *decpose_w, *decpose_b, *decshape_w, *decshape_b, *deccam_w, *deccam_b;
    const float *init_pose, *init_shape, *init_cam; /* [144], [10], [3] */
    /* SMPL constants (host, smplx layout) */
    const float* v_template;        /* [6890][3]       */
    const float* shapedirs;         /* [6890][3][10]   */
    const float* posedirs;          /* [207][20670]    */
    const float* J_regressor;       /* [24][6890]      */
    const float* lbs_weights;       /* [6890][24]      */
    const float* J_regressor_extra; /* [9][6890]       */
    const int32_t* parents;         /* [24]            */
    const int32_t* joint_map;       /* [49] into the 54 candidate joints (constants.py:29-105)      */
    const int32_t* vertex_ids;      /* [21]            */
} specb200_hmr_params_t;

/* Output pointers (device, fp32) with per-image strides in floats: lets the caller write either separate
 * contiguous tensors or one packed per-image record (the multi-GPU all-gather buffer). */
typedef struct specb200_hmr_outputs {
    float* smpl_vertices; int64_t ld_vertices; /* [6890][3] */
    float* smpl_joints3d; int64_t ld_joints3d; /* [49][3]   */
    float* smpl_joints2d; int64_t ld_joints2d; /* [49][2]   */
    float* pred_cam_t;    int64_t ld_cam_t;    /* [3]       */
    float* pred_pose;     int64_t ld_pose;     /* [24][3][3]*/
    float* pred_cam;      int64_t ld_cam;      /* [3]       */
    float* pred_shape;    int64_t ld_shape;    /* [10]      */
    float* pred_pose_6d;  int64_t ld_pose_6d;  /* [144]     */
} specb200_hmr_outputs_t;

int specb200_hmrtail_create(specb200_hmrtail_t** out, const specb200_hmr_params_t* params);
int64_t specb200_hmrtail_workspace_bytes(specb200_hmrtail_t* t, int32_t batch);
/* The head's input row buffer X lives at the start of the workspace: the trunk writes the pooled feature of
 * image b to ((float*)workspace)[b * specb200_hmrtail_x_ld() .. + C]. */
int32_t specb200_hmrtail_x_ld(specb200_hmrtail_t* t);
/* cam_rotmat/cam_intrinsics [batch][9], bbox_scale [batch], bbox_center [batch][2], img_w/img_h [batch]; all
 * fp32 device, may be NULL when use_cam == 0 and use_cam_feats == 0. */
int specb200_hmrtail_forward(specb200_hmrtail_t* t, int32_t batch, void* workspace_dev, int64_t workspace_bytes,
                             const float* cam_rotmat_dev, const float* cam_intrinsics_dev, const float* bbox_scale_dev,
                             const float* bbox_center_dev, const float* img_w_dev, const float* img_h_dev,
                             const specb200_hmr_outputs_t* outputs, void* stream);
int64_t specb200_hmrtail_last_launches(specb200_hmrtail_t* t);
void specb200_hmrtail_destroy(specb200_hmrtail_t* t);

/* ---- SMPL body model: smplx.SMPL forward from caller-given parameters, as the evaluation side calls it
 *      (/root/reference/spec/utils/compute_error.py:148-181: axis-angle pose, pose2rot=True; spec/trainer.py:249-254:
 *      rotation matrices, pose2rot=False).  Same kernels as the HMR tail's SMPL stage.  Any number of body handles (e.g.
 *      neutral, male, female) and HMR tail handles may live side by side. --------------------------------------------- */
/* host, smplx layout: v_template [6890][3], shapedirs [6890][3][10], posedirs [207][20670], J_regressor [24][6890],
 * lbs_weights [6890][24], parents [24] (the standard SMPL tree) */
int specb200_body_create(specb200_body_t** out, const float* v_template, const float* shapedirs, const float* posedirs,
                         const float* J_regressor, const float* lbs_weights, const int32_t* parents);
int64_t specb200_body_workspace_bytes(specb200_body_t* t, int32_t batch);
#define SPECB200_POSE_AXIS_ANGLE 0 /* pose_dev: [batch][72] axis-angle (global_orient first), smplx batch_rodrigues */
#define SPECB200_POSE_ROTMAT 1     /* pose_dev: [batch][24][9] rotation matrices                                   */
/* betas_dev [batch][10].  Outputs (device fp32, per-image strides in floats): verts [6890][3]; joints24 [24][3] = the posed
 * kinematic joints (smplx's joints[:, :24]).  workspace_dev: 256-byte aligned, >= specb200_body_workspace_bytes. */
int specb200_body_forward(specb200_body_t* t, int32_t batch, const float* betas_dev, const float* pose_dev, int32_t pose_kind,
                          void* workspace_dev, int64_t workspace_bytes, float* verts_dev, int64_t ld_verts, float* joints24_dev,
                          int64_t ld_joints24, void* stream);
/* joints24_out_dev [batch][24][3] = rot . (J_regressor . verts) (compute_error.py:184-187: einsum('bik,ji->bjk')); verts_dev
 * [batch][6890][3] with per-image stride ld_verts floats; rot_dev [batch][9] or NULL (no rotation). */
int specb200_body_regress_joints(specb200_body_t* t, int32_t batch, const float* verts_dev, int64_t ld_verts, const float* rot_dev,
                                 float* joints24_out_dev, void* stream);
void specb200_body_destroy(specb200_body_t* t);

/* ---- eval-side metrics on the device (SURVEY.md section 8f-1): replaces the J_regressor_h36m matmul, pelvis centring, MPJPE,
 *      numpy Procrustes (PA-MPJPE) and per-vertex error of /root/reference/spec/trainer.py:272-316 and
 *      /root/reference/spec/utils/compute_error.py:33-86 -------------------------------------------------------------- */
typedef struct specb200_eval specb200_eval_t;
/* J_regressor_h36m_host: [17][6890] fp32; joint_mapper14_host: 14 indices into the 17 joints (constants.py:109-111). */
int specb200_eval_create(specb200_eval_t** out, const float* J_regressor_h36m_host, const int32_t* joint_mapper14_host);
int64_t specb200_eval_workspace_bytes(specb200_eval_t* t, int32_t batch);
/* pred_verts_dev: [batch][6890][3] with per-image stride ld_pred floats.  Ground truth: either gt_keypoints14_dev
 * ([batch][14][3], already root-centred, trainer.py:274) or gt_verts_dev (joints regressed and centred like
 * compute_error.py:49-57).  Outputs (device, fp32): mpjpe[batch], pampjpe[batch], v2v[batch] (NULL to skip; needs
 * gt_verts; center_v2v = 1 subtracts the pelvis of each mesh first, compute_error.py:64-68), pred_keypoints14 (NULL ok). */
int specb200_eval_forward(specb200_eval_t* t, int32_t batch, const float* pred_verts_dev, int64_t ld_pred,
                          const float* gt_keypoints14_dev, const float* gt_verts_dev, int64_t ld_gt, int32_t center_v2v,
                          void* workspace_dev, int64_t workspace_bytes, float* mpjpe_dev, float* pampjpe_dev, float* v2v_dev,
                          float* pred_keypoints14_dev, void* stream);
/* joint_mapper_host: n_map (14 or 17) indices into the 17 joints: H36M_TO_J14, or H36M_TO_J17 (trainer.py:259-260). */
int specb200_eval_create_mapped(specb200_eval_t** out, const float* J_regressor_h36m_host, const int32_t* joint_mapper_host,
                                int32_t n_map);
/* specb200_eval_forward plus: pred_rot_dev / gt_rot_dev ([batch][9] or NULL) rotate each mesh before the regression, centring
 * and v2v (compute_error.py:164,186: the camera-frame metrics); gt_rot_dev also rotates given keypoints; per-joint
 * distances before / after the Procrustes alignment, mpjpe_pj_dev / pampjpe_pj_dev [batch][n_map] (NULL to skip);
 * gt keypoints and pred_keypoints are [batch][n_map][3]; n_map must equal the handle's mapper length. */
int specb200_eval_forward_ex(specb200_eval_t* t, int32_t batch, const float* pred_verts_dev, int64_t ld_pred, const float* pred_rot_dev,
                             const float* gt_keypoints_dev, const float* gt_verts_dev, int64_t ld_gt, const float* gt_rot_dev,
                             int32_t center_v2v, void* workspace_dev, int64_t workspace_bytes, float* mpjpe_dev, float* pampjpe_dev,
                             float* v2v_dev, float* pred_keypoints_dev, float* mpjpe_pj_dev, float* pampjpe_pj_dev, int32_t n_map,
                             void* stream);
/* Stateless: MPJPE / PA-MPJPE of already-regressed joints pred_dev, gt_dev [batch][n][3] (n = 14, 17 or 24), e.g. the 24 SMPL
 * joints of specb200_body_*.  rot_pred_dev / rot_gt_dev ([batch][9] or NULL) rotate each side first; center != 0 subtracts
 * joint 0 on both sides (compute_error.py:33-49 eval_j_24).  Per-joint outputs [batch][n] may be NULL. */
int specb200_eval_joint_errors(int32_t batch, int32_t n, const float* pred_dev, const float* gt_dev, const float* rot_pred_dev,
                               const float* rot_gt_dev, int32_t center, float* mpjpe_dev, float* pampjpe_dev, float* mpjpe_pj_dev,
                               float* pampjpe_pj_dev, void* stream);
void specb200_eval_destroy(specb200_eval_t* t);

/* ---- input side on the device (SURVEY.md section 8f-2): uint8 frame -> network inputs, BIT-EXACT with the
 *      libraries the reference calls (cv2.warpAffine 8-bit fixed-point path; Pillow ImagingResample 8-bit path;
 *      torchvision ToTensor + Normalize in float32) ------------------------------------------------------------- */
typedef struct specb200_preproc specb200_preproc_t;
/* mean3/std3: host float[3] (spec/constants.py:20-21).  Builds the 3x256 float32 ToTensor+Normalize table. */
int specb200_preproc_create(specb200_preproc_t** out, const float* mean3, const float* std3);
/* Person crops = get_single_image_crop_demo(img, bbox, kp_2d=None, scale, crop_size) of pare.utils.vibe_image_utils as
 * called at /root/reference/spec/tester.py:118-125 (gen_trans_from_patch_cv -> cv2.getAffineTransform ->
 * cv2.warpAffine(INTER_LINEAR, BORDER_CONSTANT 0) -> ToTensor -> Normalize), all n detections of a frame in one launch
 * per 32 boxes.  image_dev: uint8 [height][width][3] with row pitch row_stride_bytes (bgr != 0: channels are B,G,R as
 * cv2.imread returns them and are swapped like the cv2.cvtColor(BGR2RGB) of tester.py:105).  boxes_host: HOST
 * double [n][4] = (c_x, c_y, w, h) in pixels.  out_dev: float32 [n][3][crop][crop]; raw_dev: uint8 [n][crop][crop][3]
 * RGB (the "raw_img" return value) or NULL. */
int specb200_preproc_crop(specb200_preproc_t* t, const uint8_t* image_dev, int32_t height, int32_t width,
                          int64_t row_stride_bytes, int32_t bgr, const double* boxes_host, int32_t n, double scale,
                          int32_t crop_size, float* out_dev, uint8_t* raw_dev, void* stream);
/* Host only: the forward 2x3 matrices ("trans", what kp_2d is mapped with) and/or the dst->src matrices of the boxes;
 * either output may be NULL.  [n][6] row-major doubles. */
int specb200_preproc_crop_transforms(const double* boxes_host, int32_t n, double scale, int32_t crop_size,
                                     double* trans_host, double* inv_host);
/* CamCalib input = transforms.Compose([Resize(min_size), ToTensor(), Normalize(...)]) on a PIL image,
 * /root/reference/camcalib/pano_dataset.py:156-162.  resized_shape is torchvision's rule (short side -> min_size). */
int specb200_preproc_resized_shape(int32_t height, int32_t width, int32_t min_size, int32_t* out_h, int32_t* out_w);
int64_t specb200_preproc_resize_workspace_bytes(int32_t height, int32_t width, int32_t out_h, int32_t out_w);
/* out_dev: float32 [3][out_h][out_w]; raw_dev: uint8 [out_h][out_w][3] RGB or NULL.  The first call for a new
 * (size -> size) pair uploads its coefficient table with a blocking copy (do it outside stream capture). */
int specb200_preproc_resize(specb200_preproc_t* t, const uint8_t* image_dev, int32_t height, int32_t width,
                            int64_t row_stride_bytes, int32_t bgr, int32_t out_h, int32_t out_w, void* workspace_dev,
                            int64_t workspace_bytes, float* out_dev, uint8_t* raw_dev, void* stream);
void specb200_preproc_destroy(specb200_preproc_t* t);

/* ---- multi-GPU: all-gather of the packed per-image output records over NVLink peer memory (SURVEY.md section 8b, 8e).
 *      The reference has no collective (one process, /root/reference/spec/tester.py:143-167); BASELINE.json's multi-GPU
 *      configs shard the batch over one process per GPU and gather the records.  Each rank owns a receive region
 *      (slots x world x block_bytes) that every peer maps through CUDA IPC; a gather is a PUT of this rank's block into all
 *      peers' regions followed by a sequence-number flag exchange, all enqueued on the caller's stream (no host sync). ---- */
typedef struct specb200_gather specb200_gather_t;
#define SPECB200_IPC_HANDLE_BYTES 64
#define SPECB200_GATHER_COPY_ENGINE 0 /* world-1 peer cudaMemcpyAsync (copy engines; SM-free) + 1-CTA signal / wait kernels */
#define SPECB200_GATHER_PUSH_KERNEL 1 /* one kernel stores the block to every peer (16-byte stores) and signals           */
/* Allocates this rank's receive region on the current device and writes its CUDA IPC handle (64 bytes) to
 * ipc_handle_out_host.  block_bytes (multiple of 16) = bytes each rank contributes per gather. */
int specb200_gather_create(specb200_gather_t** out, int32_t rank, int32_t world, int64_t block_bytes, int32_t slots,
                           uint8_t* ipc_handle_out_host);
/* all_handles_host: world x 64 bytes, the handles of all ranks in rank order (exchanged by the caller out of band --
 * spec_b200 uses torch.distributed.all_gather_object); maps every peer's region (needs NVLink / PCIe peer access). */
int specb200_gather_connect(specb200_gather_t* g, const uint8_t* all_handles_host);
/* device pointer of receive slot `slot`: world x block_bytes, rank-major (= image order under a contiguous batch split) */
void* specb200_gather_recv_ptr(specb200_gather_t* g, int32_t slot);
/* Enqueues on `stream`: src_dev (block_bytes) -> slot `slot` of EVERY rank's region at this rank's offset; publishes `seq`
 * (must grow by one per use of a slot) to all peers; waits until all peers published it.  When the stream reaches the end
 * of this call's work, recv_ptr(slot) holds the blocks of all ranks.  A slot may be reused once every rank has enqueued
 * its consumers of the previous content before its own next call (three slots make that automatic for a pipelined loop). */
int specb200_allgather_outputs(specb200_gather_t* g, const void* src_dev, int32_t slot, uint32_t seq, int32_t mode, void* stream);
int specb200_gather_set_push_ctas(specb200_gather_t* g, int32_t ctas);
void specb200_gather_destroy(specb200_gather_t* g);

/* ---- standalone ops (unit tests / building blocks) -------------------------------------------- */
/* out[m][n] = sum_k a[m][k] w[n][k] + bias[n] ; fp32 */
int specb200_linear_f32(const float* a_dev, int32_t lda, const float* w_dev, int32_t ldw, const float* bias_dev,
                        float* out_dev, int32_t ldo, int32_t m, int32_t n, int32_t k, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPECB200_H */
