// Declarations of the fp32 tail kernels (tail.cu).
#pragma once
#include <cuda_runtime.h>

namespace sb {

constexpr int SMPL_NV = 6890;        // SMPL vertices
constexpr int SMPL_VP = 6912;        // padded to 108 tiles of 64
constexpr int SMPL_NVT = 108;        // vertex tiles
constexpr int PF_LD = 208;           // pose feature (207) padded to a multiple of 16
constexpr int BODY_XLD = 160;        // body-model row buffer: betas at column 144 (the HMR state layout with C = 0)

bool tail_upload_tables(const int* joint_map49, const int* vertex_ids21);

bool camcalib_decode_launch(const float* logits, int ld, int D, const float* img_h, const float* img_w, float* angles,
                            float* rotmat, float* intr, float* fpix, int B, cudaStream_t s);
bool head_iter_launch(float* X, int ldx, int C, const float* G, int gsplit, const float* AsT, const float* init157,
                      const float* cam_rotmat, const float* cam_intr, const float* img_h, int use_cam_feats, int B,
                      cudaStream_t s);
bool smpl_prep_launch(const float* X, int ldx, int C, const float* Jt, const float* Js, float* pf, float* Amat,
                      float* Jposed, float* o_pose, long long ld_pose, float* o_pose6d, long long ld_pose6d,
                      float* o_shape, long long ld_shape, float* o_cam, long long ld_cam, int B, cudaStream_t s);
bool body_prep_launch(const float* betas, const float* pose, int pose_kind, const float* Jt, const float* Js, float* X, float* pf,
                      float* Amat, float* joints, long long ld_joints, int B, cudaStream_t s);
bool smpl_verts_launch(const float* Vt, const float* Sd, const float* Pd, const float* Wl, const float* X, int ldx, int C,
                       const float* pf, const float* Amat, float* o_verts, long long ld_verts, int B, cudaStream_t s);
bool smpl_joints_launch(const float* verts, long long ld_verts, const float* Jposed, const float* Jx, float* ej_ws /*[B][4][27]*/, const float* X,
                        int ldx, int C, const float* cam_rotmat, const float* cam_intr, const float* bbox_scale,
                        const float* bbox_center, const float* img_w, const float* img_h, float* o_j3d, long long ld_j3d,
                        float* o_j2d, long long ld_j2d, float* o_camt, long long ld_camt, int use_cam, float focal_length,
                        float img_res, int B, cudaStream_t s);

}  // namespace sb
