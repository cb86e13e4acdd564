// Fused fp32 "tail" kernels: everything after the backbone.
//
//  * CamCalib decode: soft-argmax over 256 bins -> angles -> f_pix, R = euler(pitch,0,roll), K
//    (/root/reference/camcalib/cam_utils.py:110-145, scripts/camcalib_demo.py:127-129,
//     spec/utils/cam_params.py:24-50)
//  * HMR head state init (init_pose/shape/cam + camera features R6d, vfov;
//    /root/reference/spec/models/hmr.py:95-96 and pare HMRHead, SURVEY.md A.3)
//  * SMPL: rot6d -> rotmat, rest joints, kinematic chain, pose/shape blendshapes + linear-blend
//    skinning, 49-joint assembly, weak-perspective -> full-image camera, perspective projection
//    (pare SMPLCamHead / smplx.lbs, SURVEY.md A.4-A.6; call site spec/models/hmr.py:101-112)
//
// All HBM access is coalesced over the vertex index (SMPL constants are repacked coordinate-planar at
// create time), reductions are warp shuffles, and every reduction order is fixed (deterministic output).
#include "common.cuh"
#include "internal.h"
#include "tail.h"

namespace sb {

__constant__ int c_parents[24] = {-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21};
// joint_map (49) and the 21 selected vertex ids are uploaded at create time (bit-exact integer tables).
__constant__ int c_joint_map[49];
__constant__ int c_vertex_ids[21];

bool tail_upload_tables(const int* joint_map49, const int* vertex_ids21) {
    if (!check_cuda(cudaMemcpyToSymbol(c_joint_map, joint_map49, 49 * sizeof(int)), "joint_map upload")) return false;
    return check_cuda(cudaMemcpyToSymbol(c_vertex_ids, vertex_ids21, 21 * sizeof(int)), "vertex_ids upload");
}

// ------------------------------------------------------------------ CamCalib decode
__device__ __forceinline__ void euler_to_rotmat(float ex, float ey, float ez, float* R) {
    // batch_euler2matrix (SURVEY.md A.8): euler -> quaternion (w,x,y,z) -> normalise -> matrix
    const float hx = ex * 0.5f, hy = ey * 0.5f, hz = ez * 0.5f;
    const float cx = cosf(hx), cy = cosf(hy), cz = cosf(hz);
    const float sx = sinf(hx), sy = sinf(hy), sz = sinf(hz);
    float qw = cx * cy * cz - sx * sy * sz;
    float qx = cx * sy * sz + cy * cz * sx;
    float qy = cx * cz * sy - sx * cy * sz;
    float qz = cx * cy * sz + sx * cz * sy;
    const float nrm = sqrtf(qw * qw + qx * qx + qy * qy + qz * qz);
    qw /= nrm; qx /= nrm; qy /= nrm; qz /= nrm;
    const float w2 = qw * qw, x2 = qx * qx, y2 = qy * qy, z2 = qz * qz;
    const float wx = qw * qx, wy = qw * qy, wz = qw * qz, xy = qx * qy, xz = qx * qz, yz = qy * qz;
    R[0] = w2 + x2 - y2 - z2; R[1] = 2 * xy - 2 * wz;     R[2] = 2 * wy + 2 * xz;
    R[3] = 2 * wz + 2 * xy;     R[4] = w2 - x2 + y2 - z2; R[5] = 2 * yz - 2 * wx;
    R[6] = 2 * xz - 2 * wy;     R[7] = 2 * wx + 2 * yz;     R[8] = w2 - x2 - y2 + z2;
}

// grid = B, block = 96 (warp w decodes logits[:, w*D : (w+1)*D]).  logits row stride = ld.
__global__ void __launch_bounds__(96)
camcalib_decode_kernel(const float* __restrict__ logits, int ld, int D, const float* __restrict__ img_h,
                       const float* __restrict__ img_w, float* __restrict__ angles, float* __restrict__ rotmat,
                       float* __restrict__ intr, float* __restrict__ fpix, int B)
{
    __shared__ float s_ang[3];
    const int b = blockIdx.x, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* x = logits + static_cast<size_t>(b) * ld + w * D;
    float mx = -INFINITY;
    for (int i = lane; i < D; i += 32) mx = fmaxf(mx, x[i]);
    mx = warp_max(mx);
    float se = 0.f, sk = 0.f;
    for (int i = lane; i < D; i += 32) {
        const float e = expf(x[i] - mx);
        se += e;
        sk += e * static_cast<float>(i);
    }
    se = warp_sum(se);
    sk = warp_sum(sk);
    if (lane == 0) {
        float k = sk / se;                                       // soft-argmax index
        k = k / static_cast<float>(D - 1) * 2.f - 1.f;           // normalize_keypoints
        const float lo = (w == 0) ? 0.2617f : -0.6f;             // cam_utils.py:55,39,133
        const float hi = (w == 0) ? 2.1f : 0.6f;
        const float range = (w == 0) ? static_cast<float>(2.1 - 0.2617) : static_cast<float>(0.6 - (-0.6));
        s_ang[w] = range * ((k + 1.f) / 2.f) + lo;
        (void)hi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const float vfov = s_ang[0], pitch = s_ang[1], roll = s_ang[2];
        angles[b * 3 + 0] = vfov; angles[b * 3 + 1] = pitch; angles[b * 3 + 2] = roll;
        if (rotmat != nullptr) {
            const float h = img_h[b], wd = img_w[b];
            const float f = h / 2.f / tanf(vfov / 2.f);          // camcalib_demo.py:129
            float R[9];
            euler_to_rotmat(pitch, 0.f, roll, R);                // cam_params.py:37
            for (int i = 0; i < 9; ++i) rotmat[b * 9 + i] = R[i];
            float* K = intr + b * 9;                             // cam_params.py:39-46 (K[2,2] stays 0)
            K[0] = f; K[1] = 0.f; K[2] = wd / 2.f;
            K[3] = 0.f; K[4] = f; K[5] = h / 2.f;
            K[6] = 0.f; K[7] = 0.f; K[8] = 0.f;
            if (fpix) fpix[b] = f;
        }
    }
}

bool camcalib_decode_launch(const float* logits, int ld, int D, const float* img_h, const float* img_w, float* angles,
                            float* rotmat, float* intr, float* fpix, int B, cudaStream_t s) {
    camcalib_decode_kernel<<<B, 96, 0, s>>>(logits, ld, D, img_h, img_w, angles, rotmat, intr, fpix, B);
    return check_cuda(cudaGetLastError(), "camcalib_decode");
}

// ------------------------------------------------------------------ HMR head (folded iterative regressor)
// X row layout: [xf (C) | pose6d (144) | shape (10) | cam (3) | R6d (6) | vfov (1)]   (last 7 only with cam feats)
// The reference iterates  xc = fc2(fc1(cat[xf, s, camfeat]));  s += dec(xc)  three times with dropout = identity and
// NO non-linearity in between (pare HMRHead, SURVEY.md A.3), so one iteration is affine in (xf, s, camfeat):
//     s <- s + G + As [s; camfeat],   G = (D W2 W1[:, :C]) xf + (D (W2 b1 + b2) + bd),   As = D W2 W1[:, C:]
// The products are folded once at create time in fp64 (api.cu); per forward this leaves ONE (B x C) x (C x 157)
// GEMM for G and three 157 x 164 mat-vecs per image, done here (one CTA per image, AsT is [k][160] so lanes read
// unit-stride).  Same trick as BatchNorm folding: exact in real arithmetic, rounding differs at the 1e-7 level.
__global__ void __launch_bounds__(192)
head_iter_kernel(float* __restrict__ X, int ldx, int C, const float* __restrict__ G /*[gsplit][B][160]*/, int gsplit,
                 const float* __restrict__ AsT /*[ns][160]*/, const float* __restrict__ init157,
                 const float* __restrict__ cam_rotmat, const float* __restrict__ cam_intr,
                 const float* __restrict__ img_h, int use_cam_feats, int n_iter, int B)
{
    __shared__ float v[164];
    const int b = blockIdx.x, j = threadIdx.x;
    const int ns = 157 + (use_cam_feats ? 7 : 0);
    if (j < 157) v[j] = init157[j];
    else if (j < ns) {
        const int i = j - 157;
        v[j] = (i < 6) ? cam_rotmat[b * 9 + (i >> 1) * 3 + (i & 1)]                           // R[:, :2] row-major
                       : 2.f * atanf(img_h[b] / (2.f * cam_intr[b * 9]));                      // hmr.py:95
    }
    float g = 0.f;                                             // sum the split-K slices in a fixed order
    if (j < 157)
        for (int z = 0; z < gsplit; ++z) g += G[(static_cast<size_t>(z) * B + b) * 160 + j];
    for (int it = 0; it < n_iter; ++it) {
        __syncthreads();
        float acc = g;
        if (j < 157) {
#pragma unroll 4
            for (int k = 0; k < ns; ++k) acc = fmaf(AsT[k * 160 + j], v[k], acc);
        }
        __syncthreads();
        if (j < 157) v[j] += acc;
    }
    __syncthreads();
    float* row = X + static_cast<size_t>(b) * ldx + C;
    if (j < 157) row[j] = v[j];
}
bool head_iter_launch(float* X, int ldx, int C, const float* G, int gsplit, const float* AsT, const float* init157,
                      const float* cam_rotmat, const float* cam_intr, const float* img_h, int use_cam_feats, int B,
                      cudaStream_t s) {
    head_iter_kernel<<<B, 192, 0, s>>>(X, ldx, C, G, gsplit, AsT, init157, cam_rotmat, cam_intr, img_h, use_cam_feats, 3, B);
    return check_cuda(cudaGetLastError(), "head_iter");
}

// ------------------------------------------------------------------ SMPL kinematic chain (shared by both prep kernels)
// One warp per image.  In: sR = the 24 joint rotations, sJ = the 24 rest joints.  Out: A[24][12] = the skinning transforms
// G - G.[J;0] (rows of the 3x4 top) and Jposed[24][3] = the posed joints (the translation column of G).
__device__ __forceinline__ void smpl_chain(const float (*sR)[9], const float (*sJ)[3], float (*sG)[12], float* __restrict__ A_out,
                                           float* __restrict__ Jposed, int lane)
{
    // kinematic chain: G_0 = [R_0 | J_0];  G_i = G_par * [R_i | J_i - J_par]
    if (lane < 9) sG[0][(lane / 3) * 4 + (lane % 3)] = sR[0][lane];
    else if (lane < 12) sG[0][(lane - 9) * 4 + 3] = sJ[0][lane - 9];
    __syncwarp();
    for (int i = 1; i < 24; ++i) {
        const int par = c_parents[i];
        float v = 0.f;
        if (lane < 9) {
            const int r = lane / 3, c = lane % 3;
            v = sG[par][r * 4 + 0] * sR[i][0 * 3 + c] + sG[par][r * 4 + 1] * sR[i][1 * 3 + c] + sG[par][r * 4 + 2] * sR[i][2 * 3 + c];
        } else if (lane < 12) {
            const int r = lane - 9;
            const float rx = sJ[i][0] - sJ[par][0], ry = sJ[i][1] - sJ[par][1], rz = sJ[i][2] - sJ[par][2];
            v = sG[par][r * 4 + 0] * rx + sG[par][r * 4 + 1] * ry + sG[par][r * 4 + 2] * rz + sG[par][r * 4 + 3];
        }
        __syncwarp();
        if (lane < 9) sG[i][(lane / 3) * 4 + (lane % 3)] = v;
        else if (lane < 12) sG[i][(lane - 9) * 4 + 3] = v;
        __syncwarp();
    }
    if (lane < 24) {
        const float* G = sG[lane];
        float* A = A_out + lane * 12;
        const float jx = sJ[lane][0], jy = sJ[lane][1], jz = sJ[lane][2];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            A[r * 4 + 0] = G[r * 4 + 0]; A[r * 4 + 1] = G[r * 4 + 1]; A[r * 4 + 2] = G[r * 4 + 2];
            A[r * 4 + 3] = G[r * 4 + 3] - (G[r * 4 + 0] * jx + G[r * 4 + 1] * jy + G[r * 4 + 2] * jz);
            Jposed[lane * 3 + r] = G[r * 4 + 3];
        }
    }
}

// ------------------------------------------------------------------ SMPL prep: rot6d, rest joints, kinematic chain
// grid = B, block = 32.
__global__ void __launch_bounds__(32)
smpl_prep_kernel(const float* __restrict__ X, int ldx, int C, const float* __restrict__ Jt /*[24][3]*/,
                 const float* __restrict__ Js /*[24][3][10]*/, float* __restrict__ pf /*[B][PF_LD]*/,
                 float* __restrict__ Amat /*[B][24][12]*/, float* __restrict__ Jposed /*[B][24][3]*/,
                 float* __restrict__ o_pose, long long ld_pose, float* __restrict__ o_pose6d, long long ld_pose6d,
                 float* __restrict__ o_shape, long long ld_shape, float* __restrict__ o_cam, long long ld_cam, int B)
{
    __shared__ float sR[24][9];
    __shared__ float sJ[24][3];
    __shared__ float sG[24][12];
    __shared__ float sBeta[10];
    const int b = blockIdx.x, lane = threadIdx.x;
    const float* st = X + static_cast<size_t>(b) * ldx + C;
    if (lane < 10) sBeta[lane] = st[144 + lane];
    for (int i = lane; i < 144; i += 32) o_pose6d[b * ld_pose6d + i] = st[i];
    if (lane < 10) o_shape[b * ld_shape + lane] = st[144 + lane];
    if (lane < 3) o_cam[b * ld_cam + lane] = st[154 + lane];
    __syncwarp();
    if (lane < 24) {
        // rot6d_to_rotmat: x.view(3,2): a1 = x[:,0] = (x0,x2,x4), a2 = x[:,1] = (x1,x3,x5)
        const float* x = st + lane * 6;
        const float a1x = x[0], a1y = x[2], a1z = x[4];
        const float a2x = x[1], a2y = x[3], a2z = x[5];
        const float n1 = fmaxf(sqrtf(a1x * a1x + a1y * a1y + a1z * a1z), 1e-12f);
        const float b1x = a1x / n1, b1y = a1y / n1, b1z = a1z / n1;
        const float d = b1x * a2x + b1y * a2y + b1z * a2z;
        const float ux = a2x - d * b1x, uy = a2y - d * b1y, uz = a2z - d * b1z;
        const float n2 = fmaxf(sqrtf(ux * ux + uy * uy + uz * uz), 1e-12f);
        const float b2x = ux / n2, b2y = uy / n2, b2z = uz / n2;
        const float b3x = b1y * b2z - b1z * b2y, b3y = b1z * b2x - b1x * b2z, b3z = b1x * b2y - b1y * b2x;
        float* R = sR[lane];                                    // columns b1,b2,b3
        R[0] = b1x; R[1] = b2x; R[2] = b3x;
        R[3] = b1y; R[4] = b2y; R[5] = b3y;
        R[6] = b1z; R[7] = b2z; R[8] = b3z;
        float* op = o_pose + b * ld_pose + lane * 9;
#pragma unroll
        for (int e = 0; e < 9; ++e) op[e] = R[e];
        if (lane >= 1) {
            float* p = pf + static_cast<size_t>(b) * PF_LD + (lane - 1) * 9;
#pragma unroll
            for (int e = 0; e < 9; ++e) p[e] = R[e] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
        }
        // rest joints J = Jt + Js . beta
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float acc = Jt[lane * 3 + c];
#pragma unroll
            for (int l = 0; l < 10; ++l) acc = fmaf(Js[(lane * 3 + c) * 10 + l], sBeta[l], acc);
            sJ[lane][c] = acc;
        }
    }
    if (lane == 0) pf[static_cast<size_t>(b) * PF_LD + 207] = 0.f;   // K padding column
    __syncwarp();
    smpl_chain(sR, sJ, sG, Amat + static_cast<size_t>(b) * 288, Jposed + static_cast<size_t>(b) * 72, lane);
}

bool smpl_prep_launch(const float* X, int ldx, int C, const float* Jt, const float* Js, float* pf, float* Amat,
                      float* Jposed, float* o_pose, long long ld_pose, float* o_pose6d, long long ld_pose6d,
                      float* o_shape, long long ld_shape, float* o_cam, long long ld_cam, int B, cudaStream_t s) {
    smpl_prep_kernel<<<B, 32, 0, s>>>(X, ldx, C, Jt, Js, pf, Amat, Jposed, o_pose, ld_pose, o_pose6d, ld_pose6d,
                                      o_shape, ld_shape, o_cam, ld_cam, B);
    return check_cuda(cudaGetLastError(), "smpl_prep");
}

// ------------------------------------------------------------------ body-model prep: axis-angle / rotation matrices + betas
// The smplx SMPL forward (lbs with pose2rot) from caller-given parameters, for the evaluation side (BodyModel).  grid = B,
// block = 32.  pose_kind 0: pose = axis-angle [B][72], turned into rotations with smplx's batch_rodrigues
//     angle = |r + 1e-8|,  k = r / angle,  R = I + sin(angle) K + (1 - cos(angle)) K^2   (K = [k]_x);
// pose_kind 1: pose = rotation matrices [B][24][9], copied (pose2rot=False).  The betas are staged in the X row buffer
// ([B][BODY_XLD], read by smpl_verts_kernel at column 144 with C = 0); the posed joints go to joints[b * ld_joints].
__global__ void __launch_bounds__(32)
body_prep_kernel(const float* __restrict__ betas, const float* __restrict__ pose, int pose_kind, const float* __restrict__ Jt,
                 const float* __restrict__ Js, float* __restrict__ X, float* __restrict__ pf, float* __restrict__ Amat,
                 float* __restrict__ joints, long long ld_joints, int B)
{
    __shared__ float sR[24][9];
    __shared__ float sJ[24][3];
    __shared__ float sG[24][12];
    __shared__ float sBeta[10];
    const int b = blockIdx.x, lane = threadIdx.x;
    if (lane < 10) {
        const float be = betas[b * 10 + lane];
        sBeta[lane] = be;
        X[static_cast<size_t>(b) * BODY_XLD + 144 + lane] = be;
    }
    __syncwarp();
    if (lane < 24) {
        float* R = sR[lane];
        if (pose_kind == 0) {
            const float* r = pose + static_cast<size_t>(b) * 72 + lane * 3;
            const float ax = r[0] + 1e-8f, ay = r[1] + 1e-8f, az = r[2] + 1e-8f;
            const float angle = sqrtf(ax * ax + ay * ay + az * az);
            const float kx = r[0] / angle, ky = r[1] / angle, kz = r[2] / angle;
            const float sn = sinf(angle), omc = 1.f - cosf(angle);
            // K = [[0,-kz,ky],[kz,0,-kx],[-ky,kx,0]];  K^2 = k k^T - |k|^2 I
            R[0] = 1.f + omc * (-kz * kz - ky * ky); R[1] = -sn * kz + omc * (ky * kx);        R[2] = sn * ky + omc * (kz * kx);
            R[3] = sn * kz + omc * (kx * ky);        R[4] = 1.f + omc * (-kz * kz - kx * kx); R[5] = -sn * kx + omc * (kz * ky);
            R[6] = -sn * ky + omc * (kx * kz);       R[7] = sn * kx + omc * (ky * kz);        R[8] = 1.f + omc * (-ky * ky - kx * kx);
        } else {
            const float* m = pose + (static_cast<size_t>(b) * 24 + lane) * 9;
#pragma unroll
            for (int e = 0; e < 9; ++e) R[e] = m[e];
        }
        if (lane >= 1) {
            float* p = pf + static_cast<size_t>(b) * PF_LD + (lane - 1) * 9;
#pragma unroll
            for (int e = 0; e < 9; ++e) p[e] = R[e] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
        }
        // rest joints J = Jt + Js . beta (as smpl_prep_kernel)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float acc = Jt[lane * 3 + c];
#pragma unroll
            for (int l = 0; l < 10; ++l) acc = fmaf(Js[(lane * 3 + c) * 10 + l], sBeta[l], acc);
            sJ[lane][c] = acc;
        }
    }
    if (lane == 0) pf[static_cast<size_t>(b) * PF_LD + 207] = 0.f;   // K padding column
    __syncwarp();
    smpl_chain(sR, sJ, sG, Amat + static_cast<size_t>(b) * 288, joints + b * ld_joints, lane);
}

bool body_prep_launch(const float* betas, const float* pose, int pose_kind, const float* Jt, const float* Js, float* X, float* pf,
                      float* Amat, float* joints, long long ld_joints, int B, cudaStream_t s) {
    body_prep_kernel<<<B, 32, 0, s>>>(betas, pose, pose_kind, Jt, Js, X, pf, Amat, joints, ld_joints, B);
    return check_cuda(cudaGetLastError(), "body_prep");
}

// ------------------------------------------------------------------ SMPL vertices
// Tile: 64 vertices x 64 images per CTA; 256 threads: lane -> the adjacent vertices (2*lane, 2*lane+1), warp -> 8 images.
//
// v_posed = v_template + shapedirs . beta + posedirs . pose_feature is ONE k-loop over 14 chunks of 16 "features": chunks
// 0..12 are the 207 pose features, chunk 13 holds the 10 betas and a constant 1 against shapedirs / v_template (added last:
// the small pose offsets are summed before the O(1) template is added).  Per k a warp issues 2 LDS.128 (8 image features,
// broadcast) + 3 LDS.64 (3 coordinates x 2 vertices) for 48 FFMA; the round-1 shape (4 images per warp: 4 LDS per 24 FFMA,
// 7 shared-memory wavefronts per 24 FFMA) was bound by the shared-memory pipe, not by the FP32 pipe.  The next chunk is
// fetched into registers while the current one is consumed.  Skinning is applied as out = sum_j w_j (A_j [v;1]) -- the same
// 12 FFMA per (joint, vertex) as building T = sum_j w_j A_j first, but 6 accumulators instead of 24, and A_j is read once for
// the thread's two vertices (5 wavefronts per 24 FFMA).  The extra-joint regression moved to smpl_joints_kernel (it cost
// 540 shuffles per thread here).  Vertices leave through a per-warp shared-memory transpose as full 128-byte rows.
constexpr int SV_TV = 64, SV_TB = 64, SV_BK = 16, SV_NCH = 14;
struct SvSmem {
    float A[SV_TB][24][12];          // skinning transforms of the tile's images (72 KB)
    float P[SV_BK][3][SV_TV];        // basis chunk (12 KB); reused as the output transpose buffer
    float pf[SV_BK][SV_TB];          // feature chunk, [k][image]
    float W[24][SV_TV];              // skinning weights of the tile's vertices
};

__global__ void __launch_bounds__(256, 2)
smpl_verts_kernel(const float* __restrict__ Vt, const float* __restrict__ Sd, const float* __restrict__ Pd,
                  const float* __restrict__ Wl, const float* __restrict__ X, int ldx, int C,
                  const float* __restrict__ pf, const float* __restrict__ Amat, float* __restrict__ o_verts,
                  long long ld_verts, int B)
{
    extern __shared__ __align__(16) uint8_t sv_raw[];
    SvSmem& sm = *reinterpret_cast<SvSmem*>(sv_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int v0 = blockIdx.x * SV_TV;
    const int b0 = blockIdx.y * SV_TB;

    // stage per-image transforms and per-vertex weights
    for (int i = tid; i < SV_TB * 72; i += 256) {
        const int bi = i / 72;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b0 + bi < B) v = reinterpret_cast<const float4*>(Amat + static_cast<size_t>(b0) * 288)[i];
        reinterpret_cast<float4*>(sm.A)[i] = v;
    }
    for (int i = tid; i < 24 * (SV_TV / 4); i += 256) {
        const int j = i / (SV_TV / 4), vq = (i - j * (SV_TV / 4)) * 4;
        *reinterpret_cast<float4*>(&sm.W[j][vq]) = *reinterpret_cast<const float4*>(Wl + static_cast<size_t>(j) * SMPL_VP + v0 + vq);
    }

    float4 rp[3], rf;                                           // the chunk in flight: 3 basis float4 + 4 features of one image
    const int f_bi = tid >> 2, f_kq = (tid & 3) * 4;
    auto fetch = [&](int ch) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const int idx = tid + q * 256;                     // 768 float4 = 16 x 3 x 64 floats
            const int kk = idx / 48, rem = idx - kk * 48;
            const int c = rem / 16, vq = (rem - c * 16) * 4;
            const float* src = nullptr;
            if (ch < SV_NCH - 1) {
                const int k = ch * SV_BK + kk;
                if (k < 207) src = Pd + (static_cast<size_t>(k) * 3 + c) * SMPL_VP;
            } else if (kk < 10) {
                src = Sd + (static_cast<size_t>(kk) * 3 + c) * SMPL_VP;
            } else if (kk == 10) {
                src = Vt + static_cast<size_t>(c) * SMPL_VP;
            }
            rp[q] = src ? *reinterpret_cast<const float4*>(src + v0 + vq) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        rf = make_float4(0.f, 0.f, 0.f, 0.f);
        const int b = b0 + f_bi;
        if (b < B) {
            if (ch < SV_NCH - 1) {
                rf = *reinterpret_cast<const float4*>(pf + static_cast<size_t>(b) * PF_LD + ch * SV_BK + f_kq);
            } else {
                const float* beta = X + static_cast<size_t>(b) * ldx + C + 144;
                float e[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { const int k = f_kq + i; e[i] = k < 10 ? beta[k] : (k == 10 ? 1.f : 0.f); }
                rf = make_float4(e[0], e[1], e[2], e[3]);
            }
        }
    };
    auto stash = [&]() {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const int idx = tid + q * 256;
            const int kk = idx / 48, rem = idx - kk * 48;
            const int c = rem / 16, vq = (rem - c * 16) * 4;
            *reinterpret_cast<float4*>(&sm.P[kk][c][vq]) = rp[q];
        }
        sm.pf[f_kq + 0][f_bi] = rf.x; sm.pf[f_kq + 1][f_bi] = rf.y; sm.pf[f_kq + 2][f_bi] = rf.z; sm.pf[f_kq + 3][f_bi] = rf.w;
    };

    float acc[8][2][3];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int c = 0; c < 3; ++c) acc[i][h][c] = 0.f;

    const bool live = b0 + warp * 8 < B;                        // warps whose 8 images are all past the batch only help staging
    fetch(0);
    stash();
    for (int ch = 0; ch < SV_NCH; ++ch) {
        __syncthreads();                                        // chunk ch is in shared memory
        if (ch + 1 < SV_NCH) fetch(ch + 1);
        if (live) {
#pragma unroll
            for (int kk = 0; kk < SV_BK; ++kk) {
                const float4 a0 = *reinterpret_cast<const float4*>(&sm.pf[kk][warp * 8]);
                const float4 a1 = *reinterpret_cast<const float4*>(&sm.pf[kk][warp * 8 + 4]);
                const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                float p[3][2];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float2 p2 = *reinterpret_cast<const float2*>(&sm.P[kk][c][2 * lane]);
                    p[c][0] = p2.x; p[c][1] = p2.y;
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int h = 0; h < 2; ++h)
#pragma unroll
                        for (int c = 0; c < 3; ++c) acc[i][h][c] = fmaf(a[i], p[c][h], acc[i][h][c]);
            }
        }
        __syncthreads();                                        // everyone is done reading chunk ch
        if (ch + 1 < SV_NCH) stash();
    }
    if (!live) return;

    // skinning + store, one image at a time; sm.P is free now: 192 floats per warp for the output transpose
    float* tr = &sm.P[0][0][0] + warp * 192;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int img = warp * 8 + i;
        float o[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
#pragma unroll 4
        for (int j = 0; j < 24; ++j) {
            const float2 w = *reinterpret_cast<const float2*>(&sm.W[j][2 * lane]);
            const float4* Aj = reinterpret_cast<const float4*>(&sm.A[img][j][0]);
            const float4 r0 = Aj[0], r1 = Aj[1], r2 = Aj[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float x = acc[i][h][0], y = acc[i][h][1], z = acc[i][h][2], wh = h ? w.y : w.x;
                o[h][0] = fmaf(wh, fmaf(r0.x, x, fmaf(r0.y, y, fmaf(r0.z, z, r0.w))), o[h][0]);
                o[h][1] = fmaf(wh, fmaf(r1.x, x, fmaf(r1.y, y, fmaf(r1.z, z, r1.w))), o[h][1]);
                o[h][2] = fmaf(wh, fmaf(r2.x, x, fmaf(r2.y, y, fmaf(r2.z, z, r2.w))), o[h][2]);
            }
        }
        const int b = b0 + img;
        __syncwarp();
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int c = 0; c < 3; ++c) tr[(2 * lane + h) * 3 + c] = o[h][c];
        __syncwarp();
        if (b < B) {
            float* dst = o_verts + b * ld_verts + static_cast<size_t>(v0) * 3;
#pragma unroll
            for (int q = 0; q < 6; ++q) {
                const int f = q * 32 + lane;
                if (v0 * 3 + f < SMPL_NV * 3) dst[f] = tr[f];
            }
        }
    }
}

bool smpl_verts_launch(const float* Vt, const float* Sd, const float* Pd, const float* Wl, const float* X, int ldx, int C,
                       const float* pf, const float* Amat, float* o_verts, long long ld_verts, int B, cudaStream_t s) {
    static DeviceOnce attr;
    if (attr.need()) {
        if (!check_cuda(cudaFuncSetAttribute(smpl_verts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(sizeof(SvSmem))), "smpl_verts attr")) return false;
    }
    dim3 grid(SMPL_NVT, (B + SV_TB - 1) / SV_TB);
    smpl_verts_kernel<<<grid, 256, sizeof(SvSmem), s>>>(Vt, Sd, Pd, Wl, X, ldx, C, pf, Amat, o_verts, ld_verts, B);
    return check_cuda(cudaGetLastError(), "smpl_verts");
}

// ------------------------------------------------------------------ 49 joints, camera, projection
// The 9 extra joints (J_regressor_extra @ vertices): CTA (x, y) handles the images 8x .. 8x+7 (one per warp) and the y-th
// quarter of the vertices (7 chunks of 256), so the regressor is read once per 8 images (one image per CTA re-read all 248 KB
// of it from L2 per image: 34 us at B = 256) and 4 * B/8 CTAs share the work.  Per chunk a lane first issues all 24 loads of
// its 8 vertices, then the chunk of the regressor is staged through shared memory, then 8 x 27 FMAs.  One fixed-order shuffle
// tree per output; the four quarter sums are added in order by smpl_joints_kernel -- deterministic.
constexpr int EJ_SPLIT = 4, EJ_CHUNKS = (SMPL_VP / 256 + EJ_SPLIT - 1) / EJ_SPLIT;
__global__ void __launch_bounds__(256)
smpl_extra_joints_kernel(const float* __restrict__ verts, long long ld_verts, const float* __restrict__ Jx,
                         float* __restrict__ ej_out /*[B][EJ_SPLIT][27]*/, int B)
{
    __shared__ float sJ[9][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + warp;
    const float* vb = verts + (b < B ? b : 0) * ld_verts;
    float ej[27];
#pragma unroll
    for (int q = 0; q < 27; ++q) ej[q] = 0.f;
    const int c_begin = blockIdx.y * EJ_CHUNKS * 256;
    const int c_end = min(SMPL_NV, c_begin + EJ_CHUNKS * 256);
    for (int c0 = c_begin; c0 < c_end; c0 += 256) {
        float vx[8][3];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int v = c0 + k * 32 + lane;
#pragma unroll
            for (int c = 0; c < 3; ++c) vx[k][c] = (v < SMPL_NV) ? vb[static_cast<size_t>(v) * 3 + c] : 0.f;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < 9 * 256; i += 256) {
            const int q = i >> 8, v = i & 255;
            sJ[q][v] = (c0 + v < SMPL_NV) ? Jx[static_cast<size_t>(q) * SMPL_VP + c0 + v] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 8; ++k) {
#pragma unroll
            for (int q = 0; q < 9; ++q) {
                const float w = sJ[q][k * 32 + lane];
                ej[q * 3 + 0] = fmaf(w, vx[k][0], ej[q * 3 + 0]); ej[q * 3 + 1] = fmaf(w, vx[k][1], ej[q * 3 + 1]);
                ej[q * 3 + 2] = fmaf(w, vx[k][2], ej[q * 3 + 2]);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 27; ++q) {
        const float s = warp_sum(ej[q]);
        if (lane == 0 && b < B) ej_out[(static_cast<size_t>(b) * EJ_SPLIT + blockIdx.y) * 27 + q] = s;
    }
}

// grid = B, block = 64.
__global__ void __launch_bounds__(64)
smpl_joints_kernel(const float* __restrict__ verts, long long ld_verts, const float* __restrict__ Jposed,
                   const float* __restrict__ ej, const float* __restrict__ X, int ldx, int C,
                   const float* __restrict__ cam_rotmat, const float* __restrict__ cam_intr,
                   const float* __restrict__ bbox_scale, const float* __restrict__ bbox_center,
                   const float* __restrict__ img_w, const float* __restrict__ img_h,
                   float* __restrict__ o_j3d, long long ld_j3d, float* __restrict__ o_j2d, long long ld_j2d,
                   float* __restrict__ o_camt, long long ld_camt, int use_cam, float focal_length, float img_res, int B)
{
    __shared__ float j54[54][3];
    __shared__ float s_t[3];
    const int b = blockIdx.x, t = threadIdx.x;
    if (t < 24) {
#pragma unroll
        for (int c = 0; c < 3; ++c) j54[t][c] = Jposed[(static_cast<size_t>(b) * 24 + t) * 3 + c];
    } else if (t < 45) {
        const float* v = verts + b * ld_verts + static_cast<size_t>(c_vertex_ids[t - 24]) * 3;
        j54[t][0] = v[0]; j54[t][1] = v[1]; j54[t][2] = v[2];
    } else if (t < 54) {
        const int q = t - 45;
        const float* e = ej + static_cast<size_t>(b) * EJ_SPLIT * 27 + q * 3;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int y = 0; y < EJ_SPLIT; ++y) { s0 += e[y * 27 + 0]; s1 += e[y * 27 + 1]; s2 += e[y * 27 + 2]; }
        j54[t][0] = s0; j54[t][1] = s1; j54[t][2] = s2;
    }
    const float* cam = X + static_cast<size_t>(b) * ldx + C + 154;
    if (t == 63) {
        const float sc = cam[0], tx = cam[1], ty = cam[2];
        float ct[3];
        if (use_cam) {
            // convert_pare_to_full_img_cam (SURVEY.md A.5), bbox_height = bbox_scale * 200
            const float bh = bbox_scale[b] * 200.f;
            const float f = cam_intr[b * 9];
            const float r = bh / img_res;
            ct[2] = 2.f * f / (r * img_res * sc);
            ct[0] = tx + 2.f * (bbox_center[b * 2 + 0] - img_w[b] / 2.f) / (sc * bh);
            ct[1] = ty + 2.f * (bbox_center[b * 2 + 1] - img_h[b] / 2.f) / (sc * bh);
        } else {
            ct[0] = tx; ct[1] = ty; ct[2] = 2.f * focal_length / (img_res * sc + 1e-9f);
        }
        s_t[0] = ct[0]; s_t[1] = ct[1]; s_t[2] = ct[2];
        o_camt[b * ld_camt + 0] = ct[0]; o_camt[b * ld_camt + 1] = ct[1]; o_camt[b * ld_camt + 2] = ct[2];
    }
    __syncthreads();
    if (t < 49) {
        const int src = c_joint_map[t];
        const float x = j54[src][0], y = j54[src][1], z = j54[src][2];
        float* o3 = o_j3d + b * ld_j3d + t * 3;
        o3[0] = x; o3[1] = y; o3[2] = z;
        float R[9], K[6];
        if (use_cam) {
#pragma unroll
            for (int i = 0; i < 9; ++i) R[i] = cam_rotmat[b * 9 + i];
#pragma unroll
            for (int i = 0; i < 6; ++i) K[i] = cam_intr[b * 9 + i];
        } else {
            R[0] = 1.f; R[1] = 0.f; R[2] = 0.f; R[3] = 0.f; R[4] = 1.f; R[5] = 0.f; R[6] = 0.f; R[7] = 0.f; R[8] = 1.f;
            K[0] = focal_length; K[1] = 0.f; K[2] = 0.f; K[3] = 0.f; K[4] = focal_length; K[5] = 0.f;
        }
        // perspective_projection (SURVEY.md A.6)
        float px = R[0] * x + R[1] * y + R[2] * z + s_t[0];
        float py = R[3] * x + R[4] * y + R[5] * z + s_t[1];
        float pz = R[6] * x + R[7] * y + R[8] * z + s_t[2];
        px = px / pz; py = py / pz; pz = pz / pz;
        float u = K[0] * px + K[1] * py + K[2] * pz;
        float v = K[3] * px + K[4] * py + K[5] * pz;
        if (!use_cam) { u = u / (img_res / 2.f); v = v / (img_res / 2.f); }
        o_j2d[b * ld_j2d + t * 2 + 0] = u;
        o_j2d[b * ld_j2d + t * 2 + 1] = v;
    }
}

bool smpl_joints_launch(const float* verts, long long ld_verts, const float* Jposed, const float* Jx, float* ej_ws, const float* X,
                        int ldx, int C, const float* cam_rotmat, const float* cam_intr, const float* bbox_scale,
                        const float* bbox_center, const float* img_w, const float* img_h, float* o_j3d, long long ld_j3d,
                        float* o_j2d, long long ld_j2d, float* o_camt, long long ld_camt, int use_cam, float focal_length,
                        float img_res, int B, cudaStream_t s) {
    smpl_extra_joints_kernel<<<dim3((B + 7) / 8, EJ_SPLIT), 256, 0, s>>>(verts, ld_verts, Jx, ej_ws, B);
    smpl_joints_kernel<<<B, 64, 0, s>>>(verts, ld_verts, Jposed, ej_ws, X, ldx, C, cam_rotmat, cam_intr, bbox_scale,
                                        bbox_center, img_w, img_h, o_j3d, ld_j3d, o_j2d, ld_j2d, o_camt, ld_camt,
                                        use_cam, focal_length, img_res, B);
    return check_cuda(cudaGetLastError(), "smpl_joints");
}

}  // namespace sb
