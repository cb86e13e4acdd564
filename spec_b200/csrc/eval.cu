// Eval-side metrics on the device (SURVEY.md section 8f, rank 1): H36M joint regression from the predicted mesh,
// pelvis centring, MPJPE, Procrustes-aligned MPJPE and per-vertex error -- what
// /root/reference/spec/trainer.py:272-316 and /root/reference/spec/utils/compute_error.py:33-86 do after copying the
// 21 MB of vertices per batch to the host (numpy SVD per sample).  Only three floats per image come back.
#include "common.cuh"
#include "internal.h"
#include "tail.h"

namespace sb {

// ------------------------------------------------------------------ joint regression: out = R . (J_regressor . verts)
// NJ joints (17: J_regressor_h36m, 24: SMPL's own J_regressor), JT is [6890][LDJ] (the regressor transposed, rows padded to a
// multiple of 4).  grid (B, nsets), block 256.  set 0 = v0 (e.g. the predicted mesh), set 1 = v1 (the ground-truth mesh,
// optional).  rot0 / rot1: optional per-image 3x3 rotations [B][9] applied to the regressed joints of their set (the joints
// of the rotated mesh: J (R v) = R (J v)).  out: [nsets][B][NJ][3].
template <int NJ, int LDJ>
__global__ void __launch_bounds__(256)
regress_joints_kernel(const float* __restrict__ v0, long long ld0, const float* __restrict__ rot0, const float* __restrict__ v1,
                      long long ld1, const float* __restrict__ rot1, const float* __restrict__ JT, float* __restrict__ out, int B)
{
    constexpr int NO = NJ * 3;
    __shared__ float red[8][NO];
    __shared__ float tot[NO];
    const int b = blockIdx.x, set = blockIdx.y;
    const float* verts = (set == 0 ? v0 + b * ld0 : v1 + b * ld1);
    const float* rot = (set == 0 ? rot0 : rot1);
    float acc[NO];
#pragma unroll
    for (int i = 0; i < NO; ++i) acc[i] = 0.f;
    for (int v = threadIdx.x; v < SMPL_NV; v += 256) {
        const float x = verts[v * 3 + 0], y = verts[v * 3 + 1], z = verts[v * 3 + 2];
        const float4* jr = reinterpret_cast<const float4*>(JT + static_cast<size_t>(v) * LDJ);
        float w[LDJ];
#pragma unroll
        for (int q = 0; q < LDJ / 4; ++q) { const float4 t = jr[q]; w[4 * q] = t.x; w[4 * q + 1] = t.y; w[4 * q + 2] = t.z; w[4 * q + 3] = t.w; }
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            acc[j * 3 + 0] = fmaf(w[j], x, acc[j * 3 + 0]);
            acc[j * 3 + 1] = fmaf(w[j], y, acc[j * 3 + 1]);
            acc[j * 3 + 2] = fmaf(w[j], z, acc[j * 3 + 2]);
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < NO; ++i) {
        const float s = warp_sum(acc[i]);
        if (lane == 0) red[warp][i] = s;
    }
    __syncthreads();
    float* o = out + (static_cast<size_t>(set) * B + b) * NO;
    if (threadIdx.x < NO) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
        if (rot == nullptr) o[threadIdx.x] = s;
        else tot[threadIdx.x] = s;
    }
    if (rot != nullptr) {                       // block-uniform
        __syncthreads();
        if (threadIdx.x < NO) {
            const int j = threadIdx.x / 3, r = threadIdx.x - j * 3;
            const float* R = rot + static_cast<size_t>(b) * 9 + r * 3;
            o[threadIdx.x] = R[0] * tot[j * 3 + 0] + R[1] * tot[j * 3 + 1] + R[2] * tot[j * 3 + 2];
        }
    }
}

// ------------------------------------------------------------------ 3x3 helpers (one thread per image)
__device__ inline void jacobi_eig3(float A[3][3], float V[3][3], float lam[3]) {
    // cyclic Jacobi on a symmetric 3x3; V accumulates the rotations (det +1)
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) V[i][j] = (i == j) ? 1.f : 0.f;
    for (int sweep = 0; sweep < 12; ++sweep) {
        const float off = fabsf(A[0][1]) + fabsf(A[0][2]) + fabsf(A[1][2]);
        if (off < 1e-20f) break;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = (pq == 2) ? 1 : 0, q = (pq == 0) ? 1 : 2;
            const float apq = A[p][q];
            if (fabsf(apq) < 1e-30f) continue;
            const float theta = (A[q][q] - A[p][p]) / (2.f * apq);
            const float t = copysignf(1.f, theta) / (fabsf(theta) + sqrtf(theta * theta + 1.f));
            const float c = rsqrtf(t * t + 1.f), s = t * c;
#pragma unroll
            for (int k = 0; k < 3; ++k) {           // A <- A J
                const float akp = A[k][p], akq = A[k][q];
                A[k][p] = c * akp - s * akq;
                A[k][q] = s * akp + c * akq;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {           // A <- J^T A
                const float apk = A[p][k], aqk = A[q][k];
                A[p][k] = c * apk - s * aqk;
                A[q][k] = s * apk + c * aqk;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float vkp = V[k][p], vkq = V[k][q];
                V[k][p] = c * vkp - s * vkq;
                V[k][q] = s * vkp + c * vkq;
            }
        }
    }
    lam[0] = A[0][0]; lam[1] = A[1][1]; lam[2] = A[2][2];
}

// One side of a joint comparison.  Joint j of image b is  R_b . src[b][map[j]]  (map == null: j), minus R_b . src[b][0] when
// `center` is set (root / pelvis centring).  rot == null: no rotation.  `ld` = floats per image.
struct JointSide { const float* src; int ld; const int* map; int center; const float* rot; };

// grid ceil(B/64), block 64: thread = image.  N = evaluated joints (14, 17 or 24).
// MPJPE and Procrustes-aligned MPJPE (pare/SPIN compute_similarity_transform, one alignment per image) of the pred side
// against the gt side; optional per-joint distances before / after the alignment (reconstruction_error(reduction=None)),
// the pred joints as evaluated and both roots.
template <int N>
__global__ void __launch_bounds__(64)
eval_metrics_kernel(JointSide ps, JointSide gs, float* __restrict__ mpjpe, float* __restrict__ pampjpe,
                    float* __restrict__ mpjpe_pj, float* __restrict__ pampjpe_pj, float* __restrict__ pred_out,
                    float* __restrict__ pelvis_out /*[2][B][3]*/, int B)
{
    const int b = blockIdx.x * 64 + threadIdx.x;
    if (b >= B) return;
    float P[N][3], G[N][3];
    const float* pj = ps.src + static_cast<size_t>(b) * ps.ld;
    const float* gj = gs.src + static_cast<size_t>(b) * gs.ld;
    const float* pR = ps.rot ? ps.rot + static_cast<size_t>(b) * 9 : nullptr;
    const float* gR = gs.rot ? gs.rot + static_cast<size_t>(b) * 9 : nullptr;
    auto fetch = [](const float* x, const float* __restrict__ Rm, float o[3]) {
        if (Rm) {
            o[0] = Rm[0] * x[0] + Rm[1] * x[1] + Rm[2] * x[2];
            o[1] = Rm[3] * x[0] + Rm[4] * x[1] + Rm[5] * x[2];
            o[2] = Rm[6] * x[0] + Rm[7] * x[1] + Rm[8] * x[2];
        } else {
            o[0] = x[0]; o[1] = x[1]; o[2] = x[2];
        }
    };
    float pp[3] = {0.f, 0.f, 0.f}, gp[3] = {0.f, 0.f, 0.f};          // roots: pred pelvis = joint 0 (trainer.py:277)
    if (ps.center) fetch(pj, pR, pp);
    if (gs.center) fetch(gj, gR, gp);
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const int mp = ps.map ? ps.map[j] : j, mg = gs.map ? gs.map[j] : j;
        float x[3];
        fetch(pj + mp * 3, pR, x);
        if (ps.center) { P[j][0] = x[0] - pp[0]; P[j][1] = x[1] - pp[1]; P[j][2] = x[2] - pp[2]; }
        else { P[j][0] = x[0]; P[j][1] = x[1]; P[j][2] = x[2]; }
        fetch(gj + mg * 3, gR, x);
        if (gs.center) { G[j][0] = x[0] - gp[0]; G[j][1] = x[1] - gp[1]; G[j][2] = x[2] - gp[2]; }
        else { G[j][0] = x[0]; G[j][1] = x[1]; G[j][2] = x[2]; }
        if (pred_out) {
            float* o = pred_out + (static_cast<size_t>(b) * N + j) * 3;
            o[0] = P[j][0]; o[1] = P[j][1]; o[2] = P[j][2];
        }
    }
    if (pelvis_out) {
        pelvis_out[b * 3 + 0] = pp[0]; pelvis_out[b * 3 + 1] = pp[1]; pelvis_out[b * 3 + 2] = pp[2];
        pelvis_out[(static_cast<size_t>(B) + b) * 3 + 0] = gp[0]; pelvis_out[(static_cast<size_t>(B) + b) * 3 + 1] = gp[1];
        pelvis_out[(static_cast<size_t>(B) + b) * 3 + 2] = gp[2];
    }
    // MPJPE
    float e = 0.f;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const float dx = P[j][0] - G[j][0], dy = P[j][1] - G[j][1], dz = P[j][2] - G[j][2];
        const float d = sqrtf(dx * dx + dy * dy + dz * dz);
        if (mpjpe_pj) mpjpe_pj[static_cast<size_t>(b) * N + j] = d;
        e += d;
    }
    mpjpe[b] = e / static_cast<float>(N);
    // Procrustes (pare/SPIN compute_similarity_transform): align P (S1) to G (S2)
    float mu1[3] = {0.f, 0.f, 0.f}, mu2[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < N; ++j)
        for (int c = 0; c < 3; ++c) { mu1[c] += P[j][c]; mu2[c] += G[j][c]; }
    for (int c = 0; c < 3; ++c) { mu1[c] /= static_cast<float>(N); mu2[c] /= static_cast<float>(N); }
    float K[3][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    float var1 = 0.f;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        float x1[3], x2[3];
        for (int c = 0; c < 3; ++c) { x1[c] = P[j][c] - mu1[c]; x2[c] = G[j][c] - mu2[c]; var1 += x1[c] * x1[c]; }
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) K[r][c] = fmaf(x1[r], x2[c], K[r][c]);          // K = X1 X2^T
    }
    // K = U S V^T : eigen-decomposition of K^T K = V S^2 V^T
    float KtK[3][3], V[3][3], lam[3];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) KtK[r][c] = K[0][r] * K[0][c] + K[1][r] * K[1][c] + K[2][r] * K[2][c];
    jacobi_eig3(KtK, V, lam);
    int o0 = 0, o1 = 1, o2 = 2;                                   // sort descending
    if (lam[o0] < lam[o1]) { int t = o0; o0 = o1; o1 = t; }
    if (lam[o0] < lam[o2]) { int t = o0; o0 = o2; o2 = t; }
    if (lam[o1] < lam[o2]) { int t = o1; o1 = o2; o2 = t; }
    float v[3][3];                                                // columns v1,v2,v3 (as rows of v[])
    for (int k = 0; k < 3; ++k) { v[0][k] = V[k][o0]; v[1][k] = V[k][o1]; v[2][k] = V[k][o2]; }
    {   // keep det(V) = +1 after the permutation
        const float det = v[0][0] * (v[1][1] * v[2][2] - v[1][2] * v[2][1]) - v[0][1] * (v[1][0] * v[2][2] - v[1][2] * v[2][0]) +
                          v[0][2] * (v[1][0] * v[2][1] - v[1][1] * v[2][0]);
        if (det < 0.f) { v[2][0] = -v[2][0]; v[2][1] = -v[2][1]; v[2][2] = -v[2][2]; }
    }
    const float s1 = sqrtf(fmaxf(lam[o0], 0.f)), s2 = sqrtf(fmaxf(lam[o1], 0.f)), s3 = sqrtf(fmaxf(lam[o2], 0.f));
    float u1[3], u2[3], u3[3];
    for (int r = 0; r < 3; ++r) {
        u1[r] = (K[r][0] * v[0][0] + K[r][1] * v[0][1] + K[r][2] * v[0][2]) / fmaxf(s1, 1e-30f);
        u2[r] = (K[r][0] * v[1][0] + K[r][1] * v[1][1] + K[r][2] * v[1][2]) / fmaxf(s2, 1e-30f);
    }
    {   // re-orthonormalise u2 against u1 (fp32), u3 = u1 x u2
        const float n1 = rsqrtf(fmaxf(u1[0] * u1[0] + u1[1] * u1[1] + u1[2] * u1[2], 1e-30f));
        for (int r = 0; r < 3; ++r) u1[r] *= n1;
        const float d = u1[0] * u2[0] + u1[1] * u2[1] + u1[2] * u2[2];
        for (int r = 0; r < 3; ++r) u2[r] -= d * u1[r];
        const float n2 = rsqrtf(fmaxf(u2[0] * u2[0] + u2[1] * u2[1] + u2[2] * u2[2], 1e-30f));
        for (int r = 0; r < 3; ++r) u2[r] *= n2;
        u3[0] = u1[1] * u2[2] - u1[2] * u2[1]; u3[1] = u1[2] * u2[0] - u1[0] * u2[2]; u3[2] = u1[0] * u2[1] - u1[1] * u2[0];
    }
    // R = V Z U^T with Z = diag(1,1,sign det(U V^T)) == v1 u1^T + v2 u2^T + v3 (u1 x u2)^T ; trace(R K) = s1 + s2 + d s3
    float R[3][3];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r][c] = v[0][r] * u1[c] + v[1][r] * u2[c] + v[2][r] * u3[c];
    const float detK = K[0][0] * (K[1][1] * K[2][2] - K[1][2] * K[2][1]) - K[0][1] * (K[1][0] * K[2][2] - K[1][2] * K[2][0]) +
                       K[0][2] * (K[1][0] * K[2][1] - K[1][1] * K[2][0]);
    const float dsg = detK < 0.f ? -1.f : 1.f;
    const float scale = (s1 + s2 + dsg * s3) / fmaxf(var1, 1e-30f);
    float tr[3];
    for (int r = 0; r < 3; ++r) tr[r] = mu2[r] - scale * (R[r][0] * mu1[0] + R[r][1] * mu1[1] + R[r][2] * mu1[2]);
    float re = 0.f;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        float d2 = 0.f;
        for (int r = 0; r < 3; ++r) {
            const float h = scale * (R[r][0] * P[j][0] + R[r][1] * P[j][1] + R[r][2] * P[j][2]) + tr[r] - G[j][r];
            d2 += h * h;
        }
        const float d = sqrtf(d2);
        if (pampjpe_pj) pampjpe_pj[static_cast<size_t>(b) * N + j] = d;
        re += d;
    }
    pampjpe[b] = re / static_cast<float>(N);
}

// ------------------------------------------------------------------ per-vertex error (compute_error_verts): mean_v |p_v - g_v|
// rotp / rotg: optional per-image rotations [B][9] of each mesh, applied before the pelvis centring (compute_error.py:186-190);
// the pelvis is then that of the rotated mesh (the regression kernel rotated its joints).
__global__ void __launch_bounds__(256)
v2v_kernel(const float* __restrict__ pv, long long ldp, const float* __restrict__ rotp, const float* __restrict__ gv, long long ldg,
           const float* __restrict__ rotg, const float* __restrict__ pelvis /*[2][B][3] or null*/, float* __restrict__ out, int B)
{
    __shared__ float red[8];
    const int b = blockIdx.x;
    float ox = 0.f, oy = 0.f, oz = 0.f;
    if (pelvis) {       // (p - pelvis_p) - (g - pelvis_g)
        ox = pelvis[b * 3 + 0] - pelvis[(static_cast<size_t>(B) + b) * 3 + 0];
        oy = pelvis[b * 3 + 1] - pelvis[(static_cast<size_t>(B) + b) * 3 + 1];
        oz = pelvis[b * 3 + 2] - pelvis[(static_cast<size_t>(B) + b) * 3 + 2];
    }
    const float* p = pv + b * ldp;
    const float* g = gv + b * ldg;
    float acc = 0.f;
    if (rotp == nullptr && rotg == nullptr) {
        for (int v = threadIdx.x; v < SMPL_NV; v += 256) {
            const float dx = p[v * 3] - g[v * 3] - ox, dy = p[v * 3 + 1] - g[v * 3 + 1] - oy, dz = p[v * 3 + 2] - g[v * 3 + 2] - oz;
            acc += sqrtf(dx * dx + dy * dy + dz * dz);
        }
    } else {
        float Rp[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f}, Rg[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
        if (rotp) for (int i = 0; i < 9; ++i) Rp[i] = rotp[static_cast<size_t>(b) * 9 + i];
        if (rotg) for (int i = 0; i < 9; ++i) Rg[i] = rotg[static_cast<size_t>(b) * 9 + i];
        for (int v = threadIdx.x; v < SMPL_NV; v += 256) {
            const float px = p[v * 3], py = p[v * 3 + 1], pz = p[v * 3 + 2];
            const float gx = g[v * 3], gy = g[v * 3 + 1], gz = g[v * 3 + 2];
            const float dx = (Rp[0] * px + Rp[1] * py + Rp[2] * pz) - (Rg[0] * gx + Rg[1] * gy + Rg[2] * gz) - ox;
            const float dy = (Rp[3] * px + Rp[4] * py + Rp[5] * pz) - (Rg[3] * gx + Rg[4] * gy + Rg[5] * gz) - oy;
            const float dz = (Rp[6] * px + Rp[7] * py + Rp[8] * pz) - (Rg[6] * gx + Rg[7] * gy + Rg[8] * gz) - oz;
            acc += sqrtf(dx * dx + dy * dy + dz * dz);
        }
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int w = 0; w < 8; ++w) s += red[w];
        out[b] = s / static_cast<float>(SMPL_NV);
    }
}

template <int N>
static bool metrics_launch(const JointSide& ps, const JointSide& gs, float* mpjpe, float* pampjpe, float* mpjpe_pj, float* pampjpe_pj,
                           float* pred_out, float* pelvis_out, int B, cudaStream_t s) {
    eval_metrics_kernel<N><<<(B + 63) / 64, 64, 0, s>>>(ps, gs, mpjpe, pampjpe, mpjpe_pj, pampjpe_pj, pred_out, pelvis_out, B);
    return check_cuda(cudaGetLastError(), "eval_metrics");
}

bool eval_launch(const float* JT, const int* map, int n_map, int B, const float* pred_verts, long long ld_pred, const float* pred_rot,
                 const float* gt_kp, const float* gt_verts, long long ld_gt, const float* gt_rot, int center_v2v,
                 float* ws /*[2][B][51] + [2][B][3]*/, float* mpjpe, float* pampjpe, float* v2v, float* pred_kp, float* mpjpe_pj,
                 float* pampjpe_pj, cudaStream_t s) {
    float* j17 = ws;
    float* pelvis = ws + static_cast<size_t>(2) * B * 51;
    const bool regress_gt = (gt_kp == nullptr);
    if (regress_gt && gt_verts == nullptr) { set_error("eval: need gt keypoints or gt vertices"); return false; }
    if (n_map != 14 && n_map != 17) { set_error("eval: the joint mapper must have 14 or 17 entries"); return false; }
    dim3 grid(B, regress_gt ? 2 : 1);
    regress_joints_kernel<17, 20><<<grid, 256, 0, s>>>(pred_verts, ld_pred, pred_rot, gt_verts, ld_gt, gt_rot, JT, j17, B);
    if (!check_cuda(cudaGetLastError(), "h36m_joints")) return false;
    const JointSide ps{j17, 51, map, 1, nullptr};
    const JointSide gs = regress_gt ? JointSide{j17 + static_cast<size_t>(B) * 51, 51, map, 1, nullptr}
                                    : JointSide{gt_kp, n_map * 3, nullptr, 0, gt_rot};
    const bool ok = (n_map == 14) ? metrics_launch<14>(ps, gs, mpjpe, pampjpe, mpjpe_pj, pampjpe_pj, pred_kp, pelvis, B, s)
                                  : metrics_launch<17>(ps, gs, mpjpe, pampjpe, mpjpe_pj, pampjpe_pj, pred_kp, pelvis, B, s);
    if (!ok) return false;
    if (v2v != nullptr && gt_verts != nullptr) {
        v2v_kernel<<<B, 256, 0, s>>>(pred_verts, ld_pred, pred_rot, gt_verts, ld_gt, gt_rot, (center_v2v && regress_gt) ? pelvis : nullptr,
                                     v2v, B);
        if (!check_cuda(cudaGetLastError(), "v2v")) return false;
    }
    return true;
}

bool joint_errors_launch(int n, int B, const float* pred, const float* gt, const float* rot_pred, const float* rot_gt, int center,
                         float* mpjpe, float* pampjpe, float* mpjpe_pj, float* pampjpe_pj, cudaStream_t s) {
    const JointSide ps{pred, n * 3, nullptr, center, rot_pred}, gs{gt, n * 3, nullptr, center, rot_gt};
    switch (n) {
        case 14: return metrics_launch<14>(ps, gs, mpjpe, pampjpe, mpjpe_pj, pampjpe_pj, nullptr, nullptr, B, s);
        case 17: return metrics_launch<17>(ps, gs, mpjpe, pampjpe, mpjpe_pj, pampjpe_pj, nullptr, nullptr, B, s);
        case 24: return metrics_launch<24>(ps, gs, mpjpe, pampjpe, mpjpe_pj, pampjpe_pj, nullptr, nullptr, B, s);
        default: set_error("joint_errors: the joint count must be 14, 17 or 24"); return false;
    }
}

bool regress_joints24_launch(const float* JT24, int B, const float* verts, long long ld, const float* rot, float* out, cudaStream_t s) {
    regress_joints_kernel<24, 24><<<dim3(B, 1), 256, 0, s>>>(verts, ld, rot, nullptr, 0, nullptr, JT24, out, B);
    return check_cuda(cudaGetLastError(), "regress_joints24");
}

}  // namespace sb
