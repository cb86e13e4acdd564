// Internal (non-ABI) declarations shared by the .cu files of libspecb200.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <string>
#include <vector>

namespace sb {

enum Precision { PREC_F32 = 0, PREC_BF16 = 1, PREC_F16 = 2 };

// One convolution (+ folded-BN bias, + residual, + ReLU) over NHWC activations.
struct ConvParams {
    const void* in;      // [N,H,W,Cin]   (Cin dense)
    void* out;           // [N,Ho,Wo,*]   channel stride out_ld, channel offset out_coff
    const void* res;     // residual, same spatial/channel extent as the conv output; ld = res_ld; may be null
    const float* bias;   // [Cout]
    int N, H, W, Cin;
    int Ho, Wo, Cout;
    int kh, kw, stride, pad;
    int kwp;             // stem layout only: kw padded to a power of two (K index = (kh*kwp + kw)*4 + c)
    int K;               // GEMM K (kh*kw*Cin; kh*kwp*4 for the stem layout)
    int M;               // N*Ho*Wo
    int out_ld, out_coff, res_ld;
    int relu;
};

// Packed weights of one conv, owned by the trunk handle.
struct ConvWeights {
    int cout = 0, cin = 0, kh = 0, kw = 0;
    int K = 0, K_pad = 0, cout_pad = 0, block_n = 0;
    int kwp = 0;               // > 0: stem layout (Cin stored = 4, kw padded to kwp)
    bool stem7 = false;        // packed for conv_stem7_kernel: k = (c*7 + kh)*8 + kw, K = 168 -> 192
    void* w_tc = nullptr;      // [cout_pad][K_pad] 16-bit, K-major (tcgen05 path)
    float* w_f32 = nullptr;    // [K][cout] fp32 (SIMT parity path)
    float* bias = nullptr;     // [cout]
    std::vector<float> bias_host;   // same values on the host (kernels that take their biases as launch parameters)
    CUtensorMap tmap_b;        // TMA descriptor over w_tc (box 64 x block_n, 128B swizzle)
    bool has_tmap = false;
};

void set_error(const std::string& msg);

// NVTX range per stage of the path (SURVEY.md section 5): visible in nsys / ncu --nvtx timelines, a no-op (one
// predictable branch in the header-only NVTX3 stub) when no tool is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name);
    ~NvtxRange();
};

// cudaFuncSetAttribute is per DEVICE: remember per (function instantiation, device) whether the opt-in was done.
struct DeviceOnce {
    bool done[64] = {};
    bool need() {
        int dev = 0;
        cudaGetDevice(&dev);
        dev &= 63;
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};
bool check_cuda(cudaError_t e, const char* what);

// Launch with programmatic dependent launch allowed (common.cuh: griddep_launch / griddep_wait).  ONLY for kernels that execute
// griddep_wait() before they touch global activations; SPECB200_PDL=0 turns the attribute off (plain stream order).
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline void launch_dep(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    (void)cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);     // errors surface through cudaGetLastError at the call site
}

// tcgen05 implicit-GEMM conv (conv_tc.cu).  prec is PREC_BF16 or PREC_F16.
bool conv_tc_launch(const ConvParams& p, const ConvWeights& w, int prec, cudaStream_t s);
bool conv_tc_make_weight_tmap(ConvWeights& w);
int conv_tc_pick_block_n(int cout, int K);

// 3x3/1 conv with on-chip halo reuse (conv_halo.cu)
bool conv_halo_applicable(const ConvParams& p, const ConvWeights& w);
bool conv_halo_launch(const ConvParams& p, const ConvWeights& w, int prec, cudaStream_t s);

// 4-D tiled TMA descriptor over an NHWC 16-bit tensor: box = 64 channels x box_w x box_h x 1, 128-byte swizzle (conv_halo.cu)
bool make_tmap_nhwc(CUtensorMap* m, const void* ptr, int C_ld, int W, int H, int N, int box_w, int box_h);
// same tensor, box = box_c channels x box_w x box_h x 1 WITHOUT swizzle (dense rows of box_c * 2 bytes in shared memory)
bool make_tmap_nhwc_plain(CUtensorMap* m, const void* ptr, int C_ld, int W, int H, int N, int box_c, int box_w, int box_h);

// 2-D 16-bit K-major matrix [rows][ld] (ld elements per row): box = 64 columns x box_rows rows, 128-byte swizzle (conv_tc.cu)
bool make_tmap_2d_k64(CUtensorMap* m, const void* ptr, int rows, int ld, int box_rows);

// whole 64-channel bottleneck in one launch (conv_bneck.cu): y = relu(conv3(relu(conv2(relu(conv1(x))))) + (wd ? wd(x) : x))
struct BottleneckArgs {
    const void* x = nullptr;      // NHWC [N][H][W][Cin], Cin = 256 (identity residual) or 64 (with downsample conv wd)
    void* out = nullptr;          // NHWC [N][H][W][256]
    int N = 0, H = 0, W = 0, Cin = 0;
    const ConvWeights *w1 = nullptr, *w2 = nullptr, *w3 = nullptr, *wd = nullptr;
};
bool bottleneck_applicable(const BottleneckArgs& a);
bool bottleneck_launch(const BottleneckArgs& a, int prec, cudaStream_t s);

// dedicated 7x7/2 stem (conv_stem.cu): reads the fp32 NCHW image directly, writes NHWC 16-bit [N,Ho,Wo,64]
bool conv_stem7_launch(const float* img, void* out, const ConvWeights& w, int N, int H, int W, int Ho, int Wo, int prec,
                       cudaStream_t s);

// fp32 SIMT implicit-GEMM conv and linear (conv_simt.cu).
bool conv_f32_launch(const ConvParams& p, const ConvWeights& w, cudaStream_t s);
// out[M, n0:n0+N] (ld out_ld) = A[M,K](ld lda) @ W[N,K]^T (ld ldw) + bias[N] + add[M,N](ld add_ld) ; fp32
// ksplit > 1: split-K partial sums, slice z written to out + z*split_stride (consumer adds them in order); the number of slices
// actually written is returned in *ksplit_used (<= ksplit) -- the consumer must sum exactly that many.
// red != nullptr (and split_stride == 0): the launch picks its own split-K factor and reduces inside the kernel, in a fixed
// order, through this scratch: `partial` needs no initialisation, `counters` must be zero before the first launch (the kernel
// leaves them zero) and must not be shared by launches that can run concurrently.
struct LinearRedWs { float* partial; size_t partial_floats; unsigned* counters; int n_counters; };
bool linear_f32_launch(const float* A, int lda, const float* W, int ldw, const float* bias, const float* add,
                       int add_ld, float* out, int out_ld, int M, int N, int K, cudaStream_t s, int ksplit = 1,
                       size_t split_stride = 0, int* ksplit_used = nullptr, const LinearRedWs* red = nullptr);

// eval-side metrics (eval.cu)
// n_map = 14 or 17 entries of `map` (into the 17 H36M joints); pred_rot / gt_rot: optional [B][9] rotations of the meshes.
bool eval_launch(const float* JT, const int* map, int n_map, int B, const float* pred_verts, long long ld_pred, const float* pred_rot,
                 const float* gt_kp, const float* gt_verts, long long ld_gt, const float* gt_rot, int center_v2v, float* ws,
                 float* mpjpe, float* pampjpe, float* v2v, float* pred_kp, float* mpjpe_pj, float* pampjpe_pj, cudaStream_t s);
// MPJPE / PA-MPJPE of already-regressed joints [B][n][3] (n = 14, 17 or 24); center = subtract joint 0 on both sides
bool joint_errors_launch(int n, int B, const float* pred, const float* gt, const float* rot_pred, const float* rot_gt, int center,
                         float* mpjpe, float* pampjpe, float* mpjpe_pj, float* pampjpe_pj, cudaStream_t s);
// out [B][24][3] = rot . (J_regressor . verts); JT24 is the SMPL J_regressor transposed, [6890][24]; rot may be null
bool regress_joints24_launch(const float* JT24, int B, const float* verts, long long ld, const float* rot, float* out, cudaStream_t s);

// elementwise / layout kernels (elementwise.cu)
bool images_to_nhwc_launch(const float* img_nchw, void* out_nhwc, int N, int H, int W, int cpad, int prec, cudaStream_t s);
// nonneg_input: the source tensor is the output of a conv + ReLU (enables the TMA-tiled kernel, whose zero-filled borders act as padding)
bool maxpool3x3s2_launch(const void* in, void* out, int N, int H, int W, int C, int Ho, int Wo, int prec, cudaStream_t s,
                         bool nonneg_input = false);
bool upsample_add_launch(const void* lo, void* acc, int N, int Ho, int Wo, int C, int shift, int relu, int prec, cudaStream_t s);
bool bilinear_launch(const void* in, void* out, int N, int H, int W, int C, int Ho, int Wo, int out_ld, int out_coff,
                     int prec, cudaStream_t s);
bool copy_channels_launch(const void* in, void* out, int rows, int C, int out_ld, int out_coff, int prec, cudaStream_t s);
bool avgpool_launch(const void* in, float* out, int out_ld, int N, int HW, int C, int prec, cudaStream_t s);
bool nhwc_to_nchw_f32_launch(const void* in, float* out, int N, int H, int W, int C, int prec, cudaStream_t s);

}  // namespace sb
