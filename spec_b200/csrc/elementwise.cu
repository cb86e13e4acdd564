// Layout / elementwise kernels around the convolutions (all NHWC, 16-byte vectorised):
// image NCHW fp32 -> NHWC, 3x3/2 max-pool (ResNet stem), HRNet fuse (nearest-upsample + add),
// bilinear resize (hrnet-interp tail), channel-slice copy (concat), global average pool, NHWC->NCHW export.
// Reference ops replaced: ATen max_pool2d / adaptive_avg_pool2d / upsample / cat (SURVEY.md section 2.2).
#include "common.cuh"
#include "internal.h"
#include <stdlib.h>

namespace sb {

template <typename T> struct V16;           // 16-byte vector of T
template <> struct V16<float> {
    static constexpr int N = 4;
    __device__ static void load(const float* p, float (&f)[4]) { float4 v = *reinterpret_cast<const float4*>(p); f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w; }
    __device__ static void store(float* p, const float (&f)[4]) { *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]); }
};
template <typename T> struct V16 {
    static constexpr int N = 8;
    __device__ static void load(const T* p, float (&f)[8]) {
        uint4 v = *reinterpret_cast<const uint4*>(p);
        const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) { float2 t = DT<T>::unpack2(u[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
    }
    __device__ static void store(T* p, const float (&f)[8]) {
        uint4 v;
        v.x = DT<T>::pack2(f[0], f[1]); v.y = DT<T>::pack2(f[2], f[3]);
        v.z = DT<T>::pack2(f[4], f[5]); v.w = DT<T>::pack2(f[6], f[7]);
        *reinterpret_cast<uint4*>(p) = v;
    }
};

#define SB_DISPATCH_PREC(prec, ...)                                                    \
    do {                                                                               \
        if ((prec) == PREC_F32) { using T = float; __VA_ARGS__; }                      \
        else if ((prec) == PREC_BF16) { using T = __nv_bfloat16; __VA_ARGS__; }        \
        else if ((prec) == PREC_F16) { using T = __half; __VA_ARGS__; }                \
        else { set_error("bad precision"); return false; }                             \
    } while (0)

static inline unsigned nblk(long long n, int t) { return static_cast<unsigned>((n + t - 1) / t); }

// ------------------------------------------------------------------ images NCHW f32 -> NHWC(cpad)
template <typename T>
__global__ void images_to_nhwc_kernel(const float* __restrict__ img, T* __restrict__ out, long long npix, int HW) {
    griddep_launch();
    griddep_wait();
    // NHWC with 4 channels (RGB + one zero): 16 B / pixel in fp32, 8 B / pixel in the 16-bit modes
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    const long long n = i / HW;
    const int hw = static_cast<int>(i - n * HW);
    const float* src = img + n * 3 * HW + hw;
    const float r = src[0], g = src[HW], b = src[2 * static_cast<size_t>(HW)];
    if constexpr (sizeof(T) == 4) {
        *reinterpret_cast<float4*>(out + i * 4) = make_float4(r, g, b, 0.f);
    } else {
        uint2 v;
        v.x = DT<T>::pack2(r, g);
        v.y = DT<T>::pack2(b, 0.f);
        *reinterpret_cast<uint2*>(out + i * 4) = v;
    }
}
bool images_to_nhwc_launch(const float* img, void* out, int N, int H, int W, int cpad, int prec, cudaStream_t s) {
    const long long npix = static_cast<long long>(N) * H * W;
    if (cpad != 4) { set_error("images_to_nhwc: the image buffer must have 4 channels"); return false; }
    SB_DISPATCH_PREC(prec, (launch_dep(images_to_nhwc_kernel<T>, dim3(nblk(npix, 256)), dim3(256), 0, s, img, static_cast<T*>(out), npix, H * W)));
    return check_cuda(cudaGetLastError(), "images_to_nhwc");
}

// ------------------------------------------------------------------ maxpool 3x3 s2 p1
template <typename T>
__global__ void maxpool_kernel(const T* __restrict__ in, T* __restrict__ out, int N, int H, int W, int C, int Ho, int Wo) {
    constexpr int V = V16<T>::N;
    const int cv = C / V;
    const long long total = static_cast<long long>(N) * Ho * Wo * cv;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = static_cast<int>(i % cv) * V;
    long long t = i / cv;
    const int ow = static_cast<int>(t % Wo); t /= Wo;
    const int oh = static_cast<int>(t % Ho);
    const long long n = t / Ho;
    float m[V];
#pragma unroll
    for (int e = 0; e < V; ++e) m[e] = -INFINITY;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
        const int ih = oh * 2 - 1 + dy;
        if (ih < 0 || ih >= H) continue;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
            const int iw = ow * 2 - 1 + dx;
            if (iw < 0 || iw >= W) continue;
            float f[V];
            V16<T>::load(in + ((n * H + ih) * W + iw) * C + c, f);
#pragma unroll
            for (int e = 0; e < V; ++e) m[e] = fmaxf(m[e], f[e]);
        }
    }
    V16<T>::store(out + ((n * Ho + oh) * Wo + ow) * C + c, m);
}
// (A column-strip variant -- one thread walks down the rows carrying the horizontal 3-max, 6 instead of 9 reads per
// output -- was measured SLOWER, 0.21 vs 0.14 ms at B=256: the serial row walk costs more latency than the re-reads.)

// (Two horizontally adjacent outputs per thread -- a 3x5 window read once, 15 loads for two outputs instead of 18 -- was
// also measured SLOWER, 0.162 vs 0.139 ms: half the threads, less latency hiding.)
// TMA-tiled variant for the ResNet stem (C = 64, 16-bit, NON-NEGATIVE input = the output of a conv + ReLU): the kernel above re-reads
// every input pixel up to nine times through L1 (0.137 ms at B=256 = 0.56 of the HBM roofline).  Here a persistent CTA per SM
// pulls the 17 x 33-pixel input patch of an 8 x 16 output tile into shared memory with ONE 4-D TMA box (72 KB, 128B-swizzled rows
// of 64 channels; out-of-image pixels are zero-filled, which equals max-pool's -inf padding BECAUSE the values are >= 0 and every
// window holds a real pixel), double-buffered one tile ahead; 256 threads take the 3x3 maxima from shared memory (16-byte chunk
// per thread: eight threads per pixel, conflict-free) into a swizzled staging tile that leaves through one TMA store.
constexpr int MP_TH = 8, MP_TW = 16;
constexpr int MP_PH = 2 * MP_TH + 1, MP_PW = 2 * MP_TW + 1;          // 17 x 33 input pixels
constexpr int MP_PATCH_TX = MP_PH * MP_PW * 128;                     // 71808
constexpr int MP_PATCH_BYTES = (MP_PATCH_TX + 1023) / 1024 * 1024;   // 72704
constexpr int MP_ST_BYTES = MP_TH * MP_TW * 128;                     // 16384
constexpr int MP_DYN_BYTES = 2 * MP_PATCH_BYTES + 2 * MP_ST_BYTES + 64 + 1024;

template <typename T>
__global__ void __launch_bounds__(256, 1)
maxpool_tma_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_out, int tiles_w, int tiles_h,
                   int total_tiles)
{
    griddep_launch();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t patch_s = sbase, st_s = sbase + 2 * MP_PATCH_BYTES, bar_full = st_s + 2 * MP_ST_BYTES;
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar_full, 1); mbar_init(bar_full + 8, 1);
        mbar_fence_init();
        tma_prefetch_desc(&tmap_in); tma_prefetch_desc(&tmap_out);
    }
    __syncthreads();
    griddep_wait();
    auto issue = [&](int tile, uint32_t b) {
        const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, n = tile / (tiles_w * tiles_h);
        mbar_arrive_expect_tx(bar_full + b * 8, MP_PATCH_TX);
        tma_load_4d(patch_s + b * MP_PATCH_BYTES, &tmap_in, bar_full + b * 8, 0, 2 * tw * MP_TW - 1, 2 * th * MP_TH - 1, n);
    };
    if (tid == 0 && static_cast<int>(blockIdx.x) < total_tiles) issue(blockIdx.x, 0);
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const uint32_t b = it & 1, ph = (it >> 1) & 1;
        if (tid == 0) {
            if (tile + static_cast<int>(gridDim.x) < total_tiles) issue(tile + gridDim.x, b ^ 1);   // buffer b^1 was released by the barrier below
            tma_store_wait_read<1>();                                   // the store of tile it-2 has read staging[b]
        }
        mbar_wait(bar_full + b * 8, ph);
        __syncthreads();                                                // staging[b] is free for everybody
        const uint32_t patch = patch_s + b * MP_PATCH_BYTES, st = st_s + b * MP_ST_BYTES;
#pragma unroll
        for (int rep = 0; rep < 4; ++rep) {
            const int item = tid + rep * 256;
            const int p = item >> 3, k = item & 7;                      // output pixel of the tile, 16-byte channel chunk
            const int pr = p >> 4, pc = p & 15;
            uint32_t m[4] = {0u, 0u, 0u, 0u};                           // +0.0: the identity for non-negative inputs
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const uint32_t R = static_cast<uint32_t>((2 * pr + dy) * MP_PW + 2 * pc + dx);
                    uint32_t v[4];
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
                                 : "r"(patch + R * 128u + ((static_cast<uint32_t>(k) ^ (R & 7u)) << 4)));
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if constexpr (sizeof(T) == 2 && DT<T>::umma_fmt == 1) {
                            __nv_bfloat162 r2 = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&m[e]), *reinterpret_cast<__nv_bfloat162*>(&v[e]));
                            m[e] = *reinterpret_cast<uint32_t*>(&r2);
                        } else {
                            __half2 r2 = __hmax2(*reinterpret_cast<__half2*>(&m[e]), *reinterpret_cast<__half2*>(&v[e]));
                            m[e] = *reinterpret_cast<uint32_t*>(&r2);
                        }
                    }
                }
            asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(st + static_cast<uint32_t>(p) * 128u + ((static_cast<uint32_t>(k) ^ (static_cast<uint32_t>(p) & 7u)) << 4)),
                         "r"(m[0]), "r"(m[1]), "r"(m[2]), "r"(m[3]) : "memory");
        }
        fence_proxy_async_smem();
        __syncthreads();                                                // staging[b] complete; patch[b] no longer read
        if (tid == 0) {
            const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, n = tile / (tiles_w * tiles_h);
            tma_store_4d(&tmap_out, st, 0, tw * MP_TW, th * MP_TH, n);
            tma_store_commit();
        }
    }
    if (tid == 0) tma_store_wait_read0();
}

bool maxpool3x3s2_launch(const void* in, void* out, int N, int H, int W, int C, int Ho, int Wo, int prec, cudaStream_t s, bool nonneg_input) {
    if (nonneg_input && C == 64 && prec != PREC_F32 && H >= MP_PH && W >= MP_PW) {
        CUtensorMap tin, tout;
        if (!make_tmap_nhwc(&tin, in, 64, W, H, N, MP_PW, MP_PH)) return false;
        if (!make_tmap_nhwc(&tout, out, 64, Wo, Ho, N, MP_TW, MP_TH)) return false;
        static DeviceOnce attr;
        if (attr.need()) {
            if (!check_cuda(cudaFuncSetAttribute(maxpool_tma_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, MP_DYN_BYTES), "maxpool attr")) return false;
            if (!check_cuda(cudaFuncSetAttribute(maxpool_tma_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, MP_DYN_BYTES), "maxpool attr")) return false;
        }
        static int num_sms = 0;
        if (num_sms == 0) {
            int dev = 0;
            cudaGetDevice(&dev);
            if (!check_cuda(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev), "sm count")) return false;
        }
        const int tiles_w = (Wo + MP_TW - 1) / MP_TW, tiles_h = (Ho + MP_TH - 1) / MP_TH;
        const long long total = static_cast<long long>(N) * tiles_w * tiles_h;
        if (total > 0x7fffffffLL) { set_error("maxpool: too many tiles"); return false; }
        const unsigned grid = static_cast<unsigned>(total < num_sms ? total : num_sms);
        if (prec == PREC_BF16) launch_dep(maxpool_tma_kernel<__nv_bfloat16>, dim3(grid), dim3(256), MP_DYN_BYTES, s, tin, tout, tiles_w, tiles_h, static_cast<int>(total));
        else launch_dep(maxpool_tma_kernel<__half>, dim3(grid), dim3(256), MP_DYN_BYTES, s, tin, tout, tiles_w, tiles_h, static_cast<int>(total));
        return check_cuda(cudaGetLastError(), "maxpool (tma)");
    }
    SB_DISPATCH_PREC(prec, {
        const long long total = static_cast<long long>(N) * Ho * Wo * (C / V16<T>::N);
        maxpool_kernel<T><<<nblk(total, 256), 256, 0, s>>>(static_cast<const T*>(in), static_cast<T*>(out), N, H, W, C, Ho, Wo);
    });
    return check_cuda(cudaGetLastError(), "maxpool");
}

// ------------------------------------------------------------------ acc += nearest_upsample(lo, 2^shift) [; relu]
template <typename T>
__global__ void upsample_add_kernel(const T* __restrict__ lo, T* __restrict__ acc, int N, int Ho, int Wo, int C, int shift, int relu) {
    griddep_launch();
    griddep_wait();
    constexpr int V = V16<T>::N;
    const int cv = C / V;
    const long long total = static_cast<long long>(N) * Ho * Wo * cv;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = static_cast<int>(i % cv) * V;
    long long t = i / cv;
    const int ow = static_cast<int>(t % Wo); t /= Wo;
    const int oh = static_cast<int>(t % Ho);
    const long long n = t / Ho;
    const int Hl = Ho >> shift, Wl = Wo >> shift;
    float a[V], b[V];
    T* ap = acc + ((n * Ho + oh) * Wo + ow) * C + c;
    V16<T>::load(ap, a);
    V16<T>::load(lo + ((n * Hl + (oh >> shift)) * Wl + (ow >> shift)) * C + c, b);
#pragma unroll
    for (int e = 0; e < V; ++e) { a[e] += b[e]; if (relu) a[e] = fmaxf(a[e], 0.f); }
    V16<T>::store(ap, a);
}
bool upsample_add_launch(const void* lo, void* acc, int N, int Ho, int Wo, int C, int shift, int relu, int prec, cudaStream_t s) {
    SB_DISPATCH_PREC(prec, {
        const long long total = static_cast<long long>(N) * Ho * Wo * (C / V16<T>::N);
        launch_dep(upsample_add_kernel<T>, dim3(nblk(total, 256)), dim3(256), 0, s, static_cast<const T*>(lo), static_cast<T*>(acc), N, Ho, Wo, C, shift, relu);
    });
    return check_cuda(cudaGetLastError(), "upsample_add");
}

// ------------------------------------------------------------------ bilinear (align_corners=True) into a concat slice
template <typename T>
__global__ void bilinear_kernel(const T* __restrict__ in, T* __restrict__ out, int N, int H, int W, int C, int Ho, int Wo,
                                int out_ld, int out_coff) {
    griddep_launch();
    griddep_wait();
    constexpr int V = V16<T>::N;
    const int cv = C / V;
    const long long total = static_cast<long long>(N) * Ho * Wo * cv;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = static_cast<int>(i % cv) * V;
    long long t = i / cv;
    const int ow = static_cast<int>(t % Wo); t /= Wo;
    const int oh = static_cast<int>(t % Ho);
    const long long n = t / Ho;
    const float sy = Ho > 1 ? static_cast<float>(H - 1) / static_cast<float>(Ho - 1) : 0.f;
    const float sx = Wo > 1 ? static_cast<float>(W - 1) / static_cast<float>(Wo - 1) : 0.f;
    const float fy = sy * oh, fx = sx * ow;
    const int y0 = static_cast<int>(fy), x0 = static_cast<int>(fx);
    const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
    const float ly = fy - y0, lx = fx - x0;
    float a[V], b[V], cc[V], d[V], o[V];
    const T* base = in + n * H * W * C + c;
    V16<T>::load(base + (static_cast<size_t>(y0) * W + x0) * C, a);
    V16<T>::load(base + (static_cast<size_t>(y0) * W + x1) * C, b);
    V16<T>::load(base + (static_cast<size_t>(y1) * W + x0) * C, cc);
    V16<T>::load(base + (static_cast<size_t>(y1) * W + x1) * C, d);
#pragma unroll
    for (int e = 0; e < V; ++e)
        o[e] = (1.f - ly) * ((1.f - lx) * a[e] + lx * b[e]) + ly * ((1.f - lx) * cc[e] + lx * d[e]);
    V16<T>::store(out + ((n * Ho + oh) * Wo + ow) * out_ld + out_coff + c, o);
}
bool bilinear_launch(const void* in, void* out, int N, int H, int W, int C, int Ho, int Wo, int out_ld, int out_coff,
                     int prec, cudaStream_t s) {
    SB_DISPATCH_PREC(prec, {
        const long long total = static_cast<long long>(N) * Ho * Wo * (C / V16<T>::N);
        launch_dep(bilinear_kernel<T>, dim3(nblk(total, 256)), dim3(256), 0, s, static_cast<const T*>(in), static_cast<T*>(out), N, H, W, C, Ho, Wo, out_ld, out_coff);
    });
    return check_cuda(cudaGetLastError(), "bilinear");
}

// ------------------------------------------------------------------ copy [rows, C] into a channel slice
template <typename T>
__global__ void copy_channels_kernel(const T* __restrict__ in, T* __restrict__ out, long long rows, int C, int out_ld, int out_coff) {
    griddep_launch();
    griddep_wait();
    constexpr int V = V16<T>::N;
    const int cv = C / V;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= rows * cv) return;
    const int c = static_cast<int>(i % cv) * V;
    const long long r = i / cv;
    *reinterpret_cast<uint4*>(out + r * out_ld + out_coff + c) = *reinterpret_cast<const uint4*>(in + r * C + c);
}
bool copy_channels_launch(const void* in, void* out, int rows, int C, int out_ld, int out_coff, int prec, cudaStream_t s) {
    SB_DISPATCH_PREC(prec, {
        const long long total = static_cast<long long>(rows) * (C / V16<T>::N);
        launch_dep(copy_channels_kernel<T>, dim3(nblk(total, 256)), dim3(256), 0, s, static_cast<const T*>(in), static_cast<T*>(out), rows, C, out_ld, out_coff);
    });
    return check_cuda(cudaGetLastError(), "copy_channels");
}

// ------------------------------------------------------------------ global average pool -> fp32 [N][out_ld]
template <typename T>
__global__ void avgpool_kernel(const T* __restrict__ in, float* __restrict__ out, int out_ld, int N, int HW, int C) {
    griddep_launch();
    griddep_wait();
    constexpr int V = V16<T>::N;
    const int cv = C / V;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(N) * cv) return;
    const int c = static_cast<int>(i % cv) * V;
    const long long n = i / cv;
    float acc[V];
#pragma unroll
    for (int e = 0; e < V; ++e) acc[e] = 0.f;
    const T* p = in + n * HW * C + c;
    for (int h = 0; h < HW; ++h) {
        float f[V];
        V16<T>::load(p + static_cast<size_t>(h) * C, f);
#pragma unroll
        for (int e = 0; e < V; ++e) acc[e] += f[e];
    }
    const float inv = 1.f / static_cast<float>(HW);
#pragma unroll
    for (int e = 0; e < V; ++e) out[n * out_ld + c + e] = acc[e] * inv;
}
bool avgpool_launch(const void* in, float* out, int out_ld, int N, int HW, int C, int prec, cudaStream_t s) {
    SB_DISPATCH_PREC(prec, {
        const long long total = static_cast<long long>(N) * (C / V16<T>::N);
        launch_dep(avgpool_kernel<T>, dim3(nblk(total, 128)), dim3(128), 0, s, static_cast<const T*>(in), out, out_ld, N, HW, C);
    });
    return check_cuda(cudaGetLastError(), "avgpool");
}

// ------------------------------------------------------------------ NHWC -> NCHW fp32 (backbone-only API)
template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ in, float* __restrict__ out, int N, int HW, int C) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(N) * HW * C) return;
    const int hw = static_cast<int>(i % HW);
    const long long t = i / HW;
    const int c = static_cast<int>(t % C);
    const long long n = t / C;
    out[i] = DT<T>::to_f(in[(n * HW + hw) * C + c]);
}
bool nhwc_to_nchw_f32_launch(const void* in, float* out, int N, int H, int W, int C, int prec, cudaStream_t s) {
    SB_DISPATCH_PREC(prec, {
        const long long total = static_cast<long long>(N) * H * W * C;
        nhwc_to_nchw_kernel<T><<<nblk(total, 256), 256, 0, s>>>(static_cast<const T*>(in), out, N, H * W, C);
    });
    return check_cuda(cudaGetLastError(), "nhwc_to_nchw");
}

}  // namespace sb
