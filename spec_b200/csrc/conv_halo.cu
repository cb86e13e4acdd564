// 3x3 / stride 1 / pad 1 convolution with ON-CHIP HALO REUSE (tcgen05 + TMA), Cin = Cout = 64.
//
// The implicit-GEMM kernels in conv_tc.cu re-load the activation tile once per filter tap (9x the L2->smem traffic
// and 9x the smem write bandwidth for A).  Here one haloed input tile is loaded ONCE and the nine taps are fed to the
// tensor core as ROW-SHIFTED VIEWS of it:
//   output tile = 8 rows x 14 cols of one image, laid on a padded grid of pitch 16:  q = r*16 + c  (128 GEMM rows,
//   the 2 x 8 positions with c >= 14 are scratch);  input patch = 10 x 16 pixels (one 4-D TMA box, out-of-image parts
//   zero-filled = the conv padding) stored [160 pixels][64 ch] = 128-byte rows, 128B-swizzled;  tap (kh,kw) of output
//   q reads patch row q + kh*16 + kw, i.e. the A operand of that tap is the SAME smem buffer with the UMMA descriptor's
//   start address advanced by (kh*16+kw)*128 bytes.  The 128B swizzle is a function of the absolute smem address, so a
//   start that is not 8-row aligned still addresses the right bytes (verified on B200 by tools/umma_shift_test.cu,
//   base_offset field = 0).
// Weights: [Cout][9*Cin] K-major as everywhere (k = tap*Cin + c); the whole 72 KB tensor stays resident in smem for
// the life of the persistent CTA.
// Persistent, warp-specialised like conv_tcp_kernel: warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM owner,
// warps 4-11 epilogue (double-buffered TMEM accumulator and staging tile, residual TMA-prefetched, TMA store of a
// dense [TH][TW][64ch] box so image borders are clipped by the hardware).
//
// Users: ResNet layer1, HRNet's 64-channel branches and its 32-channel branches, which api.cu views pixel-paired as
// 64 -> 64 convs.  Measured (B=256): 1.4x faster than the im2col path (0.142 -> 0.100 ms per layer1 conv).  Convs with
// 128/256 channels stay on the im2col kernels: there the weights no longer fit beside the patch ring, and with them
// streamed the 76-88 % tile efficiency (14/16 columns, 8-row tiles on 14/28-row images) and the single resident CTA's
// shallower weight ring lost to conv_tc.cu.
#include "common.cuh"
#include "internal.h"

namespace sb {

// Tile geometry (TH output rows x TW = PW-2 output cols on a padded grid of pitch PW, TH*PW = 128 GEMM rows):
//   G = 0:  8 x 14 (pitch 16)  -- narrow maps (W = 14)          G = 1:  4 x 30 (pitch 32)  -- W >= 28 (93.75 % of the rows useful)
template <int G> struct HaloGeom;
template <> struct HaloGeom<0> { static constexpr int TH = 8, PW = 16; };
template <> struct HaloGeom<1> { static constexpr int TH = 4, PW = 32; };
template <int G> struct HaloDims {
    static constexpr int TH = HaloGeom<G>::TH, PW = HaloGeom<G>::PW, TW = PW - 2;
    static constexpr int PATCH_ROWS = (TH + 2) * PW;               // pixels loaded per tile
    static constexpr int PATCH_TX = PATCH_ROWS * 128;              // bytes per TMA load
    static constexpr int PATCH_BYTES = ((128 + 2 * PW + 2) * 128 + 1023) / 1024 * 1024;   // slot: taps read up to row 127 + 2*PW + 2
    static constexpr int PW_SHIFT = (PW == 16) ? 4 : 5;
};
constexpr int HL_THREADS = 384;
constexpr int HL_C = 64;                                   // Cin = Cout

template <int G>
struct HaloSmem {
    static constexpr int PA = 4;                            // patch ring depth
    static constexpr int B_SLOT = HL_C * 128;               // one tap's [64 Cout][64 Cin] weight tile
    static constexpr int EPI_BYTES = 128 * HL_C * 2;        // staging box of 128 rows x 128 B (TH*TW rows used)
    static constexpr int A_OFF = 0;
    static constexpr int B_OFF = PA * HaloDims<G>::PATCH_BYTES;
    static constexpr int EPI_OFF = B_OFF + 9 * B_SLOT;
    static constexpr int BAR_OFF = EPI_OFF + 2 * EPI_BYTES;  // a_full[PA] a_empty[PA] b_full tfull[2] tempty[2] rfull[2]
    static constexpr int NBAR = 2 * PA + 7;
    static constexpr int TMEMPTR_OFF = BAR_OFF + NBAR * 8;
    static constexpr int BIAS_OFF = (TMEMPTR_OFF + 8 + 15) / 16 * 16;
    static constexpr int TOTAL = BIAS_OFF + HL_C * 4;
    static constexpr int DYN_BYTES = TOTAL + 1024;
    static_assert(DYN_BYTES <= 232448, "exceeds the 227 KB dynamic shared memory limit");
    static_assert((B_OFF % 1024) == 0 && (EPI_OFF % 1024) == 0, "swizzled tiles must be 1024-byte aligned");
};

struct HaloMaps {
    CUtensorMap a;      // input  (C, W, H, N)        box {64, 16, 10, 1}
    CUtensorMap b;      // weights [Cout][9*Cin]      box {64, 64}
    CUtensorMap out;    // output (out_ld, Wo, Ho, N) box {64, 14, 8, 1}
    CUtensorMap res;    // residual, same box
};

template <typename T, int G>
__global__ void __launch_bounds__(HL_THREADS, 1)
conv3x3_halo_kernel(const ConvParams p, const __grid_constant__ HaloMaps maps, int tiles_w, int tiles_h, int total_tiles)
{
    griddep_launch();
    using L = HaloSmem<G>;
    using D = HaloDims<G>;
    constexpr int PA = L::PA;
    constexpr int HL_TH = D::TH, HL_TW = D::TW, HL_PW = D::PW, HL_PATCH_TX = D::PATCH_TX, HL_PATCH_BYTES = D::PATCH_BYTES;
    constexpr int TMEM_COLS = 2 * HL_C;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
    const uint32_t a_base = sbase + L::A_OFF, b_base = sbase + L::B_OFF, e_base = sbase + L::EPI_OFF;
    const uint32_t bar_afull = sbase + L::BAR_OFF, bar_aempty = bar_afull + PA * 8, bar_bfull = bar_aempty + PA * 8;
    const uint32_t bar_tfull = bar_bfull + 8, bar_tempty = bar_tfull + 16, bar_rfull = bar_tempty + 16;
    volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(sgen + L::TMEMPTR_OFF);
    float* sbias = reinterpret_cast<float*>(sgen + L::BIAS_OFF);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool has_res = p.res != nullptr;

    if (threadIdx.x == 0) {
        for (int s = 0; s < PA; ++s) { mbar_init(bar_afull + s * 8, 1); mbar_init(bar_aempty + s * 8, 1); }
        mbar_init(bar_bfull, 1);
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + a * 8, 1); mbar_init(bar_tempty + a * 8, 8); mbar_init(bar_rfull + a * 8, 1); }
        mbar_fence_init();
    }
    if (threadIdx.x < HL_C) sbias[threadIdx.x] = p.bias[threadIdx.x];
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a); tma_prefetch_desc(&maps.b); tma_prefetch_desc(&maps.out);
        if (has_res) tma_prefetch_desc(&maps.res);
    }
    if (warp == 2) { tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_s)), TMEM_COLS); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    griddep_wait();
    const uint32_t tmem_base = *tmem_ptr_s;

    auto decode = [&](int tile, int& n, int& oh0, int& ow0) {
        const int tw = tile % tiles_w;
        const int th = (tile / tiles_w) % tiles_h;
        n = tile / (tiles_w * tiles_h);
        oh0 = th * HL_TH; ow0 = tw * HL_TW;
    };

    if (warp == 0) {
        // ================= TMA producer
        if (lane == 0) {
            mbar_arrive_expect_tx(bar_bfull, 9 * L::B_SLOT);        // the nine tap tiles are the whole weight tensor
            for (int tap = 0; tap < 9; ++tap) tma_load_2d(b_base + tap * L::B_SLOT, &maps.b, bar_bfull, tap * 64, 0);
            uint32_t ac = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++ac) {
                int n, oh0, ow0;
                decode(tile, n, oh0, ow0);
                const uint32_t sa = ac % PA, ita = ac / PA;
                mbar_wait(bar_aempty + sa * 8, (ita & 1) ^ 1);
                mbar_arrive_expect_tx(bar_afull + sa * 8, HL_PATCH_TX);
                tma_load_4d(a_base + sa * HL_PATCH_BYTES, &maps.a, bar_afull + sa * 8, 0, ow0 - 1, oh0 - 1, n);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_f16(DT<T>::umma_fmt, 128, HL_C);
            mbar_wait(bar_bfull, 0);
            tc_fence_after();
            uint32_t tc = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tc) {
                const uint32_t a = tc & 1, aph = (tc >> 1) & 1;
                mbar_wait(bar_tempty + a * 8, aph ^ 1);
                tc_fence_after();
                const uint32_t tmem_acc = tmem_base + a * HL_C;
                const uint32_t sa = tc % PA, ita = tc / PA;
                mbar_wait(bar_afull + sa * 8, ita & 1);
                tc_fence_after();
                const uint32_t patch = a_base + sa * HL_PATCH_BYTES;
#pragma unroll 1
                for (int tap = 0; tap < 9; ++tap) {
                    const uint32_t b_s = b_base + tap * L::B_SLOT;
                    const int kh = tap / 3, kw = tap - kh * 3;
                    const uint32_t a_s = patch + static_cast<uint32_t>(kh * HL_PW + kw) * 128u;   // row-shifted view
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_f16(tmem_acc, umma_desc_sw128(a_s + k * 32), umma_desc_sw128(b_s + k * 32), idesc,
                                 static_cast<uint32_t>((tap | k) != 0));
                }
                umma_commit(bar_aempty + sa * 8);
                umma_commit(bar_tfull + a * 8);
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ================= epilogue (256 threads; accumulator row q = padded-grid position; group grp converts 32 columns)
        const int q4 = warp & 3;
        const int grp = (warp - 4) >> 2;
        const int q = q4 * 32 + lane;
        const int r = q >> D::PW_SHIFT, c = q & (HL_PW - 1);
        const bool valid = c < HL_TW;
        const int d = r * HL_TW + c;                              // dense row inside the [TH][TW] store box
        const bool leader = (warp == 4 && lane == 0);
        auto issue_res = [&](int tile, uint32_t e) {
            int n, oh0, ow0;
            decode(tile, n, oh0, ow0);
            mbar_arrive_expect_tx(bar_rfull + e * 8, HL_TH * HL_TW * 128);
            tma_load_4d(e_base + e * L::EPI_BYTES, &maps.res, bar_rfull + e * 8, 0, ow0, oh0, n);
        };
        if (leader && has_res && static_cast<int>(blockIdx.x) < total_tiles) issue_res(blockIdx.x, 0);
        uint32_t tc = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tc) {
            const uint32_t a = tc & 1, aph = (tc >> 1) & 1;       // accumulator a and staging buffer a
            int n, oh0, ow0;
            decode(tile, n, oh0, ow0);
            if (leader) {
                tma_store_wait_read0();
                if (has_res && tile + static_cast<int>(gridDim.x) < total_tiles) issue_res(tile + gridDim.x, a ^ 1);
            }
            mbar_wait(bar_tfull + a * 8, aph);
            tc_fence_after();
            if (has_res) mbar_wait(bar_rfull + a * 8, aph);
            const uint32_t row_addr = e_base + a * L::EPI_BYTES + static_cast<uint32_t>(d) * 128u;
            const uint32_t sw = static_cast<uint32_t>(d) & 7u;
            uint32_t v[32];
            tmem_ld_32x32(tmem_base + a * HL_C + (static_cast<uint32_t>(q4 * 32) << 16) + grp * 32, v);
            tmem_ld_wait();
            if (valid) {
#pragma unroll
                for (int qq = 0; qq < 4; ++qq) {
                    const int col = grp * 32 + qq * 8;
                    const uint32_t addr = row_addr + (((col >> 3) ^ sw) << 4);
                    float f[8];
                    const float4 b0 = *reinterpret_cast<const float4*>(sbias + col);
                    const float4 b1 = *reinterpret_cast<const float4*>(sbias + col + 4);
                    f[0] = __uint_as_float(v[qq * 8 + 0]) + b0.x; f[1] = __uint_as_float(v[qq * 8 + 1]) + b0.y;
                    f[2] = __uint_as_float(v[qq * 8 + 2]) + b0.z; f[3] = __uint_as_float(v[qq * 8 + 3]) + b0.w;
                    f[4] = __uint_as_float(v[qq * 8 + 4]) + b1.x; f[5] = __uint_as_float(v[qq * 8 + 5]) + b1.y;
                    f[6] = __uint_as_float(v[qq * 8 + 6]) + b1.z; f[7] = __uint_as_float(v[qq * 8 + 7]) + b1.w;
                    if (has_res) {
                        uint32_t ru[4];
                        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(ru[0]), "=r"(ru[1]), "=r"(ru[2]), "=r"(ru[3]) : "r"(addr));
#pragma unroll
                        for (int x = 0; x < 4; ++x) {
                            const float2 rf = DT<T>::unpack2(ru[x]);
                            f[2 * x] += rf.x;
                            f[2 * x + 1] += rf.y;
                        }
                    }
                    if (p.relu) {
#pragma unroll
                        for (int x = 0; x < 8; ++x) f[x] = fmaxf(f[x], 0.f);
                    }
                    const uint32_t o0 = DT<T>::pack2(f[0], f[1]), o1 = DT<T>::pack2(f[2], f[3]);
                    const uint32_t o2 = DT<T>::pack2(f[4], f[5]), o3 = DT<T>::pack2(f[6], f[7]);
                    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty + a * 8);
            fence_proxy_async_smem();
            named_bar_sync(1, 256);
            if (leader) {
                tma_store_4d(&maps.out, e_base + a * L::EPI_BYTES, p.out_coff, ow0, oh0, n);
                tma_store_commit();
            }
        }
        if (leader) tma_store_wait_read0();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// ------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn4)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static bool make_tmap_nhwc_impl(CUtensorMap* m, const void* ptr, int C_ld, int W, int H, int N, int box_c, int box_w, int box_h, bool swizzle128);

bool make_tmap_nhwc(CUtensorMap* m, const void* ptr, int C_ld, int W, int H, int N, int box_w, int box_h) {
    return make_tmap_nhwc_impl(m, ptr, C_ld, W, H, N, 64, box_w, box_h, true);
}
bool make_tmap_nhwc_plain(CUtensorMap* m, const void* ptr, int C_ld, int W, int H, int N, int box_c, int box_w, int box_h) {
    return make_tmap_nhwc_impl(m, ptr, C_ld, W, H, N, box_c, box_w, box_h, false);
}

static bool make_tmap_nhwc_impl(CUtensorMap* m, const void* ptr, int C_ld, int W, int H, int N, int box_c, int box_w, int box_h, bool swizzle128) {
    static EncodeTiledFn4 fn = nullptr;
    if (!fn) {
        void* q = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qres) != cudaSuccess || !q) {
            set_error("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed");
            return false;
        }
        fn = reinterpret_cast<EncodeTiledFn4>(q);
    }
    cuuint64_t dims[4] = {static_cast<cuuint64_t>(C_ld), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(N)};
    cuuint64_t strides[3] = {static_cast<cuuint64_t>(C_ld) * 2, static_cast<cuuint64_t>(W) * C_ld * 2, static_cast<cuuint64_t>(H) * W * C_ld * 2};
    cuuint32_t box[4] = {static_cast<cuuint32_t>(box_c), static_cast<cuuint32_t>(box_w), static_cast<cuuint32_t>(box_h), 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(4d) failed (code " + std::to_string(static_cast<int>(r)) + ")"); return false; }
    return true;
}

bool conv_halo_applicable(const ConvParams& p, const ConvWeights& w) {
    return p.kh == 3 && p.kw == 3 && p.stride == 1 && p.pad == 1 && p.Cin == HL_C && p.Cout == HL_C && w.block_n == HL_C &&
           p.W >= 14 && (p.out_coff % 8) == 0;
}

template <typename T, int G>
static bool halo_launch_cfg(const ConvParams& p, const ConvWeights& w, cudaStream_t s) {
    using L = HaloSmem<G>;
    constexpr int HL_TH = HaloDims<G>::TH, HL_TW = HaloDims<G>::TW, HL_PW = HaloDims<G>::PW;
    HaloMaps maps;
    maps.b = w.tmap_b;
    if (!make_tmap_nhwc(&maps.a, p.in, p.Cin, p.W, p.H, p.N, HL_PW, HL_TH + 2)) return false;
    if (!make_tmap_nhwc(&maps.out, p.out, p.out_ld, p.Wo, p.Ho, p.N, HL_TW, HL_TH)) return false;
    maps.res = maps.out;
    if (p.res != nullptr && !make_tmap_nhwc(&maps.res, p.res, p.res_ld, p.Wo, p.Ho, p.N, HL_TW, HL_TH)) return false;
    auto kern = conv3x3_halo_kernel<T, G>;
    static DeviceOnce attr;
    if (attr.need()) {
        if (!check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "halo smem attr")) return false;
    }
    static int num_sms = 0;
    if (num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (!check_cuda(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev), "sm count")) return false;
    }
    const int tiles_w = (p.Wo + HL_TW - 1) / HL_TW, tiles_h = (p.Ho + HL_TH - 1) / HL_TH;
    const long long total = static_cast<long long>(p.N) * tiles_w * tiles_h;
    if (total > 0x7fffffffLL) { set_error("conv_halo: too many tiles"); return false; }
    const unsigned grid = static_cast<unsigned>(total < num_sms ? total : num_sms);
    launch_dep(kern, dim3(grid), dim3(HL_THREADS), L::DYN_BYTES, s, p, maps, tiles_w, tiles_h, static_cast<int>(total));
    return check_cuda(cudaGetLastError(), "conv_halo launch");
}

static double halo_tile_eff(int H, int W, int th, int tw) {
    return (static_cast<double>(W) / (tw * ((W + tw - 1) / tw))) * (static_cast<double>(H) / (th * ((H + th - 1) / th))) * tw / (tw + 2.0);
}

template <typename T>
static bool halo_launch_dt(const ConvParams& p, const ConvWeights& w, cudaStream_t s) {
    const bool wide = halo_tile_eff(p.Ho, p.Wo, 4, 30) > halo_tile_eff(p.Ho, p.Wo, 8, 14);     // fraction of GEMM rows that are real outputs
    return wide ? halo_launch_cfg<T, 1>(p, w, s) : halo_launch_cfg<T, 0>(p, w, s);
}

bool conv_halo_launch(const ConvParams& p, const ConvWeights& w, int prec, cudaStream_t s) {
    if (prec == PREC_BF16) return halo_launch_dt<__nv_bfloat16>(p, w, s);
    if (prec == PREC_F16) return halo_launch_dt<__half>(p, w, s);
    set_error("conv_halo: 16-bit precisions only");
    return false;
}

}  // namespace sb
