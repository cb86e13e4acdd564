// ResNet stem on the tensor cores: conv 7x7 / stride 2 / pad 3 (3 -> 64) + folded BN + ReLU, reading the
// fp32 NCHW image directly and writing NHWC 16-bit (replaces the first cuDNN conv + BN + ReLU of
// pare's resnet trunk; call sites /root/reference/camcalib/model.py:73, /root/reference/spec/models/hmr.py:92).
//
// With Cin = 3 the generic implicit-GEMM paths spend their time producing the A operand (K = 147 is
// neither TMA-im2col-able nor 16-byte granular).  This kernel builds A from an on-chip input patch instead:
//   tile = 8 x 16 output pixels (one 128-row UMMA tile) of one image
//   1. all threads load the (2*8+5) x (2*16+5) x 3 input patch (fp32 NCHW, rounded to 16 bit) into smem;
//   2. each A row (output pixel) is assembled from the patch: K is ordered (c, kh, kw padded to 8), so one
//      16-byte chunk = 8 consecutive patch elements of one (c, kh) filter row; K = 21 chunks -> 192;
//   3. one thread issues 12 tcgen05.mma (M=128, N=64, K=16) against the weight matrix that stays resident in
//      smem (24 KB, TMA-loaded once per CTA);
//   4. epilogue: tcgen05.ld -> +bias -> ReLU -> 16 bit -> swizzled smem -> coalesced 16-byte global stores.
// The CTA is sequential per tile; two to three co-resident CTAs per SM (93 KB smem each) overlap the phases.
#include "common.cuh"
#include "internal.h"
#include <string>
#include <stdlib.h>

namespace sb {

constexpr int ST_TH = 8, ST_TW = 16;                 // output tile
constexpr int ST_PR = 2 * ST_TH + 5;                 // 21 patch rows
constexpr int ST_PC = 2 * ST_TW + 5;                 // 37 patch cols
constexpr int ST_PP = 48;                            // patch row pitch (elements): 2 rows = 48 words -> the two
                                                     // half-warps of the A build hit disjoint banks
constexpr int ST_KB = 3;                             // K = 192 = 3 x 64
constexpr int ST_A_BYTES = ST_KB * 128 * 128;        // 49152
constexpr int ST_B_BYTES = ST_KB * 64 * 128;         // 24576
constexpr int ST_STAGE_BYTES = 128 * 128;            // 16384
constexpr int ST_OFF_B = ST_A_BYTES;
constexpr int ST_OFF_STAGE = ST_OFF_B + ST_B_BYTES;
constexpr int ST_OFF_PATCH = ST_OFF_STAGE + ST_STAGE_BYTES;
constexpr int ST_OFF_BIAS = ST_OFF_PATCH + 6144;      // patch = 3*21*48*2 = 6048 B
constexpr int ST_OFF_BAR = ST_OFF_BIAS + 256;
constexpr int ST_DYN_BYTES = ST_OFF_BAR + 64 + 1024;

template <typename T>
__global__ void __launch_bounds__(256)
conv_stem7_kernel(const float* __restrict__ img, T* __restrict__ out, const float* __restrict__ bias,
                  const __grid_constant__ CUtensorMap tmap_b, int N, int H, int W, int Ho, int Wo,
                  int tiles_h, int tiles_w, int total_tiles)
{
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
    const uint32_t a_base = sbase;
    const uint32_t b_base = sbase + ST_OFF_B;
    const uint32_t st_base = sbase + ST_OFF_STAGE;
    T* patch = reinterpret_cast<T*>(sgen + ST_OFF_PATCH);
    float* sbias = reinterpret_cast<float*>(sgen + ST_OFF_BIAS);
    const uint32_t bar_b = sbase + ST_OFF_BAR;
    const uint32_t bar_mma = bar_b + 8;
    volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(sgen + ST_OFF_BAR + 16);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        mbar_init(bar_b, 1);
        mbar_init(bar_mma, 1);
        mbar_fence_init();
    }
    if (tid < 64) sbias[tid] = bias[tid];
    for (int i = tid; i < 3 * ST_PR * ST_PP; i += 256) patch[i] = DT<T>::from_f(0.f);   // pad columns stay zero
    if (warp == 1) {
        tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_s)), 64);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_acc = *tmem_ptr_s;
    if (tid == 0) {                                      // weights: resident for the whole kernel
        tma_prefetch_desc(&tmap_b);
        mbar_arrive_expect_tx(bar_b, ST_B_BYTES);
        for (int kb = 0; kb < ST_KB; ++kb) tma_load_2d(b_base + kb * 8192, &tmap_b, bar_b, kb * 64, 0);
    }
    mbar_wait(bar_b, 0);

    const size_t plane = static_cast<size_t>(H) * W;
    // patch loader role: warp w owns patch rows w, w+8, ... (63 rows = 3 channels x 21); lanes cover cols lane, lane+32
    float pre[16];
    auto prefetch = [&](int tile) {
        const int tw = tile % tiles_w;
        const int th = (tile / tiles_w) % tiles_h;
        const int n = tile / (tiles_w * tiles_h);
        const int ih0 = 2 * th * ST_TH - 3, iw0 = 2 * tw * ST_TW - 3;
        const float* src = img + static_cast<size_t>(n) * 3 * plane;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int row = warp + 8 * k;                        // < 63 checked below
            const int c = row >= 42 ? 2 : (row >= 21 ? 1 : 0);
            const int r = row - c * 21;
            const int ih = ih0 + r;
            const bool rok = row < 63 && static_cast<unsigned>(ih) < static_cast<unsigned>(H);
            const float* rp = src + c * plane + static_cast<size_t>(rok ? ih : 0) * W;
            const int iwa = iw0 + lane, iwb = iw0 + lane + 32;
            pre[2 * k] = (rok && static_cast<unsigned>(iwa) < static_cast<unsigned>(W)) ? __ldg(rp + iwa) : 0.f;
            pre[2 * k + 1] = (rok && lane < ST_PC - 32 && static_cast<unsigned>(iwb) < static_cast<unsigned>(W)) ? __ldg(rp + iwb) : 0.f;
        }
    };
    if (static_cast<int>(blockIdx.x) < total_tiles) prefetch(blockIdx.x);
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int tw = tile % tiles_w;
        const int th = (tile / tiles_w) % tiles_h;
        const int n = tile / (tiles_w * tiles_h);
        const int oh0 = th * ST_TH, ow0 = tw * ST_TW;
        // ---- 1. input patch (prefetched into registers during the previous tile) -> smem, 16 bit
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int row = warp + 8 * k;
            if (row < 63) {
                patch[row * ST_PP + lane] = DT<T>::from_f(pre[2 * k]);
                if (lane < ST_PC - 32) patch[row * ST_PP + lane + 32] = DT<T>::from_f(pre[2 * k + 1]);
            }
        }
        __syncthreads();
        if (tile + static_cast<int>(gridDim.x) < total_tiles) prefetch(tile + gridDim.x);   // overlaps phases 2-5
        // ---- 2. A rows from the patch: thread pair (t, half) builds 12 of the 24 chunks of row t
        {
            const int t = tid & 127, half = tid >> 7;
            const int lr = t >> 4, lc = t & 15;
            const uint32_t sw = static_cast<uint32_t>(t) & 7u;
#pragma unroll
            for (int jj = 0; jj < 12; ++jj) {
                const int j = half * 12 + jj;
                uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
                if (j < 21) {
                    const int c = j / 7, kh = j - c * 7;
                    const uint32_t* s = reinterpret_cast<const uint32_t*>(patch + (c * ST_PR + 2 * lr + kh) * ST_PP + 2 * lc);
                    w0 = s[0]; w1 = s[1]; w2 = s[2]; w3 = s[3];
                }
                const uint32_t dst = a_base + (j >> 3) * 16384 + static_cast<uint32_t>(t) * 128u + (((j & 7) ^ sw) << 4);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(w0), "r"(w1), "r"(w2), "r"(w3) : "memory");
            }
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- 3. MMA
        if (tid == 0) {
            tc_fence_after();
            constexpr uint32_t idesc = umma_idesc_f16(DT<T>::umma_fmt, 128, 64);
#pragma unroll
            for (int kb = 0; kb < ST_KB; ++kb)
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    umma_f16(tmem_acc, umma_desc_sw128(a_base + kb * 16384 + k * 32), umma_desc_sw128(b_base + kb * 8192 + k * 32),
                             idesc, static_cast<uint32_t>((kb | k) != 0));
            umma_commit(bar_mma);
        }
        mbar_wait(bar_mma, it & 1);
        tc_fence_after();
        // ---- 4. epilogue: warp w -> TMEM lane quarter (w & 3), column half (w >> 2)
        {
            const int row = (warp & 3) * 32 + lane;
            const int ch = warp >> 2;
            uint32_t v[32];
            tmem_ld_32x32(tmem_acc + (static_cast<uint32_t>((warp & 3) * 32) << 16) + ch * 32, v);
            tmem_ld_wait();
            const uint32_t sw = static_cast<uint32_t>(row) & 7u;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float f[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) f[e] = fmaxf(__uint_as_float(v[q * 8 + e]) + sbias[ch * 32 + q * 8 + e], 0.f);
                const uint32_t dst = st_base + static_cast<uint32_t>(row) * 128u + (((ch * 4 + q) ^ sw) << 4);
                const uint32_t o0 = DT<T>::pack2(f[0], f[1]), o1 = DT<T>::pack2(f[2], f[3]);
                const uint32_t o2 = DT<T>::pack2(f[4], f[5]), o3 = DT<T>::pack2(f[6], f[7]);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
            }
        }
        tc_fence_before();
        __syncthreads();
        // ---- 5. coalesced store of the 128 x 64 tile (16 B per thread, 4 iterations)
#pragma unroll
        for (int rep = 0; rep < 4; ++rep) {
            const int i = rep * 256 + tid;
            const int row = i >> 3, chk = i & 7;
            const int oh = oh0 + (row >> 4), ow = ow0 + (row & 15);
            if (oh < Ho && ow < Wo) {
                uint4 val;
                const uint32_t srca = st_base + static_cast<uint32_t>(row) * 128u + ((chk ^ (row & 7)) << 4);
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w) : "r"(srca));
                *reinterpret_cast<uint4*>(out + ((static_cast<size_t>(n) * Ho + oh) * Wo + ow) * 64 + chk * 8) = val;
            }
        }
        // the next iteration's two __syncthreads (after patch load / after A build) order the smem reuse
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_acc, 64);
    }
}

// ------------------------------------------------------------------------------------------ pipelined version
// Same arithmetic, warp-specialised and double-buffered so that the phases of consecutive tiles overlap inside ONE
// persistent CTA per SM (the first version ran them back to back in two co-resident CTAs and sat at 3.4x its floor,
// profiles/README.md):
//   warps 4-11 (builders): input patch -> smem (double-buffered), A rows of tile i into A[i & 1]
//   warp  12   (MMA)     : 11 x tcgen05.mma (the 12th K-step is all padding and is skipped) into TMEM[i & 1]
//   warps 0-3  (epilogue): TMEM -> +bias -> ReLU -> 16 bit -> swizzled staging[i & 1] -> ONE 4-D TMA store (clips edges)
// so the per-tile cost is max(build, MMA ~ 960 cycles, epilogue) instead of their sum.
constexpr int STP_BW = 8;                                       // builder warps (16 measured slower: 0.255 vs 0.205 ms)
constexpr int STP_MMA_WARP = 4 + STP_BW;
constexpr int STP_THREADS = (STP_MMA_WARP + 1) * 32;
constexpr int STP_OFF_A = 0;                                   // 2 x 49152
constexpr int STP_OFF_B = 2 * ST_A_BYTES;                      // 24576
constexpr int STP_OFF_STAGE = STP_OFF_B + ST_B_BYTES;          // 2 x 16384
constexpr int STP_OFF_PATCH = STP_OFF_STAGE + 2 * ST_STAGE_BYTES;   // 2 x 6144
constexpr int STP_RING = 4;                                     // fp32 input patches in flight (TMA), 3 tiles ahead
constexpr int STP_RP = 40;                                      // ring row pitch (floats) = TMA box width: 37 used
constexpr int STP_BOX_BYTES = 3 * ST_PR * STP_RP * 4;           // 10080: one 40 x 21 x 3 fp32 box
constexpr int STP_RING_BYTES = 64 * STP_RP * 4;                 // slot pitch (10240)
constexpr int STP_OFF_RING = STP_OFF_PATCH + 2 * 6144;
constexpr int STP_OFF_BIAS = STP_OFF_RING + STP_RING * STP_RING_BYTES;
constexpr int STP_OFF_BAR = STP_OFF_BIAS + 256;                // b, a_full[2], a_empty[2], t_full[2], t_empty[2], tmem ptr, ring_full[4]
constexpr int STP_DYN_BYTES = STP_OFF_BAR + 128 + 1024;
static_assert(STP_DYN_BYTES <= 232448, "stem: shared memory");

template <typename T>
__global__ void __launch_bounds__(STP_THREADS, 1)
conv_stem7p_kernel(const __grid_constant__ CUtensorMap tmap_img, const float* __restrict__ bias,
                   const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_out,
                   int tiles_h, int tiles_w, int total_tiles)
{
    griddep_launch();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
    const uint32_t a_base = sbase + STP_OFF_A;
    const uint32_t b_base = sbase + STP_OFF_B;
    const uint32_t st_base = sbase + STP_OFF_STAGE;
    T* patch0 = reinterpret_cast<T*>(sgen + STP_OFF_PATCH);
    float* sbias = reinterpret_cast<float*>(sgen + STP_OFF_BIAS);
    const uint32_t bar_b = sbase + STP_OFF_BAR;
    const uint32_t bar_afull = bar_b + 8, bar_aempty = bar_b + 24, bar_tfull = bar_b + 40, bar_tempty = bar_b + 56;
    volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(sgen + STP_OFF_BAR + 72);
    const uint32_t bar_ring = bar_b + 80;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        mbar_init(bar_b, 1);
        for (int i = 0; i < STP_RING; ++i) mbar_init(bar_ring + i * 8, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar_afull + i * 8, STP_BW);               // one arrival per builder warp
            mbar_init(bar_aempty + i * 8, 1);                   // tcgen05.commit
            mbar_init(bar_tfull + i * 8, 1);                    // tcgen05.commit
            mbar_init(bar_tempty + i * 8, 4);                   // one arrival per epilogue warp
        }
        mbar_fence_init();
    }
    if (tid < 64) sbias[tid] = bias[tid];
    for (int i = tid; i < 2 * (6144 / 2); i += STP_THREADS) patch0[i] = DT<T>::from_f(0.f);          // both patch buffers: pad columns stay zero
    if (warp == STP_MMA_WARP) {
        tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_s)), 128);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    griddep_wait();
    const uint32_t tmem_base = *tmem_ptr_s;

    if (warp >= 4 && warp < STP_MMA_WARP) {
        // ================= builders
        const int wb = warp - 4, bt = tid - 128;
        const uint32_t ring_base = sbase + STP_OFF_RING;
        const float* ring_gen = reinterpret_cast<const float*>(sgen + STP_OFF_RING);
        // The fp32 image is the only HBM read of this kernel and one tile's patch is under 10 KB: with a single tile in
        // flight per SM (register prefetch, first version) the builders waited a full memory latency per tile.  One
        // builder thread therefore keeps the patches of the next THREE tiles in flight as 4-D TMA boxes (40 x 21 x 3 fp32,
        // out-of-image pixels zero-filled by the TMA unit = the conv's padding) into a ring of four slots.
        // (4-byte cp.async was tried for this ring and is element-rate bound: 0.36 ms vs 0.27 ms.)
        auto issue = [&](int tile, uint32_t slot) {
            if (tile >= total_tiles) return;
            const int tw = tile % tiles_w;
            const int th = (tile / tiles_w) % tiles_h;
            const int n = tile / (tiles_w * tiles_h);
            mbar_arrive_expect_tx(bar_ring + slot * 8, STP_BOX_BYTES);
            // the box start must be 16-byte aligned in global memory (tools/tma_img_test.cu): load from x = 32 tw - 4, one
            // column left of the patch, and read the ring at column + 1
            tma_load_4d(ring_base + slot * STP_RING_BYTES, &tmap_img, bar_ring + slot * 8, 2 * tw * ST_TW - 4, 2 * th * ST_TH - 3, 0, n);
        };
        if (bt == 0) {
            tma_prefetch_desc(&tmap_img);
            for (int d = 0; d < STP_RING - 1; ++d) issue(static_cast<int>(blockIdx.x + d * gridDim.x), d);
        }
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const uint32_t s = it & 1, ph = (it >> 1) & 1;
            const uint32_t slot = it % STP_RING;
            T* patch = patch0 + s * (6144 / 2);
            mbar_wait(bar_ring + slot * 8, (it / STP_RING) & 1);   // this tile's fp32 patch has landed
            const float* mine = ring_gen + slot * (STP_RING_BYTES / 4) + wb * STP_RP + lane + 1;       // rows wb, wb + STP_BW, ...
            {   // all loads first, then all stores: the LDS latencies overlap instead of adding up
                constexpr int RK = (63 + STP_BW - 1) / STP_BW;
                float pa[RK], pb[RK];
#pragma unroll
                for (int k = 0; k < RK; ++k) {
                    const bool rok = wb + STP_BW * k < 63;
                    pa[k] = rok ? mine[k * STP_BW * STP_RP] : 0.f;
                    pb[k] = (rok && lane < ST_PC - 32) ? mine[k * STP_BW * STP_RP + 32] : 0.f;
                }
#pragma unroll
                for (int k = 0; k < RK; ++k) {
                    const int row = wb + STP_BW * k;
                    if (row < 63) {
                        patch[row * ST_PP + lane] = DT<T>::from_f(pa[k]);
                        if (lane < ST_PC - 32) patch[row * ST_PP + lane + 32] = DT<T>::from_f(pb[k]);
                    }
                }
            }
            named_bar_sync(2, 32 * STP_BW);                     // patch[s] complete; also orders the reuse of patch[s ^ 1]
            // every builder has read ring slots <= it: the slot of tile it-1 may be refilled (tile it+3)
            if (bt == 0) issue(tile + (STP_RING - 1) * static_cast<int>(gridDim.x), (it + STP_RING - 1) % STP_RING);
            mbar_wait(bar_aempty + s * 8, ph ^ 1);              // the MMAs of tile it-2 have consumed A[s]
            {
                constexpr int PARTS = STP_BW / 4, CPT = (22 + PARTS - 1) / PARTS;     // chunks per thread
                const int t = bt & 127, part = bt >> 7;
                const int lr = t >> 4, lc = t & 15;
                const uint32_t sw = static_cast<uint32_t>(t) & 7u;
                const uint32_t a_s = a_base + s * ST_A_BYTES;
                uint32_t w[CPT][4];
#pragma unroll
                for (int jj = 0; jj < CPT; ++jj) {              // all loads in flight before the first store
                    const int j = part * CPT + jj;              // 21 real chunks + one zero chunk (second half of K-step 11)
                    w[jj][0] = w[jj][1] = w[jj][2] = w[jj][3] = 0;
                    if (j < 21) {
                        const int c = j / 7, kh = j - c * 7;
                        const uint32_t* sp = reinterpret_cast<const uint32_t*>(patch + (c * ST_PR + 2 * lr + kh) * ST_PP + 2 * lc);
                        w[jj][0] = sp[0]; w[jj][1] = sp[1]; w[jj][2] = sp[2]; w[jj][3] = sp[3];
                    }
                }
#pragma unroll
                for (int jj = 0; jj < CPT; ++jj) {
                    const int j = part * CPT + jj;
                    if (j < 22) {
                        const uint32_t dst = a_s + (j >> 3) * 16384 + static_cast<uint32_t>(t) * 128u + (((j & 7) ^ sw) << 4);
                        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(w[jj][0]), "r"(w[jj][1]), "r"(w[jj][2]), "r"(w[jj][3]) : "memory");
                    }
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_afull + s * 8);
        }
    } else if (warp == STP_MMA_WARP) {
        // ================= MMA issuer
        if (lane == 0) {
            tma_prefetch_desc(&tmap_b);
            mbar_arrive_expect_tx(bar_b, ST_B_BYTES);            // weights: resident for the whole kernel
            for (int kb = 0; kb < ST_KB; ++kb) tma_load_2d(b_base + kb * 8192, &tmap_b, bar_b, kb * 64, 0);
            mbar_wait(bar_b, 0);
            constexpr uint32_t idesc = umma_idesc_f16(DT<T>::umma_fmt, 128, 64);
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
                const uint32_t s = it & 1, ph = (it >> 1) & 1;
                mbar_wait(bar_tempty + s * 8, ph ^ 1);          // epilogue drained accumulator s
                mbar_wait(bar_afull + s * 8, ph);
                tc_fence_after();
                const uint32_t a_s = a_base + s * ST_A_BYTES;
                const uint32_t acc = tmem_base + s * 64;
#pragma unroll
                for (int ks = 0; ks < 11; ++ks)
                    umma_f16(acc, umma_desc_sw128(a_s + (ks >> 2) * 16384 + (ks & 3) * 32),
                             umma_desc_sw128(b_base + (ks >> 2) * 8192 + (ks & 3) * 32), idesc, static_cast<uint32_t>(ks != 0));
                umma_commit(bar_aempty + s * 8);
                umma_commit(bar_tfull + s * 8);
            }
        }
        __syncwarp();
    } else {
        // ================= epilogue (warps 0-3: TMEM lane quarter = warp)
        const int row = warp * 32 + lane;
        const uint32_t sw = static_cast<uint32_t>(row) & 7u;
        const bool leader = tid == 0;
        if (leader) tma_prefetch_desc(&tmap_out);
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const uint32_t s = it & 1, ph = (it >> 1) & 1;
            const int tw = tile % tiles_w;
            const int th = (tile / tiles_w) % tiles_h;
            const int n = tile / (tiles_w * tiles_h);
            mbar_wait(bar_tfull + s * 8, ph);
            tc_fence_after();
            uint32_t va[32], vb[32];
            const uint32_t acc = tmem_base + s * 64 + (static_cast<uint32_t>(warp * 32) << 16);
            tmem_ld_32x32(acc, va);
            tmem_ld_32x32(acc + 32, vb);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty + s * 8);     // accumulator s may be overwritten
            if (leader) tma_store_wait_read<1>();               // the store of tile it-2 has finished reading staging[s]
            named_bar_sync(3, 128);
            const uint32_t st_s = st_base + s * ST_STAGE_BYTES + static_cast<uint32_t>(row) * 128u;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                float f[8];
                const float4 b0 = *reinterpret_cast<const float4*>(sbias + q * 8);      // two broadcast LDS.128 per 8 channels
                const float4 b1 = *reinterpret_cast<const float4*>(sbias + q * 8 + 4);
                const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    f[e] = fmaxf(__uint_as_float(q < 4 ? va[(q & 3) * 8 + e] : vb[(q & 3) * 8 + e]) + bb[e], 0.f);
                const uint32_t o0 = DT<T>::pack2(f[0], f[1]), o1 = DT<T>::pack2(f[2], f[3]);
                const uint32_t o2 = DT<T>::pack2(f[4], f[5]), o3 = DT<T>::pack2(f[6], f[7]);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(st_s + ((static_cast<uint32_t>(q) ^ sw) << 4)), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
            }
            fence_proxy_async_smem();
            named_bar_sync(3, 128);
            if (leader) {
                tma_store_4d(&tmap_out, st_base + s * ST_STAGE_BYTES, 0, tw * ST_TW, th * ST_TH, n);
                tma_store_commit();
            }
        }
        if (leader) tma_store_wait_read0();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == STP_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 128);
    }
}

// 4-D tiled TMA descriptor over the fp32 NCHW image: box = 40 x 21 x 3 x 1 (one stem tile's input patch), no swizzle,
// out-of-bounds elements read as zero (= the convolution's zero padding).
static bool make_tmap_image_f32(CUtensorMap* m, const float* img, int W, int H, int N) {
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* q = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qres) != cudaSuccess || !q) {
            set_error("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed");
            return false;
        }
        fn = reinterpret_cast<EncodeTiledFn>(q);
    }
    cuuint64_t dims[4] = {static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), 3, static_cast<cuuint64_t>(N)};
    cuuint64_t strides[3] = {static_cast<cuuint64_t>(W) * 4, static_cast<cuuint64_t>(H) * W * 4, static_cast<cuuint64_t>(H) * W * 12};
    cuuint32_t box[4] = {STP_RP, ST_PR, 3, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(img), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(image) failed (code " + std::to_string(static_cast<int>(r)) + ")"); return false; }
    return true;
}

bool conv_stem7_launch(const float* img, void* out, const ConvWeights& w, int N, int H, int W, int Ho, int Wo, int prec,
                       cudaStream_t s) {
    if (!w.has_tmap || !w.stem7) { set_error("conv_stem7: weights not packed for the stem kernel"); return false; }
    static int num_sms = 0;
    if (num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (!check_cuda(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev), "sm count")) return false;
    }
    const int tiles_h = (Ho + ST_TH - 1) / ST_TH, tiles_w = (Wo + ST_TW - 1) / ST_TW;
    const long long total = static_cast<long long>(N) * tiles_h * tiles_w;
    if (total > 0x7fffffffLL) { set_error("conv_stem7: too many tiles"); return false; }
    // the TMA-fed kernel needs 16-byte aligned image rows (W % 4 == 0) and an image at least one box (40 x 21) large;
    // other shapes keep the first kernel
    if ((W % 4) == 0 && W >= STP_RP && H >= ST_PR && (reinterpret_cast<uintptr_t>(img) & 15) == 0) {
        CUtensorMap tmap_out, tmap_img;
        if (!make_tmap_nhwc(&tmap_out, out, 64, Wo, Ho, N, ST_TW, ST_TH)) return false;
        if (!make_tmap_image_f32(&tmap_img, img, W, H, N)) return false;
        static DeviceOnce attr_p;
        if (attr_p.need()) {
            if (!check_cuda(cudaFuncSetAttribute(conv_stem7p_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, STP_DYN_BYTES), "stem attr")) return false;
            if (!check_cuda(cudaFuncSetAttribute(conv_stem7p_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, STP_DYN_BYTES), "stem attr")) return false;
        }
        const unsigned gridp = static_cast<unsigned>(total < num_sms ? total : num_sms);
        if (prec == PREC_BF16)
            launch_dep(conv_stem7p_kernel<__nv_bfloat16>, dim3(gridp), dim3(STP_THREADS), STP_DYN_BYTES, s, tmap_img, w.bias, w.tmap_b, tmap_out, tiles_h, tiles_w, static_cast<int>(total));
        else if (prec == PREC_F16)
            launch_dep(conv_stem7p_kernel<__half>, dim3(gridp), dim3(STP_THREADS), STP_DYN_BYTES, s, tmap_img, w.bias, w.tmap_b, tmap_out, tiles_h, tiles_w, static_cast<int>(total));
        else { set_error("conv_stem7: 16-bit precisions only"); return false; }
        return check_cuda(cudaGetLastError(), "conv_stem7p launch");
    }
    const unsigned grid = static_cast<unsigned>(total < 2LL * num_sms ? total : 2LL * num_sms);
    static DeviceOnce attr;
    if (attr.need()) {
        if (!check_cuda(cudaFuncSetAttribute(conv_stem7_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_DYN_BYTES), "stem attr")) return false;
        if (!check_cuda(cudaFuncSetAttribute(conv_stem7_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_DYN_BYTES), "stem attr")) return false;
    }
    if (prec == PREC_BF16)
        conv_stem7_kernel<__nv_bfloat16><<<grid, 256, ST_DYN_BYTES, s>>>(img, static_cast<__nv_bfloat16*>(out), w.bias, w.tmap_b, N, H, W, Ho, Wo, tiles_h, tiles_w, static_cast<int>(total));
    else if (prec == PREC_F16)
        conv_stem7_kernel<__half><<<grid, 256, ST_DYN_BYTES, s>>>(img, static_cast<__half*>(out), w.bias, w.tmap_b, N, H, W, Ho, Wo, tiles_h, tiles_w, static_cast<int>(total));
    else { set_error("conv_stem7: 16-bit precisions only"); return false; }
    return check_cuda(cudaGetLastError(), "conv_stem7 launch");
}

}  // namespace sb
