// WHOLE-BOTTLENECK kernel for the 64-channel bottlenecks (ResNet-50 layer1, HRNet layer1): ONE launch computes
//     y = relu( conv3_1x1( relu( conv2_3x3( relu( conv1_1x1(x) ) ) ) ) + residual ),   residual = x  or  downsample_1x1(x)
// replacing the three (four with the downsample) conv+BN+ReLU(+add) launches of a torchvision Bottleneck (SURVEY.md 7.1 step
// 5 / B.2: "fuse 1x1 -> 3x3 -> 1x1(+res) within a bottleneck").  Un-fused, a 256 -> 64 -> 64 -> 256 block at 56x56, batch 256,
// moves 1.65 GB through HBM (x read twice, the 64-channel intermediates t1 / t2 written and re-read) and took 0.36 ms on
// three HBM-bound launches (profiles/layers_resnet50_b256_bf16_v25.txt); fused it reads x once and writes y once (0.82 GB):
// the intermediates never leave the SM.
//
// Tile = 8 x 14 output pixels of one image on a padded grid of pitch 16 (GEMM row q = r*16 + c, 128 rows, the two columns
// c >= 14 of each row are scratch) -- the geometry of conv3x3_halo_kernel (conv_halo.cu):
//   conv1  x halo patch 10 x 16 pixels (4-D TMA box per 64 input channels, out-of-image = zero fill) -> 160 GEMM rows =
//          two M=128 MMAs per k-step (patch rows 0..127 and 32..159; rows 128..159 = lanes 96..127 of the second); epilogue 1 adds the
//          bias, applies ReLU, ZEROES the rows that lie outside the image (conv2 pads t1 with zeros, not with relu(b1)),
//          rounds to 16 bit and writes t1 as a K-major 128B-swizzled operand tile [162 rows][64 ch] in shared memory;
//   conv2  nine taps = nine row-shifted UMMA-descriptor views of t1 (start address + (kh*16+kw)*128 B; tools/umma_shift_test.cu)
//          against the resident [64][576] weight tensor; epilogue 2 -> t2 [128 rows][64 ch], same layout, over t1's memory;
//   conv3  one K=64 step, N = 256, accumulating ON TOP of the downsample conv when the block has one (the downsample's A
//          operand is the centre of the x patch = the same buffer shifted by 17 rows; both GEMMs share one accumulator, the
//          biases are summed); identity residuals are read from global memory (L2: the tile was fetched microseconds ago)
//          straight into the epilogue threads' registers (256-bit loads), one 32-column group ahead; epilogue 3: + bias +
//          residual, ReLU, 16 bit, [8][14][16 ch] staging boxes -> TMA stores (image borders clipped by the hardware).
// All weights (W1 <= 32 KB, W2 72 KB, W3 32 KB, Wds 32 KB) stay resident in shared memory for the life of the persistent CTA;
// x streams through a two/three-slot TMA ring, so the next tile's patch loads under this tile's conv2 / conv3.
//   warp 0  TMA producer      warp 1  MMA issuer (one thread)      warp 2  TMEM owner      warp 15  epilogue 1 of halo rows 128..159
//   warps 3-6  "front" epilogues 1 and 2 (they sit on the MMA thread's critical path: conv2 waits for t1, conv3 for t2)
//   warps 7-14 "back" epilogue 3 (two groups alternating 16-column steps, each through its own small staging box + TMA store)
// TMEM (512 columns): conv1 accumulators 0..127, conv2 128..191, conv3 (+downsample) 256..511 -- all disjoint, so the MMA
// thread issues conv1 of tile i+1 while the back warps drain conv3 of tile i.
// (First version, measured on B200: all eight epilogue warps ran the three epilogues in sequence and epilogue 3 went through
// one staging box with two named barriers and a TMA-store drain per 64-column chunk -- the chain epi1 -> conv2 -> epi2 ->
// conv3 -> epi3 -> epi1(next) was 11.6 k / 15.2 k cycles per tile (downsample / identity block) against 5.2 k / 7.0 k cycles
// of MMA issue: 0.29 / 0.375 ms per block, the identity block SLOWER than its three un-fused launches (0.363 ms).)
#include "common.cuh"
#include "internal.h"
#include <stdio.h>
#include <vector>

namespace sb {

namespace {
constexpr int BK_THREADS = 512;                                     // 16 warps: 0 TMA, 1 MMA, 2 TMEM owner, 3-6 front, 7-14 back, 15 epilogue 1 of halo rows 128..159
constexpr int BK_TH = 8, BK_TW = 14, BK_PW = 16;
constexpr int BK_PATCH_BYTES = (BK_TH + 2) * BK_PW * 128;          // 160 pixels x 64 ch x 2 B = 20480
constexpr int BK_T1_BYTES = 21 * 1024;                              // 168 rows (taps read up to row 127 + 34)
constexpr int BK_ST_BYTES = BK_TH * BK_TW * 32;                     // one output staging box: [8][14] pixels x 16 channels, dense 32-byte rows = 3584

template <int CIN>
struct BneckSmem {
    static constexpr int NCB = CIN / 64;
    static constexpr bool DS = (CIN == 64);                         // block with a downsample conv on the residual path
    static constexpr int NS = DS ? 2 : 3;                           // x ring slots (one 64-channel block per tile with a downsample, four without)
    // identity block: the [64][64] W1 k-block travels WITH its x block through the ring (slot = 20 KB patch + 8 KB weights,
    // re-fetched from L2 per tile) instead of 32 KB of resident W1 -- that is what pays for the double-buffered staging boxes
    static constexpr bool W1_RESIDENT = DS;
    static constexpr int SLOT_BYTES = BK_PATCH_BYTES + (W1_RESIDENT ? 0 : 8192);
    static constexpr int W1_OFF = 0;
    static constexpr int W2_OFF = W1_OFF + (W1_RESIDENT ? NCB * 8192 : 0);
    static constexpr int W3_OFF = W2_OFF + 9 * 8192;
    static constexpr int WD_OFF = W3_OFF + 32768;
    static constexpr int X_OFF = WD_OFF + (DS ? 32768 : 0);
    static constexpr int T1_OFF = X_OFF + NS * SLOT_BYTES;
    static constexpr int ST_OFF = T1_OFF + BK_T1_BYTES;             // staging boxes: 2 back warp groups x 2 buffers
    static constexpr int BAR_OFF = ST_OFF + 4 * BK_ST_BYTES;        // w_full, x_full[NS], x_empty[NS], acc1_full, t1_full, acc2_full, t2_full, acc3_full, acc3_empty
    static constexpr int NBAR = 1 + 2 * NS + 6;
    static constexpr int TMEMPTR_OFF = BAR_OFF + NBAR * 8;
    static constexpr int TOTAL = TMEMPTR_OFF + 16;
    static constexpr int DYN_BYTES = TOTAL + 1024;
    static_assert(DYN_BYTES <= 232448, "exceeds the 227 KB dynamic shared memory limit");
    static_assert((X_OFF % 1024) == 0 && (SLOT_BYTES % 1024) == 0 && (T1_OFF % 1024) == 0 && (ST_OFF % 128) == 0 && (BK_ST_BYTES % 128) == 0, "tile alignment");
};

struct BneckMaps {
    CUtensorMap x;      // input  (Cin, W, H, N)   box {64, 16, 10, 1}
    CUtensorMap w1;     // [64][Cin]    box {64, 64}
    CUtensorMap w2;     // [64][576]    box {64, 64}
    CUtensorMap w3;     // [256][64]    box {64, 256}
    CUtensorMap wd;     // [256][64]    box {64, 256}   (downsample; == w3 when unused)
    CUtensorMap out;    // output (256, W, H, N)   box {16, 14, 8, 1}, no swizzle (dense 32-byte rows)
};

// Folded-BN biases as LAUNCH PARAMETERS (constant bank): every use is an immediate operand of an FADD -- the epilogues issue no
// shared-memory loads for them (the front warps' LSU instructions queue behind the back warps' global traffic).
struct BneckBias { float b1[64], b2[64], b3[256]; };

struct BneckParams {
    const void* x;          // NHWC [N][H][W][CIN]: conv1 input; identity residual when there is no downsample
    void* out;              // NHWC [N][H][W][256]
    int N, H, W;
    int tiles_w, tiles_h, total_tiles;
    long long* trace;       // TRACE instantiation only: clock64() stamps of CTA 0, [tile < BK_TRACE_TILES][BK_TRACE_SLOTS]
};
constexpr int BK_TRACE_TILES = 24, BK_TRACE_SLOTS = 16;

// TRACE = true: diagnostic instantiation (SPECB200_BNECK_TRACE=<file>): CTA 0 stamps clock64() at every phase boundary of its
// first tiles -- the per-tile timeline the epilogue/MMA hand-over analysis in profiles/ was made from.
template <typename T, int CIN, bool TRACE = false>
__global__ void __launch_bounds__(BK_THREADS, 1)
bottleneck64_kernel(const BneckParams p, const __grid_constant__ BneckMaps maps, const __grid_constant__ BneckBias bias)
{
    griddep_launch();
    auto stamp = [&](uint32_t tc, int slot) {
        if constexpr (TRACE) {
            if (blockIdx.x == 0 && tc < BK_TRACE_TILES) p.trace[tc * BK_TRACE_SLOTS + slot] = clock64();
        }
    };
    using L = BneckSmem<CIN>;
    constexpr int NCB = L::NCB;
    constexpr bool DS = L::DS;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
    const uint32_t w1_s = sbase + L::W1_OFF, w2_s = sbase + L::W2_OFF, w3_s = sbase + L::W3_OFF, wd_s = sbase + L::WD_OFF;
    const uint32_t x_s = sbase + L::X_OFF, t1_s = sbase + L::T1_OFF, st_s = sbase + L::ST_OFF;
    const uint32_t bar_w = sbase + L::BAR_OFF;
    const uint32_t bar_xfull = bar_w + 8, bar_xempty = bar_xfull + L::NS * 8;
    const uint32_t bar_acc1 = bar_xempty + L::NS * 8, bar_t1 = bar_acc1 + 8, bar_acc2 = bar_t1 + 8, bar_t2 = bar_acc2 + 8;
    const uint32_t bar_acc3 = bar_t2 + 8, bar_acc3e = bar_acc3 + 8;
    volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(sgen + L::TMEMPTR_OFF);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(bar_w, 1);
        for (int s = 0; s < L::NS; ++s) { mbar_init(bar_xfull + s * 8, 1); mbar_init(bar_xempty + s * 8, 1); }
        mbar_init(bar_acc1, 1); mbar_init(bar_t1, 5); mbar_init(bar_acc2, 1); mbar_init(bar_t2, 4);     // front warps 3-6 (+ warp 15 for t1)
        mbar_init(bar_acc3, 1); mbar_init(bar_acc3e, 8);                                                   // back warps 7-14
        mbar_fence_init();
    }
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.x); tma_prefetch_desc(&maps.w1); tma_prefetch_desc(&maps.w2); tma_prefetch_desc(&maps.w3);
        tma_prefetch_desc(&maps.out);
        if (DS) tma_prefetch_desc(&maps.wd);
    }
    if (warp == 2) { tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_s)), 512); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    griddep_wait();
    const uint32_t tmem_base = *tmem_ptr_s;
    const uint32_t acc1 = tmem_base, acc2 = tmem_base + 128, acc3 = tmem_base + 256;

    auto decode = [&](int tile, int& n, int& oh0, int& ow0) {
        const int tw = tile % p.tiles_w;
        const int th = (tile / p.tiles_w) % p.tiles_h;
        n = tile / (p.tiles_w * p.tiles_h);
        oh0 = th * BK_TH; ow0 = tw * BK_TW;
    };

    if (warp == 0) {
        // ================= TMA producer: the weights once, then the x patches of this CTA's tiles
        if (lane == 0) {
            mbar_arrive_expect_tx(bar_w, ((L::W1_RESIDENT ? NCB : 0) + 9) * 8192 + 32768 + (DS ? 32768 : 0));
            if (L::W1_RESIDENT)
                for (int cb = 0; cb < NCB; ++cb) tma_load_2d(w1_s + cb * 8192, &maps.w1, bar_w, cb * 64, 0);
            for (int tap = 0; tap < 9; ++tap) tma_load_2d(w2_s + tap * 8192, &maps.w2, bar_w, tap * 64, 0);
            tma_load_2d(w3_s, &maps.w3, bar_w, 0, 0);
            if (DS) tma_load_2d(wd_s, &maps.wd, bar_w, 0, 0);
            uint32_t xc = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                int n, oh0, ow0;
                decode(tile, n, oh0, ow0);
                for (int cb = 0; cb < NCB; ++cb, ++xc) {
                    const uint32_t s = xc % L::NS, it = xc / L::NS;
                    mbar_wait(bar_xempty + s * 8, (it & 1) ^ 1);
                    mbar_arrive_expect_tx(bar_xfull + s * 8, L::SLOT_BYTES);
                    tma_load_4d(x_s + s * L::SLOT_BYTES, &maps.x, bar_xfull + s * 8, cb * 64, ow0 - 1, oh0 - 1, n);
                    if (!L::W1_RESIDENT) tma_load_2d(x_s + s * L::SLOT_BYTES + BK_PATCH_BYTES, &maps.w1, bar_xfull + s * 8, cb * 64, 0);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc64 = umma_idesc_f16(DT<T>::umma_fmt, 128, 64);
            constexpr uint32_t idesc256 = umma_idesc_f16(DT<T>::umma_fmt, 128, 256);
            mbar_wait(bar_w, 0);
            tc_fence_after();
            uint32_t xc = 0, tc = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++tc) {
                const uint32_t ph = tc & 1;
                uint32_t ds_slot = 0;
                stamp(tc, 0);
                // ---- conv1: [160 halo pixels] x [CIN] . W1^T -> acc1.  Two M tiles: patch rows 0..127 and rows 32..159 -- of the
                // second only TMEM lanes 96..127 (rows 128..159) are read (by warp 15, whose lane quarter that is)
                for (int cb = 0; cb < NCB; ++cb, ++xc) {
                    const uint32_t s = xc % L::NS, it = xc / L::NS;
                    mbar_wait(bar_xfull + s * 8, it & 1);
                    tc_fence_after();
                    const uint32_t xs = x_s + s * L::SLOT_BYTES;
                    const uint32_t w1b = L::W1_RESIDENT ? w1_s + cb * 8192 : xs + BK_PATCH_BYTES;
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            umma_f16(acc1 + mt * 64, umma_desc_sw128(xs + mt * 4096 + k * 32), umma_desc_sw128(w1b + k * 32),
                                     idesc64, static_cast<uint32_t>((cb | k) != 0));
                    if (DS) ds_slot = s;                               // the downsample conv still needs this patch (released below)
                    else umma_commit(bar_xempty + s * 8);
                }
                umma_commit(bar_acc1);
                stamp(tc, 1);
                // ---- conv2: nine row-shifted views of t1 . W2^T -> acc2
                mbar_wait(bar_t1, ph);
                tc_fence_after();
                stamp(tc, 2);
#pragma unroll 1
                for (int tap = 0; tap < 9; ++tap) {
                    const int kh = tap / 3, kw = tap - kh * 3;
                    const uint32_t a_s = t1_s + static_cast<uint32_t>(kh * BK_PW + kw) * 128u;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_f16(acc2, umma_desc_sw128(a_s + k * 32), umma_desc_sw128(w2_s + tap * 8192 + k * 32), idesc64,
                                 static_cast<uint32_t>((tap | k) != 0));
                }
                umma_commit(bar_acc2);
                stamp(tc, 3);
                // ---- the conv3 accumulator must have been drained by the back warps (tile i-1); then the downsample conv on the
                // tile's centre pixels (patch row q + 17) opens it, and conv3 accumulates on top
                mbar_wait(bar_acc3e, ph ^ 1);
                tc_fence_after();
                if (DS) {
                    const uint32_t xs = x_s + ds_slot * L::SLOT_BYTES;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_f16(acc3, umma_desc_sw128(xs + 17 * 128 + k * 32), umma_desc_sw128(wd_s + k * 32), idesc256,
                                 static_cast<uint32_t>(k != 0));
                    umma_commit(bar_xempty + ds_slot * 8);
                }
                stamp(tc, 4);
                // ---- conv3: t2 . W3^T -> acc3
                mbar_wait(bar_t2, ph);
                tc_fence_after();
                stamp(tc, 5);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    umma_f16(acc3, umma_desc_sw128(t1_s + k * 32), umma_desc_sw128(w3_s + k * 32), idesc256,
                             static_cast<uint32_t>(DS || k != 0));
                umma_commit(bar_acc3);
                stamp(tc, 6);
            }
        }
        __syncwarp();
    } else if ((warp >= 3 && warp < 7) || warp == 15) {
        // ================= front epilogues (on the MMA thread's critical path): acc1 -> t1, acc2 -> t2
        // warps 3-6: GEMM rows 0..127 (TMEM lane quarter = warp % 4), all 64 columns; warp 15: halo rows 128..159 = lanes 96..127 of
        // the second conv1 accumulator (epilogue 1 only).  Warp 15 sits on the scheduler partition with the fewest warps; with
        // that job on warp 2 (same partition as front warp 6) t1 was complete ~700 cycles after the other front warps.
        const bool extra = (warp == 15);
        const int q = extra ? 128 + lane : (warp & 3) * 32 + lane;          // t1 row written by this thread
        const uint32_t lane_off = static_cast<uint32_t>(extra ? 96 : (warp & 3) * 32) << 16;
        const uint32_t row_addr = t1_s + static_cast<uint32_t>(q) * 128u;
        const uint32_t sw = static_cast<uint32_t>(q) & 7u;
        // 64 accumulator columns of one row: +bias, ReLU, optional zeroing, 16 bit, swizzled row store
        auto store_row = [&](const uint32_t (&va)[32], const uint32_t (&vb)[32], const float (&bs)[64], bool zero) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float f[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const uint32_t u = j < 4 ? va[(j & 3) * 8 + e] : vb[(j & 3) * 8 + e];
                    f[e] = zero ? 0.f : fmaxf(__uint_as_float(u) + bs[j * 8 + e], 0.f);      // bs[...]: constant-bank operand
                }
                const uint32_t o0 = DT<T>::pack2(f[0], f[1]), o1 = DT<T>::pack2(f[2], f[3]);
                const uint32_t o2 = DT<T>::pack2(f[4], f[5]), o3 = DT<T>::pack2(f[6], f[7]);
                const uint32_t addr = row_addr + ((static_cast<uint32_t>(j) ^ sw) << 4);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
            }
        };
        uint32_t tc = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++tc) {
            const uint32_t ph = tc & 1;
            int n, oh0, ow0;
            decode(tile, n, oh0, ow0);
            // ---------------- epilogue 1: rows = halo-patch pixels; out-of-image rows are conv2's zero padding
            mbar_wait(bar_acc1, ph);
            tc_fence_after();
            if (warp == 3 && lane == 0) stamp(tc, 7);
            {
                uint32_t va[32], vb[32];
                const uint32_t src = acc1 + (extra ? 64u : 0u) + lane_off;
                tmem_ld_32x32(src, va);
                tmem_ld_32x32(src + 32, vb);
                tmem_ld_wait();
                const int ih = oh0 - 1 + (q >> 4), iw = ow0 - 1 + (q & 15);
                const bool outside = static_cast<unsigned>(ih) >= static_cast<unsigned>(p.H) || static_cast<unsigned>(iw) >= static_cast<unsigned>(p.W);
                store_row(va, vb, bias.b1, outside);
            }
            tc_fence_before();
            fence_proxy_async_smem();                              // generic-proxy writes of t1 -> UMMA (async proxy) reads
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_t1);
            if (warp == 3 && lane == 0) stamp(tc, 8);
            if (extra) continue;
            // ---------------- epilogue 2: acc2 -> t2 (over t1: every conv2 MMA has retired when acc2 is full)
            mbar_wait(bar_acc2, ph);
            tc_fence_after();
            if (warp == 3 && lane == 0) stamp(tc, 9);
            {
                uint32_t va[32], vb[32];
                tmem_ld_32x32(acc2 + lane_off, va);
                tmem_ld_32x32(acc2 + lane_off + 32, vb);
                tmem_ld_wait();
                store_row(va, vb, bias.b2, false);
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_t2);
            if (warp == 3 && lane == 0) stamp(tc, 10);
        }
    } else if (warp >= 7 && warp < 15) {
        // ================= back epilogue: acc3 (+ residual) -> y, under the next tile's conv1 / conv2.
        // Two groups of four warps (group = (warp - 7) / 4; TMEM lane quarter = warp % 4) take alternate 16-COLUMN steps, each
        // group through its own pair of 3.5 KB staging boxes (the store of step k drains while step k+1 fills the other box): tcgen05.ld x16 -> + bias (constant bank) + residual -> ReLU -> 16 bit -> two
        // 16-byte st.shared into dense 32-byte rows (conflict-free: a warp writes 1 KB contiguous) -> ONE TMA store of the
        // [8][14][16 ch] box (borders clipped by the hardware).  While one group's box drains, the other group computes.  The
        // only per-thread global access left is the identity residual: one 256-bit load per step, one step ahead.
        // Why so small-grained -- measured history (tools/bneck_trace.py, cycles per tile of CTA 0 on B200; MMA issue alone
        // = 5.2 k / 7.0 k for the downsample / identity block):
        //   v1  all eight epilogue warps ran the three epilogues in sequence, epilogue 3 through one 16 KB staging box with two
        //       named barriers and a TMA-store drain per 64 columns: 11.6 k / 15.2 k;
        //   v2  front / back warp groups, back group with 16-byte per-thread global loads and stores (512-byte lane stride = 32
        //       L1 wavefronts per warp instruction): ncu L1/TEX 85 % busy, the FRONT warps' shared-memory stores queued behind
        //       that traffic and epilogue 1 took 3.8 k cycles instead of 1.1 k: 10.8 k / 14.0 k;
        //   v3  back group through one 16 KB staging box + TMA store: L1 quiet (epilogue 1 = 1.2 k) but the box must drain before
        //       the next chunk is written -- epilogue 3 took 7.5 k / 12.2 k cycles holding the accumulator, and the box cost the
        //       third x-ring slot (conv1 3.3 k -> 4.4-5.3 k): 8.2 k / 12.6 k;
        //   v4-v5  256-bit per-thread accesses, also time-shifted into the front warps' idle windows: still 2048-4096 L1 wavefront
        //       cycles per tile in bursts of 256 per warp; epilogue 1 2.6-4.5 k: 8.4 k / 12.2 k;
        //   v6  this scheme with ONE box per group: epilogue 1 / 2 at 0.8 k / 0.6 k, but every step waited for its own previous
        //       store to drain: epilogue 3 5.8 k / 8.7 k cycles = the new critical resource: 7.5 k / 9.4 k.
        const int q4 = warp & 3;
        const int grp = (warp - 7) >> 2;
        const int q = q4 * 32 + lane;
        const uint32_t lane_off = static_cast<uint32_t>(q4 * 32) << 16;
        const int r = q >> 4, c = q & 15;
        const bool valid = c < BK_TW;
        const uint32_t st_grp = st_s + grp * 2 * BK_ST_BYTES;                               // this group's two boxes
        const uint32_t row_off = static_cast<uint32_t>(r * BK_TW + c) * 32u;                // dense row of the [8][14] store box
        const bool leader = (warp == 7 + grp * 4 && lane == 0);
        const int bar_id = 1 + grp;
        const T* __restrict__ xg = static_cast<const T*>(p.x);
        uint32_t tc = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++tc) {
            const uint32_t ph = tc & 1;
            int n, oh0, ow0;
            decode(tile, n, oh0, ow0);
            const bool live = valid && (oh0 + r) < p.H && (ow0 + c) < p.W;            // a real pixel inside the image
            const T* res_px = xg + ((static_cast<size_t>(n) * p.H + (oh0 + r)) * p.W + (ow0 + c)) * CIN;
            // identity residual: 16 channels = one 256-bit load per step, THREE steps ahead (an L2 round trip is ~1 k cycles, a
            // step ~0.5 k: one step ahead left every step waiting for its residual -- epilogue 3 took 9.5 k cycles per tile)
            uint32_t rq[3][8];
            auto load_res = [&](int slot, int step) {               // channels [step*16, +16) of this pixel
                if (!DS && live)
                    asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                                 : "=r"(rq[slot][0]), "=r"(rq[slot][1]), "=r"(rq[slot][2]), "=r"(rq[slot][3]),
                                   "=r"(rq[slot][4]), "=r"(rq[slot][5]), "=r"(rq[slot][6]), "=r"(rq[slot][7])
                                 : "l"(res_px + step * 16));
            };
            load_res(0, grp); load_res(1, grp + 2); load_res(2, grp + 4);
            mbar_wait(bar_acc3, ph);
            tc_fence_after();
            if (warp == 7 && lane == 0) stamp(tc, 11);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int step = 2 * k + grp;                       // output channels [step*16, +16)
                uint32_t v[16];
                tmem_ld_32x16(acc3 + lane_off + step * 16, v);
                tmem_ld_wait();
                if (k == 7) {                                      // the accumulator is in registers: the next tile may overwrite it
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_acc3e);
                }
                uint32_t rc[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) rc[j] = rq[k % 3][j];
                if (k + 3 < 8) load_res(k % 3, step + 6);
                uint32_t o[8];                                      // 16 outputs, packed (computed BEFORE waiting for the box to drain)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    float f[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[j * 8 + e]) + bias.b3[step * 16 + j * 8 + e];
                    if (!DS && live) {
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 rf = DT<T>::unpack2(rc[j * 4 + e]);
                            f[2 * e] += rf.x;
                            f[2 * e + 1] += rf.y;
                        }
                    }
#pragma unroll
                    for (int e = 0; e < 4; ++e) o[j * 4 + e] = DT<T>::pack2(fmaxf(f[2 * e], 0.f), fmaxf(f[2 * e + 1], 0.f));
                }
                const uint32_t st_buf = st_grp + (k & 1) * BK_ST_BYTES;
                if (leader) tma_store_wait_read<1>();              // the store issued two steps ago (same box) has read it
                named_bar_sync(bar_id, 128);
                if (valid) {
                    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(st_buf + row_off), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
                    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(st_buf + row_off + 16), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
                }
                fence_proxy_async_smem();
                named_bar_sync(bar_id, 128);
                if (leader) {
                    tma_store_4d(&maps.out, st_buf, step * 16, ow0, oh0, n);
                    tma_store_commit();
                }
            }
            if (warp == 7 && lane == 0) stamp(tc, 12);
        }
        if (leader) tma_store_wait_read0();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// diagnostic launch: instrumented kernel, synchronises, appends one line per traced tile to `path`
template <typename T, int CIN>
bool bneck_trace_run(BneckParams p, const BneckMaps& maps, const BneckBias& bias, const char* path, cudaStream_t s) {
    using L = BneckSmem<CIN>;
    auto kern = bottleneck64_kernel<T, CIN, true>;
    if (!check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "bottleneck smem attr")) return false;
    const size_t n = static_cast<size_t>(BK_TRACE_TILES) * BK_TRACE_SLOTS;
    if (!check_cuda(cudaMalloc(&p.trace, n * 8), "trace alloc") || !check_cuda(cudaMemset(p.trace, 0, n * 8), "trace memset")) return false;
    int num_sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned grid = static_cast<unsigned>(p.total_tiles < num_sms ? p.total_tiles : num_sms);
    launch_dep(kern, dim3(grid), dim3(BK_THREADS), L::DYN_BYTES, s, p, maps, bias);
    bool ok = check_cuda(cudaStreamSynchronize(s), "bottleneck trace run");
    std::vector<long long> h(n);
    ok = ok && check_cuda(cudaMemcpy(h.data(), p.trace, n * 8, cudaMemcpyDeviceToHost), "trace copy");
    cudaFree(p.trace);
    if (ok) {
        FILE* f = fopen(path, "a");
        if (f) {
            fprintf(f, "# bottleneck64 CIN=%d: per tile of CTA 0, cycles relative to the tile's MMA start: conv1_issued t1_ready conv2_issued acc3e_ds t2_ready conv3_issued | front: acc1_full epi1_done acc2_full epi2_done | back: acc3_full epi3_done | next tile start\n", CIN);
            for (int t = 0; t + 1 < BK_TRACE_TILES; ++t) {
                const long long* r = &h[static_cast<size_t>(t) * BK_TRACE_SLOTS];
                if (r[0] == 0) break;
                for (int k = 1; k <= 12; ++k) fprintf(f, "%lld ", r[k] - r[0]);
                fprintf(f, "| %lld\n", h[static_cast<size_t>(t + 1) * BK_TRACE_SLOTS] - r[0]);
            }
            fclose(f);
        }
    }
    return ok;
}

template <typename T, int CIN>
bool bneck_launch_t(const BottleneckArgs& a, cudaStream_t s) {
    using L = BneckSmem<CIN>;
    BneckMaps maps;
    if (!make_tmap_nhwc(&maps.x, a.x, CIN, a.W, a.H, a.N, BK_PW, BK_TH + 2)) return false;
    if (!make_tmap_nhwc_plain(&maps.out, a.out, 256, a.W, a.H, a.N, 16, BK_TW, BK_TH)) return false;
    if (!make_tmap_2d_k64(&maps.w1, a.w1->w_tc, 64, a.w1->K_pad, 64)) return false;
    if (!make_tmap_2d_k64(&maps.w2, a.w2->w_tc, 64, a.w2->K_pad, 64)) return false;
    if (!make_tmap_2d_k64(&maps.w3, a.w3->w_tc, 256, a.w3->K_pad, 256)) return false;
    maps.wd = maps.w3;
    if (a.wd != nullptr && !make_tmap_2d_k64(&maps.wd, a.wd->w_tc, 256, a.wd->K_pad, 256)) return false;
    BneckParams p;
    p.x = a.x; p.out = a.out;
    BneckBias bias;
    if (a.w1->bias_host.size() != 64 || a.w2->bias_host.size() != 64 || a.w3->bias_host.size() != 256 ||
        (a.wd != nullptr && a.wd->bias_host.size() != 256)) { set_error("bottleneck: host biases missing"); return false; }
    for (int i = 0; i < 64; ++i) { bias.b1[i] = a.w1->bias_host[i]; bias.b2[i] = a.w2->bias_host[i]; }
    for (int i = 0; i < 256; ++i) bias.b3[i] = a.w3->bias_host[i] + (a.wd != nullptr ? a.wd->bias_host[i] : 0.f);
    p.N = a.N; p.H = a.H; p.W = a.W;
    p.tiles_w = (a.W + BK_TW - 1) / BK_TW; p.tiles_h = (a.H + BK_TH - 1) / BK_TH;
    const long long total = static_cast<long long>(a.N) * p.tiles_w * p.tiles_h;
    if (total > 0x7fffffffLL) { set_error("bottleneck: too many tiles"); return false; }
    p.total_tiles = static_cast<int>(total);
    p.trace = nullptr;
    static const char* trace_path = getenv("SPECB200_BNECK_TRACE");
    if (trace_path != nullptr && trace_path[0] != 0) return bneck_trace_run<T, CIN>(p, maps, bias, trace_path, s);
    auto kern = bottleneck64_kernel<T, CIN>;
    static DeviceOnce attr;
    if (attr.need() && !check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "bottleneck smem attr")) return false;
    static int num_sms = 0;
    if (num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (!check_cuda(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev), "sm count")) return false;
    }
    const unsigned grid = static_cast<unsigned>(total < num_sms ? total : num_sms);
    launch_dep(kern, dim3(grid), dim3(BK_THREADS), L::DYN_BYTES, s, p, maps, bias);
    return check_cuda(cudaGetLastError(), "bottleneck launch");
}
}  // namespace

bool bottleneck_applicable(const BottleneckArgs& a) {
    const bool ds = a.wd != nullptr;
    const int cin = ds ? 64 : 256;
    auto ok16 = [](const ConvWeights* w, int cout, int cin_, int k) {
        return w && w->w_tc && w->bias && w->cout == cout && w->cin == cin_ && w->kh == k && w->kw == k && w->kwp == 0 && !w->stem7 &&
               w->K_pad == k * k * cin_;
    };
    return a.Cin == cin && a.N > 0 && a.H >= 1 && a.W >= 1 && ok16(a.w1, 64, cin, 1) && ok16(a.w2, 64, 64, 3) && ok16(a.w3, 256, 64, 1) &&
           (!ds || ok16(a.wd, 256, 64, 1));
}

bool bottleneck_launch(const BottleneckArgs& a, int prec, cudaStream_t s) {
    if (!bottleneck_applicable(a)) { set_error("bottleneck: not applicable"); return false; }
    const bool ds = a.wd != nullptr;
    if (prec == PREC_BF16) return ds ? bneck_launch_t<__nv_bfloat16, 64>(a, s) : bneck_launch_t<__nv_bfloat16, 256>(a, s);
    if (prec == PREC_F16) return ds ? bneck_launch_t<__half, 64>(a, s) : bneck_launch_t<__half, 256>(a, s);
    set_error("bottleneck: 16-bit precisions only");
    return false;
}

}  // namespace sb
