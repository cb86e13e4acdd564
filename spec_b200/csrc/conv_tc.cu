// Implicit-GEMM convolution on the sm_100a tensor cores (tcgen05 + TMEM + TMA).
//
// Replaces the cuDNN conv + separate BN / ReLU / residual-add kernels the reference runs for every
// backbone convolution (call sites /root/reference/camcalib/model.py:73 and
// /root/reference/spec/models/hmr.py:92; op inventory SURVEY.md section 2.2).
//
// GEMM view:  D[M, Cout] = A[M, K] * W[Cout, K]^T,  M = N*Ho*Wo output pixels, K = kh*kw*Cin with
// k = (tap, channel).  Activations are NHWC 16-bit, weights K-major 16-bit (BN folded), accumulation
// fp32 in tensor memory.  One CTA computes a 128 x BLOCK_N output tile.
//
// A operand (128 pixels x 64 channels per pipeline stage, 128B-swizzled K-major rows):
//   A_TILED   1x1 stride-1 convs: A is the plain [M, Cin] matrix -> TMA tiled 2-D load.
//   A_IM2COL  any conv with Cin % 64 == 0: TMA im2col-mode load straight from the NHWC tensor (the
//             hardware walks output pixels, applies the filter-tap offset and zero-fills the padding).
//   A_GATHER  everything else (e.g. Cin = 32): warps 0-3 do the im2col in software with zero-filling
//             cp.async into the same swizzled layout.
//   A_STEM    the 3-channel stem conv: the image is stored NHWC with 4 channels (8 bytes / pixel) and K is
//             ordered (kh, kw padded to a power of two, c4), so the kw pixels of one filter row are
//             contiguous in memory and are gathered pixel-wise (8-byte cp.async) -- K = 224 -> 256 for
//             the 7x7 stem instead of 7*7*8 = 392 -> 448 with channel-padded 16-byte chunks.
// B operand: TMA tiled 2-D load of the [Cout, K] weight matrix.
//
//   warps 0-3  (A_GATHER producers, then) epilogue: tcgen05.ld accumulator rows -> +bias (+residual)
//              -> ReLU -> 16-bit.  EPI_TMA: the residual tile is TMA-loaded into the (by then free)
//              pipeline smem, combined in place, and the finished tile leaves through a TMA store --
//              fully coalesced 128-byte lines in both directions.  BLOCK_N = 32 keeps direct stores.
//   warp 4     TMA producer (A, and B in the gather modes); owns the TMEM allocation.
//   warp 5     MMA issuer: one thread issues tcgen05.mma (M=128, N=BLOCK_N, K=16) x4 per stage and
//              commits stage release / accumulator-ready to mbarriers.
//   warps 6-9  second epilogue group: in the TMA-store epilogue they convert the upper half of the columns.
//              In the TMA-fed modes warp 6 first issues the weight tiles (second producer).
//
// Second producer: one thread that waits, arms and issues two TMA loads per k-block tops out at ~350 ns per block
// (tools/tma_mcast_test.cu); issuing A and B from two threads gave -7..-11 % on the 3x3 CTA-pair convs (B200, round 2).
// All three tcgen05 conv kernels split their producers this way.
//
// BLOCK_N = 256 (3x3 convs with Cout >= 256): at 128 x 128 tiles the tensor pipe consumes 128 B/cycle of operands,
// so covering ~1.5k cycles of TMA latency needs ~190 KB in flight -- more than one SM's smem; a 128 x 256 tile needs
// 96 B/cycle.  One CTA per SM then (4 stages x 48 KB), so the epilogue gets both groups to stay short.
//
// Pipeline: STAGES-deep smem ring with full/empty mbarriers; smem footprint <= ~100 KB so two CTAs
// share an SM and one CTA's epilogue overlaps the other's main loop.
#include "common.cuh"
#include "internal.h"

namespace sb {

constexpr int TILE_M = 128;
constexpr int TILE_K = 64;                      // 64 x 16-bit = 128 B = one swizzle row
constexpr int A_STAGE_BYTES = TILE_M * TILE_K * 2;
constexpr int GATHER_LAG = 2;                   // cp.async groups kept in flight per producer thread
constexpr int CONV_TC_THREADS = 320;           // warps 0-3 epilogue A (+gather), 4 TMA, 5 MMA, 6-9 epilogue B
enum { A_TILED = 0, A_IM2COL = 1, A_GATHER = 2, A_STEM = 3 };

template <int BLOCK_N, int STAGES>
struct ConvTcSmem {
    static constexpr int B_STAGE_BYTES = BLOCK_N * TILE_K * 2;
    static constexpr int A_OFF = 0;
    static constexpr int B_OFF = STAGES * A_STAGE_BYTES;
    static constexpr int BAR_OFF = B_OFF + STAGES * B_STAGE_BYTES;          // full[STAGES], empty[STAGES], tmem_full, res_full
    static constexpr int TMEMPTR_OFF = BAR_OFF + (2 * STAGES + 2) * 8;
    static constexpr int BIAS_OFF = TMEMPTR_OFF + 8;
    static constexpr int TOTAL = BIAS_OFF + BLOCK_N * 4;
    static constexpr int DYN_BYTES = TOTAL + 1024;                           // slack for manual 1024 B alignment
    static constexpr int EPI_BYTES = TILE_M * BLOCK_N * 2;                   // output staging tile (aliases the A stages)
    static_assert(EPI_BYTES <= STAGES * A_STAGE_BYTES, "staging tile must fit in the A stages");
};

struct ConvTcMaps {
    CUtensorMap a;      // A_TILED: [M][Cin] tiled;  A_IM2COL: NHWC im2col;  A_GATHER: unused
    CUtensorMap b;      // weights [Cout_pad][K_pad]
    CUtensorMap out;    // EPI_TMA: [M][out_ld] box 64 x 128
    CUtensorMap res;    // EPI_TMA + residual: [M][res_ld] box 64 x 128
};

// (A variant of this kernel in clusters of two CTAs that shared the weight tile by TMA multicast -- each CTA loading half of it per
// k-block, stage release by a multicast commit onto both empty barriers -- was written in round 1, parity-tested and timed on B200
// in round 2: clean, but SLOWER on the layers that use this kernel (layer2 3x3: 0.081-0.093 ms against 0.072-0.084 ms), so it
// was removed; profiles/README.md has the numbers and tools/tma_mcast_test.cu the probe.)
template <typename T, int BLOCK_N, int STAGES, int A_MODE>
__global__ void __launch_bounds__(CONV_TC_THREADS)
conv_tc_kernel(const ConvParams p, const __grid_constant__ ConvTcMaps maps, int n_tiles)
{
    griddep_launch();
    static_assert(GATHER_LAG <= STAGES - 1, "producer lag must leave one free stage");
    using L = ConvTcSmem<BLOCK_N, STAGES>;
    constexpr int TMEM_COLS = BLOCK_N < 32 ? 32 : BLOCK_N;
    constexpr bool EPI_TMA_CAPABLE = BLOCK_N >= 64;
    const bool epi_tma = EPI_TMA_CAPABLE && (p.Cout & 63) == 0;   // whole 64-column boxes only (concat slices stay intact)
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
    const uint32_t a_base = sbase + L::A_OFF;
    const uint32_t b_base = sbase + L::B_OFF;
    const uint32_t bar_full = sbase + L::BAR_OFF;
    const uint32_t bar_empty = bar_full + STAGES * 8;
    const uint32_t bar_tmem = bar_empty + STAGES * 8;
    const uint32_t bar_res = bar_tmem + 8;
    volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(sgen + L::TMEMPTR_OFF);
    float* sbias = reinterpret_cast<float*>(sgen + L::BIAS_OFF);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int tile_id = static_cast<int>(blockIdx.x);
    const int n_tile = tile_id % n_tiles;
    const int m_tile = tile_id / n_tiles;
    const int n0 = n_tile * BLOCK_N;
    const int num_kb = (p.K + TILE_K - 1) / TILE_K;

    // ---------------- one-time setup
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + s * 8, (A_MODE == A_GATHER || A_MODE == A_STEM) ? 5 : 1);   // 4 gather warps + the TMA thread
            mbar_init(bar_empty + s * 8, 1);
        }
        mbar_init(bar_tmem, 1);
        mbar_init(bar_res, 1);
        mbar_fence_init();
    }
    if (threadIdx.x < BLOCK_N) {
        const int c = n0 + threadIdx.x;
        sbias[threadIdx.x] = (c < p.Cout) ? p.bias[c] : 0.f;
    }
    if (warp == 4) {
        if (lane == 0) {
            tma_prefetch_desc(&maps.b);
            if (A_MODE == A_TILED || A_MODE == A_IM2COL) tma_prefetch_desc(&maps.a);
            if (epi_tma) { tma_prefetch_desc(&maps.out); if (p.res != nullptr) tma_prefetch_desc(&maps.res); }
        }
        __syncwarp();
        tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_s)), TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    griddep_wait();
    const uint32_t tmem_acc = *tmem_ptr_s;

    if (warp < 4 || warp >= 6) {
        const int grp = warp >= 6 ? 1 : 0;                       // epilogue group (column half in the TMA epilogue)
        const int q4 = warp & 3;                                 // TMEM lane quarter this warp may access
        const int t = q4 * 32 + lane;                            // tile row == TMEM lane
        const long long r = static_cast<long long>(m_tile) * TILE_M + t;
        const bool row_ok = r < p.M;
        // ---------------- second TMA producer: warp 6 issues the weight tiles while warp 4 issues A; its epilogue share starts
        // afterwards (every load is issued long before the last MMA retires)
        if constexpr (A_MODE == A_TILED || A_MODE == A_IM2COL) {
            if (warp == 6) {
                if (lane == 0) {
                    for (int kb = 0; kb < num_kb; ++kb) {
                        const int s = kb % STAGES;
                        const int it = kb / STAGES;
                        mbar_wait(bar_empty + s * 8, (it & 1) ^ 1);
                        tma_load_2d(b_base + s * L::B_STAGE_BYTES, &maps.b, bar_full + s * 8, kb * TILE_K, n0);
                    }
                }
                __syncwarp();
            }
        }
        // ---------------- A producer (software im2col)
        if (grp == 0)
        if constexpr (A_MODE == A_GATHER || A_MODE == A_STEM) {
            const T* __restrict__ in = static_cast<const T*>(p.in);
            int n = 0, oh = 0, ow = 0;
            if (row_ok) {
                const int hw = p.Ho * p.Wo;
                n = static_cast<int>(r / hw);
                const int rem = static_cast<int>(r - static_cast<long long>(n) * hw);
                oh = rem / p.Wo;
                ow = rem - oh * p.Wo;
            }
            const int ih0 = oh * p.stride - p.pad, iw0 = ow * p.stride - p.pad;
            const T* base = in + static_cast<size_t>(n) * p.H * p.W * p.Cin;
            const uint32_t row_off = static_cast<uint32_t>(t) * 128u;
            const uint32_t sw = static_cast<uint32_t>(t) & 7u;
            const bool uniform_tap = (p.Cin % TILE_K) == 0;
            const int taps = p.kh * p.kw;
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % STAGES;
                const int it = kb / STAGES;
                mbar_wait(bar_empty + s * 8, (it & 1) ^ 1);
                const uint32_t dst = a_base + s * A_STAGE_BYTES + row_off;
                if constexpr (A_MODE == A_STEM) {
                    const int kw_mask = p.kwp - 1;
                    const int kw_shift = 31 - __clz(p.kwp);
#pragma unroll
                    for (int pp = 0; pp < 16; ++pp) {             // 16 pixels (8 B each) per 128-byte K slice
                        const int idx = kb * 16 + pp;
                        const int khi = idx >> kw_shift, kwi = idx & kw_mask;
                        const int ih = ih0 + khi, iw = iw0 + kwi;
                        const bool ok = row_ok && khi < p.kh && static_cast<unsigned>(ih) < static_cast<unsigned>(p.H) &&
                                        static_cast<unsigned>(iw) < static_cast<unsigned>(p.W);
                        const T* src = ok ? base + (static_cast<size_t>(ih) * p.W + iw) * 4 : in;
                        cp_async8(dst + (((pp >> 1) ^ sw) << 4) + (pp & 1) * 8, src, ok);
                    }
                } else if (uniform_tap) {
                    const int k0 = kb * TILE_K;
                    const int tap = k0 / p.Cin;
                    const int c0 = k0 - tap * p.Cin;
                    const int khi = tap / p.kw, kwi = tap - khi * p.kw;
                    const int ih = ih0 + khi, iw = iw0 + kwi;
                    const bool ok = row_ok && static_cast<unsigned>(ih) < static_cast<unsigned>(p.H) &&
                                    static_cast<unsigned>(iw) < static_cast<unsigned>(p.W);
                    const T* src = ok ? base + (static_cast<size_t>(ih) * p.W + iw) * p.Cin + c0 : in;
#pragma unroll
                    for (int j = 0; j < 8; ++j) cp_async16(dst + ((j ^ sw) << 4), src + j * 8, ok);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int kidx = kb * TILE_K + j * 8;
                        const int tap = kidx / p.Cin;
                        const int c = kidx - tap * p.Cin;
                        const int khi = tap / p.kw, kwi = tap - khi * p.kw;
                        const int ih = ih0 + khi, iw = iw0 + kwi;
                        const bool ok = row_ok && tap < taps && static_cast<unsigned>(ih) < static_cast<unsigned>(p.H) &&
                                        static_cast<unsigned>(iw) < static_cast<unsigned>(p.W);
                        const T* src = ok ? base + (static_cast<size_t>(ih) * p.W + iw) * p.Cin + c : in;
                        cp_async16(dst + ((j ^ sw) << 4), src, ok);
                    }
                }
                cp_async_commit();
                if (kb >= GATHER_LAG) {
                    cp_async_wait<GATHER_LAG>();
                    fence_proxy_async_smem();                     // generic-proxy writes -> async-proxy (UMMA) reads
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_full + ((kb - GATHER_LAG) % STAGES) * 8);
                }
            }
            // drain the last min(GATHER_LAG, num_kb) groups
            for (int kb = (num_kb > GATHER_LAG ? num_kb - GATHER_LAG : 0); kb < num_kb; ++kb) {
                const int pending = num_kb - 1 - kb;
                if (pending >= 1) cp_async_wait<1>(); else cp_async_wait<0>();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_full + (kb % STAGES) * 8);
            }
        }
        // ---------------- epilogue
        mbar_wait(bar_tmem, 0);                                   // all MMAs retired: accumulator ready, pipeline smem free
        tc_fence_after();
        if (epi_tma) {
            const uint32_t stage_tile = a_base;                   // [BLOCK_N/64][128 rows][128 B], 128B-swizzled
            const bool has_res = p.res != nullptr;
            if (has_res) {
                if (grp == 0 && t == 0) {
                    mbar_arrive_expect_tx(bar_res, L::EPI_BYTES);
#pragma unroll
                    for (int bx = 0; bx < (BLOCK_N >= 64 ? BLOCK_N / 64 : 1); ++bx)
                        tma_load_2d(stage_tile + bx * (TILE_M * 128), &maps.res, bar_res, n0 + bx * 64, m_tile * TILE_M);
                }
                mbar_wait(bar_res, 0);
            }
            const uint32_t row_addr = stage_tile + static_cast<uint32_t>(t) * 128u;
            const uint32_t sw = static_cast<uint32_t>(t) & 7u;
#pragma unroll 1
            for (int c = grp * (BLOCK_N / 64); c < (grp + 1) * (BLOCK_N / 64); ++c) {
                uint32_t v[32];
                tmem_ld_32x32(tmem_acc + (static_cast<uint32_t>(q4 * 32) << 16) + c * 32, v);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int col = c * 32 + q * 8;               // column inside the tile
                    const uint32_t addr = row_addr + (col >> 6) * (TILE_M * 128) + ((((col & 63) >> 3) ^ sw) << 4);
                    float f[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[q * 8 + e]) + sbias[col + e];
                    if (has_res) {
                        uint32_t ru[4];
                        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(ru[0]), "=r"(ru[1]), "=r"(ru[2]), "=r"(ru[3]) : "r"(addr));
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 rf = DT<T>::unpack2(ru[e]);
                            f[2 * e] += rf.x;
                            f[2 * e + 1] += rf.y;
                        }
                    }
                    if (p.relu) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.f);
                    }
                    const uint32_t o0 = DT<T>::pack2(f[0], f[1]), o1 = DT<T>::pack2(f[2], f[3]);
                    const uint32_t o2 = DT<T>::pack2(f[4], f[5]), o3 = DT<T>::pack2(f[6], f[7]);
                    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
                }
            }
            fence_proxy_async_smem();                             // generic-proxy smem writes -> TMA store reads
            named_bar_sync(1, 256);
            if (grp == 0 && t == 0) {
#pragma unroll
                for (int bx = 0; bx < (BLOCK_N >= 64 ? BLOCK_N / 64 : 1); ++bx)
                    if (n0 + bx * 64 < p.Cout)
                        tma_store_2d(&maps.out, stage_tile + bx * (TILE_M * 128), p.out_coff + n0 + bx * 64, m_tile * TILE_M);
                tma_store_commit();
                tma_store_wait_read0();                           // smem must stay valid until the store has read it
            }
        } else if (grp == 0) {
            T* __restrict__ out = static_cast<T*>(p.out);
            const T* __restrict__ res = static_cast<const T*>(p.res);
            const size_t out_row = static_cast<size_t>(r) * p.out_ld + p.out_coff;
            const size_t res_row = static_cast<size_t>(r) * p.res_ld;
#pragma unroll 1
            for (int c = 0; c < BLOCK_N / 32; ++c) {
                uint32_t v[32];
                tmem_ld_32x32(tmem_acc + (static_cast<uint32_t>(q4 * 32) << 16) + c * 32, v);
                tmem_ld_wait();
                if (row_ok) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int col = n0 + c * 32 + q * 8;
                        if (col < p.Cout) {
                            float f[8];
#pragma unroll
                            for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[q * 8 + e]) + sbias[c * 32 + q * 8 + e];
                            if (res != nullptr) {
                                const uint4 rv = *reinterpret_cast<const uint4*>(res + res_row + col);
                                const uint32_t ru[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const float2 rf = DT<T>::unpack2(ru[e]);
                                    f[2 * e] += rf.x;
                                    f[2 * e + 1] += rf.y;
                                }
                            }
                            if (p.relu) {
#pragma unroll
                                for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.f);
                            }
                            uint4 ov;
                            ov.x = DT<T>::pack2(f[0], f[1]);
                            ov.y = DT<T>::pack2(f[2], f[3]);
                            ov.z = DT<T>::pack2(f[4], f[5]);
                            ov.w = DT<T>::pack2(f[6], f[7]);
                            *reinterpret_cast<uint4*>(out + out_row + col) = ov;
                        }
                    }
                }
            }
        }
    } else if (warp == 4) {
        // ---------------- TMA producer
        if (lane == 0) {
            constexpr uint32_t tx_bytes = L::B_STAGE_BYTES + ((A_MODE == A_TILED || A_MODE == A_IM2COL) ? A_STAGE_BYTES : 0);
            int pw = 0, ph = 0, pn = 0;                           // im2col base pixel of the tile's first row
            if constexpr (A_MODE == A_IM2COL) {
                const long long r0 = static_cast<long long>(m_tile) * TILE_M;
                const int hw = p.Ho * p.Wo;
                pn = static_cast<int>(r0 / hw);
                const int rem = static_cast<int>(r0 - static_cast<long long>(pn) * hw);
                const int oh = rem / p.Wo, ow = rem - oh * p.Wo;
                pw = ow * p.stride - p.pad;
                ph = oh * p.stride - p.pad;
            }
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % STAGES;
                const int it = kb / STAGES;
                mbar_wait(bar_empty + s * 8, (it & 1) ^ 1);
                mbar_arrive_expect_tx(bar_full + s * 8, tx_bytes);
                if constexpr (A_MODE == A_GATHER || A_MODE == A_STEM)
                    tma_load_2d(b_base + s * L::B_STAGE_BYTES, &maps.b, bar_full + s * 8, kb * TILE_K, n0);
                if constexpr (A_MODE == A_TILED) {
                    tma_load_2d(a_base + s * A_STAGE_BYTES, &maps.a, bar_full + s * 8, kb * TILE_K, m_tile * TILE_M);
                } else if constexpr (A_MODE == A_IM2COL) {
                    const int k0 = kb * TILE_K;
                    const int tap = k0 / p.Cin;
                    const int c0 = k0 - tap * p.Cin;
                    const int khi = tap / p.kw, kwi = tap - khi * p.kw;
                    tma_load_im2col_4d(a_base + s * A_STAGE_BYTES, &maps.a, bar_full + s * 8, c0, pw, ph, pn,
                                       static_cast<uint16_t>(kwi), static_cast<uint16_t>(khi));
                }
            }
        }
        __syncwarp();
    } else {
        // ---------------- MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_f16(DT<T>::umma_fmt, TILE_M, BLOCK_N < 16 ? 16 : BLOCK_N);
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % STAGES;
                const int it = kb / STAGES;
                mbar_wait(bar_full + s * 8, it & 1);
                tc_fence_after();
                const uint32_t a_s = a_base + s * A_STAGE_BYTES;
                const uint32_t b_s = b_base + s * L::B_STAGE_BYTES;
#pragma unroll
                for (int k = 0; k < TILE_K / 16; ++k) {
                    umma_f16(tmem_acc, umma_desc_sw128(a_s + k * 32), umma_desc_sw128(b_s + k * 32), idesc,
                             static_cast<uint32_t>((kb | k) != 0));
                }
                umma_commit(bar_empty + s * 8);                   // frees the smem stage when these MMAs retire
            }
            umma_commit(bar_tmem);                                // accumulator complete
        }
        __syncwarp();
    }

    // ---------------- teardown
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc(tmem_acc, TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------ persistent kernel
// One CTA per SM loops over output tiles (tile = blockIdx.x + i*gridDim.x, Cout tiles fastest so CTAs running
// concurrently share the A tile in L2).  Compared with the one-tile kernel above it
//   * pays barrier init / TMEM alloc / descriptor fetch once per SM instead of once per tile,
//   * double-buffers the accumulator in TMEM (2 x BLOCK_N columns): the MMA warp starts tile i+1 while the
//     epilogue warps drain tile i,
//   * double-buffers the epilogue staging tile: the residual of tile i+1 is TMA-prefetched while tile i is being
//     combined, and the TMA store of tile i overlaps the main loop of tile i+1.
// A comes by TMA (tiled or im2col), so there are no gather warps: warp 0 = TMA producer, warp 1 = MMA issuer,
// warp 2 = TMEM owner, warps 4-11 = epilogue (two groups of four warps, each group owns half of the columns:
// short-K layers are bound by the epilogue's conversion work, so it gets 8 warps).
constexpr int CONV_TCP_THREADS = 384;          // warps 0-3: TMA / MMA / TMEM / idle; warps 4-11: epilogue (2 column halves)

// Epilogue staging: NBUF buffers of TILE_M x EPI_N 16-bit values (one 128B-swizzled TMA box each).  Life cycle of a
// buffer: [residual TMA load ->] combine in place -> TMA store.  With four 64-column buffers the residual of item i+2 is
// requested at the top of item i into the buffer whose store was issued at the end of item i-2 (long drained), so the
// leader never waits for a store and 32 KB of residual per SM are in flight ahead of the combine; the first version
// (two 128-column buffers, same 64 KB) stalled for the previous item's store at the top of EVERY item and had at most
// one residual tile in flight (ncu: 'barrier' was the top stall of the 1x1 convs, profiles/ncu_r01c.md).
template <int BLOCK_N, int STAGES, int NBUF = 4>
struct ConvTcpSmem {
    static constexpr int B_STAGE_BYTES = BLOCK_N * TILE_K * 2;
    static constexpr int EPI_N = 64;                                  // epilogue sub-tile width (columns)
    static constexpr int EPI_BUFS = NBUF;
    static constexpr int EPI_BYTES = TILE_M * EPI_N * 2;
    static constexpr int A_OFF = 0;
    static constexpr int B_OFF = STAGES * A_STAGE_BYTES;
    static constexpr int EPI_OFF = B_OFF + STAGES * B_STAGE_BYTES;
    static constexpr int BAR_OFF = EPI_OFF + NBUF * EPI_BYTES;     // full[S], empty[S], tfull[2], tempty[2], rfull[NBUF]
    static constexpr int TMEMPTR_OFF = BAR_OFF + (2 * STAGES + 4 + NBUF) * 8;
    static constexpr int BIAS_OFF = (TMEMPTR_OFF + 8 + 15) / 16 * 16;
    static constexpr int MAX_COUT = 2048;
    static constexpr int TOTAL = BIAS_OFF + MAX_COUT * 4;
    static constexpr int DYN_BYTES = TOTAL + 1024;
    static_assert(DYN_BYTES <= 232448, "exceeds the 227 KB dynamic shared memory limit");
};

template <typename T, int BLOCK_N, int STAGES, int A_MODE>
__global__ void __launch_bounds__(CONV_TCP_THREADS, 1)
conv_tcp_kernel(const ConvParams p, const __grid_constant__ ConvTcMaps maps, int n_tiles, int total_tiles)
{
    griddep_launch();
    static_assert(A_MODE == A_TILED || A_MODE == A_IM2COL, "persistent kernel is TMA-fed");
    using L = ConvTcpSmem<BLOCK_N, STAGES>;
    constexpr int NBUF = L::EPI_BUFS;
    constexpr int RES_AHEAD = NBUF > 2 ? NBUF - 2 : 1;            // residual prefetch distance in epilogue items
    constexpr int ST_PENDING = NBUF - RES_AHEAD - 1;              // bulk-store groups that may still be reading smem
    constexpr int TMEM_COLS = 2 * BLOCK_N;
    constexpr int EPI_N = L::EPI_N;
    constexpr int NSUB = BLOCK_N / EPI_N;                        // 128-column epilogue sub-tiles per accumulator
    constexpr int BOXES = EPI_N / 64;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
    const uint32_t a_base = sbase + L::A_OFF;
    const uint32_t b_base = sbase + L::B_OFF;
    const uint32_t e_base = sbase + L::EPI_OFF;
    const uint32_t bar_full = sbase + L::BAR_OFF;
    const uint32_t bar_empty = bar_full + STAGES * 8;
    const uint32_t bar_tfull = bar_empty + STAGES * 8;
    const uint32_t bar_tempty = bar_tfull + 16;
    const uint32_t bar_rfull = bar_tempty + 16;
    volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(sgen + L::TMEMPTR_OFF);
    float* sbias = reinterpret_cast<float*>(sgen + L::BIAS_OFF);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_kb = (p.K + TILE_K - 1) / TILE_K;
    const bool has_res = p.res != nullptr;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + s * 8, 1); mbar_init(bar_empty + s * 8, 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + a * 8, 1); mbar_init(bar_tempty + a * 8, 8); }
        for (int a = 0; a < NBUF; ++a) mbar_init(bar_rfull + a * 8, 1);
        mbar_fence_init();
    }
    for (int c = threadIdx.x; c < p.Cout; c += CONV_TCP_THREADS) sbias[c] = p.bias[c];
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a); tma_prefetch_desc(&maps.b); tma_prefetch_desc(&maps.out);
        if (has_res) tma_prefetch_desc(&maps.res);
    }
    if (warp == 2) {
        tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_s)), TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    griddep_wait();
    const uint32_t tmem_base = *tmem_ptr_s;

    if (warp == 0) {
        // ================= TMA producer (A; arms the full barrier for both operands)
        if (lane == 0) {
            constexpr uint32_t tx_bytes = L::B_STAGE_BYTES + A_STAGE_BYTES;
            const int hw = p.Ho * p.Wo;
            uint32_t kc = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int m_tile = tile / n_tiles;
                int pw = 0, ph = 0, pn = 0;
                if constexpr (A_MODE == A_IM2COL) {
                    const long long r0 = static_cast<long long>(m_tile) * TILE_M;
                    pn = static_cast<int>(r0 / hw);
                    const int rem = static_cast<int>(r0 - static_cast<long long>(pn) * hw);
                    const int oh = rem / p.Wo, ow = rem - oh * p.Wo;
                    pw = ow * p.stride - p.pad;
                    ph = oh * p.stride - p.pad;
                }
                for (int kb = 0; kb < num_kb; ++kb, ++kc) {
                    const uint32_t s = kc % STAGES, it = kc / STAGES;
                    mbar_wait(bar_empty + s * 8, (it & 1) ^ 1);
                    mbar_arrive_expect_tx(bar_full + s * 8, tx_bytes);
                    if constexpr (A_MODE == A_TILED) {
                        tma_load_2d(a_base + s * A_STAGE_BYTES, &maps.a, bar_full + s * 8, kb * TILE_K, m_tile * TILE_M);
                    } else {
                        const int k0 = kb * TILE_K;
                        const int tap = k0 / p.Cin;
                        const int c0 = k0 - tap * p.Cin;
                        const int khi = tap / p.kw, kwi = tap - khi * p.kw;
                        tma_load_im2col_4d(a_base + s * A_STAGE_BYTES, &maps.a, bar_full + s * 8, c0, pw, ph, pn,
                                           static_cast<uint16_t>(kwi), static_cast<uint16_t>(khi));
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 3) {
        // ================= second producer: the weight tiles, same stage / phase sequence as warp 0
        if (lane == 0) {
            uint32_t kc = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int n0 = (tile % n_tiles) * BLOCK_N;
                for (int kb = 0; kb < num_kb; ++kb, ++kc) {
                    const uint32_t s = kc % STAGES, it = kc / STAGES;
                    mbar_wait(bar_empty + s * 8, (it & 1) ^ 1);
                    tma_load_2d(b_base + s * L::B_STAGE_BYTES, &maps.b, bar_full + s * 8, kb * TILE_K, n0);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_f16(DT<T>::umma_fmt, TILE_M, BLOCK_N);
            uint32_t kc = 0, tc = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tc) {
                const uint32_t a = tc & 1, aph = (tc >> 1) & 1;
                mbar_wait(bar_tempty + a * 8, aph ^ 1);            // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t tmem_acc = tmem_base + a * BLOCK_N;
                for (int kb = 0; kb < num_kb; ++kb, ++kc) {
                    const uint32_t s = kc % STAGES, it = kc / STAGES;
                    mbar_wait(bar_full + s * 8, it & 1);
                    tc_fence_after();
                    const uint32_t a_s = a_base + s * A_STAGE_BYTES;
                    const uint32_t b_s = b_base + s * L::B_STAGE_BYTES;
#pragma unroll
                    for (int k = 0; k < TILE_K / 16; ++k)
                        umma_f16(tmem_acc, umma_desc_sw128(a_s + k * 32), umma_desc_sw128(b_s + k * 32), idesc,
                                 static_cast<uint32_t>((kb | k) != 0));
                    umma_commit(bar_empty + s * 8);
                }
                umma_commit(bar_tfull + a * 8);
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ================= epilogue (256 threads; row t == TMEM lane t; column half `grp`)
        const int q4 = warp & 3;                                   // TMEM lane quarter this warp may access
        const int grp = (warp - 4) >> 2;                           // 0: columns [0, N/2), 1: [N/2, N)
        const int t = q4 * 32 + lane;
        const bool leader = (warp == 4 && lane == 0);
        const uint32_t sw = static_cast<uint32_t>(t) & 7u;
        // epilogue work items are (tile, 64-column sub-tile h); item j uses staging buffer / residual barrier j % NBUF
        auto issue_res = [&](uint32_t j) {                          // residual of this CTA's item j
            const int tile = static_cast<int>(blockIdx.x + (j / NSUB) * gridDim.x);
            if (tile >= total_tiles) return;
            const int h = static_cast<int>(j % NSUB);
            const uint32_t e = j % NBUF;
            const int n_tile = tile % n_tiles, m_tile = tile / n_tiles;
            mbar_arrive_expect_tx(bar_rfull + e * 8, L::EPI_BYTES);
#pragma unroll
            for (int bx = 0; bx < BOXES; ++bx)
                tma_load_2d(e_base + e * L::EPI_BYTES + bx * (TILE_M * 128), &maps.res, bar_rfull + e * 8,
                            n_tile * BLOCK_N + h * EPI_N + bx * 64, m_tile * TILE_M);
        };
        // two buffers and no residual: the drain check moves to just before the barrier (see below)
        const bool wait_at_top = has_res || NBUF > 2;
        if (leader && has_res)
            for (int d = 0; d < RES_AHEAD; ++d) issue_res(d);
        uint32_t tc = 0, ec = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tc) {
            const uint32_t a = tc & 1, aph = (tc >> 1) & 1;
            const int n_tile = tile % n_tiles, m_tile = tile / n_tiles;
            const int n0 = n_tile * BLOCK_N;
#pragma unroll 1
            for (int h = 0; h < NSUB; ++h, ++ec) {
                const uint32_t e = ec % NBUF, eph = (ec / NBUF) & 1;
                if (leader && wait_at_top) {
                    tma_store_wait_read<ST_PENDING>();             // the last store out of buffer (ec + RES_AHEAD) % NBUF has drained
                    if (has_res) issue_res(ec + RES_AHEAD);
                }
                if (h == 0) {
                    mbar_wait(bar_tfull + a * 8, aph);
                    tc_fence_after();
                }
                if (has_res) mbar_wait(bar_rfull + e * 8, eph);
                const uint32_t row_addr = e_base + e * L::EPI_BYTES + static_cast<uint32_t>(t) * 128u;
                const uint32_t tmem_acc = tmem_base + a * BLOCK_N + h * EPI_N + (static_cast<uint32_t>(q4 * 32) << 16);
#pragma unroll 1
                for (int c = grp * (EPI_N / 64); c < (grp + 1) * (EPI_N / 64); ++c) {
                    uint32_t v[32];
                    tmem_ld_32x32(tmem_acc + c * 32, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int col = c * 32 + q * 8;
                        const uint32_t addr = row_addr + (col >> 6) * (TILE_M * 128) + ((((col & 63) >> 3) ^ sw) << 4);
                        float f[8];
                        const float4 b0 = *reinterpret_cast<const float4*>(sbias + n0 + h * EPI_N + col);
                        const float4 b1 = *reinterpret_cast<const float4*>(sbias + n0 + h * EPI_N + col + 4);
                        f[0] = __uint_as_float(v[q * 8 + 0]) + b0.x; f[1] = __uint_as_float(v[q * 8 + 1]) + b0.y;
                        f[2] = __uint_as_float(v[q * 8 + 2]) + b0.z; f[3] = __uint_as_float(v[q * 8 + 3]) + b0.w;
                        f[4] = __uint_as_float(v[q * 8 + 4]) + b1.x; f[5] = __uint_as_float(v[q * 8 + 5]) + b1.y;
                        f[6] = __uint_as_float(v[q * 8 + 6]) + b1.z; f[7] = __uint_as_float(v[q * 8 + 7]) + b1.w;
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
                if (h == NSUB - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_tempty + a * 8);    // accumulator a may be overwritten
                }
                fence_proxy_async_smem();
                // two buffers, no residual: the store of the previous item (out of the buffer the NEXT item writes) had this
                // whole item to drain; checking it here, after the leader's own share of the work, costs nothing
                if (leader && !wait_at_top) tma_store_wait_read0();
                named_bar_sync(1, 256);
                if (leader) {
#pragma unroll
                    for (int bx = 0; bx < BOXES; ++bx)
                        tma_store_2d(&maps.out, e_base + e * L::EPI_BYTES + bx * (TILE_M * 128),
                                     p.out_coff + n0 + h * EPI_N + bx * 64, m_tile * TILE_M);
                    tma_store_commit();
                }
            }
        }
        if (leader) tma_store_wait_read0();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

#include "conv_tc2.cuh"

// ------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static void* get_driver_fn(const char* name) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint(name, &ptr, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || ptr == nullptr) {
        set_error(std::string("cudaGetDriverEntryPoint(") + name + ") failed");
        return nullptr;
    }
    return ptr;
}

// 2-D 16-bit row-major tensor [rows][ld] viewed as cols columns; box = 64 cols x box_rows rows, 128-byte swizzle.
static bool make_tmap_2d(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) fn = reinterpret_cast<EncodeTiledFn>(get_driver_fn("cuTensorMapEncodeTiled"));
    if (!fn) return false;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * 2};
    cuuint32_t box[2] = {TILE_K, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (code " + std::to_string(static_cast<int>(r)) + ")");
        return false;
    }
    return true;
}

bool make_tmap_2d_k64(CUtensorMap* m, const void* ptr, int rows, int ld, int box_rows) {
    return make_tmap_2d(m, ptr, static_cast<uint64_t>(rows), static_cast<uint64_t>(ld), static_cast<uint64_t>(ld), static_cast<uint32_t>(box_rows));
}

// NHWC activation tensor in im2col mode: 64 channels x 128 output pixels per load.
static bool make_tmap_im2col(CUtensorMap* m, const ConvParams& p) {
    static EncodeIm2colFn fn = nullptr;
    if (!fn) fn = reinterpret_cast<EncodeIm2colFn>(get_driver_fn("cuTensorMapEncodeIm2col"));
    if (!fn) return false;
    cuuint64_t dims[4] = {static_cast<cuuint64_t>(p.Cin), static_cast<cuuint64_t>(p.W), static_cast<cuuint64_t>(p.H),
                          static_cast<cuuint64_t>(p.N)};
    cuuint64_t strides[3] = {static_cast<cuuint64_t>(p.Cin) * 2, static_cast<cuuint64_t>(p.W) * p.Cin * 2,
                             static_cast<cuuint64_t>(p.H) * p.W * p.Cin * 2};
    // bounding box of the filter's top-left corner ("base pixel"): [-pad, dim - 1 + pad - (k-1)]
    int lower[2] = {-p.pad, -p.pad};
    int upper[2] = {p.pad - (p.kw - 1), p.pad - (p.kh - 1)};
    cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(p.stride), static_cast<cuuint32_t>(p.stride), 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(p.in), dims, strides, lower, upper,
                    TILE_K, TILE_M, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeIm2col failed (code " + std::to_string(static_cast<int>(r)) + ")");
        return false;
    }
    return true;
}

int conv_tc_pick_block_n(int cout, int K) {
    if (cout <= 32) return 32;
    if (cout <= 64) return 64;
    // 128 x 256 tiles when there are >= 4 k-blocks to amortise the wider epilogue (measured: K = 64 / 128 expansions
    // are faster at N = 128, everything with K >= 256 and Cout % 256 == 0 is faster at N = 256)
    if (cout >= 256 && (cout % 256) == 0 && K >= 256) return 256;
    return 128;
}

bool conv_tc_make_weight_tmap(ConvWeights& w) {
    if (!make_tmap_2d(&w.tmap_b, w.w_tc, static_cast<uint64_t>(w.cout_pad), static_cast<uint64_t>(w.K_pad),
                      static_cast<uint64_t>(w.K_pad), static_cast<uint32_t>(w.block_n)))
        return false;
    w.has_tmap = true;
    return true;
}

static int g_num_sms = 0;

// CTA-pair (cta_group::2) persistent kernel: 256 x BLOCK_N tiles over clusters of two CTAs
template <typename T, int BLOCK_N, int STAGES>
static bool launch_pair(const ConvParams& p, ConvTcMaps maps, const ConvWeights& w, int mode, int m_tiles, int n_tiles, cudaStream_t s) {
    using L = ConvTc2Smem<BLOCK_N, STAGES>;
    // each CTA loads HALF of the weight tile: box of BLOCK_N/2 rows
    if (!make_tmap_2d(&maps.b, w.w_tc, static_cast<uint64_t>(w.cout_pad), static_cast<uint64_t>(w.K_pad), static_cast<uint64_t>(w.K_pad), BLOCK_N / 2)) return false;
    auto k0 = conv_tcp2_kernel<T, BLOCK_N, STAGES, A_TILED>;
    auto k1 = conv_tcp2_kernel<T, BLOCK_N, STAGES, A_IM2COL>;
    static DeviceOnce attr_done;
    if (attr_done.need()) {
        if (!check_cuda(cudaFuncSetAttribute(k0, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
        if (!check_cuda(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
    }
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (!check_cuda(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev), "sm count")) return false;
    }
    const long long total = static_cast<long long>((m_tiles + 1) / 2) * n_tiles;       // pair tiles
    if (total > 0x7fffffffLL) { set_error("conv_tc: too many tiles"); return false; }
    const long long pairs = g_num_sms / 2;
    const unsigned grid = 2u * static_cast<unsigned>(total < pairs ? total : pairs);
    if (mode == A_TILED) launch_dep(k0, dim3(grid), dim3(CONV_TCP_THREADS), L::DYN_BYTES, s, p, maps, n_tiles, static_cast<int>(total));
    else launch_dep(k1, dim3(grid), dim3(CONV_TCP_THREADS), L::DYN_BYTES, s, p, maps, n_tiles, static_cast<int>(total));
    return check_cuda(cudaGetLastError(), "conv_tcp2 launch");
}

template <typename T, int BLOCK_N, int STAGES>
static bool launch_persistent(const ConvParams& p, const ConvTcMaps& maps, int mode, int m_tiles, int n_tiles, cudaStream_t s) {
    using L = ConvTcpSmem<BLOCK_N, STAGES>;
    auto k0 = conv_tcp_kernel<T, BLOCK_N, STAGES, A_TILED>;
    auto k1 = conv_tcp_kernel<T, BLOCK_N, STAGES, A_IM2COL>;
    static DeviceOnce attr_done;
    if (attr_done.need()) {
        if (!check_cuda(cudaFuncSetAttribute(k0, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
        if (!check_cuda(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
    }
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (!check_cuda(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev), "sm count")) return false;
    }
    const long long total = static_cast<long long>(m_tiles) * n_tiles;
    if (total > 0x7fffffffLL) { set_error("conv_tc: too many tiles"); return false; }
    const unsigned grid = static_cast<unsigned>(total < g_num_sms ? total : g_num_sms);
    if (mode == A_TILED) launch_dep(k0, dim3(grid), dim3(CONV_TCP_THREADS), L::DYN_BYTES, s, p, maps, n_tiles, static_cast<int>(total));
    else launch_dep(k1, dim3(grid), dim3(CONV_TCP_THREADS), L::DYN_BYTES, s, p, maps, n_tiles, static_cast<int>(total));
    return check_cuda(cudaGetLastError(), "conv_tcp launch");
}

template <typename T, int BLOCK_N, int STAGES>
static bool launch_cfg(const ConvParams& p, const ConvWeights& w, cudaStream_t s) {
    using L = ConvTcSmem<BLOCK_N, STAGES>;
    int mode = A_GATHER;
    if (w.kwp > 0) mode = A_STEM;
    else if (p.kh == 1 && p.kw == 1 && p.stride == 1 && p.pad == 0 && (p.Cin % TILE_K) == 0) mode = A_TILED;
    else if ((p.Cin % TILE_K) == 0) mode = A_IM2COL;
    const int m_tiles = (p.M + TILE_M - 1) / TILE_M;
    const int n_tiles = (p.Cout + BLOCK_N - 1) / BLOCK_N;
    ConvTcMaps maps;
    maps.b = w.tmap_b;
    maps.a = w.tmap_b; maps.out = w.tmap_b; maps.res = w.tmap_b;      // placeholders for unused slots
    if (mode == A_TILED) {
        if (!make_tmap_2d(&maps.a, p.in, static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.Cin), static_cast<uint64_t>(p.Cin), TILE_M)) return false;
    } else if (mode == A_IM2COL) {
        if (!make_tmap_im2col(&maps.a, p)) return false;
    }
    if (BLOCK_N >= 64 && (p.Cout & 63) == 0) {
        if (!make_tmap_2d(&maps.out, p.out, static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.out_ld), static_cast<uint64_t>(p.out_ld), TILE_M)) return false;
        if (p.res != nullptr &&
            !make_tmap_2d(&maps.res, p.res, static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.res_ld), static_cast<uint64_t>(p.res_ld), TILE_M)) return false;
    }
    if constexpr (BLOCK_N == 64 || BLOCK_N == 128 || BLOCK_N == 256) {
        // k>1 convs at N<=128: two co-resident one-tile CTAs feed the tensor pipe better than one persistent CTA (measured);
        // at N=256 the operand bytes per MMA cycle drop to 96 B and the persistent kernels (overlapped epilogue) win.
        const bool tma_fed = (mode == A_TILED || mode == A_IM2COL) && (p.Cout & 63) == 0 && p.Cout <= 2048;
        const bool one_tile_better = p.kh * p.kw > 1 && BLOCK_N < 256;
        if (tma_fed && !one_tile_better) {
            if (BLOCK_N == 256 && m_tiles >= 2) return launch_pair<T, 256, 4>(p, maps, w, mode, m_tiles, n_tiles, s);
            return launch_persistent<T, BLOCK_N, (BLOCK_N == 256 ? 3 : (BLOCK_N == 128 ? 4 : 6))>(p, maps, mode, m_tiles, n_tiles, s);
        }
    }
    auto k0 = conv_tc_kernel<T, BLOCK_N, STAGES, A_TILED>;
    auto k1 = conv_tc_kernel<T, BLOCK_N, STAGES, A_IM2COL>;
    auto k2 = conv_tc_kernel<T, BLOCK_N, STAGES, A_GATHER>;
    auto k3 = conv_tc_kernel<T, BLOCK_N, STAGES, A_STEM>;
    static DeviceOnce attr_done;
    if (attr_done.need()) {
        if (!check_cuda(cudaFuncSetAttribute(k0, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
        if (!check_cuda(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
        if (!check_cuda(cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
        if (!check_cuda(cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES), "smem attr")) return false;
    }
    const long long grid = static_cast<long long>(m_tiles) * n_tiles;
    if (grid > 0x7fffffffLL) { set_error("conv_tc: grid too large"); return false; }
    const unsigned g = static_cast<unsigned>(grid);
    if (mode == A_TILED) launch_dep(k0, g, dim3(CONV_TC_THREADS), L::DYN_BYTES, s, p, maps, n_tiles);
    else if (mode == A_IM2COL) launch_dep(k1, g, dim3(CONV_TC_THREADS), L::DYN_BYTES, s, p, maps, n_tiles);
    else if (mode == A_STEM) launch_dep(k3, g, dim3(CONV_TC_THREADS), L::DYN_BYTES, s, p, maps, n_tiles);
    else launch_dep(k2, g, dim3(CONV_TC_THREADS), L::DYN_BYTES, s, p, maps, n_tiles);
    return check_cuda(cudaGetLastError(), "conv_tc launch");
}

template <typename T>
static bool launch_dt(const ConvParams& p, const ConvWeights& w, cudaStream_t s) {
    switch (w.block_n) {
        case 32: return launch_cfg<T, 32, 4>(p, w, s);
        case 64: return launch_cfg<T, 64, 4>(p, w, s);
        case 128: return launch_cfg<T, 128, 3>(p, w, s);
        case 256: return launch_cfg<T, 256, 4>(p, w, s);
        default: set_error("conv_tc: unsupported block_n"); return false;
    }
}

bool conv_tc_launch(const ConvParams& p, const ConvWeights& w, int prec, cudaStream_t s) {
    if (!w.has_tmap) { set_error("conv_tc: weights not packed"); return false; }
    if (((p.Cin % 8) != 0 && w.kwp == 0) || (w.kwp > 0 && p.Cin != 4) || (p.Cout % 8) != 0 || (p.out_ld % 8) != 0 || (p.out_coff % 8) != 0 ||
        (p.res != nullptr && (p.res_ld % 8) != 0)) {
        set_error("conv_tc: channel counts / strides must be multiples of 8");
        return false;
    }
    if (prec == PREC_BF16) return launch_dt<__nv_bfloat16>(p, w, s);
    if (prec == PREC_F16) return launch_dt<__half>(p, w, s);
    set_error("conv_tc: precision must be bf16 or fp16");
    return false;
}

}  // namespace sb
