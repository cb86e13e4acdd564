// CTA-PAIR (cta_group::2) persistent implicit-GEMM conv kernel; included by conv_tc.cu.
//
// Same structure as conv_tcp_kernel, but two CTAs on one SM pair (cluster 2x1x1) compute one 256 x BLOCK_N tile:
//   CTA r loads A rows [128r, 128r+128) of the tile and HALF of the weight tile (rows [r*N/2, (r+1)*N/2)) -- the
//   tensor cores of the pair exchange the B halves, so each SM fetches 4 KB (A) + N*16 B (B half) of operands per
//   MMA instead of 4 KB + N*32 B.  At N = 256 that is 8 KB per 128-cycle MMA = 64 B/cycle, the rate the one-CTA kernels
//   were measured to be capped at (they need 12 KB per 128 cycles => ~67 % of the tensor pipe; profiles/README.md).
//   The leader CTA (rank 0) issues tcgen05.mma.cta_group::2 (M = 256); completion is multicast to both CTAs' barriers;
//   both producers signal the LEADER's full barrier (TMA .cta_group::2 + remote arrive.expect_tx); each CTA drains its
//   own 128 accumulator rows through the same double-buffered TMA-store epilogue.
#pragma once

template <int BLOCK_N, int STAGES, int NBUF = 4>
struct ConvTc2Smem {
    static constexpr int B_STAGE_BYTES = (BLOCK_N / 2) * TILE_K * 2;      // half of the weight tile per CTA
    static constexpr int EPI_N = 64;                                       // see ConvTcpSmem: four 64-column staging buffers
    static constexpr int EPI_BUFS = NBUF;
    static constexpr int EPI_BYTES = TILE_M * EPI_N * 2;
    static constexpr int A_OFF = 0;
    static constexpr int B_OFF = STAGES * A_STAGE_BYTES;
    static constexpr int EPI_OFF = B_OFF + STAGES * B_STAGE_BYTES;
    static constexpr int BAR_OFF = EPI_OFF + NBUF * EPI_BYTES;             // full[S], empty[S], tfull[2], tempty[2], rfull[NBUF]
    static constexpr int TMEMPTR_OFF = BAR_OFF + (2 * STAGES + 4 + NBUF) * 8;
    static constexpr int BIAS_OFF = (TMEMPTR_OFF + 8 + 15) / 16 * 16;
    static constexpr int MAX_COUT = 2048;
    static constexpr int TOTAL = BIAS_OFF + MAX_COUT * 4;
    static constexpr int DYN_BYTES = TOTAL + 1024;
    static_assert(DYN_BYTES <= 232448, "exceeds the 227 KB dynamic shared memory limit");
    static_assert((B_OFF % 1024) == 0 && (EPI_OFF % 1024) == 0 && (B_STAGE_BYTES % 1024) == 0, "swizzled tiles must be 1024-byte aligned");
};

template <typename T, int BLOCK_N, int STAGES, int A_MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CONV_TCP_THREADS, 1)
conv_tcp2_kernel(const ConvParams p, const __grid_constant__ ConvTcMaps maps, int n_tiles, int total_tiles /* pair tiles */)
{
    griddep_launch();
    static_assert(A_MODE == A_TILED || A_MODE == A_IM2COL, "pair kernel is TMA-fed");
    using L = ConvTc2Smem<BLOCK_N, STAGES>;
    constexpr int NBUF = L::EPI_BUFS;
    constexpr int RES_AHEAD = NBUF > 2 ? NBUF - 2 : 1;            // residual prefetch distance in epilogue items
    constexpr int ST_PENDING = NBUF - RES_AHEAD - 1;              // bulk-store groups that may still be reading smem
    constexpr int TMEM_COLS = 2 * BLOCK_N;
    constexpr int EPI_N = L::EPI_N;
    constexpr int NSUB = BLOCK_N / EPI_N;
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
    const uint32_t rank = cluster_ctarank();
    const int first_tile = static_cast<int>(cluster_id_x());
    const int tile_step = static_cast<int>(cluster_nclusters_x());
    const int num_kb = (p.K + TILE_K - 1) / TILE_K;
    const bool has_res = p.res != nullptr;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + s * 8, 2); mbar_init(bar_empty + s * 8, 1); }   // full: both producers
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + a * 8, 1); mbar_init(bar_tempty + a * 8, 16); }
        for (int a = 0; a < NBUF; ++a) mbar_init(bar_rfull + a * 8, 1);
        mbar_fence_init();
    }
    for (int c = threadIdx.x; c < p.Cout; c += CONV_TCP_THREADS) sbias[c] = p.bias[c];
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a); tma_prefetch_desc(&maps.b); tma_prefetch_desc(&maps.out);
        if (has_res) tma_prefetch_desc(&maps.res);
    }
    if (warp == 2) tmem_alloc_2cta(smem_u32(const_cast<uint32_t*>(tmem_ptr_s)), TMEM_COLS);
    tc_fence_before();
    cluster_sync_all();                                            // both CTAs' barriers and TMEM are ready
    tc_fence_after();
    griddep_wait();
    const uint32_t tmem_base = *tmem_ptr_s;

    if (warp == 0) {
        // ================= TMA producer (A; one per CTA, arms the leader's full barrier for both operands)
        if (lane == 0) {
            constexpr uint32_t tx_bytes = L::B_STAGE_BYTES + A_STAGE_BYTES;
            const int hw = p.Ho * p.Wo;
            uint32_t kc = 0;
            for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
                const int m_tile = (tile / n_tiles) * 2 + static_cast<int>(rank);
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
                    mbar_wait(bar_empty + s * 8, (it & 1) ^ 1);                  // own stage released (multicast commit)
                    const uint32_t lead_full = mapa_u32(bar_full + s * 8, 0);
                    mbar_arrive_expect_tx_cluster(lead_full, tx_bytes);
                    if constexpr (A_MODE == A_TILED) {
                        tma_load_2d_2sm(a_base + s * A_STAGE_BYTES, &maps.a, lead_full, kb * TILE_K, m_tile * TILE_M);
                    } else {
                        const int k0 = kb * TILE_K;
                        const int tap = k0 / p.Cin;
                        const int c0 = k0 - tap * p.Cin;
                        const int khi = tap / p.kw, kwi = tap - khi * p.kw;
                        tma_load_im2col_4d_2sm(a_base + s * A_STAGE_BYTES, &maps.a, lead_full, c0, pw, ph, pn,
                                               static_cast<uint16_t>(kwi), static_cast<uint16_t>(khi));
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 3) {
        // ================= second producer: the weight half-tiles, same stage / phase sequence as warp 0.
        // Bytes that land before warp 0 has armed the barrier only make the tx-count transiently negative.
        if (lane == 0) {
            uint32_t kc = 0;
            for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
                const int n_tile = tile % n_tiles;
                const int nrow0 = n_tile * BLOCK_N + static_cast<int>(rank) * (BLOCK_N / 2);
                for (int kb = 0; kb < num_kb; ++kb, ++kc) {
                    const uint32_t s = kc % STAGES, it = kc / STAGES;
                    mbar_wait(bar_empty + s * 8, (it & 1) ^ 1);
                    tma_load_2d_2sm(b_base + s * L::B_STAGE_BYTES, &maps.b, mapa_u32(bar_full + s * 8, 0), kb * TILE_K, nrow0);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer (leader CTA only)
        if (lane == 0 && rank == 0) {
            constexpr uint32_t idesc = umma_idesc_f16(DT<T>::umma_fmt, 2 * TILE_M, BLOCK_N);
            uint32_t kc = 0, tc = 0;
            for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++tc) {
                const uint32_t a = tc & 1, aph = (tc >> 1) & 1;
                mbar_wait(bar_tempty + a * 8, aph ^ 1);            // both CTAs' epilogues have drained accumulator a
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
                        umma_f16_2cta(tmem_acc, umma_desc_sw128(a_s + k * 32), umma_desc_sw128(b_s + k * 32), idesc,
                                      static_cast<uint32_t>((kb | k) != 0));
                    umma_commit_2cta(bar_empty + s * 8);           // frees the stage in BOTH CTAs
                }
                umma_commit_2cta(bar_tfull + a * 8);               // accumulator ready in BOTH CTAs
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ================= epilogue: this CTA's 128 rows of the pair tile
        const int q4 = warp & 3;
        const int grp = (warp - 4) >> 2;
        const int t = q4 * 32 + lane;
        const bool leader = (warp == 4 && lane == 0);
        const uint32_t sw = static_cast<uint32_t>(t) & 7u;
        const uint32_t lead_tempty = mapa_u32(bar_tempty, 0);
        auto issue_res = [&](uint32_t j) {                          // residual of this CTA's epilogue item j
            const int tile = first_tile + static_cast<int>(j / NSUB) * tile_step;
            if (tile >= total_tiles) return;
            const int h = static_cast<int>(j % NSUB);
            const uint32_t e = j % NBUF;
            const int n_tile = tile % n_tiles, m_tile = (tile / n_tiles) * 2 + static_cast<int>(rank);
            mbar_arrive_expect_tx(bar_rfull + e * 8, L::EPI_BYTES);
#pragma unroll
            for (int bx = 0; bx < BOXES; ++bx)
                tma_load_2d(e_base + e * L::EPI_BYTES + bx * (TILE_M * 128), &maps.res, bar_rfull + e * 8,
                            n_tile * BLOCK_N + h * EPI_N + bx * 64, m_tile * TILE_M);
        };
        const bool wait_at_top = has_res || NBUF > 2;
        if (leader && has_res)
            for (int d = 0; d < RES_AHEAD; ++d) issue_res(d);
        uint32_t tc = 0, ec = 0;
        for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++tc) {
            const uint32_t a = tc & 1, aph = (tc >> 1) & 1;
            const int n_tile = tile % n_tiles, m_tile = (tile / n_tiles) * 2 + static_cast<int>(rank);
            const int n0 = n_tile * BLOCK_N;
#pragma unroll 1
            for (int h = 0; h < NSUB; ++h, ++ec) {
                const uint32_t e = ec % NBUF, eph = (ec / NBUF) & 1;
                if (leader && wait_at_top) {
                    tma_store_wait_read<ST_PENDING>();             // the last store out of buffer (ec + RES_AHEAD) % NBUF has drained
                    if (has_res) issue_res(ec + RES_AHEAD);
                }
                if (h == 0) { mbar_wait(bar_tfull + a * 8, aph); tc_fence_after(); }
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
                    if (lane == 0) mbar_arrive_cluster(lead_tempty + a * 8);   // tell the leader's MMA thread (count 16 = 8 warps x 2 CTAs)
                }
                fence_proxy_async_smem();
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
    cluster_sync_all();                                            // nobody may still read TMEM / signal the peer
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    }
}
