// out = LayerNorm(A W^T + bias + resid) * gamma + beta in ONE kernel (tcgen05 / TMEM / TMA, bf16 in / out, fp32 accumulate).
//
// The wav2vec2 encoder layer is post-LN (HF modeling_wav2vec2.py:576-609, reached through ref:src/model/wav2vec.py:174-180):
//     h = LN(h + out_proj(attn));  h = LN(h + W2 gelu(W1 h))
// so two of its four GEMMs are followed by a LayerNorm over the full 768-wide row.  A 256-wide accumulator tile holds a
// third of a row; the statistics of a row therefore live in THREE tiles.  This kernel runs those three tiles at the same
// time in one thread-block CLUSTER of 3 CTA pairs (6 CTAs; pair p owns columns [256p, 256p+256) of a 256-row block and is
// a cta_group::2 UMMA pair exactly like gemm_tc2_kernel) and exchanges the per-row (sum, sum of squares) through
// distributed shared memory:
//   pass 1  accumulator (TMEM) + bias + residual (TMA -> swizzled staging) -> fp32 sum written BACK into TMEM
//           (tcgen05.st: TMEM is the row buffer, nothing is recomputed), per-thread partial (s1, s2) of its 128 columns
//   exchange every epilogue thread stores its partial into the stats slot of the NP CTAs that hold the same rows
//           (st.shared::cluster), one lane per warp arrives (release.cluster) on their stats mbarrier; waits (acquire.cluster) on its own
//   pass 2  TMEM -> (x - mean) * rstd * gamma + beta -> bf16 -> swizzled staging -> TMA store
// The pre-LayerNorm sum never leaves the SM and is never rounded to bf16 (round 1 stored it in bf16 and re-read it in a
// separate layernorm_kernel launch: 24 launches per forward, 6 % of the step, and the largest single contribution to the
// bf16 path's error -- tools/bf16_noise_floor.py: 1.6 % -> 1.0 % of the largest vertex offset).
// Mainloop, barriers and TMEM double buffering follow gemm_tc2_kernel (gemm_tc.cu); the ring is 4 stages deep here because
// the stats slots and the LayerNorm parameters need 13 KB of shared memory.
//
// Two kernels live here: gemm_ln_kernel (one GEMM + LayerNorm: a2f_gemm_ln, used by the training forward, which also stores
// the pre-LayerNorm sum) and enc_block_kernel further down (up to four GEMM phases of an encoder layer back to back in the
// same cluster: a2f_encoder_block, the inference path).  Both use ln_tile_epilogue for their LayerNorm tiles.
#include "a2f_common.cuh"
#include "gemm_params.cuh"

namespace a2f {

unsigned long long* debug_timeline();   // gemm_tc.cu (a2f_debug_set_timeline)

namespace {

constexpr int LBM = 128;            // rows per CTA (UMMA M = 256 over the pair)
constexpr int LBN = 256;            // columns per pair tile
constexpr int LBK = 64;             // K per stage (one 128-byte swizzle row of bf16)
constexpr int L_THREADS = 320;      // warp 0 TMA producer, warp 1 MMA issuer, warps 2..9 epilogue
constexpr int L_STAGES = 4;
constexpr int L_A_BYTES = LBM * LBK * 2;
constexpr int L_B_BYTES = (LBN / 2) * LBK * 2;
constexpr int L_STAGE_BYTES = L_A_BYTES + L_B_BYTES;
constexpr int L_EPI_BYTES = 16384;  // one 128-row x 128-byte block (64 bf16 columns)
constexpr int L_SBW = 64;           // columns per staging block

struct LnMaps {
    CUtensorMap a, b, c, r;
};

struct LnParams {
    int M, N, K;
    int tiles_m, num_k_blocks;
    const float* bias;
    const float* gamma;
    const float* beta;
    float eps;
    bf16* pre_out;                  // training: the pre-LayerNorm sum x (bf16 [M,N], row stride ldp) for the backward; else NULL
    long long ldp;
};

template <int NP> struct LnCfg {
    static constexpr int STATS_BYTES = 2 * (2 * NP) * LBM * 8;      // [parity][source pair x half][row] float2
    static constexpr int PARAM_BYTES = 3 * LBN * 4;                 // bias | gamma | beta of this pair's 256 columns
    static constexpr size_t SMEM_BYTES = (size_t)L_STAGES * L_STAGE_BYTES + 4 * L_EPI_BYTES + STATS_BYTES + PARAM_BYTES + 256;
};

A2F_D uint64_t ln_smem_desc(uint32_t saddr) {
    // K-major, SWIZZLE_128B: LBO 1 (ignored), SBO 64 (1024 B between 8-row groups), version 1, layout 2
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)1u << 16) | ((uint64_t)64u << 32) | ((uint64_t)1u << 46) |
           ((uint64_t)2u << 61);
}
A2F_D void umma_commit_pair(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}
A2F_D uint32_t map_to_rank(uint32_t saddr, uint32_t rank) {
    uint32_t d;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(d) : "r"(saddr), "r"(rank));
    return d;
}
A2F_D void st_cluster_f2(uint32_t daddr, float a, float b) {
    asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(daddr), "f"(a), "f"(b) : "memory");
}
A2F_D void mbar_arrive_cluster_release(uint32_t daddr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(daddr) : "memory");
}
A2F_D void mbar_wait_cluster_acquire(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (ok) return;
        if (++spins > (1u << 26)) __trap();      // a protocol bug becomes a launch error, not a hung GPU
    }
}

// One 128-row x 256-column tile of the LayerNorm epilogue (8 epilogue warps of one CTA; see the header): residual fetch,
// pass 1, statistics exchange over the cluster, pass 2, TMA store.  Shared by gemm_ln_kernel and enc_block_kernel.
template <int NP>
A2F_D void ln_tile_epilogue(const CUtensorMap* map_r, const CUtensorMap* map_c, const float* sParam, float2* sStats,
                            uint64_t* rbar, uint64_t* stat_bar, uint64_t* tfull, uint32_t tfull_phase, uint64_t* tempty,
                            uint32_t t_acc, int n0, int pr, int hr, int half, int q, int lane, bool leader, int bar_id,
                            uint8_t* stage_base, int row_base, uint32_t it, float inv_n, float eps, bf16* pre_out,
                            long long ldp, int M) {
    const int r_tile = q * 32 + lane;
    const uint32_t par = it & 1u, par_phase = (it >> 1) & 1u;
    // residual blocks of this tile -> the two staging buffers of this half (while the mainloop runs); a buffer is
    // free once the TMA store that last used it has finished reading it
    if (leader) {
        tma_store_wait_read1();
        mbar_expect_tx(&rbar[half * 2 + 0], L_EPI_BYTES);
        tma_load_2d(stage_base, map_r, &rbar[half * 2 + 0], n0 + half * L_SBW, row_base);
        tma_store_wait_read();
        mbar_expect_tx(&rbar[half * 2 + 1], L_EPI_BYTES);
        tma_load_2d(stage_base + L_EPI_BYTES, map_r, &rbar[half * 2 + 1], n0 + (half + 2) * L_SBW, row_base);
    }
    mbar_wait(tfull, tfull_phase);
    tc_fence_after();
    const uint32_t t_row = t_acc + ((uint32_t)(q * 32) << 16);

    // ---- pass 1: x = acc + bias + resid -> TMEM, partial row statistics ----
    float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
    for (int j = 0; j < 2; ++j) {
        const int col0 = (half + 2 * j) * L_SBW;
        const uint8_t* rowp = stage_base + j * L_EPI_BYTES + r_tile * 128;
        float v[L_SBW];
        tmem_ld_32x32(t_row + col0, v);
        tmem_ld_32x32(t_row + col0 + 32, v + 32);
        mbar_wait(&rbar[half * 2 + j], it & 1u);
        tmem_ld_wait();
#pragma unroll
        for (int ch = 0; ch < L_SBW / 8; ++ch) {
            const uint4 u = *reinterpret_cast<const uint4*>(rowp + ((ch ^ (r_tile & 7)) * 16));
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
            const float4 b0 = *reinterpret_cast<const float4*>(sParam + col0 + ch * 8);
            const float4 b1 = *reinterpret_cast<const float4*>(sParam + col0 + ch * 8 + 4);
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = __bfloat1622float2(h2[e]);
                const float x0 = v[ch * 8 + 2 * e] + bb[2 * e] + f.x;
                const float x1 = v[ch * 8 + 2 * e + 1] + bb[2 * e + 1] + f.y;
                v[ch * 8 + 2 * e] = x0;
                v[ch * 8 + 2 * e + 1] = x1;
                s1 += x0 + x1;
                s2 = fmaf(x0, x0, fmaf(x1, x1, s2));
            }
        }
        tmem_st_32x32(t_row + col0, v);
        tmem_st_32x32(t_row + col0 + 32, v + 32);
        if (pre_out != nullptr && row_base + r_tile < M) {
            // training: LayerNorm's backward needs its input; every thread writes its own row's 128 bytes
            bf16* pp = pre_out + (long long)(row_base + r_tile) * ldp + n0 + col0;
#pragma unroll
            for (int ch = 0; ch < L_SBW / 8; ++ch) {
                uint4 u;
                u.x = pack_bf16x2(v[ch * 8 + 0], v[ch * 8 + 1]);
                u.y = pack_bf16x2(v[ch * 8 + 2], v[ch * 8 + 3]);
                u.z = pack_bf16x2(v[ch * 8 + 4], v[ch * 8 + 5]);
                u.w = pack_bf16x2(v[ch * 8 + 6], v[ch * 8 + 7]);
                *reinterpret_cast<uint4*>(pp + ch * 8) = u;
            }
        }
    }
    // ---- exchange: my partial -> the stats slot of every CTA that holds these rows (same hr, all NP pairs) ----
    {
        const uint32_t slot = smem_u32(sStats + ((size_t)par * (2 * NP) + (size_t)(pr * 2 + half)) * LBM + r_tile);
        const uint32_t sbar = smem_u32(&stat_bar[par]);
#pragma unroll
        for (int d = 0; d < NP; ++d) st_cluster_f2(map_to_rank(slot, (uint32_t)(2 * d + hr)), s1, s2);
        // one arrive per warp and destination (release.cluster, cumulative over the warp's stores through __syncwarp): 8 x NP
        // remote arrives per CTA and tile instead of 256 x NP
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int d = 0; d < NP; ++d) mbar_arrive_cluster_release(map_to_rank(sbar, (uint32_t)(2 * d + hr)));
        }
    }
    tmem_st_wait();
    mbar_wait_cluster_acquire(&stat_bar[par], par_phase);
    float S1 = 0.f, S2 = 0.f;
    {
        const float2* st = sStats + (size_t)par * (2 * NP) * LBM + r_tile;
#pragma unroll
        for (int d = 0; d < 2 * NP; ++d) {
            const float2 t = st[(size_t)d * LBM];
            S1 += t.x;
            S2 += t.y;
        }
    }
    const float mean = S1 * inv_n;
    const float var = fmaxf(fmaf(-mean, mean, S2 * inv_n), 0.f);
    const float rstd = rsqrtf(var + eps);
    const float nmr = -mean * rstd;

    // ---- pass 2: normalise, affine, bf16, TMA store ----
#pragma unroll 1
    for (int j = 0; j < 2; ++j) {
        const int col0 = (half + 2 * j) * L_SBW;
        uint8_t* stage_buf = stage_base + j * L_EPI_BYTES;
        uint8_t* rowp = stage_buf + r_tile * 128;
        float v[L_SBW];
        tmem_ld_32x32(t_row + col0, v);
        tmem_ld_32x32(t_row + col0 + 32, v + 32);
        tmem_ld_wait();
        if (j == 1) {
            // last read of this accumulator: hand it back to the MMA warp before the stores
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(tempty);
        }
#pragma unroll
        for (int ch = 0; ch < L_SBW / 8; ++ch) {
            float y[8];
#pragma unroll
            for (int e = 0; e < 8; e += 4) {
                const float4 g = *reinterpret_cast<const float4*>(sParam + LBN + col0 + ch * 8 + e);
                const float4 b = *reinterpret_cast<const float4*>(sParam + 2 * LBN + col0 + ch * 8 + e);
                y[e + 0] = fmaf(fmaf(v[ch * 8 + e + 0], rstd, nmr), g.x, b.x);
                y[e + 1] = fmaf(fmaf(v[ch * 8 + e + 1], rstd, nmr), g.y, b.y);
                y[e + 2] = fmaf(fmaf(v[ch * 8 + e + 2], rstd, nmr), g.z, b.z);
                y[e + 3] = fmaf(fmaf(v[ch * 8 + e + 3], rstd, nmr), g.w, b.w);
            }
            uint4 u;
            u.x = pack_bf16x2(y[0], y[1]);
            u.y = pack_bf16x2(y[2], y[3]);
            u.z = pack_bf16x2(y[4], y[5]);
            u.w = pack_bf16x2(y[6], y[7]);
            *reinterpret_cast<uint4*>(rowp + ((ch ^ (r_tile & 7)) * 16)) = u;
        }
        fence_proxy_async_smem();
        named_bar_sync(bar_id, 128);
        if (leader) {
            tma_store_2d(map_c, stage_buf, n0 + col0, row_base);
            tma_store_commit();
        }
    }
}

template <int NP>
__global__ void __launch_bounds__(L_THREADS, 1)
gemm_ln_kernel(const __grid_constant__ LnMaps maps, const LnParams p) {
    using Cfg = LnCfg<NP>;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sA = smem;
    uint8_t* sB = smem + (size_t)L_STAGES * L_A_BYTES;
    uint8_t* sEpi = smem + (size_t)L_STAGES * L_STAGE_BYTES;                     // [half][buffer] 16 KB each
    float2* sStats = reinterpret_cast<float2*>(sEpi + 4 * L_EPI_BYTES);          // [2][2*NP][128]
    float* sParam = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(sStats) + Cfg::STATS_BYTES);   // bias | gamma | beta
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sParam) + Cfg::PARAM_BYTES);
    uint64_t* full_bar = bars;                        // [STAGES] leader only
    uint64_t* empty_bar = bars + L_STAGES;            // [STAGES] both CTAs of the pair (multicast commit)
    uint64_t* tfull_bar = bars + 2 * L_STAGES;        // [2]      both CTAs (multicast commit)
    uint64_t* tempty_bar = tfull_bar + 2;             // [2]      leader only: 8 epilogue warps x 2 CTAs
    uint64_t* rbar = tempty_bar + 2;                  // [2 halves][2 buffers] residual block landed
    uint64_t* stat_bar = rbar + 4;                    // [2 parities] all partial sums of this CTA's rows landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stat_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();          // 0 .. 2*NP-1
    const int pr = rank >> 1;                         // pair index in the cluster == column block of this pair
    const int hr = rank & 1;                          // which 128 rows of the 256-row block
    const bool is_leader = hr == 0;
    const int cl = (int)cluster_id_x(), n_cl = (int)cluster_count_x();

    if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) __trap();
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a);
        tma_prefetch_desc(&maps.b);
        tma_prefetch_desc(&maps.c);
        tma_prefetch_desc(&maps.r);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < L_STAGES; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], 16);
            mbar_init(&stat_bar[i], NP * 8);
        }
        for (int i = 0; i < 4; ++i) mbar_init(&rbar[i], 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc_2sm<512>(tmem_slot);
    tc_fence_before();
    cluster_sync_all();                               // every CTA's barriers exist before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_sync();

    const int n0 = pr * LBN;                          // first column of this pair

    if (warp == 0) {
        // ===================== TMA producer (both CTAs of the pair) =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int mb = cl; mb < p.tiles_m; mb += n_cl) {
                const int row0 = mb * 2 * LBM + hr * LBM;
                const int wrow0 = n0 + hr * (LBN / 2);
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (is_leader) mbar_expect_tx(&full_bar[stage], 2 * L_STAGE_BYTES);
                    tma_load_2d_2sm(sA + (size_t)stage * L_A_BYTES, &maps.a, &full_bar[stage], kb * LBK, row0);
                    tma_load_2d_2sm(sB + (size_t)stage * L_B_BYTES, &maps.b, &full_bar[stage], kb * LBK, wrow0);
                    if (++stage == L_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA of the pair) =====================
        if (is_leader && lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(LBN >> 3) << 17) |
                                   ((uint32_t)((2 * LBM) >> 4) << 24);
            const uint16_t pair_mask = (uint16_t)(3u << (2 * pr));
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int mb = cl; mb < p.tiles_m; mb += n_cl) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * LBN);
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t adesc = ln_smem_desc(smem_u32(sA + (size_t)stage * L_A_BYTES));
                    const uint64_t bdesc = ln_smem_desc(smem_u32(sB + (size_t)stage * L_B_BYTES));
#pragma unroll
                    for (int k = 0; k < LBK / 16; ++k)
                        umma_f16_2sm(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
                    umma_commit_pair(&empty_bar[stage], pair_mask);
                    if (++stage == L_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit_pair(&tfull_bar[acc], pair_mask);
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue: 8 warps, thread = one row x one column half (2 blocks of 64 columns) ==========
        const int ew = warp - 2;
        const int q = warp & 3;                       // TMEM lane quarter
        const int half = ew >> 2;                     // blocks {half, half + 2} of the tile's four 64-column blocks
        const bool leader = ((ew & 3) == 0) && lane == 0;
        const int bar_id = 1 + half;
        uint8_t* stage_base = sEpi + half * 2 * L_EPI_BYTES;
        // bias | gamma | beta of this pair's 256 columns: loaded once (the pair keeps its column block for every tile)
        {
            const int c = ew * 32 + lane;             // 256 epilogue threads
            sParam[c] = p.bias ? __ldg(p.bias + n0 + c) : 0.f;
            sParam[LBN + c] = __ldg(p.gamma + n0 + c);
            sParam[2 * LBN + c] = __ldg(p.beta + n0 + c);
        }
        named_bar_sync(3, 256);
        int acc = 0;
        uint32_t acc_phase = 0;
        uint32_t it = 0;                              // tiles this CTA has processed
        const float inv_n = 1.0f / (float)p.N;
        for (int mb = cl; mb < p.tiles_m; mb += n_cl, ++it) {
            ln_tile_epilogue<NP>(&maps.r, &maps.c, sParam, sStats, rbar, stat_bar, &tfull_bar[acc], acc_phase, &tempty_bar[acc],
                                 tmem_base + (uint32_t)(acc * LBN), n0, pr, hr, half, q, lane, leader, bar_id, stage_base,
                                 mb * 2 * LBM + hr * LBM, it, inv_n, p.eps, p.pre_out, p.ldp, p.M);
            acc ^= 1;
            if (acc == 0) acc_phase ^= 1;
        }
        if (leader) tma_store_wait_all();
    }

    tc_fence_before();
    cluster_sync_all();                               // nobody signals a CTA that has left; TMEM reads are complete
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2sm<512>(tmem_base);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Everything of an encoder layer that is local to a block of rows, in ONE kernel  (HF modeling_wav2vec2.py:551-609):
//     h1    = LayerNorm(h_in + att Wo^T + bo)                    phase 0   (optional)
//     f     = gelu(h1 W1^T + b1)                                 phase 1   TP = F / (256 NP) tiles per pair
//     h_out = LayerNorm(h1 + f W2^T + b2)                        phase 2
//     qkv   = h_out Wq^T + bq   (in-projection of the NEXT layer) phase 3   (optional) NQT = NQ / (256 NP) tiles per pair
// Only the attention itself mixes rows, so a layer is two launches: attention, then this kernel.  Same cluster of NP CTA
// pairs per 256-row block as gemm_ln_kernel; pair p owns columns [256 p, +256) of the LayerNorm tiles and tile t of a
// multi-tile phase = columns [256 (t NP + p), +256).  The tiles of a row block go through the same smem ring and the same two
// TMEM accumulators back to back: the tensor pipe only drains where the algorithm forces it (the two LayerNorms: every
// column of a row has to exist before the next GEMM can read the row).
// Hand-over between phases: a phase's output is stored with TMA (bf16, stays in L2); when the stores of a tile have
// COMPLETED the two epilogue leaders arrive (release.cluster) on a `pub` mbarrier of the NP CTAs that own the same 128
// rows; the producer warp of those CTAs waits (acquire.cluster) before its first TMA load of that data.  f is published
// per round t (columns [768 t, +768) = tile t of all pairs) and phase 2 waits for round t only at k-block 12 t, so the
// last round is waited for while three quarters of the K loop are still ahead.
// Results are bit-identical to a2f_gemm_ln / a2f_gemm(GELU) / a2f_gemm_ln / a2f_gemm run one after the other.
struct BlkMaps {
    CUtensorMap att, wo, hin, h1, w1, f, w2, c, wq, q;
};

struct BlkParams {
    int M, N;
    int tiles_m;
    int kb0, kb1, kb2, kb3;         // k-blocks of the four phases
    int tp, nqt;                    // tiles per pair in phases 1 and 3
    int has_p0, has_p3;
    const float* bias_o; const float* gamma1; const float* beta1;
    const float* bias1;
    const float* bias2; const float* gamma2; const float* beta2;
    const float* bias_q;
    float eps;
    unsigned long long* timeline;   // debug (a2f_debug_set_timeline): 16 stamps per CTA (clock64, then globaltimer)
};

A2F_D unsigned long long blk_gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define BLK_STAMP(slot) do { if (p.timeline) { p.timeline[blockIdx.x * 16 + (slot)] = (unsigned long long)clock64(); \
                                                p.timeline[(gridDim.x + blockIdx.x) * 16 + (slot)] = blk_gtimer(); } } while (0)

constexpr int BLK_MAX_TP = 4;       // phase-1 tiles per pair (F <= 4 N)
constexpr int BLK_MAX_NQT = 3;      // phase-3 tiles per pair (NQ <= 3 N)

template <int NP> struct BlkCfg {
    static constexpr int STATS_BYTES = LnCfg<NP>::STATS_BYTES;
    // bias_o | gamma1 | beta1 | bias2 | gamma2 | beta2 | bias1 [TP] | bias_q [NQT], 256 floats each
    static constexpr int PARAM_BYTES = (6 + BLK_MAX_TP + BLK_MAX_NQT) * LBN * 4;
    static constexpr size_t SMEM_BYTES = (size_t)L_STAGES * L_STAGE_BYTES + 4 * L_EPI_BYTES + STATS_BYTES + PARAM_BYTES + 256;
};

A2F_D void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// epilogue leader: the TMA stores of this half are in L2 -> tell the producers of the NP CTAs that hold the same rows
template <int NP> A2F_D void blk_publish(uint64_t* bar, int hr) {
    tma_store_wait_all();                              // writes complete, not only read out of shared memory
    fence_proxy_async_all();
    const uint32_t b = smem_u32(bar);
#pragma unroll
    for (int d = 0; d < NP; ++d) mbar_arrive_cluster_release(map_to_rank(b, (uint32_t)(2 * d + hr)));
}

// One 128 x 256 tile of a plain epilogue (8 epilogue warps): out = act(acc + bias) -> bf16 -> TMA store at (col_base, row_base)
template <bool GELU>
A2F_D void blk_plain_tile(const CUtensorMap* map_out, const float* tb, uint64_t* tfull, uint32_t tfull_phase, uint64_t* tempty,
                          uint32_t t_acc, int col_base, int row_base, int half, int q, int lane, bool leader, int bar_id,
                          uint8_t* stage_base) {
    const int r_tile = q * 32 + lane;
    if (leader) tma_store_wait_read();                 // both staging buffers of this half are free again
    named_bar_sync(bar_id, 128);
    mbar_wait(tfull, tfull_phase);
    tc_fence_after();
    const uint32_t t_row = t_acc + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
    for (int j = 0; j < 2; ++j) {
        const int col0 = (half + 2 * j) * L_SBW;
        uint8_t* stage_buf = stage_base + j * L_EPI_BYTES;
        uint8_t* rowp = stage_buf + r_tile * 128;
        float v[L_SBW];
        tmem_ld_32x32(t_row + col0, v);
        tmem_ld_32x32(t_row + col0 + 32, v + 32);
        tmem_ld_wait();
        if (j == 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(tempty);
        }
#pragma unroll
        for (int e = 0; e < L_SBW; e += 4) {
            const float4 f = *reinterpret_cast<const float4*>(tb + col0 + e);
            v[e] += f.x; v[e + 1] += f.y; v[e + 2] += f.z; v[e + 3] += f.w;
        }
        if (GELU) {
#pragma unroll
            for (int e = 0; e < L_SBW; e += 2) {
                const float2 r = gelu_fast2(make_float2(v[e], v[e + 1]));
                v[e] = r.x;
                v[e + 1] = r.y;
            }
        }
#pragma unroll
        for (int ch = 0; ch < L_SBW / 8; ++ch) {
            uint4 u;
            u.x = pack_bf16x2(v[ch * 8 + 0], v[ch * 8 + 1]);
            u.y = pack_bf16x2(v[ch * 8 + 2], v[ch * 8 + 3]);
            u.z = pack_bf16x2(v[ch * 8 + 4], v[ch * 8 + 5]);
            u.w = pack_bf16x2(v[ch * 8 + 6], v[ch * 8 + 7]);
            *reinterpret_cast<uint4*>(rowp + ((ch ^ (r_tile & 7)) * 16)) = u;
        }
        fence_proxy_async_smem();
        named_bar_sync(bar_id, 128);
        if (leader) {
            tma_store_2d(map_out, stage_buf, col_base + col0, row_base);
            tma_store_commit();
        }
    }
}

template <int NP>
__global__ void __launch_bounds__(L_THREADS, 1)
enc_block_kernel(const __grid_constant__ BlkMaps maps, const BlkParams p) {
    using Cfg = BlkCfg<NP>;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sA = smem;
    uint8_t* sB = smem + (size_t)L_STAGES * L_A_BYTES;
    uint8_t* sEpi = smem + (size_t)L_STAGES * L_STAGE_BYTES;
    float2* sStats = reinterpret_cast<float2*>(sEpi + 4 * L_EPI_BYTES);
    float* sP0 = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(sStats) + Cfg::STATS_BYTES);   // bias_o | gamma1 | beta1
    float* sP2 = sP0 + 3 * LBN;                                                  // bias2 | gamma2 | beta2
    float* sBias1 = sP2 + 3 * LBN;                                               // [TP][256]
    float* sBiasQ = sBias1 + BLK_MAX_TP * LBN;                                   // [NQT][256]
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sP0) + Cfg::PARAM_BYTES);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + L_STAGES;
    uint64_t* tfull_bar = bars + 2 * L_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* rbar = tempty_bar + 2;
    uint64_t* stat_bar = rbar + 4;
    uint64_t* f_bar = stat_bar + 2;                   // [TP] round t of f (this CTA's 128 rows, 256 NP columns) is in L2
    uint64_t* h1_bar = f_bar + BLK_MAX_TP;            // h1 (this CTA's 128 rows, all columns) is in L2
    uint64_t* h2_bar = h1_bar + 1;                    // h_out likewise
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(h2_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int pr = rank >> 1;
    const int hr = rank & 1;
    const bool is_leader = hr == 0;
    const int cl = (int)cluster_id_x(), n_cl = (int)cluster_count_x();
    const int TP = p.tp, NQT = p.has_p3 ? p.nqt : 0;
    const bool has_p0 = p.has_p0 != 0;

    if (threadIdx.x == 0) BLK_STAMP(0);
    if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) __trap();
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.h1);
        tma_prefetch_desc(&maps.w1);
        tma_prefetch_desc(&maps.f);
        tma_prefetch_desc(&maps.w2);
        tma_prefetch_desc(&maps.c);
        if (has_p0) {
            tma_prefetch_desc(&maps.att);
            tma_prefetch_desc(&maps.wo);
            tma_prefetch_desc(&maps.hin);
        }
        if (NQT) {
            tma_prefetch_desc(&maps.wq);
            tma_prefetch_desc(&maps.q);
        }
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < L_STAGES; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], 16);
            mbar_init(&stat_bar[i], NP * 8);
        }
        for (int i = 0; i < 4; ++i) mbar_init(&rbar[i], 1);
        for (int i = 0; i < BLK_MAX_TP + 2; ++i) mbar_init(&f_bar[i], 2 * NP);  // 2 epilogue leaders x NP CTAs with these rows
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc_2sm<512>(tmem_slot);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_sync();
    if (threadIdx.x == 0) BLK_STAMP(1);

    const int n0 = pr * LBN;                          // this pair's columns of the LayerNorm tiles
    const int kb_round = (NP * LBN) / LBK;            // k-blocks of phase 2 per round of f

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            uint32_t it = 0;
            auto load = [&](const CUtensorMap* ma, const CUtensorMap* mbm, int kb, int arow, int brow) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                if (is_leader) mbar_expect_tx(&full_bar[stage], 2 * L_STAGE_BYTES);
                tma_load_2d_2sm(sA + (size_t)stage * L_A_BYTES, ma, &full_bar[stage], kb * LBK, arow);
                tma_load_2d_2sm(sB + (size_t)stage * L_B_BYTES, mbm, &full_bar[stage], kb * LBK, brow);
                if (++stage == L_STAGES) { stage = 0; phase ^= 1; }
            };
            for (int mb = cl; mb < p.tiles_m; mb += n_cl, ++it) {
                const int row0 = mb * 2 * LBM + hr * LBM;
                const int wrow_ln = n0 + hr * (LBN / 2);
                if (has_p0) {
                    for (int kb = 0; kb < p.kb0; ++kb) load(&maps.att, &maps.wo, kb, row0, wrow_ln);
                    mbar_wait_cluster_acquire(h1_bar, it & 1u);   // h1: TMA stores of the NP CTAs with these rows, TMA loads here
                    fence_proxy_async_all();
                }
                for (int t = 0; t < TP; ++t) {
                    const int wrow0 = (t * NP + pr) * LBN + hr * (LBN / 2);
                    for (int kb = 0; kb < p.kb1; ++kb) load(&maps.h1, &maps.w1, kb, row0, wrow0);
                }
                for (int kb = 0; kb < p.kb2; ++kb) {
                    if (kb % kb_round == 0) {
                        mbar_wait_cluster_acquire(&f_bar[kb / kb_round], it & 1u);
                        fence_proxy_async_all();
                    }
                    load(&maps.f, &maps.w2, kb, row0, wrow_ln);
                }
                if (NQT) {
                    mbar_wait_cluster_acquire(h2_bar, it & 1u);
                    fence_proxy_async_all();
                    for (int t = 0; t < NQT; ++t) {
                        const int wrow0 = (t * NP + pr) * LBN + hr * (LBN / 2);
                        for (int kb = 0; kb < p.kb3; ++kb) load(&maps.c, &maps.wq, kb, row0, wrow0);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA of the pair) =====================
        if (is_leader && lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(LBN >> 3) << 17) |
                                   ((uint32_t)((2 * LBM) >> 4) << 24);
            const uint16_t pair_mask = (uint16_t)(3u << (2 * pr));
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            const int t_p1 = has_p0 ? 1 : 0, t_p2 = t_p1 + TP, n_tiles = t_p2 + 1 + NQT;
            for (int mb = cl; mb < p.tiles_m; mb += n_cl) {
                for (int t = 0; t < n_tiles; ++t) {
                    const int nkb = t < t_p1 ? p.kb0 : t < t_p2 ? p.kb1 : t == t_p2 ? p.kb2 : p.kb3;
                    mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * LBN);
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        if (mb == cl && t == 0 && kb == 0) BLK_STAMP(2);
                        const uint64_t adesc = ln_smem_desc(smem_u32(sA + (size_t)stage * L_A_BYTES));
                        const uint64_t bdesc = ln_smem_desc(smem_u32(sB + (size_t)stage * L_B_BYTES));
#pragma unroll
                        for (int k = 0; k < LBK / 16; ++k)
                            umma_f16_2sm(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
                        umma_commit_pair(&empty_bar[stage], pair_mask);
                        if (++stage == L_STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit_pair(&tfull_bar[acc], pair_mask);
                    if (mb == cl) {                    // stamps: 3 = phase 0, 4 = last phase-1 tile, 5 = phase 2, 6 = last phase-3 tile
                        if (t < t_p1) BLK_STAMP(3);
                        else if (t == t_p2 - 1) BLK_STAMP(4);
                        else if (t == t_p2) BLK_STAMP(5);
                        else if (t == n_tiles - 1) BLK_STAMP(6);
                    }
                    acc ^= 1;
                    if (acc == 0) acc_phase ^= 1;
                }
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue =====================
        const int ew = warp - 2;
        const int q = warp & 3;
        const int half = ew >> 2;
        const bool leader = ((ew & 3) == 0) && lane == 0;
        const int bar_id = 1 + half;
        uint8_t* stage_base = sEpi + half * 2 * L_EPI_BYTES;
        {
            const int c = ew * 32 + lane;
            if (has_p0) {
                sP0[c] = p.bias_o ? __ldg(p.bias_o + n0 + c) : 0.f;
                sP0[LBN + c] = __ldg(p.gamma1 + n0 + c);
                sP0[2 * LBN + c] = __ldg(p.beta1 + n0 + c);
            }
            sP2[c] = p.bias2 ? __ldg(p.bias2 + n0 + c) : 0.f;
            sP2[LBN + c] = __ldg(p.gamma2 + n0 + c);
            sP2[2 * LBN + c] = __ldg(p.beta2 + n0 + c);
            for (int t = 0; t < TP; ++t) sBias1[t * LBN + c] = p.bias1 ? __ldg(p.bias1 + (t * NP + pr) * LBN + c) : 0.f;
            for (int t = 0; t < NQT; ++t) sBiasQ[t * LBN + c] = p.bias_q ? __ldg(p.bias_q + (t * NP + pr) * LBN + c) : 0.f;
        }
        named_bar_sync(3, 256);
        int acc = 0;
        uint32_t acc_phase = 0;
        uint32_t it = 0, ln_it = 0;
        const float inv_n = 1.0f / (float)p.N;
        auto next_acc = [&]() {
            acc ^= 1;
            if (acc == 0) acc_phase ^= 1;
        };
        for (int mb = cl; mb < p.tiles_m; mb += n_cl, ++it) {
            const int row_base = mb * 2 * LBM + hr * LBM;
            const bool first = mb == cl && half == 0;
            // ---- phase 0: h1 = LayerNorm(h_in + att Wo^T + bo) ----
            if (has_p0) {
                ln_tile_epilogue<NP>(&maps.hin, &maps.h1, sP0, sStats, rbar, stat_bar, &tfull_bar[acc], acc_phase, &tempty_bar[acc],
                                     tmem_base + (uint32_t)(acc * LBN), n0, pr, hr, half, q, lane, leader, bar_id, stage_base,
                                     row_base, ln_it, inv_n, p.eps, nullptr, 0, p.M);
                ++ln_it;
                if (leader) {
                    blk_publish<NP>(h1_bar, hr);
                    if (first) BLK_STAMP(7);
                }
                next_acc();
            }
            // ---- phase 1: TP tiles of gelu(h1 W1^T + b1) -> f ----
            for (int t = 0; t < TP; ++t) {
                blk_plain_tile<true>(&maps.f, sBias1 + t * LBN, &tfull_bar[acc], acc_phase, &tempty_bar[acc],
                                     tmem_base + (uint32_t)(acc * LBN), (t * NP + pr) * LBN, row_base, half, q, lane, leader, bar_id,
                                     stage_base);
                if (leader) {
                    blk_publish<NP>(&f_bar[t], hr);
                    if (first) BLK_STAMP(8 + t);
                }
                next_acc();
            }
            // ---- phase 2: h_out = LayerNorm(h1 + f W2^T + b2) ----
            if (mb == cl && threadIdx.x == 64) BLK_STAMP(12);
            ln_tile_epilogue<NP>(&maps.h1, &maps.c, sP2, sStats, rbar, stat_bar, &tfull_bar[acc], acc_phase, &tempty_bar[acc],
                                 tmem_base + (uint32_t)(acc * LBN), n0, pr, hr, half, q, lane, leader, bar_id, stage_base,
                                 row_base, ln_it, inv_n, p.eps, nullptr, 0, p.M);
            ++ln_it;
            if (mb == cl && threadIdx.x == 64) BLK_STAMP(13);
            next_acc();
            // ---- phase 3: qkv of the next layer = h_out Wq^T + bq ----
            if (NQT) {
                if (leader) blk_publish<NP>(h2_bar, hr);
                for (int t = 0; t < NQT; ++t) {
                    blk_plain_tile<false>(&maps.q, sBiasQ + t * LBN, &tfull_bar[acc], acc_phase, &tempty_bar[acc],
                                          tmem_base + (uint32_t)(acc * LBN), (t * NP + pr) * LBN, row_base, half, q, lane, leader,
                                          bar_id, stage_base);
                    next_acc();
                }
            }
        }
        if (leader) tma_store_wait_all();
        if (threadIdx.x == 64) BLK_STAMP(14);
    }

    tc_fence_before();
    cluster_sync_all();
    if (threadIdx.x == 0) BLK_STAMP(15);
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2sm<512>(tmem_base);
    }
}

static int g_ln_max_clusters[5] = {0, 0, 0, 0, 0};

template <int NP>
int launch_gemm_ln(LnMaps& maps, const LnParams& p, cudaStream_t s) {
    using Cfg = LnCfg<NP>;
    auto kern = gemm_ln_kernel<NP>;
    static bool attr_done = false;
    if (!attr_done) {
        A2F_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES));
        attr_done = true;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.blockDim = dim3(L_THREADS, 1, 1);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2 * NP;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    if (g_ln_max_clusters[NP] == 0) {
        // clusters of 2*NP CTAs that can be resident at once (one CTA per SM, GPC boundaries): the persistent tile loop is
        // sized to that, so that no cluster waits for another one to retire
        cfg.gridDim = dim3(2 * NP * (sm_count() / (2 * NP)), 1, 1);
        cfg.numAttrs = 1;
        int n = 0;
        cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
        if (e != cudaSuccess || n < 1) {
            (void)cudaGetLastError();
            n = sm_count() / (2 * NP) - (NP > 1 ? 1 : 0);
            if (n < 1) n = 1;
        }
        g_ln_max_clusters[NP] = n;
    }
    const int n_clusters = p.tiles_m < g_ln_max_clusters[NP] ? p.tiles_m : g_ln_max_clusters[NP];
    cfg.gridDim = dim3(2 * NP * n_clusters, 1, 1);
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    A2F_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p));
    count_launch();
    return A2F_OK;
}


template <int NP>
int launch_enc_block(BlkMaps& maps, const BlkParams& p, cudaStream_t s) {
    using Cfg = BlkCfg<NP>;
    auto kern = enc_block_kernel<NP>;
    static bool attr_done = false;
    static int max_clusters = 0;
    if (!attr_done) {
        A2F_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES));
        attr_done = true;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.blockDim = dim3(L_THREADS, 1, 1);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2 * NP;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    if (max_clusters == 0) {
        cfg.gridDim = dim3(2 * NP * (sm_count() / (2 * NP)), 1, 1);
        cfg.numAttrs = 1;
        int n = 0;
        cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
        if (e != cudaSuccess || n < 1) {
            (void)cudaGetLastError();
            n = sm_count() / (2 * NP) - (NP > 1 ? 1 : 0);
            if (n < 1) n = 1;
        }
        max_clusters = n;
    }
    const int n_clusters = p.tiles_m < max_clusters ? p.tiles_m : max_clusters;
    cfg.gridDim = dim3(2 * NP * n_clusters, 1, 1);
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    A2F_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p));
    count_launch();
    return A2F_OK;
}

static int ln_map2d(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, long long ld, uint32_t box_rows) {
    uint64_t dims[2] = {cols, rows};
    uint64_t str[1] = {(uint64_t)ld * 2};
    uint32_t box[2] = {LBK, box_rows};
    return encode_tmap_bf16(m, ptr, 2, dims, str, box, 1);
}

}  // namespace

// A [M,K] bf16 (row stride lda), W [N,K] bf16 (row stride ldw), resid / out [M,N] bf16; N = 256 * NP, NP in {1,2,3}.
int gemm_ln_tc(const void* A, long long lda, const void* W, long long ldw, const float* bias, const void* resid, long long ldr,
               const float* gamma, const float* beta, float eps, void* out, long long ldo, void* pre_out, long long ldp, int M,
               int N, int K, cudaStream_t s) {
    if (M <= 0) return A2F_OK;
    A2F_REQUIRE(N % LBN == 0 && N / LBN >= 1 && N / LBN <= 3, "a2f_gemm_ln: N must be 256, 512 or 768");
    A2F_REQUIRE(K > 0 && K % 8 == 0, "a2f_gemm_ln: K must be a positive multiple of 8");
    A2F_REQUIRE(lda % 8 == 0 && ldw % 8 == 0 && ldr % 8 == 0 && ldo % 8 == 0, "a2f_gemm_ln: row strides must be multiples of 8 elements");
    A2F_REQUIRE(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(resid) |
                  reinterpret_cast<uintptr_t>(out)) & 15) == 0, "a2f_gemm_ln: operands must be 16-byte aligned");
    LnMaps maps;
    memset(&maps, 0, sizeof(maps));
    {
        uint64_t dims[2] = {(uint64_t)K, (uint64_t)M};
        uint64_t str[1] = {(uint64_t)lda * 2};
        uint32_t box[2] = {LBK, LBM};
        int rc = encode_tmap_bf16(&maps.a, A, 2, dims, str, box, 1);
        if (rc != A2F_OK) return rc;
    }
    {
        uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
        uint64_t str[1] = {(uint64_t)ldw * 2};
        uint32_t box[2] = {LBK, LBN / 2};
        int rc = encode_tmap_bf16(&maps.b, W, 2, dims, str, box, 1);
        if (rc != A2F_OK) return rc;
    }
    {
        uint64_t dims[2] = {(uint64_t)N, (uint64_t)M};
        uint64_t str[1] = {(uint64_t)ldo * 2};
        uint32_t box[2] = {L_SBW, LBM};
        int rc = encode_tmap_bf16(&maps.c, out, 2, dims, str, box, 1);
        if (rc != A2F_OK) return rc;
        uint64_t rstr[1] = {(uint64_t)ldr * 2};
        rc = encode_tmap_bf16(&maps.r, resid, 2, dims, rstr, box, 1);
        if (rc != A2F_OK) return rc;
    }
    LnParams p;
    p.M = M; p.N = N; p.K = K;
    p.tiles_m = (M + 2 * LBM - 1) / (2 * LBM);
    p.num_k_blocks = (K + LBK - 1) / LBK;
    p.bias = bias; p.gamma = gamma; p.beta = beta; p.eps = eps;
    p.pre_out = static_cast<bf16*>(pre_out);
    p.ldp = ldp;
    A2F_REQUIRE(pre_out == nullptr || (ldp % 8 == 0 && ldp >= N && (reinterpret_cast<uintptr_t>(pre_out) & 15) == 0),
                "a2f_gemm_ln: pre_out must be 16-byte aligned with a row stride that is a multiple of 8 elements");
    switch (N / LBN) {
        case 1: return launch_gemm_ln<1>(maps, p, s);
        case 2: return launch_gemm_ln<2>(maps, p, s);
        default: return launch_gemm_ln<3>(maps, p, s);
    }
}


// All operands bf16 with 16-byte aligned bases and row strides that are multiples of 8 elements (a2f.h: a2f_encoder_block_args).
int enc_block_tc(const a2f_encoder_block_args& g, cudaStream_t s) {
    const int M = g.M, N = g.N, F = g.F;
    if (M <= 0) return A2F_OK;
    const bool p0 = g.att != nullptr, p3 = g.wq != nullptr;
    A2F_REQUIRE(N % LBN == 0 && N / LBN >= 1 && N / LBN <= 3, "a2f_encoder_block: N must be 256, 512 or 768");
    A2F_REQUIRE(F > 0 && F % N == 0 && F / N <= BLK_MAX_TP, "a2f_encoder_block: F must be N, 2N, 3N or 4N");
    A2F_REQUIRE(g.h1 && g.w1 && g.f && g.w2 && g.h_out && g.ln2_g && g.ln2_b, "a2f_encoder_block: NULL operand");
    A2F_REQUIRE(!p0 || (g.wo && g.h_in && g.ln1_g && g.ln1_b), "a2f_encoder_block: att given without wo / h_in / ln1");
    A2F_REQUIRE(!p3 || (g.qkv && g.NQ > 0 && g.NQ % N == 0 && g.NQ / N <= BLK_MAX_NQT),
                "a2f_encoder_block: wq given without qkv, or NQ not N, 2N or 3N");
    const long long lds[] = {g.ld_h1, g.ld_w1, g.ld_f, g.ld_w2, g.ld_hout, p0 ? g.ld_att : 8, p0 ? g.ld_wo : 8, p0 ? g.ld_hin : 8,
                             p3 ? g.ld_wq : 8, p3 ? g.ld_qkv : 8};
    for (long long ld : lds) A2F_REQUIRE(ld > 0 && ld % 8 == 0, "a2f_encoder_block: row strides must be positive multiples of 8 elements");
    const void* ptrs[] = {g.h1, g.w1, g.f, g.w2, g.h_out, g.att, g.wo, g.h_in, g.wq, g.qkv};
    for (const void* q : ptrs) A2F_REQUIRE((reinterpret_cast<uintptr_t>(q) & 15) == 0, "a2f_encoder_block: operands must be 16-byte aligned");
    A2F_REQUIRE(g.h_out != g.h1 && g.f != g.h1 && g.f != g.h_out, "a2f_encoder_block: h1, f and h_out must be distinct buffers");
    BlkMaps maps;
    memset(&maps, 0, sizeof(maps));
    int rc;
    if ((rc = ln_map2d(&maps.h1, g.h1, (uint64_t)N, (uint64_t)M, g.ld_h1, LBM)) != A2F_OK) return rc;
    if ((rc = ln_map2d(&maps.w1, g.w1, (uint64_t)N, (uint64_t)F, g.ld_w1, LBN / 2)) != A2F_OK) return rc;
    if ((rc = ln_map2d(&maps.f, g.f, (uint64_t)F, (uint64_t)M, g.ld_f, LBM)) != A2F_OK) return rc;
    if ((rc = ln_map2d(&maps.w2, g.w2, (uint64_t)F, (uint64_t)N, g.ld_w2, LBN / 2)) != A2F_OK) return rc;
    if ((rc = ln_map2d(&maps.c, g.h_out, (uint64_t)N, (uint64_t)M, g.ld_hout, LBM)) != A2F_OK) return rc;
    if (p0) {
        if ((rc = ln_map2d(&maps.att, g.att, (uint64_t)N, (uint64_t)M, g.ld_att, LBM)) != A2F_OK) return rc;
        if ((rc = ln_map2d(&maps.wo, g.wo, (uint64_t)N, (uint64_t)N, g.ld_wo, LBN / 2)) != A2F_OK) return rc;
        if ((rc = ln_map2d(&maps.hin, g.h_in, (uint64_t)N, (uint64_t)M, g.ld_hin, LBM)) != A2F_OK) return rc;
    }
    if (p3) {
        if ((rc = ln_map2d(&maps.wq, g.wq, (uint64_t)N, (uint64_t)g.NQ, g.ld_wq, LBN / 2)) != A2F_OK) return rc;
        if ((rc = ln_map2d(&maps.q, g.qkv, (uint64_t)g.NQ, (uint64_t)M, g.ld_qkv, LBM)) != A2F_OK) return rc;
    }
    BlkParams p;
    memset(&p, 0, sizeof(p));
    p.M = M; p.N = N;
    p.tiles_m = (M + 2 * LBM - 1) / (2 * LBM);
    p.kb0 = p.kb1 = p.kb3 = N / LBK;
    p.kb2 = F / LBK;
    p.tp = F / N;
    p.nqt = p3 ? g.NQ / N : 0;
    p.has_p0 = p0 ? 1 : 0;
    p.has_p3 = p3 ? 1 : 0;
    p.bias_o = g.bo; p.gamma1 = g.ln1_g; p.beta1 = g.ln1_b;
    p.bias1 = g.b1;
    p.bias2 = g.b2; p.gamma2 = g.ln2_g; p.beta2 = g.ln2_b;
    p.bias_q = g.bq;
    p.eps = g.eps;
    p.timeline = debug_timeline();
    switch (N / LBN) {
        case 1: return launch_enc_block<1>(maps, p, s);
        case 2: return launch_enc_block<2>(maps, p, s);
        default: return launch_enc_block<3>(maps, p, s);
    }
}

}  // namespace a2f

extern "C" int a2f_gemm_ln(const void* A, long long lda, const void* W, long long ldw, const float* bias, const void* resid,
                           long long ldr, const float* gamma, const float* beta, float eps, void* out, long long ldo,
                           void* pre_out, long long ldp, int M, int N, int K, void* stream) {
    int rc = a2f::require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(A && W && resid && gamma && beta && out, "a2f_gemm_ln: A, W, resid, gamma, beta and out must be non-NULL");
    A2F_REQUIRE(M >= 0 && N > 0 && K > 0, "a2f_gemm_ln: bad M/N/K");
    return a2f::gemm_ln_tc(A, lda, W, ldw, bias, resid, ldr, gamma, beta, eps, out, ldo, pre_out, ldp, M, N, K,
                           a2f::as_stream(stream));
}

extern "C" int a2f_encoder_block(const a2f_encoder_block_args* args, void* stream) {
    int rc = a2f::require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(args != nullptr, "a2f_encoder_block: NULL args");
    A2F_REQUIRE(args->M >= 0 && args->N > 0 && args->F > 0, "a2f_encoder_block: bad M/N/F");
    return a2f::enc_block_tc(*args, a2f::as_stream(stream));
}
