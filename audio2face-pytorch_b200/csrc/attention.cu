// Encoder self-attention of wav2vec2 (HF modeling_wav2vec2.py:438-549): softmax(Q K^T * scale) V per (batch, head),
// no mask, head_dim 64.  The reference materialises and returns the [B,12,T,T] probabilities of all 12 layers
// (ref:src/model/wav2vec.py:101 forces output_attentions=True) although nothing reads them
// (ref:src/model/faceformer.py:149-151 keeps only last_hidden_state); here the probabilities never leave the SM.
//
//   fp32  : SIMT online-softmax kernel, one warp per query row (the 1e-5 parity path)
//   bf16  : flash-style kernel on mma.sync.m16n8k16 bf16 tensor-core tiles, 64 queries x 64 keys per step,
//           K/V tiles streamed through shared memory with cp.async double buffering, fp32 softmax statistics.
//           (A tcgen05/TMEM version of this kernel is the planned replacement; at T=300 attention is 4% of the
//            encoder FLOPs, SURVEY.md App. C.)
#include "a2f_common.cuh"

namespace a2f {

// ------------------------------------------------------------------------------------------------ dropout of P
// Training with encoder dropout: O = (P o Z / (1 - p)) V with the LSE of the UNDROPPED softmax (HF modeling_wav2vec2.py
// attention dropout).  Z follows the RNG contract of include/a2f.h over the logical tensor [B, H, T, Tp], Tp = ceil(T/8)*8:
// keys 8k .. 8k+7 of query row t of (b, h) are ONE Philox call, g = ((b*H + h)*T + t)*Tp/8 + k, so the forward and both
// backward passes regenerate the same bits from (seed, offset, site) whatever their tiling.  so == nullptr = off.
struct AttnDrop {
    const unsigned long long* so;     // {seed, offset} in device memory
    uint32_t site, threshold;
    float scale;                      // 1 / (1 - p)
};
struct AttnDropRt {                   // what a thread reads once at kernel start
    unsigned long long seed;
    uint32_t offset;
};
A2F_D AttnDropRt attn_drop_load(const AttnDrop& d) { return AttnDropRt{d.so[0], (uint32_t)d.so[1]}; }
A2F_D uint32_t attn_keep8(const AttnDrop& d, const AttnDropRt& r, int bh, int T, int t, int ktile) {
    const unsigned long long g = ((unsigned long long)bh * T + t) * (unsigned long long)((T + 7) >> 3) + ktile;
    return dropout_keep8(r.seed, r.offset, d.site, g, d.threshold);
}
// Z of an m16n8k16 accumulator tile whose rows are queries (row_base + lane/4, +8) and whose n-tile nt holds keys
// 8*(ktile0 + nt) + (lane&3)*2 + {0,1}: z[0] / z[1] = keep bits of the two rows' 8-key groups.  Each pair of n-tiles needs
// 32 distinct Philox calls per warp, one per lane (call = row lane/4 bits 2-4, row half bit 1, n-tile parity bit 0),
// computed at the even n-tile into `held` and handed out by shuffles.
A2F_D void mma_rows_keep(const AttnDrop& d, const AttnDropRt& r, int bh, int T, int row_base, int ktile0, int nt, int lane,
                         uint32_t& held, uint32_t* z) {
    if ((nt & 1) == 0)
        held = attn_keep8(d, r, bh, T, row_base + (lane >> 2) + 8 * ((lane >> 1) & 1), ktile0 + nt + (lane & 1));
    z[0] = __shfl_sync(0xffffffffu, held, (lane & ~3) | (nt & 1));
    z[1] = __shfl_sync(0xffffffffu, held, (lane & ~3) | 2 | (nt & 1));
}
A2F_D void mask_pair(uint32_t z, int lane, float& a, float& b) {
    const int c = (lane & 3) * 2;
    if (!((z >> c) & 1u)) a = 0.f;
    if (!((z >> (c + 1)) & 1u)) b = 0.f;
}

// ------------------------------------------------------------------------------------------------ fp32 SIMT
// qkv: [B,T,3*H*64] fp32.  One warp per (b,h,query).  Lane l scores keys j = j0+l; output dims (2l, 2l+1).
__global__ void __launch_bounds__(256) mha_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out,
                                                      float* __restrict__ lse, int B, int T, int H, float scale,
                                                      AttnDrop drop) {
    const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int total = B * H * T;
    if (warp_global >= total) return;
    const int t = warp_global % T;
    const int h = (warp_global / T) % H;
    const int b = warp_global / (T * H);
    const int ld = 3 * H * 64;
    const float* base = qkv + (long long)b * T * ld;
    const float* qp = base + (long long)t * ld + h * 64;
    float q[64];
#pragma unroll
    for (int d = 0; d < 64; d += 4) {
        const float4 f = *reinterpret_cast<const float4*>(qp + d);
        q[d] = f.x; q[d + 1] = f.y; q[d + 2] = f.z; q[d + 3] = f.w;
    }
    const bool dropping = drop.so != nullptr;
    const AttnDropRt dr = dropping ? attn_drop_load(drop) : AttnDropRt{0ull, 0u};
    float m = -INFINITY, l = 0.f, o0 = 0.f, o1 = 0.f;
    for (int j0 = 0; j0 < T; j0 += 32) {
        const int j = j0 + lane;
        float s = -INFINITY;
        if (j < T) {
            const float* kp = base + (long long)j * ld + H * 64 + h * 64;
            float acc = 0.f;
#pragma unroll
            for (int d = 0; d < 64; d += 4) {
                const float4 f = *reinterpret_cast<const float4*>(kp + d);
                acc = fmaf(q[d], f.x, acc);
                acc = fmaf(q[d + 1], f.y, acc);
                acc = fmaf(q[d + 2], f.z, acc);
                acc = fmaf(q[d + 3], f.w, acc);
            }
            s = acc * scale;
        }
        const float m_new = fmaxf(m, warp_max(s));
        const float corr = __expf(m - m_new);      // first chunk: exp(-inf) = 0
        const float pj = (j < T) ? __expf(s - m_new) : 0.f;
        l = l * corr + warp_sum(pj);
        float pd = pj;                                    // the dropped probability feeds O, the undropped one l / LSE
        if (dropping && j < T && !((attn_keep8(drop, dr, b * H + h, T, t, j >> 3) >> (j & 7)) & 1u)) pd = 0.f;
        o0 *= corr;
        o1 *= corr;
        const int nj = min(32, T - j0);
        for (int jj = 0; jj < nj; ++jj) {
            const float pv = __shfl_sync(0xffffffffu, pd, jj);
            const float2 vv = *reinterpret_cast<const float2*>(base + (long long)(j0 + jj) * ld + 2 * H * 64 + h * 64 + 2 * lane);
            o0 = fmaf(pv, vv.x, o0);
            o1 = fmaf(pv, vv.y, o1);
        }
        m = m_new;
    }
    const float inv = (dropping ? drop.scale : 1.f) / l;
    float* op = out + ((long long)b * T + t) * (H * 64) + h * 64 + 2 * lane;
    *reinterpret_cast<float2*>(op) = make_float2(o0 * inv, o1 * inv);
    if (lse != nullptr && lane == 0) lse[((long long)b * H + h) * T + t] = m + logf(l);
}

// ------------------------------------------------------------------------------------------------ bf16 tensor-core
constexpr int FA_BM = 64;      // queries per CTA (4 warps x 16 rows)
constexpr int FA_BN = 64;      // keys per step
constexpr int FA_D = 64;
constexpr int FA_LD = 72;      // padded smem row (bf16 elements): 144-byte pitch -> conflict-free ldmatrix

A2F_D void ldmatrix_x4(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(smem_u32(p)));
}
A2F_D void ldmatrix_x4_trans(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(smem_u32(p)));
}
A2F_D void mma_bf16_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
A2F_D void cp_async_16(void* smem_dst, const void* gsrc, bool valid) {
    const int sz = valid ? 16 : 0;     // src-size 0 -> zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(sz) : "memory");
}
A2F_D void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> A2F_D void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// grid: (ceil(T/64), H, B); 128 threads.
template <bool DROP>
__global__ void __launch_bounds__(128) mha_bf16_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out,
                                                       float* __restrict__ lse, float* __restrict__ out32, int T, int H,
                                                       float scale_log2, AttnDrop drop) {
    pdl_sync();   // PDL: wait for the previous kernel's results, let the next kernel's prologue start
    __shared__ __align__(16) bf16 sQ[FA_BM * FA_LD];
    __shared__ __align__(16) bf16 sK[2][FA_BN * FA_LD];
    __shared__ __align__(16) bf16 sV[2][FA_BN * FA_LD];

    const int q0 = blockIdx.x * FA_BM, h = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ld = 3 * H * FA_D;
    const bf16* base = qkv + (long long)b * T * ld;
    const bf16* gQ = base + h * FA_D;
    const bf16* gK = base + H * FA_D + h * FA_D;
    const bf16* gV = base + 2 * H * FA_D + h * FA_D;

    // 64 rows x 64 cols bf16 = 512 chunks of 16 B; 128 threads x 4
    auto load_tile = [&](bf16* dst, const bf16* src, int row0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = threadIdx.x + i * 128;
            const int r = idx >> 3, c = (idx & 7) * 8;
            const bool ok = (row0 + r) < T;
            cp_async_16(dst + r * FA_LD + c, src + (long long)(ok ? row0 + r : 0) * ld + c, ok);
        }
    };

    load_tile(sQ, gQ, q0);
    load_tile(sK[0], gK, 0);
    load_tile(sV[0], gV, 0);
    cp_async_commit();

    const int ntiles = (T + FA_BN - 1) / FA_BN;
    uint32_t qf[4][4];                 // Q fragments: 4 k-steps (16 dims each)
    float o[8][4];                     // 16 x 64 output accumulator: 8 n-tiles
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
    AttnDropRt dr{0ull, 0u};
    if (DROP) dr = attn_drop_load(drop);

    for (int it = 0; it < ntiles; ++it) {
        const int cur = it & 1;
        if (it + 1 < ntiles) {
            load_tile(sK[cur ^ 1], gK, (it + 1) * FA_BN);
            load_tile(sV[cur ^ 1], gV, (it + 1) * FA_BN);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        if (it == 0) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int c = ks * 16 + (lane >> 4) * 8;
                ldmatrix_x4(qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3], sQ + r * FA_LD + c);
            }
        }
        // S = Q K^T : 16 x 64 per warp
        float s[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int np = 0; np < 4; ++np) {     // pairs of 8-key n-tiles
                uint32_t b0, b1, b2, b3;
                // matrices: (keys np*16+0..7, d ks*16+0..7), (same keys, d +8), (keys +8, d), (keys +8, d +8)
                const int r = np * 16 + (lane & 7) + (lane >> 4) * 8;
                const int c = ks * 16 + ((lane >> 3) & 1) * 8;
                ldmatrix_x4(b0, b1, b2, b3, sK[cur] + r * FA_LD + c);
                mma_bf16_16816(s[2 * np], qf[ks], b0, b1);
                mma_bf16_16816(s[2 * np + 1], qf[ks], b2, b3);
            }
        }
        // mask keys beyond T (last tile only) and online softmax; rows g = lane/4 and g+8
        const int key0 = it * FA_BN;
        if (key0 + FA_BN > T) {
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int kc = key0 + nt * 8 + (lane & 3) * 2;
                if (kc >= T) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
                if (kc + 1 >= T) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
            }
        }
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            mx[0] = fmaxf(mx[0], fmaxf(s[nt][0], s[nt][1]));
            mx[1] = fmaxf(mx[1], fmaxf(s[nt][2], s[nt][3]));
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
        }
        float corr[2], msc[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const float m_new = fmaxf(m_run[r], mx[r]);
            corr[r] = exp2f((m_run[r] - m_new) * scale_log2);
            m_run[r] = m_new;
            msc[r] = m_new * scale_log2;
        }
        float rs[2] = {0.f, 0.f};
        uint32_t pf[4][4];                 // P as A fragments: 4 k-steps of 16 keys
        uint32_t zheld = 0;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            float p0 = exp2f(fmaf(s[nt][0], scale_log2, -msc[0]));
            float p1 = exp2f(fmaf(s[nt][1], scale_log2, -msc[0]));
            float p2 = exp2f(fmaf(s[nt][2], scale_log2, -msc[1]));
            float p3 = exp2f(fmaf(s[nt][3], scale_log2, -msc[1]));
            rs[0] += p0 + p1;
            rs[1] += p2 + p3;
            if (DROP) {
                uint32_t z[2];
                mma_rows_keep(drop, dr, b * H + h, T, q0 + warp * 16, key0 / 8, nt, lane, zheld, z);
                mask_pair(z[0], lane, p0, p1);
                mask_pair(z[1], lane, p2, p3);
            }
            const int ks = nt >> 1, hi = nt & 1;
            pf[ks][hi * 2 + 0] = pack_bf16x2(p0, p1);
            pf[ks][hi * 2 + 1] = pack_bf16x2(p2, p3);
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) l_run[r] = l_run[r] * corr[r] + rs[r];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            o[nt][0] *= corr[0]; o[nt][1] *= corr[0];
            o[nt][2] *= corr[1]; o[nt][3] *= corr[1];
        }
        // O += P V : B fragments of V (k = key, n = d) through ldmatrix.trans on the row-major [key][d] tile
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int dp = 0; dp < 4; ++dp) {    // pairs of 8-wide d tiles
                uint32_t b0, b1, b2, b3;
                // matrices: (keys ks*16+0..7, d dp*16+0..7), (keys +8, same d), (keys, d +8), (keys +8, d +8)
                const int r = ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int c = dp * 16 + (lane >> 4) * 8;
                ldmatrix_x4_trans(b0, b1, b2, b3, sV[cur] + r * FA_LD + c);
                mma_bf16_16816(o[2 * dp], pf[ks], b0, b1);
                mma_bf16_16816(o[2 * dp + 1], pf[ks], b2, b3);
            }
        }
        __syncthreads();     // everyone is done with buffer `cur` before it is refilled two iterations later
    }

    // finalise: row sums across the 4 lanes of a quad, normalise, store bf16
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
        l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    }
    const int row0 = q0 + warp * 16 + (lane >> 2);
    const float osc = DROP ? drop.scale : 1.f;
    const float inv0 = osc / l_run[0], inv1 = osc / l_run[1];
    if (lse != nullptr && (lane & 3) == 0) {
        // natural-log LSE of the scaled scores: m*scale + ln(l)
        float* lp = lse + ((long long)b * H + h) * T;
        if (row0 < T) lp[row0] = m_run[0] * scale_log2 * 0.69314718055994531f + logf(l_run[0]);
        if (row0 + 8 < T) lp[row0 + 8] = m_run[1] * scale_log2 * 0.69314718055994531f + logf(l_run[1]);
    }
    bf16* ob = out + (long long)b * T * (H * FA_D) + h * FA_D;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const int c = nt * 8 + (lane & 3) * 2;
        if (row0 < T)
            *reinterpret_cast<uint32_t*>(ob + (long long)row0 * (H * FA_D) + c) = pack_bf16x2(o[nt][0] * inv0, o[nt][1] * inv0);
        if (row0 + 8 < T)
            *reinterpret_cast<uint32_t*>(ob + (long long)(row0 + 8) * (H * FA_D) + c) = pack_bf16x2(o[nt][2] * inv1, o[nt][3] * inv1);
    }
    if (out32 != nullptr) {      // training: un-rounded output for the backward's delta = rowsum(dO o O) term
        float* o32 = out32 + (long long)b * T * (H * FA_D) + h * FA_D;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int c = nt * 8 + (lane & 3) * 2;
            if (row0 < T)
                *reinterpret_cast<float2*>(o32 + (long long)row0 * (H * FA_D) + c) = make_float2(o[nt][0] * inv0, o[nt][1] * inv0);
            if (row0 + 8 < T)
                *reinterpret_cast<float2*>(o32 + (long long)(row0 + 8) * (H * FA_D) + c) = make_float2(o[nt][2] * inv1, o[nt][3] * inv1);
        }
    }
}


// ------------------------------------------------------------------------------------------------ short sequences
// Clips of at most 160 frames (5 s at 30 fps is T = 150): every key of a (batch, head) fits in shared memory and a warp's
// whole score row block (16 x NKT*16) fits in registers, so the softmax is single-pass (no running max / rescale) and
// nothing is re-synchronised per key block.  One CTA = 80 queries (5 warps x 16 rows) of one (b, h) against all keys:
// at T = 150 that is 768 CTAs of 160x160 useful work instead of the flash kernel's 1152 CTAs over 192x192 padded work
// with three barrier-separated key steps each (22 us -> see profiles/).  K is waited for separately from V, so QK^T and the
// softmax overlap the V load.
constexpr int FS_NW = 5;                 // warps per CTA
constexpr int FS_BM = 16 * FS_NW;        // queries per CTA
// NQB = query blocks of 80 rows a CTA walks through: with T > 80 one CTA takes ALL queries of its (b, h) (NQB = 2), so K and
// V are loaded once per (b, h) instead of once per 80 queries, and the grid of the bench shape (32 x 12 = 384 CTAs, three
// resident per SM) is a single wave instead of 768 CTAs in 1.7 waves.
template <int NKT, int NQB> struct FsCfg {
    static constexpr int KEYS = NKT * 16;
    static constexpr size_t SMEM_BYTES = (size_t)(NQB * FS_BM + 2 * KEYS) * FA_LD * sizeof(bf16);
};

// grid: (ceil(T/(80*NQB)), H, B); 160 threads; T <= NKT*16.
template <int NKT, int NQB, bool DROP>
__global__ void __launch_bounds__(32 * FS_NW, 3) mha_short_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out,
                                                                   float* __restrict__ lse, float* __restrict__ out32, int T,
                                                                   int H, float scale_log2, AttnDrop drop) {
    constexpr int KEYS = NKT * 16;
    extern __shared__ __align__(16) uint8_t fs_smem[];
    bf16* sQ = reinterpret_cast<bf16*>(fs_smem);
    bf16* sK = sQ + NQB * FS_BM * FA_LD;
    bf16* sV = sK + KEYS * FA_LD;
    pdl_sync();   // PDL: wait for the previous kernel's results, let the next kernel's prologue start

    const int q0 = blockIdx.x * (NQB * FS_BM), h = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ld = 3 * H * FA_D;
    const bf16* base = qkv + (long long)b * T * ld;
    const bf16* gQ = base + h * FA_D;
    const bf16* gK = base + H * FA_D + h * FA_D;
    const bf16* gV = base + 2 * H * FA_D + h * FA_D;

    // rows x 8 chunks of 16 B; rows beyond T are zero-filled (V must be finite: its rows meet zero probabilities)
    auto load_rows = [&](bf16* dst, const bf16* src, int row0, int rows) {
        for (int idx = threadIdx.x; idx < rows * 8; idx += 32 * FS_NW) {
            const int r = idx >> 3, c = (idx & 7) * 8;
            const bool ok = (row0 + r) < T;
            cp_async_16(dst + r * FA_LD + c, src + (long long)(ok ? row0 + r : 0) * ld + c, ok);
        }
    };
    load_rows(sQ, gQ, q0, NQB * FS_BM);
    load_rows(sK, gK, 0, KEYS);
    cp_async_commit();
    load_rows(sV, gV, 0, KEYS);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();

#pragma unroll 1
  for (int qb = 0; qb < NQB; ++qb) {
    const int qrow = qb * FS_BM + warp * 16;         // first query row of this warp's block inside the CTA's query slab
    const bool active = q0 + qrow < T;               // warp-uniform
    uint32_t pf[NKT][4];                             // P as A fragments: NKT k-steps of 16 keys
    float rs[2] = {0.f, 0.f}, mx[2] = {-INFINITY, -INFINITY};
    if (active) {
        uint32_t qf[4][4];
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            const int r = qrow + (lane & 7) + ((lane >> 3) & 1) * 8;
            const int c = ks * 16 + (lane >> 4) * 8;
            ldmatrix_x4(qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3], sQ + r * FA_LD + c);
        }
        float s[2 * NKT][4];
#pragma unroll
        for (int i = 0; i < 2 * NKT; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int np = 0; np < NKT; ++np) {
                uint32_t b0, b1, b2, b3;
                const int r = np * 16 + (lane & 7) + (lane >> 4) * 8;
                const int c = ks * 16 + ((lane >> 3) & 1) * 8;
                ldmatrix_x4(b0, b1, b2, b3, sK + r * FA_LD + c);
                mma_bf16_16816(s[2 * np], qf[ks], b0, b1);
                mma_bf16_16816(s[2 * np + 1], qf[ks], b2, b3);
            }
        }
        // mask keys beyond T, row max (rows g = lane/4 and g+8), probabilities, row sums
#pragma unroll
        for (int nt = 0; nt < 2 * NKT; ++nt) {
            const int kc = nt * 8 + (lane & 3) * 2;
            if (kc >= T) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
            if (kc + 1 >= T) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
            mx[0] = fmaxf(mx[0], fmaxf(s[nt][0], s[nt][1]));
            mx[1] = fmaxf(mx[1], fmaxf(s[nt][2], s[nt][3]));
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
        }
        const float msc0 = mx[0] * scale_log2, msc1 = mx[1] * scale_log2;
        AttnDropRt dr{0ull, 0u};
        if (DROP) dr = attn_drop_load(drop);
        uint32_t zheld = 0;
#pragma unroll
        for (int nt = 0; nt < 2 * NKT; ++nt) {
            float p0 = exp2f(fmaf(s[nt][0], scale_log2, -msc0));
            float p1 = exp2f(fmaf(s[nt][1], scale_log2, -msc0));
            float p2 = exp2f(fmaf(s[nt][2], scale_log2, -msc1));
            float p3 = exp2f(fmaf(s[nt][3], scale_log2, -msc1));
            rs[0] += p0 + p1;
            rs[1] += p2 + p3;
            if (DROP) {
                uint32_t z[2];
                mma_rows_keep(drop, dr, b * H + h, T, q0 + qrow, 0, nt, lane, zheld, z);
                mask_pair(z[0], lane, p0, p1);
                mask_pair(z[1], lane, p2, p3);
            }
            const int ks = nt >> 1, hi = nt & 1;
            pf[ks][hi * 2 + 0] = pack_bf16x2(p0, p1);
            pf[ks][hi * 2 + 1] = pack_bf16x2(p2, p3);
        }
    }
    if (qb == 0) {
        cp_async_wait<0>();
        __syncthreads();                             // V has landed
    }
    if (!active) continue;

    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
#pragma unroll
    for (int ks = 0; ks < NKT; ++ks) {
#pragma unroll
        for (int dp = 0; dp < 4; ++dp) {
            uint32_t b0, b1, b2, b3;
            const int r = ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
            const int c = dp * 16 + (lane >> 4) * 8;
            ldmatrix_x4_trans(b0, b1, b2, b3, sV + r * FA_LD + c);
            mma_bf16_16816(o[2 * dp], pf[ks], b0, b1);
            mma_bf16_16816(o[2 * dp + 1], pf[ks], b2, b3);
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 1);
        rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 2);
    }
    const int row0 = q0 + qrow + (lane >> 2);
    const float osc = DROP ? drop.scale : 1.f;
    const float inv0 = osc / rs[0], inv1 = osc / rs[1];
    if (lse != nullptr && (lane & 3) == 0) {
        float* lp = lse + ((long long)b * H + h) * T;
        if (row0 < T) lp[row0] = mx[0] * scale_log2 * 0.69314718055994531f + logf(rs[0]);
        if (row0 + 8 < T) lp[row0 + 8] = mx[1] * scale_log2 * 0.69314718055994531f + logf(rs[1]);
    }
    bf16* ob = out + (long long)b * T * (H * FA_D) + h * FA_D;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const int c = nt * 8 + (lane & 3) * 2;
        if (row0 < T)
            *reinterpret_cast<uint32_t*>(ob + (long long)row0 * (H * FA_D) + c) = pack_bf16x2(o[nt][0] * inv0, o[nt][1] * inv0);
        if (row0 + 8 < T)
            *reinterpret_cast<uint32_t*>(ob + (long long)(row0 + 8) * (H * FA_D) + c) = pack_bf16x2(o[nt][2] * inv1, o[nt][3] * inv1);
    }
    if (out32 != nullptr) {
        float* o32 = out32 + (long long)b * T * (H * FA_D) + h * FA_D;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int c = nt * 8 + (lane & 3) * 2;
            if (row0 < T)
                *reinterpret_cast<float2*>(o32 + (long long)row0 * (H * FA_D) + c) = make_float2(o[nt][0] * inv0, o[nt][1] * inv0);
            if (row0 + 8 < T)
                *reinterpret_cast<float2*>(o32 + (long long)(row0 + 8) * (H * FA_D) + c) = make_float2(o[nt][2] * inv1, o[nt][3] * inv1);
        }
    }
  }   // qb
}

template <int NKT, int NQB, bool DROP>
static int launch_mha_short_q(const bf16* qkv, bf16* out, float* lse, float* out32, int B, int T, int H, float scale_log2,
                              const AttnDrop& drop, cudaStream_t s) {
    auto kern = mha_short_kernel<NKT, NQB, DROP>;
    static bool attr_done = false;
    if (!attr_done) {
        A2F_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FsCfg<NKT, NQB>::SMEM_BYTES));
        attr_done = true;
    }
    const dim3 grid((T + NQB * FS_BM - 1) / (NQB * FS_BM), H, B);
    A2F_CHECK_CUDA(launch_pdl(kern, grid, dim3(32 * FS_NW), FsCfg<NKT, NQB>::SMEM_BYTES, s, qkv, out, lse, out32, T, H, scale_log2,
                              drop));
    return A2F_OK;
}

static int g_mha_short_nqb = 0;   // debug: 0 = automatic (2 query blocks per CTA when T > 80), 1 = one block per CTA (round 1)
void set_mha_short_nqb(int v) { g_mha_short_nqb = v; }

template <int NKT, bool DROP>
static int launch_mha_short(const bf16* qkv, bf16* out, float* lse, float* out32, int B, int T, int H, float scale_log2,
                            const AttnDrop& drop, cudaStream_t s) {
    if (T > FS_BM && g_mha_short_nqb != 1)
        return launch_mha_short_q<NKT, 2, DROP>(qkv, out, lse, out32, B, T, H, scale_log2, drop, s);
    return launch_mha_short_q<NKT, 1, DROP>(qkv, out, lse, out32, B, T, H, scale_log2, drop, s);
}


// ================================================================================================ backward
// delta[b,h,t] = sum_d dO[b,t,h,d] * O[b,t,h,d]   (one warp per (b,t,h))
template <typename TO, typename T>
__global__ void __launch_bounds__(256) mha_delta_kernel(const TO* __restrict__ o, const T* __restrict__ dout,
                                                        float* __restrict__ delta, int B, int Tn, int H) {
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= (long long)B * Tn * H) return;
    const int h = (int)(w % H);
    const long long bt = w / H;
    const int t = (int)(bt % Tn), b = (int)(bt / Tn);
    const TO* op = o + bt * (H * 64) + h * 64 + 2 * lane;
    const T* dp = dout + bt * (H * 64) + h * 64 + 2 * lane;
    float s = ld_as_float(op) * ld_as_float(dp) + ld_as_float(op + 1) * ld_as_float(dp + 1);
    s = warp_sum(s);
    if (lane == 0) delta[((long long)b * H + h) * Tn + t] = s;
}

// fp32 parity path: one warp per (b,h,query); lanes own keys; dK / dV through fp32 atomics (dqkv must be zeroed).
__global__ void __launch_bounds__(128) mha_bwd_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ dout,
                                                          const float* __restrict__ lse, const float* __restrict__ delta,
                                                          float* __restrict__ dqkv, int B, int T, int H, float scale,
                                                          AttnDrop drop) {
    __shared__ float qs[4][64], dos[4][64];
    const int wl = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wg = blockIdx.x * 4 + wl;
    if (wg >= B * H * T) return;
    const int t = wg % T, h = (wg / T) % H, b = wg / (T * H);
    const int ld = 3 * H * 64;
    const float* base = qkv + (long long)b * T * ld;
    float* dbase = dqkv + (long long)b * T * ld;
    qs[wl][lane] = base[(long long)t * ld + h * 64 + lane];
    qs[wl][lane + 32] = base[(long long)t * ld + h * 64 + lane + 32];
    dos[wl][lane] = dout[((long long)b * T + t) * (H * 64) + h * 64 + lane];
    dos[wl][lane + 32] = dout[((long long)b * T + t) * (H * 64) + h * 64 + lane + 32];
    __syncwarp();
    const float L = lse[((long long)b * H + h) * T + t], dl = delta[((long long)b * H + h) * T + t];
    const bool dropping = drop.so != nullptr;
    const AttnDropRt dr = dropping ? attn_drop_load(drop) : AttnDropRt{0ull, 0u};
    float dq[64];
#pragma unroll
    for (int d = 0; d < 64; ++d) dq[d] = 0.f;
    for (int j = lane; j < T; j += 32) {
        const float* kp = base + (long long)j * ld + H * 64 + h * 64;
        const float* vp = base + (long long)j * ld + 2 * H * 64 + h * 64;
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int d = 0; d < 64; d += 4) {
            const float4 kf = *reinterpret_cast<const float4*>(kp + d);
            const float4 vf = *reinterpret_cast<const float4*>(vp + d);
            s = fmaf(qs[wl][d], kf.x, s); s = fmaf(qs[wl][d + 1], kf.y, s);
            s = fmaf(qs[wl][d + 2], kf.z, s); s = fmaf(qs[wl][d + 3], kf.w, s);
            dp = fmaf(dos[wl][d], vf.x, dp); dp = fmaf(dos[wl][d + 1], vf.y, dp);
            dp = fmaf(dos[wl][d + 2], vf.z, dp); dp = fmaf(dos[wl][d + 3], vf.w, dp);
        }
        const float p = __expf(s * scale - L);
        // dropout: O = (P o Z/(1-p)) V, so dV sees the dropped P and dP = (dO V^T) o Z/(1-p); delta = rowsum(dO o O) holds
        float pv = p;
        if (dropping) {
            const float z = ((attn_keep8(drop, dr, b * H + h, T, t, j >> 3) >> (j & 7)) & 1u) ? drop.scale : 0.f;
            pv = p * z;
            dp *= z;
        }
        const float ds = p * (dp - dl) * scale;
        float* dkp = dbase + (long long)j * ld + H * 64 + h * 64;
        float* dvp = dbase + (long long)j * ld + 2 * H * 64 + h * 64;
#pragma unroll
        for (int d = 0; d < 64; ++d) {
            dq[d] = fmaf(ds, kp[d], dq[d]);
            atomicAdd(dkp + d, ds * qs[wl][d]);
            atomicAdd(dvp + d, pv * dos[wl][d]);
        }
    }
    float* dqp = dbase + (long long)t * ld + h * 64;
#pragma unroll
    for (int d = 0; d < 64; ++d) {
        const float v = warp_sum(dq[d]);
        if (lane == (d & 31)) dqp[d] = v;
    }
}

constexpr int FAB_TILE = FA_BM * FA_LD;     // bf16 elements of one 64 x 64 (padded) tile

// bf16 tensor-core backward, query-major pass: dQ = (P o (dO V^T - delta)) K * scale.   grid (ceil(T/64), H, B), 128 thr.
template <bool DROP>
__global__ void __launch_bounds__(128) mha_bwd_dq_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ dout,
                                                         const float* __restrict__ lse, const float* __restrict__ delta,
                                                         bf16* __restrict__ dqkv, int T, int H, float scale, AttnDrop drop) {
    extern __shared__ __align__(16) bf16 fab_smem[];
    bf16* sQ = fab_smem;
    bf16* sdO = sQ + FAB_TILE;
    bf16* sK = sdO + FAB_TILE;           // [2]
    bf16* sV = sK + 2 * FAB_TILE;        // [2]
    const int q0 = blockIdx.x * FA_BM, h = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ld = 3 * H * FA_D, ldo = H * FA_D;
    const bf16* base = qkv + (long long)b * T * ld;
    const bf16* gQ = base + h * FA_D;
    const bf16* gK = base + H * FA_D + h * FA_D;
    const bf16* gV = base + 2 * H * FA_D + h * FA_D;
    const bf16* gdO = dout + (long long)b * T * ldo + h * FA_D;
    auto load_tile = [&](bf16* dst, const bf16* src, int row0, int lds) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = threadIdx.x + i * 128;
            const int r = idx >> 3, c = (idx & 7) * 8;
            const bool ok = (row0 + r) < T;
            cp_async_16(dst + r * FA_LD + c, src + (long long)(ok ? row0 + r : 0) * lds + c, ok);
        }
    };
    load_tile(sQ, gQ, q0, ld);
    load_tile(sdO, gdO, q0, ldo);
    load_tile(sK, gK, 0, ld);
    load_tile(sV, gV, 0, ld);
    cp_async_commit();
    const float scale_log2 = scale * 1.4426950408889634f;
    const int r0 = q0 + warp * 16 + (lane >> 2);
    const float* lp = lse + ((long long)b * H + h) * T;
    const float* dp_ = delta + ((long long)b * H + h) * T;
    float lse2[2], dl[2];
    lse2[0] = r0 < T ? lp[r0] * 1.4426950408889634f : 0.f;
    lse2[1] = r0 + 8 < T ? lp[r0 + 8] * 1.4426950408889634f : 0.f;
    dl[0] = r0 < T ? dp_[r0] : 0.f;
    dl[1] = r0 + 8 < T ? dp_[r0 + 8] : 0.f;
    AttnDropRt dr{0ull, 0u};
    if (DROP) dr = attn_drop_load(drop);
    uint32_t qf[4][4], dof[4][4];
    float dq[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dq[i][j] = 0.f;
    const int ntiles = (T + FA_BN - 1) / FA_BN;
    for (int it = 0; it < ntiles; ++it) {
        const int cur = it & 1;
        if (it + 1 < ntiles) {
            load_tile(sK + (cur ^ 1) * FAB_TILE, gK, (it + 1) * FA_BN, ld);
            load_tile(sV + (cur ^ 1) * FAB_TILE, gV, (it + 1) * FA_BN, ld);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        if (it == 0) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int c = ks * 16 + (lane >> 4) * 8;
                ldmatrix_x4(qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3], sQ + r * FA_LD + c);
                ldmatrix_x4(dof[ks][0], dof[ks][1], dof[ks][2], dof[ks][3], sdO + r * FA_LD + c);
            }
        }
        const bf16* cK = sK + cur * FAB_TILE;
        const bf16* cV = sV + cur * FAB_TILE;
        float s[8][4], dp[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { s[i][j] = 0.f; dp[i][j] = 0.f; }
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int np = 0; np < 4; ++np) {
                uint32_t b0, b1, b2, b3;
                const int r = np * 16 + (lane & 7) + (lane >> 4) * 8;
                const int c = ks * 16 + ((lane >> 3) & 1) * 8;
                ldmatrix_x4(b0, b1, b2, b3, cK + r * FA_LD + c);
                mma_bf16_16816(s[2 * np], qf[ks], b0, b1);
                mma_bf16_16816(s[2 * np + 1], qf[ks], b2, b3);
                ldmatrix_x4(b0, b1, b2, b3, cV + r * FA_LD + c);
                mma_bf16_16816(dp[2 * np], dof[ks], b0, b1);
                mma_bf16_16816(dp[2 * np + 1], dof[ks], b2, b3);
            }
        }
        const int key0 = it * FA_BN;
        uint32_t dsf[4][4];
        uint32_t zheld = 0;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int kc = key0 + nt * 8 + (lane & 3) * 2;
            float zs[4] = {1.f, 1.f, 1.f, 1.f};
            if (DROP) {                    // dP = (dO V^T) o Z/(1-p)
                uint32_t z[2];
                mma_rows_keep(drop, dr, b * H + h, T, q0 + warp * 16, key0 / 8, nt, lane, zheld, z);
                const int c = (lane & 3) * 2;
#pragma unroll
                for (int e = 0; e < 4; ++e) zs[e] = ((z[e >> 1] >> (c + (e & 1))) & 1u) ? drop.scale : 0.f;
            }
            float d4[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int rr = e >> 1;
                const bool ok = (kc + (e & 1)) < T;
                const float p = ok ? exp2f(fmaf(s[nt][e], scale_log2, -lse2[rr])) : 0.f;
                d4[e] = p * (dp[nt][e] * zs[e] - dl[rr]) * scale;
            }
            const int ks = nt >> 1, hi = nt & 1;
            dsf[ks][hi * 2 + 0] = pack_bf16x2(d4[0], d4[1]);
            dsf[ks][hi * 2 + 1] = pack_bf16x2(d4[2], d4[3]);
        }
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int dpp = 0; dpp < 4; ++dpp) {
                uint32_t b0, b1, b2, b3;
                const int r = ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int c = dpp * 16 + (lane >> 4) * 8;
                ldmatrix_x4_trans(b0, b1, b2, b3, cK + r * FA_LD + c);
                mma_bf16_16816(dq[2 * dpp], dsf[ks], b0, b1);
                mma_bf16_16816(dq[2 * dpp + 1], dsf[ks], b2, b3);
            }
        }
        __syncthreads();
    }
    bf16* ob = dqkv + (long long)b * T * ld + h * FA_D;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const int c = nt * 8 + (lane & 3) * 2;
        if (r0 < T) *reinterpret_cast<uint32_t*>(ob + (long long)r0 * ld + c) = pack_bf16x2(dq[nt][0], dq[nt][1]);
        if (r0 + 8 < T) *reinterpret_cast<uint32_t*>(ob + (long long)(r0 + 8) * ld + c) = pack_bf16x2(dq[nt][2], dq[nt][3]);
    }
}

// key-major pass: dV = P^T dO, dK = (P o (dO V^T - delta))^T Q * scale.   grid (ceil(T/64), H, B), 128 threads.
template <bool DROP>
__global__ void __launch_bounds__(128) mha_bwd_dkv_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ dout,
                                                          const float* __restrict__ lse, const float* __restrict__ delta,
                                                          bf16* __restrict__ dqkv, int T, int H, float scale, AttnDrop drop) {
    extern __shared__ __align__(16) bf16 fab_smem[];
    bf16* sK = fab_smem;
    bf16* sV = sK + FAB_TILE;
    bf16* sQ = sV + FAB_TILE;            // [2]
    bf16* sdO = sQ + 2 * FAB_TILE;       // [2]
    float* sL = reinterpret_cast<float*>(sdO + 2 * FAB_TILE);   // [2][64] lse * log2e
    float* sD = sL + 128;                                       // [2][64] delta
    const int k0 = blockIdx.x * FA_BN, h = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ld = 3 * H * FA_D, ldo = H * FA_D;
    const bf16* base = qkv + (long long)b * T * ld;
    const bf16* gQ = base + h * FA_D;
    const bf16* gK = base + H * FA_D + h * FA_D;
    const bf16* gV = base + 2 * H * FA_D + h * FA_D;
    const bf16* gdO = dout + (long long)b * T * ldo + h * FA_D;
    const float* lp = lse + ((long long)b * H + h) * T;
    const float* dlp = delta + ((long long)b * H + h) * T;
    auto load_tile = [&](bf16* dst, const bf16* src, int row0, int lds) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = threadIdx.x + i * 128;
            const int r = idx >> 3, c = (idx & 7) * 8;
            const bool ok = (row0 + r) < T;
            cp_async_16(dst + r * FA_LD + c, src + (long long)(ok ? row0 + r : 0) * lds + c, ok);
        }
    };
    auto load_stats = [&](int buf, int row0) {
        if (threadIdx.x < 64) {
            const int r = row0 + threadIdx.x;
            sL[buf * 64 + threadIdx.x] = r < T ? lp[r] * 1.4426950408889634f : 0.f;
            sD[buf * 64 + threadIdx.x] = r < T ? dlp[r] : 0.f;
        }
    };
    load_tile(sK, gK, k0, ld);
    load_tile(sV, gV, k0, ld);
    load_tile(sQ, gQ, 0, ld);
    load_tile(sdO, gdO, 0, ldo);
    load_stats(0, 0);
    cp_async_commit();
    const float scale_log2 = scale * 1.4426950408889634f;
    AttnDropRt dr{0ull, 0u};
    if (DROP) dr = attn_drop_load(drop);
    uint32_t kf[4][4], vf[4][4];
    float dk[8][4], dv[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { dk[i][j] = 0.f; dv[i][j] = 0.f; }
    const int ntiles = (T + FA_BM - 1) / FA_BM;
    for (int it = 0; it < ntiles; ++it) {
        const int cur = it & 1;
        if (it + 1 < ntiles) {
            load_tile(sQ + (cur ^ 1) * FAB_TILE, gQ, (it + 1) * FA_BM, ld);
            load_tile(sdO + (cur ^ 1) * FAB_TILE, gdO, (it + 1) * FA_BM, ldo);
            load_stats(cur ^ 1, (it + 1) * FA_BM);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        if (it == 0) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int c = ks * 16 + (lane >> 4) * 8;
                ldmatrix_x4(kf[ks][0], kf[ks][1], kf[ks][2], kf[ks][3], sK + r * FA_LD + c);
                ldmatrix_x4(vf[ks][0], vf[ks][1], vf[ks][2], vf[ks][3], sV + r * FA_LD + c);
            }
        }
        const bf16* cQ = sQ + cur * FAB_TILE;
        const bf16* cdO = sdO + cur * FAB_TILE;
        // S^T = K Q^T and dP^T = V dO^T : [16 keys x 64 queries] per warp
        float st[8][4], dpt[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { st[i][j] = 0.f; dpt[i][j] = 0.f; }
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int np = 0; np < 4; ++np) {
                uint32_t b0, b1, b2, b3;
                const int r = np * 16 + (lane & 7) + (lane >> 4) * 8;
                const int c = ks * 16 + ((lane >> 3) & 1) * 8;
                ldmatrix_x4(b0, b1, b2, b3, cQ + r * FA_LD + c);
                mma_bf16_16816(st[2 * np], kf[ks], b0, b1);
                mma_bf16_16816(st[2 * np + 1], kf[ks], b2, b3);
                ldmatrix_x4(b0, b1, b2, b3, cdO + r * FA_LD + c);
                mma_bf16_16816(dpt[2 * np], vf[ks], b0, b1);
                mma_bf16_16816(dpt[2 * np + 1], vf[ks], b2, b3);
            }
        }
        const int qbase = it * FA_BM;
        uint32_t pf[4][4], dsf[4][4];
        uint32_t zbits_dkv = 0;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int qc = nt * 8 + (lane & 3) * 2;         // query column within the tile
            float zs[4] = {1.f, 1.f, 1.f, 1.f};
            if (DROP) {
                // rows here are KEYS (k0 + warp*16 + lane/4, +8), columns queries: per pair of n-tiles one Philox call per
                // lane, call (query pair slot, query parity, key group, n-tile parity) = lane bits (0-1, 2, 3, 4)
                if ((nt & 1) == 0) {
                    const int q = qbase + (nt + (lane >> 4)) * 8 + (lane & 3) * 2 + ((lane >> 2) & 1);
                    zbits_dkv = attn_keep8(drop, dr, b * H + h, T, q, (k0 + warp * 16) / 8 + ((lane >> 3) & 1));
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int src = (lane & 3) | ((e & 1) << 2) | ((e >> 1) << 3) | ((nt & 1) << 4);
                    const uint32_t zb = __shfl_sync(0xffffffffu, zbits_dkv, src);
                    zs[e] = ((zb >> (lane >> 2)) & 1u) ? drop.scale : 0.f;
                }
            }
            float p4[4], d4[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int qq = qc + (e & 1);
                const bool ok = (qbase + qq) < T;
                const float p = ok ? exp2f(fmaf(st[nt][e], scale_log2, -sL[cur * 64 + qq])) : 0.f;
                p4[e] = p * zs[e];                                 // dV = (P o Z/(1-p))^T dO
                d4[e] = p * (dpt[nt][e] * zs[e] - sD[cur * 64 + qq]) * scale;
            }
            const int ks = nt >> 1, hi = nt & 1;
            pf[ks][hi * 2 + 0] = pack_bf16x2(p4[0], p4[1]);
            pf[ks][hi * 2 + 1] = pack_bf16x2(p4[2], p4[3]);
            dsf[ks][hi * 2 + 0] = pack_bf16x2(d4[0], d4[1]);
            dsf[ks][hi * 2 + 1] = pack_bf16x2(d4[2], d4[3]);
        }
        // dV += P^T dO ; dK += dS^T Q   (reduction over the 64 queries of the tile)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int dpp = 0; dpp < 4; ++dpp) {
                uint32_t b0, b1, b2, b3;
                const int r = ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int c = dpp * 16 + (lane >> 4) * 8;
                ldmatrix_x4_trans(b0, b1, b2, b3, cdO + r * FA_LD + c);
                mma_bf16_16816(dv[2 * dpp], pf[ks], b0, b1);
                mma_bf16_16816(dv[2 * dpp + 1], pf[ks], b2, b3);
                ldmatrix_x4_trans(b0, b1, b2, b3, cQ + r * FA_LD + c);
                mma_bf16_16816(dk[2 * dpp], dsf[ks], b0, b1);
                mma_bf16_16816(dk[2 * dpp + 1], dsf[ks], b2, b3);
            }
        }
        __syncthreads();
    }
    const int r0 = k0 + warp * 16 + (lane >> 2);
    bf16* okp = dqkv + (long long)b * T * ld + H * FA_D + h * FA_D;
    bf16* ovp = dqkv + (long long)b * T * ld + 2 * H * FA_D + h * FA_D;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const int c = nt * 8 + (lane & 3) * 2;
        if (r0 < T) {
            *reinterpret_cast<uint32_t*>(okp + (long long)r0 * ld + c) = pack_bf16x2(dk[nt][0], dk[nt][1]);
            *reinterpret_cast<uint32_t*>(ovp + (long long)r0 * ld + c) = pack_bf16x2(dv[nt][0], dv[nt][1]);
        }
        if (r0 + 8 < T) {
            *reinterpret_cast<uint32_t*>(okp + (long long)(r0 + 8) * ld + c) = pack_bf16x2(dk[nt][2], dk[nt][3]);
            *reinterpret_cast<uint32_t*>(ovp + (long long)(r0 + 8) * ld + c) = pack_bf16x2(dv[nt][2], dv[nt][3]);
        }
    }
}

}  // namespace a2f

namespace a2f {
int mha_tc_fwd(const void* qkv, void* out, int B, int T, int H, float scale, cudaStream_t s);   // attention_tc.cu
static int g_mha_impl = 0;          // 0 = automatic, 1 = always mma.sync, 2 = always tcgen05 (a2f_debug_set_umma_field 6)
static int g_mha_tc_min_t = 300;    // automatic: tcgen05 from this sequence length on (field 7)
int mha_impl() { return g_mha_impl; }
int mha_tc_min_t() { return g_mha_tc_min_t; }
void set_mha_impl(int v) { g_mha_impl = v; }
void set_mha_tc_min_t(int v) { g_mha_tc_min_t = v; }
}  // namespace a2f

using namespace a2f;

// attention dropout of a2f_dropout_args (NULL / p == 0 / NULL pointer = off)
static int attn_drop_from(const a2f_dropout_args* a, AttnDrop* d, bool* on) {
    *d = AttnDrop{nullptr, 0u, 0u, 1.f};
    *on = false;
    if (a == nullptr || a->seed_offset_dev == nullptr || a->p == 0.f) return A2F_OK;
    if (!(a->p > 0.f && a->p < 1.f)) return set_error(A2F_EINVAL, "attention dropout: p must lie in [0, 1)");
    *d = AttnDrop{static_cast<const unsigned long long*>(a->seed_offset_dev), a->site, dropout_threshold(a->p), 1.f / (1.f - a->p)};
    *on = true;
    return A2F_OK;
}

extern "C" int a2f_mha_fwd(const void* qkv, void* out, int dtype, int B, int T, int H, int D, float scale,
                           void* stream) {
    return a2f_mha_fwd_train(qkv, out, nullptr, nullptr, dtype, B, T, H, D, scale, stream);
}

extern "C" int a2f_mha_fwd_lse(const void* qkv, void* out, float* lse, int dtype, int B, int T, int H, int D, float scale,
                               void* stream) {
    return a2f_mha_fwd_train(qkv, out, lse, nullptr, dtype, B, T, H, D, scale, stream);
}

extern "C" int a2f_mha_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, int dtype,
                           int B, int T, int H, int D, float scale, void* workspace, size_t workspace_bytes,
                           void* stream) {
    return a2f_mha_bwd_train(qkv, out, nullptr, dout, lse, dqkv, dtype, B, T, H, D, scale, workspace, workspace_bytes, stream);
}

extern "C" int a2f_mha_bwd_train(const void* qkv, const void* out, const float* out_f32, const void* dout, const float* lse,
                                 void* dqkv, int dtype, int B, int T, int H, int D, float scale, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    return a2f_mha_bwd_train_dropout(qkv, out, out_f32, dout, lse, dqkv, dtype, B, T, H, D, scale, nullptr, workspace,
                                     workspace_bytes, stream);
}

extern "C" int a2f_mha_bwd_train_dropout(const void* qkv, const void* out, const float* out_f32, const void* dout,
                                         const float* lse, void* dqkv, int dtype, int B, int T, int H, int D, float scale,
                                         const a2f_dropout_args* dropout, void* workspace, size_t workspace_bytes,
                                         void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(qkv && out && dout && lse && dqkv && workspace && B > 0 && T > 0 && H > 0, "a2f_mha_bwd: bad arguments");
    A2F_REQUIRE(D == 64, "a2f_mha_bwd: head_dim must be 64");
    A2F_REQUIRE(workspace_bytes >= (size_t)B * H * T * sizeof(float), "a2f_mha_bwd: workspace too small (B*H*T floats)");
    AttnDrop drop;
    bool dropping;
    rc = attn_drop_from(dropout, &drop, &dropping);
    if (rc != A2F_OK) return rc;
    cudaStream_t s = as_stream(stream);
    float* delta = static_cast<float*>(workspace);
    const long long warps = (long long)B * T * H;
    const int dgrid = (int)((warps * 32 + 255) / 256);
    // delta = rowsum(dO o O) with the DROPPED output O (what the forward returned): still rowsum(dP o P) of the softmax
    if (dtype == A2F_F32) {
        mha_delta_kernel<float, float><<<dgrid, 256, 0, s>>>((const float*)out, (const float*)dout, delta, B, T, H);
        A2F_CHECK_LAUNCH("mha_delta_kernel");
        A2F_CHECK_CUDA(cudaMemsetAsync(dqkv, 0, (size_t)B * T * 3 * H * 64 * sizeof(float), s));
        mha_bwd_f32_kernel<<<(int)((warps + 3) / 4), 128, 0, s>>>((const float*)qkv, (const float*)dout, lse, delta,
                                                                  (float*)dqkv, B, T, H, scale, drop);
        A2F_CHECK_LAUNCH("mha_bwd_f32_kernel");
        count_launch(2);
    } else if (dtype == A2F_BF16) {
        if (out_f32 != nullptr)
            mha_delta_kernel<float, bf16><<<dgrid, 256, 0, s>>>(out_f32, (const bf16*)dout, delta, B, T, H);
        else
            mha_delta_kernel<bf16, bf16><<<dgrid, 256, 0, s>>>((const bf16*)out, (const bf16*)dout, delta, B, T, H);
        A2F_CHECK_LAUNCH("mha_delta_kernel");
        const size_t smem = (size_t)6 * FAB_TILE * sizeof(bf16) + 256 * sizeof(float);
        static bool attr_done = false;
        if (!attr_done) {
            A2F_CHECK_CUDA(cudaFuncSetAttribute(mha_bwd_dq_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            A2F_CHECK_CUDA(cudaFuncSetAttribute(mha_bwd_dkv_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            A2F_CHECK_CUDA(cudaFuncSetAttribute(mha_bwd_dq_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            A2F_CHECK_CUDA(cudaFuncSetAttribute(mha_bwd_dkv_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_done = true;
        }
        const dim3 grid((T + 63) / 64, H, B);
        auto dq = dropping ? mha_bwd_dq_kernel<true> : mha_bwd_dq_kernel<false>;
        auto dkv = dropping ? mha_bwd_dkv_kernel<true> : mha_bwd_dkv_kernel<false>;
        dq<<<grid, 128, smem, s>>>((const bf16*)qkv, (const bf16*)dout, lse, delta, (bf16*)dqkv, T, H, scale, drop);
        A2F_CHECK_LAUNCH("mha_bwd_dq_kernel");
        dkv<<<grid, 128, smem, s>>>((const bf16*)qkv, (const bf16*)dout, lse, delta, (bf16*)dqkv, T, H, scale, drop);
        A2F_CHECK_LAUNCH("mha_bwd_dkv_kernel");
        count_launch(3);
    } else {
        return set_error(A2F_EINVAL, "a2f_mha_bwd: bad dtype");
    }
    return A2F_OK;
}

extern "C" int a2f_mha_fwd_train(const void* qkv, void* out, float* lse, float* out_f32, int dtype, int B, int T, int H,
                                 int D, float scale, void* stream) {
    return a2f_mha_fwd_train_dropout(qkv, out, lse, out_f32, dtype, B, T, H, D, scale, nullptr, stream);
}

extern "C" int a2f_mha_fwd_train_dropout(const void* qkv, void* out, float* lse, float* out_f32, int dtype, int B, int T,
                                         int H, int D, float scale, const a2f_dropout_args* dropout, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(qkv && out && B > 0 && T > 0 && H > 0, "a2f_mha_fwd: bad arguments");
    A2F_REQUIRE(D == 64, "a2f_mha_fwd: head_dim must be 64");
    AttnDrop drop;
    bool dropping;
    rc = attn_drop_from(dropout, &drop, &dropping);
    if (rc != A2F_OK) return rc;
    cudaStream_t s = as_stream(stream);
    if (dtype == A2F_F32) {
        const long long warps = (long long)B * H * T;
        const int grid = (int)((warps * 32 + 255) / 256);
        mha_f32_kernel<<<grid, 256, 0, s>>>(static_cast<const float*>(qkv), static_cast<float*>(out), lse, B, T, H, scale, drop);
        A2F_CHECK_LAUNCH("mha_f32_kernel");
    } else if (dtype == A2F_BF16) {
        A2F_REQUIRE(reinterpret_cast<uintptr_t>(qkv) % 16 == 0, "a2f_mha_fwd: qkv must be 16-byte aligned");
        // inference forward (no log-sum-exp / fp32 side output): the tcgen05 kernel of attention_tc.cu for sequences
        // long enough to fill its 128x128 tiles; the mma.sync kernel below for short ones and for training
        const int impl = mha_impl();
        if (!dropping && lse == nullptr && out_f32 == nullptr && reinterpret_cast<uintptr_t>(out) % 16 == 0 &&
            (impl == 2 || (impl == 0 && T >= mha_tc_min_t()))) {
            rc = mha_tc_fwd(qkv, out, B, T, H, scale, s);
            if (rc != A2F_OK) return rc;
            count_launch();
            return A2F_OK;
        }
        if (impl != 1 && T <= 160) {
            // short clips: single-pass kernel with every key of a (batch, head) resident in shared memory
            const float sl2 = scale * 1.4426950408889634f;
            const bf16* q = static_cast<const bf16*>(qkv);
            bf16* o = static_cast<bf16*>(out);
            if (dropping)
                rc = T <= 80 ? launch_mha_short<5, true>(q, o, lse, out_f32, B, T, H, sl2, drop, s)
                             : launch_mha_short<10, true>(q, o, lse, out_f32, B, T, H, sl2, drop, s);
            else
                rc = T <= 80 ? launch_mha_short<5, false>(q, o, lse, out_f32, B, T, H, sl2, drop, s)
                             : launch_mha_short<10, false>(q, o, lse, out_f32, B, T, H, sl2, drop, s);
            if (rc != A2F_OK) return rc;
            count_launch();
            return A2F_OK;
        }
        const dim3 grid((T + FA_BM - 1) / FA_BM, H, B);
        auto kern = dropping ? mha_bf16_kernel<true> : mha_bf16_kernel<false>;
        A2F_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(128), 0, s, static_cast<const bf16*>(qkv), static_cast<bf16*>(out), lse,
                                  out_f32, T, H, scale * 1.4426950408889634f, drop));
        A2F_CHECK_LAUNCH("mha_bf16_kernel");
    } else {
        return set_error(A2F_EINVAL, "a2f_mha_fwd: bad dtype");
    }
    count_launch();
    return A2F_OK;
}
