// Song2Face (ref:src/model/song2face.py:5-72; registry entry "song2face" of ref:src/model/lightning_model.py:50-58):
// conv stack -> two LSTMs over the CHANNEL axis (the reference feeds [B, C=256, H=64] to a batch_first LSTM: 256 steps of
// 64 features) -> bilinear resize of the hidden axis 256 -> 32 -> four convs along it -> the Audio2Mesh output MLP + vertex
// head.  The convolutions, the LSTM input projections, the MLP and the head reuse the kernels of the other models
// (a2f_im2col1d + a2f_gemm, a2f_a2m_mlp); this file holds what is specific to the model:
//   a2f_transpose_batched   [B, R, C] -> [B, C, R] fp32 (conv output [B, H, C] -> LSTM input [B, steps = C, features = H])
//   a2f_lstm_recurrence     h_t, c_t of a batch_first single-layer LSTM given the input projections of all steps
//   a2f_song2face_resize    [B, steps, hidden] -> [B, 32, steps]: the bilinear 256 -> 32 resize of the hidden axis
//                           (F.interpolate(size=(32,1)): source index 8 i + 3.5, the mean of two neighbours) written in
//                           the channels-last layout the regression convs read
// and the pieces of the training step (model.train(), conv_training.py):
//   a2f_lstm_recurrence_train   the cluster recurrence that also saves the gates and c_t of every step
//   a2f_lstm_bptt               backpropagation through time of one LSTM on the same 8-CTA cluster layout
//   a2f_col2im1d                adjoint of a2f_im2col1d (gather form)
//   a2f_song2face_resize_bwd    adjoint of a2f_song2face_resize (gather form)
#include "a2f_common.cuh"
#include <cooperative_groups.h>
#include <stdlib.h>

namespace a2f {
namespace cg = cooperative_groups;

__global__ void __launch_bounds__(256) transpose_batched_kernel(const float* __restrict__ x, float* __restrict__ y, int R, int C) {
    __shared__ float tile[32][33];
    pdl_sync();
    const long long b = blockIdx.z;
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const float* xb = x + b * R * C;
    float* yb = y + b * R * C;
    for (int j = ty; j < 32; j += 8)
        if (r0 + j < R && c0 + tx < C) tile[j][tx] = xb[(long long)(r0 + j) * C + c0 + tx];
    __syncthreads();
    for (int j = ty; j < 32; j += 8)
        if (c0 + j < C && r0 + tx < R) yb[(long long)(c0 + j) * R + r0 + tx] = tile[tx][j];
}

// One CTA per LSTM_BT batch elements (2 for small batches: more CTAs in flight; 4 from 128 windows on: less L2 traffic --
// measured at 64 windows: BT 1 / 2 / 4 = 15.1 / 6.8 / 9.3 ms per forward); thread (u, part) owns hidden unit u and 1/LSTM_KP of the contraction (HID = 256,
// blockDim = HID * LSTM_KP).  Part 0 keeps c[b][u] in registers for the whole sequence.  Per step the four gates of unit u
// are xp[b, t, g*HID + u] (input projection with both biases, precomputed for all steps by one GEMM)
// + sum_k W_hh[g*HID + u, k] h_{t-1}[b, k]; W_hh is read TRANSPOSED ([k][4*HID], coalesced across the threads) from L2
// every step and shared by the LSTM_BT batch elements of the CTA.  The step is a chain of dependent L2 round trips, so
// the k loop is unrolled 8-fold (32 independent loads in flight per thread) and split over LSTM_KP thread groups whose
// partial sums meet in shared memory: 83 -> ~10 us per step at 64 windows.  (Next step: W_hh slices resident in the
// shared memory of an 8-CTA cluster, h exchanged through DSMEM.)  PyTorch gate order i, f, g, o; fp32 throughout.
constexpr int LSTM_KP = 4;
template <int LSTM_BT>
__global__ void __launch_bounds__(256 * LSTM_KP) lstm_recurrence_kernel(const float* __restrict__ xp, const float* __restrict__ whh_t,
                                                                       float* __restrict__ hout, int B, int T, int HID) {
    extern __shared__ float lstm_sm[];               // [2][LSTM_BT][HID] hidden states, then [LSTM_KP-1][4][LSTM_BT][HID] partials
    float* part_sm = lstm_sm + 2 * LSTM_BT * HID;
    pdl_sync();
    const int u = threadIdx.x % HID, part = threadIdx.x / HID;
    const int b0 = blockIdx.x * LSTM_BT;
    float c[LSTM_BT];
#pragma unroll
    for (int i = 0; i < LSTM_BT; ++i) {
        c[i] = 0.f;
        if (part == 0) lstm_sm[i * HID + u] = 0.f;
    }
    __syncthreads();
    const int G = 4 * HID;
    const int kper = HID / LSTM_KP, k0 = part * kper;
    for (int t = 0; t < T; ++t) {
        const float* hp = lstm_sm + (t & 1) * LSTM_BT * HID;
        float* hn = lstm_sm + ((t + 1) & 1) * LSTM_BT * HID;
        float acc[4][LSTM_BT];
#pragma unroll
        for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int i = 0; i < LSTM_BT; ++i) {
                const int b = b0 + i;
                acc[g][i] = (part == 0 && b < B) ? __ldg(xp + ((long long)b * T + t) * G + g * HID + u) : 0.f;
            }
#pragma unroll 1
        for (int kk = 0; kk < kper; kk += 8) {
            float w[8][4];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float* wr = whh_t + (long long)(k0 + kk + j) * G + u;
                w[j][0] = __ldg(wr); w[j][1] = __ldg(wr + HID); w[j][2] = __ldg(wr + 2 * HID); w[j][3] = __ldg(wr + 3 * HID);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
                for (int i = 0; i < LSTM_BT; ++i) {
                    const float h = hp[i * HID + k0 + kk + j];
                    acc[0][i] = fmaf(w[j][0], h, acc[0][i]);
                    acc[1][i] = fmaf(w[j][1], h, acc[1][i]);
                    acc[2][i] = fmaf(w[j][2], h, acc[2][i]);
                    acc[3][i] = fmaf(w[j][3], h, acc[3][i]);
                }
        }
        if (part > 0) {
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
                for (int i = 0; i < LSTM_BT; ++i) part_sm[(((part - 1) * 4 + g) * LSTM_BT + i) * HID + u] = acc[g][i];
        }
        __syncthreads();
        if (part == 0) {
#pragma unroll
            for (int i = 0; i < LSTM_BT; ++i) {
                float gsum[4];
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    float v = acc[g][i];
#pragma unroll
                    for (int pp = 0; pp < LSTM_KP - 1; ++pp) v += part_sm[((pp * 4 + g) * LSTM_BT + i) * HID + u];
                    gsum[g] = v;
                }
                const float ig = 1.f / (1.f + expf(-gsum[0])), fg = 1.f / (1.f + expf(-gsum[1]));
                const float gg = tanhf(gsum[2]), og = 1.f / (1.f + expf(-gsum[3]));
                c[i] = fmaf(fg, c[i], ig * gg);
                const float h = og * tanhf(c[i]);
                hn[i * HID + u] = h;
                const int b = b0 + i;
                if (b < B) hout[((long long)b * T + t) * HID + u] = h;
            }
        }
        __syncthreads();
    }
}

// Cluster variant: W_hh never leaves the chip.  A thread-block cluster of LC_CTAS = 8 CTAs serves LC_BT = 8 windows; CTA r
// owns hidden units [32 r, 32 r + 32) = 128 gate rows, whose W_hh rows (128 x 256 fp32, padded to a 257-float pitch:
// conflict-free for a warp of consecutive rows) sit in its shared memory for the whole sequence.  Per step: thread
// (gate row, half of the batch tile) accumulates 4 outputs over k = 0..255 (one weight LDS + one broadcast float4 LDS of
// h_{t-1} per k); the 128 x 8 gate pre-activations meet in shared memory; thread (unit, window) applies the
// nonlinearities (c stays in its registers), writes h_t to global memory and into the h buffer of ALL eight CTAs
// through distributed shared memory; one cluster barrier per step (h is double-buffered).
// TRAIN = true (training forward) also stores the post-activation gates i, f, g, o ([B, T, 4*256]) and c_t ([B, T, 256])
// for a2f_lstm_bptt; the arithmetic is the same, so hout is bit-identical to the inference instantiation.
constexpr int LC_CTAS = 8;
constexpr int LC_BT = 8;
constexpr int LC_UNITS = 32;                  // hidden units per CTA (HID = 256)
constexpr int LC_ROWS = 4 * LC_UNITS;         // gate rows per CTA
constexpr int LC_WPITCH = 257;
constexpr size_t LC_SMEM = ((size_t)LC_ROWS * LC_WPITCH + 2 * 256 * LC_BT + LC_ROWS * LC_BT) * sizeof(float);

template <bool TRAIN>
__global__ void __cluster_dims__(LC_CTAS, 1, 1) __launch_bounds__(256, 1)
lstm_cluster_kernel(const float* __restrict__ xp, const float* __restrict__ whh, float* __restrict__ hout, int B, int T,
                    float* __restrict__ gates_out, float* __restrict__ cell_out) {
    extern __shared__ __align__(16) float lc_sm[];
    float* wsm = lc_sm;                                   // [LC_ROWS][LC_WPITCH]   local row g*32 + j = gate g of unit u0 + j
    float* hsm = wsm + LC_ROWS * LC_WPITCH;               // [2][256 k][LC_BT]      hidden state, k-major, windows innermost
    float* gsm = hsm + 2 * 256 * LC_BT;                   // [LC_ROWS][LC_BT]       gate pre-activations of this step
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int b0 = ((int)blockIdx.x / LC_CTAS) * LC_BT;
    const int u0 = rank * LC_UNITS;
    const int tid = threadIdx.x;
    for (int i = tid; i < LC_ROWS * 256; i += 256) {      // W_hh rows of this CTA (module weights: safe before the PDL wait)
        const int lr = i >> 8, k = i & 255;
        const int g = lr / LC_UNITS, j = lr - g * LC_UNITS;
        wsm[lr * LC_WPITCH + k] = __ldg(whh + (long long)(g * 256 + u0 + j) * 256 + k);
    }
    for (int i = tid; i < 2 * 256 * LC_BT; i += 256) hsm[i] = 0.f;
    pdl_sync();
    cluster.sync();
    const int row = tid & (LC_ROWS - 1), bh = tid >> 7;   // MAC phase: gate row, half of the batch tile (4 windows)
    const int gu = tid & (LC_UNITS - 1), gb = tid >> 5;   // gate phase: unit, window
    const int grow = (row / LC_UNITS) * 256 + u0 + (row % LC_UNITS);     // global gate row of `row`
    float c = 0.f;
    float nxt[4];                                          // input projections of the next step, requested one step ahead
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int b = b0 + bh * 4 + i;
        nxt[i] = (b < B && T > 0) ? __ldg(xp + ((long long)b * T) * 1024 + grow) : 0.f;
    }
    for (int t = 0; t < T; ++t) {
        const float* hp = hsm + (t & 1) * 256 * LC_BT;
        float acc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            acc[i] = nxt[i];
            const int b = b0 + bh * 4 + i;
            nxt[i] = (b < B && t + 1 < T) ? __ldg(xp + ((long long)b * T + t + 1) * 1024 + grow) : 0.f;
        }
        const float* wr = wsm + row * LC_WPITCH;
#pragma unroll 8
        for (int k = 0; k < 256; ++k) {
            const float w = wr[k];
            const float4 h4 = *reinterpret_cast<const float4*>(hp + k * LC_BT + bh * 4);
            acc[0] = fmaf(w, h4.x, acc[0]);
            acc[1] = fmaf(w, h4.y, acc[1]);
            acc[2] = fmaf(w, h4.z, acc[2]);
            acc[3] = fmaf(w, h4.w, acc[3]);
        }
        *reinterpret_cast<float4*>(gsm + row * LC_BT + bh * 4) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        __syncthreads();
        {
            const float gi = gsm[(0 * LC_UNITS + gu) * LC_BT + gb], gf = gsm[(1 * LC_UNITS + gu) * LC_BT + gb];
            const float gg = gsm[(2 * LC_UNITS + gu) * LC_BT + gb], go = gsm[(3 * LC_UNITS + gu) * LC_BT + gb];
            const float ig = 1.f / (1.f + expf(-gi)), fg = 1.f / (1.f + expf(-gf));
            const float og = 1.f / (1.f + expf(-go));
            const float tg = tanhf(gg);
            c = fmaf(fg, c, ig * tg);
            const float h = og * tanhf(c);
            const int b = b0 + gb;
            if (b < B) {
                const long long bt = (long long)b * T + t;
                hout[bt * 256 + u0 + gu] = h;
                if (TRAIN) {
                    float* gp = gates_out + bt * 1024 + u0 + gu;
                    gp[0] = ig; gp[256] = fg; gp[512] = tg; gp[768] = og;
                    cell_out[bt * 256 + u0 + gu] = c;
                }
            }
            const int dst = ((t + 1) & 1) * 256 * LC_BT + (u0 + gu) * LC_BT + gb;
#pragma unroll
            for (int r = 0; r < LC_CTAS; ++r) cluster.map_shared_rank(hsm, r)[dst] = h;
        }
        cluster.sync();                                   // h_t visible in every CTA; gsm free for the next step
    }
}

// Backpropagation through time of one LSTM on the cluster layout of the forward: an 8-CTA cluster serves LC_BT = 8 windows,
// CTA r owns hidden units [32 r, 32 r + 32), their 128 W_hh rows (resident in shared memory, 257-float pitch) and their
// dc registers.  Step t (T-1 down to 0), thread (unit, window):
//   dh = dh_out[b, t, u] + dh_rec_t[b, u];  tc = tanh(c_t);  dc += dh o (1 - tc^2)
//   da_i = dc g i (1-i)   da_f = dc c_{t-1} f (1-f)   da_g = dc i (1 - g^2)   da_o = dh tc o (1-o);   dc <- dc f
// then thread k forms the partial dh_rec_{t-1}[b, k] = sum over the CTA's 128 rows of W_hh[row, k] da_t[row, b] for the 8
// windows and stores it into receive slot `rank` of the CTA that owns unit k (DSMEM).  After one cluster barrier each
// CTA sums its 8 slots in rank order: that is dh_rec_{t-1} of its own units, so a step needs no other exchange.  The
// receive buffer is double-buffered by step parity; the saved gates, c and dh_out are requested one step ahead.  No
// atomics: the result does not depend on scheduling.
constexpr size_t LB_SMEM = ((size_t)LC_ROWS * LC_WPITCH + 2 * LC_CTAS * LC_BT * LC_UNITS + LC_ROWS * LC_BT) * sizeof(float);

__global__ void __cluster_dims__(LC_CTAS, 1, 1) __launch_bounds__(256, 1)
lstm_bptt_kernel(const float* __restrict__ dh_out, const float* __restrict__ gates, const float* __restrict__ cell,
                 const float* __restrict__ whh, float* __restrict__ dgates, int B, int T) {
    extern __shared__ __align__(16) float lb_sm[];
    float* wsm = lb_sm;                                   // [LC_ROWS][LC_WPITCH]   local row g*32 + j = gate g of unit u0 + j
    float* rsm = wsm + LC_ROWS * LC_WPITCH;               // [2][LC_CTAS slot][LC_BT window][LC_UNITS]   partial dh_rec
    float* dsm = rsm + 2 * LC_CTAS * LC_BT * LC_UNITS;    // [LC_ROWS][LC_BT]       da of this step
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int b0 = ((int)blockIdx.x / LC_CTAS) * LC_BT;
    const int u0 = rank * LC_UNITS;
    const int tid = threadIdx.x;
    for (int i = tid; i < LC_ROWS * 256; i += 256) {
        const int lr = i >> 8, k = i & 255;
        const int g = lr / LC_UNITS, j = lr - g * LC_UNITS;
        wsm[lr * LC_WPITCH + k] = __ldg(whh + (long long)(g * 256 + u0 + j) * 256 + k);
    }
    for (int i = tid; i < 2 * LC_CTAS * LC_BT * LC_UNITS; i += 256) rsm[i] = 0.f;
    pdl_sync();
    cluster.sync();
    const int gu = tid & (LC_UNITS - 1), gb = tid >> 5;   // gate phase: unit, window
    const int b = b0 + gb;
    const bool live = b < B;
    const int dst_cta = tid >> 5, dst_u = tid & (LC_UNITS - 1);     // MAC phase: thread = k = 32 * dst_cta + dst_u
    float dc = 0.f;
    // values of step t, requested during step t + 1
    float ng[4], nc_prev = 0.f, ndh = 0.f, c_t = 0.f;
    {
        const long long bt = (long long)b * T + (T - 1);
#pragma unroll
        for (int g = 0; g < 4; ++g) ng[g] = live ? __ldg(gates + bt * 1024 + g * 256 + u0 + gu) : 0.f;
        c_t = live ? __ldg(cell + bt * 256 + u0 + gu) : 0.f;
        nc_prev = (live && T > 1) ? __ldg(cell + (bt - 1) * 256 + u0 + gu) : 0.f;
        ndh = live ? __ldg(dh_out + bt * 256 + u0 + gu) : 0.f;
    }
    for (int t = T - 1; t >= 0; --t) {
        const float ig = ng[0], fg = ng[1], gg = ng[2], og = ng[3];
        const float c_prev = nc_prev;
        float dh = ndh;
        if (t > 0) {
            const long long bt = (long long)b * T + (t - 1);
#pragma unroll
            for (int g = 0; g < 4; ++g) ng[g] = live ? __ldg(gates + bt * 1024 + g * 256 + u0 + gu) : 0.f;
            nc_prev = (live && t > 1) ? __ldg(cell + (bt - 1) * 256 + u0 + gu) : 0.f;
            ndh = live ? __ldg(dh_out + bt * 256 + u0 + gu) : 0.f;
        }
        const float* rp = rsm + (t & 1) * LC_CTAS * LC_BT * LC_UNITS + gb * LC_UNITS + gu;
#pragma unroll
        for (int r = 0; r < LC_CTAS; ++r) dh += rp[r * LC_BT * LC_UNITS];
        const float tc = tanhf(c_t);
        dc = fmaf(dh * og, 1.f - tc * tc, dc);
        const float da_i = dc * gg * ig * (1.f - ig);
        const float da_f = dc * c_prev * fg * (1.f - fg);
        const float da_g = dc * ig * (1.f - gg * gg);
        const float da_o = dh * tc * og * (1.f - og);
        dc *= fg;
        c_t = c_prev;
        if (live) {
            float* dp = dgates + ((long long)b * T + t) * 1024 + u0 + gu;
            dp[0] = da_i; dp[256] = da_f; dp[512] = da_g; dp[768] = da_o;
        }
        if (t == 0) break;                                // dh_rec_{-1} is not needed; every CTA leaves at the same step
        dsm[(0 * LC_UNITS + gu) * LC_BT + gb] = da_i;
        dsm[(1 * LC_UNITS + gu) * LC_BT + gb] = da_f;
        dsm[(2 * LC_UNITS + gu) * LC_BT + gb] = da_g;
        dsm[(3 * LC_UNITS + gu) * LC_BT + gb] = da_o;
        __syncthreads();
        float acc[LC_BT];
#pragma unroll
        for (int i = 0; i < LC_BT; ++i) acc[i] = 0.f;
        const float* wk = wsm + tid;
#pragma unroll 8
        for (int lr = 0; lr < LC_ROWS; ++lr) {
            const float w = wk[lr * LC_WPITCH];
            const float4 d0 = *reinterpret_cast<const float4*>(dsm + lr * LC_BT);
            const float4 d1 = *reinterpret_cast<const float4*>(dsm + lr * LC_BT + 4);
            acc[0] = fmaf(w, d0.x, acc[0]); acc[1] = fmaf(w, d0.y, acc[1]);
            acc[2] = fmaf(w, d0.z, acc[2]); acc[3] = fmaf(w, d0.w, acc[3]);
            acc[4] = fmaf(w, d1.x, acc[4]); acc[5] = fmaf(w, d1.y, acc[5]);
            acc[6] = fmaf(w, d1.z, acc[6]); acc[7] = fmaf(w, d1.w, acc[7]);
        }
        float* remote = cluster.map_shared_rank(rsm, dst_cta) + ((t - 1) & 1) * LC_CTAS * LC_BT * LC_UNITS +
                        rank * LC_BT * LC_UNITS + dst_u;
#pragma unroll
        for (int i = 0; i < LC_BT; ++i) remote[i * LC_UNITS] = acc[i];
        cluster.sync();                                   // partials visible in their owner CTAs; dsm free for the next step
    }
}

// Adjoint of im2col1d_split_kernel<false> (gather form, one thread per element of dx):
//   dx[o, l, c] = sum over (lo, tap) with lo*stride - pad + tap = l of dcol[o*L_out + lo, tap*C + c] (* scale[c])
__global__ void __launch_bounds__(256) col2im1d_kernel(const float* __restrict__ dcol, long long outer, long long outer_stride,
                                                       int ld, int C, int L, int L_out, int taps, int stride, int pad,
                                                       const float* __restrict__ scale, int kpad, float* __restrict__ dx) {
    pdl_sync();
    const long long total = outer * L * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const int l = (int)((i / C) % L);
        const long long o = i / ((long long)C * L);
        const float* dco = dcol + o * L_out * kpad + c;
        float s = 0.f;
        for (int tap = (l + pad) % stride; tap < taps; tap += stride) {
            const int lo = (l + pad - tap) / stride;
            if (lo >= 0 && lo < L_out) s += __ldg(dco + (long long)lo * kpad + tap * C);
        }
        if (scale != nullptr) s *= __ldg(scale + c);
        dx[o * outer_stride + (long long)l * ld + c] = s;
    }
}

// Adjoint of song2face_resize_kernel (gather form): dh[b, t, j] = sum_i w(i, j) dout[b, i, t] over the output rows i whose
// two bilinear taps touch j, with the forward's float arithmetic for the taps and weights.  Every column is written.
__global__ void __launch_bounds__(256) song2face_resize_bwd_kernel(const float* __restrict__ dout, int B, int T, int HID,
                                                                   int out_h, float* __restrict__ dh) {
    pdl_sync();
    const long long total = (long long)B * T * HID;
    const float scale = (float)HID / (float)out_h;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(idx % HID);
        const int t = (int)((idx / HID) % T);
        const long long b = idx / ((long long)HID * T);
        // rows whose source index lies in [j - 1, j + 1), with a margin of 2 on each side
        int i_lo = (int)floorf(((float)j - 0.5f) / scale - 0.5f) - 2;
        int i_hi = (int)ceilf(((float)j + 1.5f) / scale - 0.5f) + 2;
        if (i_lo < 0) i_lo = 0;
        if (i_hi > out_h - 1) i_hi = out_h - 1;
        float s = 0.f;
        for (int i = i_lo; i <= i_hi; ++i) {
            float src = scale * ((float)i + 0.5f) - 0.5f;
            if (src < 0.f) src = 0.f;
            int j0 = (int)src;
            if (j0 > HID - 1) j0 = HID - 1;
            const int j1 = j0 + (j0 < HID - 1 ? 1 : 0);
            const float l1 = src - (float)j0, l0 = 1.f - l1;
            const float g = __ldg(dout + (b * out_h + i) * T + t);
            if (j0 == j) s = fmaf(l0, g, s);
            if (j1 == j) s = fmaf(l1, g, s);
        }
        dh[idx] = s;
    }
}

// out[b, i, t] = 0.5 * (h[b, t, 8 i + 3] + h[b, t, 8 i + 4]) generalised: bilinear source index of F.interpolate
// (align_corners = False) along the hidden axis, output channels-last [B, out_h, steps]
__global__ void __launch_bounds__(256) song2face_resize_kernel(const float* __restrict__ h, int B, int T, int HID, int out_h,
                                                               float* __restrict__ out) {
    pdl_sync();
    const long long total = (long long)B * out_h * T;
    const float scale = (float)HID / (float)out_h;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(idx % T);
        const int i = (int)((idx / T) % out_h);
        const long long b = idx / ((long long)T * out_h);
        float src = scale * ((float)i + 0.5f) - 0.5f;
        if (src < 0.f) src = 0.f;
        int j0 = (int)src;
        if (j0 > HID - 1) j0 = HID - 1;
        const int j1 = j0 + (j0 < HID - 1 ? 1 : 0);
        const float l1 = src - (float)j0, l0 = 1.f - l1;
        const float* row = h + (b * T + t) * HID;
        out[idx] = l0 * row[j0] + l1 * row[j1];
    }
}

}  // namespace a2f

using namespace a2f;

extern "C" {

int a2f_transpose_batched(const float* x, float* y, int B, int R, int C, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(x && y && B > 0 && R > 0 && C > 0 && B < 65536, "a2f_transpose_batched: bad arguments");
    const dim3 grid((C + 31) / 32, (R + 31) / 32, B);
    A2F_CHECK_CUDA(launch_pdl(transpose_batched_kernel, grid, dim3(256), 0, as_stream(stream), x, y, R, C));
    count_launch();
    return A2F_OK;
}

static int g_lstm_impl = 0;      // debug: 1 = never use the cluster kernel
int a2f_lstm_recurrence(const float* xp, const float* whh_t, const float* whh_n, float* hout, int B, int T, int hidden,
                        void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(xp && whh_t && hout && B > 0 && T > 0, "a2f_lstm_recurrence: bad arguments");
    {
        const char* e = getenv("A2F_LSTM_IMPL");
        g_lstm_impl = (e && e[0] == '1') ? 1 : 0;
    }
    A2F_REQUIRE(hidden == 256, "a2f_lstm_recurrence: hidden size must be 256 (one thread per unit)");
    if (B >= 4 && g_lstm_impl != 1) {
        // cluster kernel: W_hh (un-transposed [4*hidden, hidden]) resident in shared memory; whh_n must be given
        A2F_REQUIRE(whh_n != nullptr, "a2f_lstm_recurrence: the cluster kernel needs W_hh in its [4*hidden, hidden] layout");
        static bool cattr = false;
        if (!cattr) {
            A2F_CHECK_CUDA(cudaFuncSetAttribute(lstm_cluster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LC_SMEM));
            cattr = true;
        }
        const int groups = (B + LC_BT - 1) / LC_BT;
        A2F_CHECK_CUDA(launch_pdl(lstm_cluster_kernel<false>, dim3(groups * LC_CTAS), dim3(256), LC_SMEM, as_stream(stream), xp, whh_n,
                                  hout, B, T, (float*)nullptr, (float*)nullptr));
        count_launch();
        return A2F_OK;
    }
    const int bt = B >= 128 ? 4 : 2;
    const size_t smem = ((size_t)2 * bt * hidden + (size_t)(LSTM_KP - 1) * 4 * bt * hidden) * sizeof(float);
    static bool attr_done = false;
    if (!attr_done) {
        A2F_CHECK_CUDA(cudaFuncSetAttribute(lstm_recurrence_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        A2F_CHECK_CUDA(cudaFuncSetAttribute(lstm_recurrence_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attr_done = true;
    }
    if (bt == 2)
        A2F_CHECK_CUDA(launch_pdl(lstm_recurrence_kernel<2>, dim3((B + 1) / 2), dim3(hidden * LSTM_KP), smem, as_stream(stream), xp,
                                  whh_t, hout, B, T, hidden));
    else
        A2F_CHECK_CUDA(launch_pdl(lstm_recurrence_kernel<4>, dim3((B + 3) / 4), dim3(hidden * LSTM_KP), smem, as_stream(stream), xp,
                                  whh_t, hout, B, T, hidden));
    count_launch();
    return A2F_OK;
}

int a2f_lstm_recurrence_train(const float* xp, const float* whh_n, float* hout, float* gates, float* cell, int B, int T, int hidden,
                              void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(xp && whh_n && hout && gates && cell && B > 0 && T > 0, "a2f_lstm_recurrence_train: bad arguments");
    A2F_REQUIRE(hidden == 256, "a2f_lstm_recurrence_train: hidden size must be 256");
    static bool attr = false;
    if (!attr) {
        A2F_CHECK_CUDA(cudaFuncSetAttribute(lstm_cluster_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LC_SMEM));
        attr = true;
    }
    const int groups = (B + LC_BT - 1) / LC_BT;
    A2F_CHECK_CUDA(launch_pdl(lstm_cluster_kernel<true>, dim3(groups * LC_CTAS), dim3(256), LC_SMEM, as_stream(stream), xp, whh_n,
                              hout, B, T, gates, cell));
    count_launch();
    return A2F_OK;
}

int a2f_lstm_bptt(const float* dh_out, const float* gates, const float* cell, const float* whh_n, float* dgates, int B, int T,
                  int hidden, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dh_out && gates && cell && whh_n && dgates && B > 0 && T > 0, "a2f_lstm_bptt: bad arguments");
    A2F_REQUIRE(hidden == 256, "a2f_lstm_bptt: hidden size must be 256");
    static bool attr = false;
    if (!attr) {
        A2F_CHECK_CUDA(cudaFuncSetAttribute(lstm_bptt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LB_SMEM));
        attr = true;
    }
    const int groups = (B + LC_BT - 1) / LC_BT;
    A2F_CHECK_CUDA(launch_pdl(lstm_bptt_kernel, dim3(groups * LC_CTAS), dim3(256), LB_SMEM, as_stream(stream), dh_out, gates, cell,
                              whh_n, dgates, B, T));
    count_launch();
    return A2F_OK;
}

int a2f_col2im1d(float* dx, long long outer, long long outer_stride, int ld, int C, int L, int taps, int stride, int pad,
                 const float* scale, const float* shift, int kpad, const float* dcol, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dx && dcol && outer > 0 && C > 0 && L > 0 && taps > 0 && stride > 0 && pad >= 0 && ld >= C, "a2f_col2im1d: bad arguments");
    A2F_REQUIRE((scale == nullptr) == (shift == nullptr), "a2f_col2im1d: scale and shift come together");
    A2F_REQUIRE(kpad >= taps * C, "a2f_col2im1d: kpad must cover taps*C");
    const int L_out = (L + 2 * pad - taps) / stride + 1;
    A2F_REQUIRE(L_out > 0, "a2f_col2im1d: empty output");
    const long long total = outer * L * C;
    long long blocks = (total + 255) / 256;
    if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
    A2F_CHECK_CUDA(launch_pdl(col2im1d_kernel, dim3((unsigned)blocks), dim3(256), 0, as_stream(stream), dcol, outer, outer_stride, ld, C,
                              L, L_out, taps, stride, pad, scale, kpad, dx));
    count_launch();
    return A2F_OK;
}

int a2f_song2face_resize_bwd(const float* dout, int B, int T, int hidden, int out_h, float* dh, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dout && dh && B > 0 && T > 0 && hidden > 0 && out_h > 0, "a2f_song2face_resize_bwd: bad arguments");
    const long long total = (long long)B * T * hidden;
    long long blocks = (total + 255) / 256;
    if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
    A2F_CHECK_CUDA(launch_pdl(song2face_resize_bwd_kernel, dim3((unsigned)blocks), dim3(256), 0, as_stream(stream), dout, B, T, hidden,
                              out_h, dh));
    count_launch();
    return A2F_OK;
}

int a2f_song2face_resize(const float* h, int B, int T, int hidden, int out_h, float* out, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(h && out && B > 0 && T > 0 && hidden > 0 && out_h > 0, "a2f_song2face_resize: bad arguments");
    const long long total = (long long)B * out_h * T;
    long long blocks = (total + 255) / 256;
    if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
    A2F_CHECK_CUDA(launch_pdl(song2face_resize_kernel, dim3((unsigned)blocks), dim3(256), 0, as_stream(stream), h, B, T, hidden,
                              out_h, out));
    count_launch();
    return A2F_OK;
}

}  // extern "C"
