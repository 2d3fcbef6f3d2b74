// Training-step kernels of the two convolutional models (ref:src/model/voca.py, ref:src/model/audio2face.py under
// Lightning's training_step, ref:src/model/lightning_model.py:150-161): train-mode BatchNorm2d (batch statistics,
// running-stat update) forward / backward over the zero-padded channels-last activations of a2m.cu, the fused
// affine + activation pass, and VOCA's input assembly.  The convolutions and Linears themselves are a2f_gemm /
// a2f_gemm_wgrad calls (implicit GEMM, gather-segment data gradients).
//
// Layout convention shared by every kernel here: element (batch b, row r, channel c) of a tensor lives at
//   base + b*batch_stride + r*ld + c,   b < batches, r < rows_per_batch, c < C
// (the caller passes `base` already advanced past the left zero padding, so padding is never touched).
#include "a2f_common.cuh"

namespace a2f {

// VOCA input (ref voca.py:40-45): x [B,29,16] features x frames, one-hot tiling emb[r][c] = oh8[(16 r + c) % 8],
// concatenated along the feature axis and permuted so that features are channels and the 16 frames are rows:
// out [B, 17, 37] channels-last with row 0 = left zero padding of the (3x1, stride 2, pad 1) convs.
__global__ void voca_assemble_kernel(const float* __restrict__ x, const float* __restrict__ one_hot, int n_onehot,
                                     float* __restrict__ out, int B) {
    const long long n = (long long)B * 17 * 37;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int c = (int)(i % 37);
        const int r = (int)((i / 37) % 17);
        const long long b = i / (37 * 17);
        float v = 0.f;
        if (r > 0) {
            const int h = r - 1;
            if (c < 29) v = x[(b * 29 + c) * 16 + h];
            else v = one_hot[b * n_onehot + ((16 * (c - 29) + h) % 8)];
        }
        out[i] = v;
    }
}

// sums[c] += sum x, sums[C + c] += sum x^2 over all (b, r): blockDim.x = 32 channels x 8 row lanes
__global__ void __launch_bounds__(256) bn_moments_kernel(const float* __restrict__ x, int C, long long rows_per_batch,
                                                         long long ld, long long batch_stride, long long batches,
                                                         double* __restrict__ sums) {
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int rl = threadIdx.x >> 5;
    const long long rows = batches * rows_per_batch;
    double s = 0.0, q = 0.0;
    if (c < C) {
        for (long long row = (long long)blockIdx.y * 8 + rl; row < rows; row += (long long)gridDim.y * 8) {
            const long long b = row / rows_per_batch, r = row - b * rows_per_batch;
            const float v = x[b * batch_stride + r * ld + c];
            s += v;
            q += (double)v * v;
        }
    }
    __shared__ double sh[2][8][32];
    sh[0][rl][threadIdx.x & 31] = s;
    sh[1][rl][threadIdx.x & 31] = q;
    __syncthreads();
    if (rl == 0 && c < C) {
#pragma unroll
        for (int j = 1; j < 8; ++j) {
            s += sh[0][j][threadIdx.x];
            q += sh[1][j][threadIdx.x];
        }
        atomicAdd(&sums[c], s);
        atomicAdd(&sums[C + c], q);
    }
}

// mean / rstd, the fused scale / shift of y = gamma*(x-mean)*rstd + beta, and the running-stat update
// (torch BatchNorm2d train mode: biased variance normalises, unbiased variance feeds running_var, momentum 0.1)
// FROZEN (eval-mode BatchNorm): mean / var are the running statistics, which are only read; `sums` is unused
template <bool FROZEN>
__global__ void bn_finalize_kernel(const double* __restrict__ sums, int C, double n, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float* __restrict__ mean_rstd,
                                   float* __restrict__ scale_shift) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double mean, var;
    if (FROZEN) {
        mean = running_mean[c];
        var = running_var[c];
    } else {
        mean = sums[c] / n;
        var = sums[C + c] / n - mean * mean;
        if (var < 0.0) var = 0.0;
    }
    const double rstd = 1.0 / sqrt(var + (double)eps);
    mean_rstd[c] = (float)mean;
    mean_rstd[C + c] = (float)rstd;
    const float sc = (float)((double)gamma[c] * rstd);
    scale_shift[c] = sc;
    scale_shift[C + c] = (float)((double)beta[c] - mean * (double)gamma[c] * rstd);
    if (!FROZEN && running_mean != nullptr) {
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
        const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
}

__global__ void __launch_bounds__(256) affine_act_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                         const float* __restrict__ scale, const float* __restrict__ shift,
                                                         int act, int C, long long rows_per_batch, long long ld_in,
                                                         long long bs_in, long long ld_out, long long bs_out,
                                                         long long batches) {
    const long long n = batches * rows_per_batch * C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int c = (int)(i % C);
        const long long row = i / C;
        const long long b = row / rows_per_batch, r = row - b * rows_per_batch;
        float v = in[b * bs_in + r * ld_in + c];
        if (scale != nullptr) v = fmaf(v, scale[c], shift[c]);
        out[b * bs_out + r * ld_out + c] = apply_act_rt(v, act);
    }
}

// sums[c] += sum dy_eff, sums[C+c] += sum dy_eff * xhat;  dy_eff = dy * (y > 0) when a ReLU followed the BatchNorm
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                                                            const float* __restrict__ z, const float* __restrict__ mean_rstd,
                                                            int C, long long rows_per_batch, long long ld,
                                                            long long batch_stride, long long batches,
                                                            double* __restrict__ sums) {
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int rl = threadIdx.x >> 5;
    const long long rows = batches * rows_per_batch;
    double s = 0.0, q = 0.0;
    if (c < C) {
        const float mean = mean_rstd[c], rstd = mean_rstd[C + c];
        for (long long row = (long long)blockIdx.y * 8 + rl; row < rows; row += (long long)gridDim.y * 8) {
            const long long b = row / rows_per_batch, r = row - b * rows_per_batch;
            const long long off = b * batch_stride + r * ld + c;
            float g = dy[off];
            if (y != nullptr && !(y[off] > 0.f)) g = 0.f;
            s += g;
            q += (double)g * ((z[off] - mean) * rstd);
        }
    }
    __shared__ double sh[2][8][32];
    sh[0][rl][threadIdx.x & 31] = s;
    sh[1][rl][threadIdx.x & 31] = q;
    __syncthreads();
    if (rl == 0 && c < C) {
#pragma unroll
        for (int j = 1; j < 8; ++j) {
            s += sh[0][j][threadIdx.x];
            q += sh[1][j][threadIdx.x];
        }
        atomicAdd(&sums[c], s);
        atomicAdd(&sums[C + c], q);
    }
}

// dz = gamma*rstd * (dy_eff - mean(dy_eff) - xhat * mean(dy_eff * xhat));  dgamma += sum dy_eff*xhat, dbeta += sum dy_eff
// FROZEN (eval-mode BatchNorm, mean / rstd from the running statistics, so constants): dz = gamma*rstd * dy_eff
template <bool FROZEN>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                                                           const float* __restrict__ z, const float* __restrict__ mean_rstd,
                                                           const float* __restrict__ gamma, const double* __restrict__ sums,
                                                           double n, int C, long long rows_per_batch, long long ld,
                                                           long long batch_stride, long long batches, float* __restrict__ dz,
                                                           float* __restrict__ dgamma, float* __restrict__ dbeta) {
    const long long total = batches * rows_per_batch * C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long j = i; j < C; j += stride) {
        dgamma[j] += (float)sums[C + j];
        dbeta[j] += (float)sums[j];
    }
    for (; i < total; i += stride) {
        const int c = (int)(i % C);
        const long long row = i / C;
        const long long b = row / rows_per_batch, r = row - b * rows_per_batch;
        const long long off = b * batch_stride + r * ld + c;
        float g = dy[off];
        if (y != nullptr && !(y[off] > 0.f)) g = 0.f;
        const float rstd = mean_rstd[C + c];
        if (FROZEN) {
            dz[off] = gamma[c] * rstd * g;
        } else {
            const float xh = (z[off] - mean_rstd[c]) * rstd;
            const float m1 = (float)(sums[c] / n), m2 = (float)(sums[C + c] / n);
            dz[off] = gamma[c] * rstd * (g - m1 - xh * m2);
        }
    }
}

static int ew_blocks(long long n) {
    long long b = (n + 255) / 256;
    const long long cap = 8LL * sm_count();
    return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

// a2f_bn_train_bwd / a2f_bn_frozen_bwd after argument checks: the same two launches (reduce, apply), differing only in
// the apply instantiation
template <bool FROZEN>
static int bn_bwd_launch(const float* dy, const float* y_relu, const float* z, const float* mean_rstd, const float* gamma,
                         int C, long long rows_per_batch, long long ld, long long batch_stride, long long batches,
                         float* dz, float* dgamma, float* dbeta, void* workspace, void* stream) {
    cudaStream_t s = as_stream(stream);
    double* sums = static_cast<double*>(workspace);
    A2F_CHECK_CUDA(cudaMemsetAsync(sums, 0, (size_t)2 * C * sizeof(double), s));
    const long long rows = batches * rows_per_batch;
    long long gy = (rows + 63) / 64;
    if (gy > 256) gy = 256;
    bn_bwd_reduce_kernel<<<dim3((C + 31) / 32, (unsigned)gy), 256, 0, s>>>(dy, y_relu, z, mean_rstd, C, rows_per_batch, ld,
                                                                            batch_stride, batches, sums);
    A2F_CHECK_LAUNCH("bn_bwd_reduce_kernel");
    bn_bwd_apply_kernel<FROZEN><<<ew_blocks(rows * C), 256, 0, s>>>(dy, y_relu, z, mean_rstd, gamma, sums, (double)rows, C,
                                                                     rows_per_batch, ld, batch_stride, batches, dz, dgamma,
                                                                     dbeta);
    A2F_CHECK_LAUNCH("bn_bwd_apply_kernel");
    count_launch(2);
    return A2F_OK;
}

}  // namespace a2f

using namespace a2f;

extern "C" {

int a2f_voca_assemble(const float* x, const float* one_hot, int n_onehot, float* out, int B, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(x && one_hot && out && n_onehot >= 8, "a2f_voca_assemble: bad arguments (needs >= 8 one-hot columns)");
    if (B <= 0) return A2F_OK;
    voca_assemble_kernel<<<ew_blocks((long long)B * 17 * 37), 256, 0, as_stream(stream)>>>(x, one_hot, n_onehot, out, B);
    A2F_CHECK_LAUNCH("voca_assemble_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_bn_train_stats(const float* x, int C, long long rows_per_batch, long long ld, long long batch_stride,
                       long long batches, const float* gamma, const float* beta, float eps, float momentum,
                       float* running_mean, float* running_var, float* mean_rstd, float* scale_shift, void* workspace,
                       size_t workspace_bytes, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(x && gamma && beta && mean_rstd && scale_shift && workspace && C > 0 && rows_per_batch > 0 && batches > 0,
                "a2f_bn_train_stats: bad arguments");
    A2F_REQUIRE(workspace_bytes >= (size_t)2 * C * sizeof(double), "a2f_bn_train_stats: workspace too small (2*C doubles)");
    A2F_REQUIRE((running_mean == nullptr) == (running_var == nullptr), "a2f_bn_train_stats: pass both running stats or none");
    cudaStream_t s = as_stream(stream);
    double* sums = static_cast<double*>(workspace);
    A2F_CHECK_CUDA(cudaMemsetAsync(sums, 0, (size_t)2 * C * sizeof(double), s));
    const long long rows = batches * rows_per_batch;
    long long gy = (rows + 63) / 64;
    if (gy > 256) gy = 256;
    bn_moments_kernel<<<dim3((C + 31) / 32, (unsigned)gy), 256, 0, s>>>(x, C, rows_per_batch, ld, batch_stride, batches, sums);
    A2F_CHECK_LAUNCH("bn_moments_kernel");
    bn_finalize_kernel<false><<<(C + 127) / 128, 128, 0, s>>>(sums, C, (double)rows, gamma, beta, eps, momentum,
                                                               running_mean, running_var, mean_rstd, scale_shift);
    A2F_CHECK_LAUNCH("bn_finalize_kernel");
    count_launch(2);
    return A2F_OK;
}

int a2f_bn_frozen_stats(const float* gamma, const float* beta, float eps, const float* running_mean,
                        const float* running_var, int C, float* mean_rstd, float* scale_shift, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(gamma && beta && running_mean && running_var && mean_rstd && scale_shift && C > 0,
                "a2f_bn_frozen_stats: bad arguments");
    bn_finalize_kernel<true><<<(C + 127) / 128, 128, 0, as_stream(stream)>>>(
        nullptr, C, 1.0, gamma, beta, eps, 0.f, const_cast<float*>(running_mean), const_cast<float*>(running_var),
        mean_rstd, scale_shift);
    A2F_CHECK_LAUNCH("bn_finalize_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_affine_act(const float* in, float* out, const float* scale, const float* shift, int act, int C,
                   long long rows_per_batch, long long ld_in, long long bs_in, long long ld_out, long long bs_out,
                   long long batches, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(in && out && C > 0 && rows_per_batch > 0 && batches >= 0 && ((scale == nullptr) == (shift == nullptr)),
                "a2f_affine_act: bad arguments");
    if (batches == 0) return A2F_OK;
    affine_act_kernel<<<ew_blocks(batches * rows_per_batch * C), 256, 0, as_stream(stream)>>>(
        in, out, scale, shift, act, C, rows_per_batch, ld_in, bs_in, ld_out, bs_out, batches);
    A2F_CHECK_LAUNCH("affine_act_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_bn_train_bwd(const float* dy, const float* y_relu, const float* z, const float* mean_rstd, const float* gamma, int C,
                     long long rows_per_batch, long long ld, long long batch_stride, long long batches, float* dz,
                     float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dy && z && mean_rstd && gamma && dz && dgamma && dbeta && workspace && C > 0 && rows_per_batch > 0 &&
                    batches > 0,
                "a2f_bn_train_bwd: bad arguments");
    A2F_REQUIRE(workspace_bytes >= (size_t)2 * C * sizeof(double), "a2f_bn_train_bwd: workspace too small (2*C doubles)");
    return bn_bwd_launch<false>(dy, y_relu, z, mean_rstd, gamma, C, rows_per_batch, ld, batch_stride, batches, dz, dgamma,
                                dbeta, workspace, stream);
}

int a2f_bn_frozen_bwd(const float* dy, const float* y_relu, const float* z, const float* mean_rstd, const float* gamma, int C,
                      long long rows_per_batch, long long ld, long long batch_stride, long long batches, float* dz,
                      float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dy && z && mean_rstd && gamma && dz && dgamma && dbeta && workspace && C > 0 && rows_per_batch > 0 &&
                    batches > 0,
                "a2f_bn_frozen_bwd: bad arguments");
    A2F_REQUIRE(workspace_bytes >= (size_t)2 * C * sizeof(double), "a2f_bn_frozen_bwd: workspace too small (2*C doubles)");
    return bn_bwd_launch<true>(dy, y_relu, z, mean_rstd, gamma, C, rows_per_batch, ld, batch_stride, batches, dz, dgamma,
                               dbeta, workspace, stream);
}

}  // extern "C"
