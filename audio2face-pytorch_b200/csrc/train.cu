// Backward-pass kernels of the audio->mesh path that are not GEMMs (those are gemm_tc.cu / gemm_wgrad.cu):
//   a2f_act_fwd / a2f_act_bwd        y = act(z) ; dz = dy * act'(z)                       (HBM-bound elementwise)
//   a2f_colsum                       bias gradients: out[n] += sum_m x[m,n]
//   a2f_layernorm_bwd                LayerNorm backward (+ dgamma, dbeta, optional column sum of dx = bias gradient)
//   a2f_interp_ln_bwd                backward of linear_interpolation + projection LayerNorm (ref:src/model/wav2vec.py:76-84)
//   a2f_conv0_bwd                    backward of normalise+Conv1d(1->512,k10,s5)+GroupNorm+GELU without ever storing the
//                                    512 x L0 pre-activation: the conv is recomputed from the audio (10 FMAs)
//   a2f_weight_norm_bwd              g*v/||v|| backward of the positional conv (HF weight_norm(dim=2))
//   a2f_transpose_cast, a2f_pack_posconv_dgrad_weight, a2f_cast_rows       operand packers of the backward GEMMs
//   a2f_adam_step                    fused Adam with L2 weight decay (ref:src/model/lightning_model.py:209-213)
#include "a2f_common.cuh"
#include "gemm_params.cuh"

namespace a2f {

template <typename T> A2F_D T* ptr_as(void* p) { return static_cast<T*>(p); }

// ------------------------------------------------------------------------------------------------ elementwise
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) act_fwd_kernel(const TI* __restrict__ z, const TO* __restrict__ resid,
                                                      TO* __restrict__ y, long long n, int act, int fast) {
    long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const long long stride = (long long)gridDim.x * blockDim.x * 4;
    for (; i < n; i += stride) {
        if (i + 4 <= n) {
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = ld_as_float(z + i + j);
            if (act == A2F_ACT_GELU && fast) {
                const float2 r0 = gelu_fast2(make_float2(v[0], v[1])), r1 = gelu_fast2(make_float2(v[2], v[3]));
                v[0] = r0.x; v[1] = r0.y; v[2] = r1.x; v[3] = r1.y;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = apply_act_rt(v[j], act);
            }
            if (resid) {
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] += ld_as_float(resid + i + j);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) st_from_float(y + i + j, v[j]);
        } else {
            for (long long k = i; k < n; ++k) {
                float v = ld_as_float(z + k);
                v = (act == A2F_ACT_GELU && fast) ? gelu_fast(v) : apply_act_rt(v, act);
                if (resid) v += ld_as_float(resid + k);
                st_from_float(y + k, v);
            }
        }
    }
}

// bf16 -> bf16, 8 elements (16 bytes) per thread: the training forward's GELU over [2400, 3072] pre-activations was 13 us
// with 2-byte loads
__global__ void __launch_bounds__(256) act_fwd_bf16x8_kernel(const bf16* __restrict__ z, const bf16* __restrict__ resid,
                                                             bf16* __restrict__ y, long long n8, int act) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n8; i += stride) {
        const uint4 u = *reinterpret_cast<const uint4*>(z + i * 8);
        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
        float v[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __bfloat1622float2(h2[e]);
            v[2 * e] = f.x;
            v[2 * e + 1] = f.y;
        }
        if (act == A2F_ACT_GELU) {
#pragma unroll
            for (int e = 0; e < 8; e += 2) {
                const float2 r = gelu_fast2(make_float2(v[e], v[e + 1]));
                v[e] = r.x;
                v[e + 1] = r.y;
            }
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = apply_act_rt(v[e], act);
        }
        if (resid) {
            const uint4 ur = *reinterpret_cast<const uint4*>(resid + i * 8);
            const __nv_bfloat162* r2 = reinterpret_cast<const __nv_bfloat162*>(&ur);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = __bfloat1622float2(r2[e]);
                v[2 * e] += f.x;
                v[2 * e + 1] += f.y;
            }
        }
        uint4 o;
        o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
        o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
        *reinterpret_cast<uint4*>(y + i * 8) = o;
    }
}

template <typename TD, typename TZ, typename TO>
__global__ void __launch_bounds__(256) act_bwd_kernel(const TD* __restrict__ dy, const TZ* __restrict__ z,
                                                      TO* __restrict__ dz, long long n, int act) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) st_from_float(dz + i, ld_as_float(dy + i) * act_grad(ld_as_float(z + i), act));
}

// rows x cols (row stride ld_in) -> out rows x ld_out (columns >= cols zero filled)
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) cast_rows_kernel(const TI* __restrict__ in, long long ld_in, TO* __restrict__ out,
                                                        long long ld_out, long long rows, int cols) {
    const long long n = rows * ld_out;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const long long r = i / ld_out;
        const int c = (int)(i - r * ld_out);
        st_from_float(out + i, c < cols ? ld_as_float(in + r * ld_in + c) : 0.f);
    }
}

// out[c*ldo + r] = in[r*ld_r + c*ld_c]   (32x32 smem tiles, coalesced on the output side)
template <typename TO>
__global__ void __launch_bounds__(256) transpose_cast_kernel(const float* __restrict__ in, long long ld_r, long long ld_c,
                                                             int R, int Cc, TO* __restrict__ out, long long ldo) {
    __shared__ float tile[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    // read: fastest-varying index follows the smaller input stride
    if (ld_c <= ld_r) {
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const int r = r0 + j, c = c0 + tx;
            if (r < R && c < Cc) tile[j][tx] = in[(long long)r * ld_r + (long long)c * ld_c];
        }
    } else {
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const int r = r0 + tx, c = c0 + j;
            if (r < R && c < Cc) tile[tx][j] = in[(long long)r * ld_r + (long long)c * ld_c];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
        const int c = c0 + j, r = r0 + tx;
        if (r < R && c < Cc) st_from_float(out + (long long)c * ldo + r, tile[tx][j]);
    }
}

// Many strided 2-D copies in ONE launch (a2f_strided_copy_jobs): dst[r*ldo_r + c*ldo_c] = src[r*ld_r + c*ld_c] for a
// device-resident table of jobs.  A training step re-derives ~150 operand layouts from the updated fp32 masters
// (bf16 casts, W^T operands of the data-gradient GEMMs, implicit-GEMM conv layouts, fused QKV); as separate launches
// they cost 1.4 ms of a 15.9 ms step, as one launch they cost the HBM traffic.  32x32 smem tiles: the read side
// follows the smaller source stride, the write side the smaller destination stride.
// One CTA walks CJ_TILES consecutive tiles, CJ_BATCH at a time: the job lookup (a binary search over the device-resident
// table) is paid once per CTA, and the loads of CJ_BATCH tiles are in flight together before the first barrier -- with one
// tile per CTA every 1024 elements cost a full load -> barrier -> store round trip (186 k tiles of a FaceFormer re-pack:
// 330 us per launch against ~90 us of HBM traffic).
constexpr int CJ_TILES = 8;
constexpr int CJ_BATCH = 4;
__global__ void __launch_bounds__(256) strided_copy_jobs_kernel(const a2f_copy_job* __restrict__ jobs, int n_jobs,
                                                                int total_tiles) {
    __shared__ float tile[CJ_BATCH][32][33];
    __shared__ int job0;
    const int t_first = (int)blockIdx.x * CJ_TILES;
    if (threadIdx.x == 0) {
        int lo = 0, hi = n_jobs - 1;                   // last job whose first tile is <= t_first
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (jobs[mid].tile0 <= t_first) lo = mid; else hi = mid - 1;
        }
        job0 = lo;
    }
    __syncthreads();
    int ji = job0;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int t_end = min(t_first + CJ_TILES, total_tiles);
    for (int tb = t_first; tb < t_end; tb += CJ_BATCH) {
        int jidx[CJ_BATCH];
#pragma unroll
        for (int i = 0; i < CJ_BATCH; ++i) {
            const int tt = tb + i;
            if (tt < t_end) {
                while (ji + 1 < n_jobs && jobs[ji + 1].tile0 <= tt) ++ji;      // uniform across the CTA
                jidx[i] = ji;
                const a2f_copy_job jb = jobs[ji];
                const int tiles_c = (jb.C + 31) >> 5;
                const int t = tt - jb.tile0;
                const int r0 = (t / tiles_c) * 32, c0 = (t % tiles_c) * 32;
                const float* __restrict__ in = jb.src;
                if (jb.ld_c == 1 && jb.ldo_c == 1 && jb.dst_dtype == A2F_BF16 && (jb.ld_r & 3) == 0 && (jb.ldo_r & 3) == 0 &&
                    ((reinterpret_cast<uintptr_t>(jb.src) & 15) | (reinterpret_cast<uintptr_t>(jb.dst) & 7)) == 0 &&
                    r0 + 32 <= jb.R && c0 + 32 <= jb.C) {
                    // plain fp32 -> bf16 cast of a full tile (half of a re-pack's volume): 16-byte loads, 8-byte stores,
                    // no trip through shared memory
                    const int r = r0 + (threadIdx.x >> 3), c = c0 + (threadIdx.x & 7) * 4;
                    const float4 f = *reinterpret_cast<const float4*>(in + (long long)r * jb.ld_r + c);
                    uint2 o;
                    o.x = pack_bf16x2(f.x, f.y);
                    o.y = pack_bf16x2(f.z, f.w);
                    *reinterpret_cast<uint2*>(static_cast<bf16*>(jb.dst) + (long long)r * jb.ldo_r + c) = o;
                    jidx[i] = -1;                                              // done
                } else if (jb.ld_c <= jb.ld_r) {
#pragma unroll
                    for (int j = ty; j < 32; j += 8) {
                        const int r = r0 + j, c = c0 + tx;
                        if (r < jb.R && c < jb.C) tile[i][j][tx] = in[(long long)r * jb.ld_r + (long long)c * jb.ld_c];
                    }
                } else {
#pragma unroll
                    for (int j = ty; j < 32; j += 8) {
                        const int r = r0 + tx, c = c0 + j;
                        if (r < jb.R && c < jb.C) tile[i][tx][j] = in[(long long)r * jb.ld_r + (long long)c * jb.ld_c];
                    }
                }
            } else {
                jidx[i] = -1;
            }
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < CJ_BATCH; ++i) {
            if (jidx[i] < 0) continue;
            const int tt = tb + i;
            const a2f_copy_job jb = jobs[jidx[i]];
            const int tiles_c = (jb.C + 31) >> 5;
            const int t = tt - jb.tile0;
            const int r0 = (t / tiles_c) * 32, c0 = (t % tiles_c) * 32;
            const bool full = r0 + 32 <= jb.R && c0 + 32 <= jb.C;
            if (jb.ldo_c <= jb.ldo_r) {
                if (full && jb.dst_dtype == A2F_BF16 && jb.ldo_c == 1 && (jb.ldo_r & 1) == 0 &&
                    (reinterpret_cast<uintptr_t>(jb.dst) & 3) == 0) {
                    // bf16 rows: two columns per thread, 4-byte stores (128 B per warp instruction instead of 64)
                    const int cp = (threadIdx.x & 15) * 2;
#pragma unroll
                    for (int j = threadIdx.x >> 4; j < 32; j += 16) {
                        const long long o = (long long)(r0 + j) * jb.ldo_r + c0 + cp;
                        *reinterpret_cast<uint32_t*>(static_cast<bf16*>(jb.dst) + o) = pack_bf16x2(tile[i][j][cp], tile[i][j][cp + 1]);
                    }
                    continue;
                }
#pragma unroll
                for (int j = ty; j < 32; j += 8) {
                    const int r = r0 + j, c = c0 + tx;
                    if (r < jb.R && c < jb.C) {
                        const long long o = (long long)r * jb.ldo_r + (long long)c * jb.ldo_c;
                        if (jb.dst_dtype == A2F_BF16) static_cast<bf16*>(jb.dst)[o] = __float2bfloat16(tile[i][j][tx]);
                        else static_cast<float*>(jb.dst)[o] = tile[i][j][tx];
                    }
                }
            } else {
                if (full && jb.dst_dtype == A2F_BF16 && jb.ldo_r == 1 && (jb.ldo_c & 1) == 0 &&
                    (reinterpret_cast<uintptr_t>(jb.dst) & 3) == 0) {
                    // transposed bf16 output (rows of the destination run along r): two r per thread
                    const int rp = (threadIdx.x & 15) * 2;
#pragma unroll
                    for (int j = threadIdx.x >> 4; j < 32; j += 16) {
                        const long long o = (long long)(c0 + j) * jb.ldo_c + r0 + rp;
                        *reinterpret_cast<uint32_t*>(static_cast<bf16*>(jb.dst) + o) = pack_bf16x2(tile[i][rp][j], tile[i][rp + 1][j]);
                    }
                    continue;
                }
#pragma unroll
                for (int j = ty; j < 32; j += 8) {
                    const int r = r0 + tx, c = c0 + j;
                    if (r < jb.R && c < jb.C) {
                        const long long o = (long long)r * jb.ldo_r + (long long)c * jb.ldo_c;
                        if (jb.dst_dtype == A2F_BF16) static_cast<bf16*>(jb.dst)[o] = __float2bfloat16(tile[i][tx][j]);
                        else static_cast<float*>(jb.dst)[o] = tile[i][tx][j];
                    }
                }
            }
        }
        __syncthreads();                               // the tile buffers are reused by the next batch
    }
}

// out[i0*so0 + i1*so1 + i2*so2] += in[i0*si0 + i1*si1 + i2*si2]   (un-permutes a packed weight gradient into .grad)
__global__ void __launch_bounds__(256) add_strided3_kernel(const float* __restrict__ in, float* __restrict__ out, int n1,
                                                           int n2, long long n, long long si0, long long si1,
                                                           long long si2, long long so0, long long so1, long long so2) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int i2 = (int)(i % n2);
        const long long r = i / n2;
        const int i1 = (int)(r % n1);
        const long long i0 = r / n1;
        out[i0 * so0 + i1 * so1 + i2 * so2] += in[i0 * si0 + i1 * si1 + i2 * si2];
    }
}

// ------------------------------------------------------------------------------------------------ column sums
// out[n] += sum_m x[m*ld + n].  CTA = 64 columns x 256-row slab.
template <typename TI>
__global__ void __launch_bounds__(256) colsum_kernel(const TI* __restrict__ x, long long ld, long long rows, int cols,
                                                     float* __restrict__ out) {
    __shared__ float sh[4][64];
    const int cx = threadIdx.x & 63, ry = threadIdx.x >> 6;
    const int c = blockIdx.x * 64 + cx;
    const long long r0 = (long long)blockIdx.y * 256;
    const long long r1 = r0 + 256 < rows ? r0 + 256 : rows;
    float s = 0.f;
    if (c < cols)
        for (long long r = r0 + ry; r < r1; r += 4) s += ld_as_float(x + r * ld + c);
    sh[ry][cx] = s;
    __syncthreads();
    if (ry == 0 && c < cols) atomicAdd(out + c, (sh[0][cx] + sh[1][cx]) + (sh[2][cx] + sh[3][cx]));
}

// 16-byte loads (8 bf16 / 4 fp32 columns per thread): CTA = 32 column groups x 8 row lanes over a 64-row slab.
struct ColsumOuts {
    float* p[3];
    int seg_cols;        // columns per output segment (cols when there is one output)
};
template <typename TI>
__global__ void __launch_bounds__(256) colsum_vec_kernel(const TI* __restrict__ x, long long ld, long long rows, int cols,
                                                         ColsumOuts outs) {
    constexpr int VEC = 16 / (int)sizeof(TI);
    __shared__ float sh[8][32 * VEC + 1];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = (blockIdx.x * 32 + tx) * VEC;
    const long long r0 = (long long)blockIdx.y * 64;
    const long long r1 = r0 + 64 < rows ? r0 + 64 : rows;
    float acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
    if (c < cols) {
#pragma unroll 4
        for (long long r = r0 + ty; r < r1; r += 8) {
            const uint4 u = *reinterpret_cast<const uint4*>(x + r * ld + c);
            if (sizeof(TI) == 2) {
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 f = __bfloat1622float2(h2[e]);
                    acc[2 * e] += f.x;
                    acc[2 * e + 1] += f.y;
                }
            } else {
                acc[0] += __uint_as_float(u.x); acc[1] += __uint_as_float(u.y);
                acc[2 % VEC] += __uint_as_float(u.z); acc[3 % VEC] += __uint_as_float(u.w);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) sh[ty][tx * VEC + j] = acc[j];
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * VEC; i += 256) {
        const int cc = blockIdx.x * 32 * VEC + i;
        if (cc < cols) {
            float t = 0.f;
#pragma unroll
            for (int k = 0; k < 8; ++k) t += sh[k][i];
            const int sg = cc / outs.seg_cols;
            atomicAdd(outs.p[sg] + (cc - sg * outs.seg_cols), t);
        }
    }
}

// ------------------------------------------------------------------------------------------------ LayerNorm backward
template <typename TI> A2F_D float4 ldv4(const TI* p);
template <> A2F_D float4 ldv4<float>(const float* p) { return *reinterpret_cast<const float4*>(p); }
template <> A2F_D float4 ldv4<bf16>(const bf16* p) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
A2F_D void stv4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
A2F_D void stv4(bf16* p, float4 v) {
    uint2 u;
    u.x = pack_bf16x2(v.x, v.y);
    u.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = u;
}

// One warp per row, rows strided over the grid; per-warp dgamma / dbeta / dbias partials live in registers and are
// combined through shared memory once per CTA, then added atomically (<= 2*148 CTAs).
// PGRAD_ONLY: dgamma / dbeta alone (the input gradient is not wanted: nothing below the LayerNorm trains); the
// per-element data-gradient arithmetic and the dx stores are left out.
template <typename TD, typename TX, typename TO, int NV, bool PGRAD_ONLY = false>
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const TD* __restrict__ dy, const TX* __restrict__ x,
                                                            const float* __restrict__ gamma, float eps,
                                                            TO* __restrict__ dx, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, float* __restrict__ dbias,
                                                            long long rows) {
    constexpr int C = NV * 128;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float4 gm[NV], ag[NV], ab[NV], as[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        gm[j] = *reinterpret_cast<const float4*>(gamma + j * 128 + lane * 4);
        ag[j] = ab[j] = as[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (long long row = (long long)blockIdx.x * 8 + warp; row < rows; row += (long long)gridDim.x * 8) {
        float4 xv[NV], dv[NV];
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            xv[j] = ldv4<TX>(x + row * C + j * 128 + lane * 4);
            dv[j] = ldv4<TD>(dy + row * C + j * 128 + lane * 4);
            s += (xv[j].x + xv[j].y) + (xv[j].z + xv[j].w);
        }
        const float mean = warp_sum(s) * (1.f / C);
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            xv[j].x -= mean; xv[j].y -= mean; xv[j].z -= mean; xv[j].w -= mean;
            q += (xv[j].x * xv[j].x + xv[j].y * xv[j].y) + (xv[j].z * xv[j].z + xv[j].w * xv[j].w);
        }
        const float rstd = rsqrtf(warp_sum(q) * (1.f / C) + eps);
        float s1 = 0.f, s2 = 0.f;      // sum g, sum g*xhat  with g = dy*gamma
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            xv[j].x *= rstd; xv[j].y *= rstd; xv[j].z *= rstd; xv[j].w *= rstd;      // xhat
            ab[j].x += dv[j].x; ab[j].y += dv[j].y; ab[j].z += dv[j].z; ab[j].w += dv[j].w;
            ag[j].x += dv[j].x * xv[j].x; ag[j].y += dv[j].y * xv[j].y; ag[j].z += dv[j].z * xv[j].z; ag[j].w += dv[j].w * xv[j].w;
            if constexpr (!PGRAD_ONLY) {
                dv[j].x *= gm[j].x; dv[j].y *= gm[j].y; dv[j].z *= gm[j].z; dv[j].w *= gm[j].w;      // g
                s1 += (dv[j].x + dv[j].y) + (dv[j].z + dv[j].w);
                s2 += (dv[j].x * xv[j].x + dv[j].y * xv[j].y) + (dv[j].z * xv[j].z + dv[j].w * xv[j].w);
            }
        }
        if constexpr (PGRAD_ONLY) continue;
        s1 = warp_sum(s1) * (1.f / C);
        s2 = warp_sum(s2) * (1.f / C);
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            float4 o;
            o.x = rstd * (dv[j].x - s1 - xv[j].x * s2);
            o.y = rstd * (dv[j].y - s1 - xv[j].y * s2);
            o.z = rstd * (dv[j].z - s1 - xv[j].z * s2);
            o.w = rstd * (dv[j].w - s1 - xv[j].w * s2);
            as[j].x += o.x; as[j].y += o.y; as[j].z += o.z; as[j].w += o.w;
            stv4(dx + row * C + j * 128 + lane * 4, o);
        }
    }
    __shared__ float sh[8][C + 4];
    auto reduce_out = [&](float4* acc, float* dst) {
        if (dst == nullptr) return;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < NV; ++j) *reinterpret_cast<float4*>(&sh[warp][j * 128 + lane * 4]) = acc[j];
        __syncthreads();
        for (int c = threadIdx.x; c < C; c += 256) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) t += sh[w][c];
            atomicAdd(dst + c, t);
        }
    };
    reduce_out(ag, dgamma);
    reduce_out(ab, dbeta);
    if constexpr (!PGRAD_ONLY) reduce_out(as, dbias);
}

// ------------------------------------------------------------------------------------------------ interp + LN backward
// Forward (w2v_frontend.cu interp_ln_kernel): v = l0*x[i0] + l1*x[i1]; y = LN(v)*gamma + beta.  One warp per frame:
// recompute v and its statistics, LayerNorm backward, scatter l0*dv / l1*dv into the fp32 gradient of the conv-stack
// output with atomics (each source row receives <= ~3 frames), accumulate dgamma / dbeta.  PGRAD_ONLY: dgamma / dbeta
// alone (the conv stack below does not train): no data-gradient arithmetic, no scatter, no din buffer.
template <typename TI, typename TD, int C, bool PGRAD_ONLY = false>
__global__ void __launch_bounds__(256) interp_ln_bwd_kernel(const TI* __restrict__ in, const TD* __restrict__ dy,
                                                            const float* __restrict__ gamma, float eps,
                                                            float* __restrict__ din, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, int B, int S, int T) {
    constexpr int PER = C / 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float ag[PER], ab[PER];
#pragma unroll
    for (int j = 0; j < PER; ++j) ag[j] = ab[j] = 0.f;
    const float scale = T > 1 ? (float)(S - 1) / (float)(T - 1) : 0.f;
    for (int f = blockIdx.x * 8 + warp; f < B * T; f += gridDim.x * 8) {
        const int b = f / T, t = f % T;
        const float src = scale * (float)t;
        int i0 = (int)src;
        if (i0 > S - 1) i0 = S - 1;
        const int i1 = i0 + (i0 < S - 1 ? 1 : 0);
        float l1 = src - (float)i0;
        l1 = fminf(fmaxf(l1, 0.f), 1.f);
        const float l0 = 1.f - l1;
        const TI* r0 = in + ((long long)b * S + i0) * C;
        const TI* r1 = in + ((long long)b * S + i1) * C;
        float v[PER], g[PER];
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int cc = j * 32 + lane;
            v[j] = l0 * ld_as_float(r0 + cc) + l1 * ld_as_float(r1 + cc);
            s += v[j];
        }
        const float mean = warp_sum(s) * (1.f / C);
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            v[j] -= mean;
            q = fmaf(v[j], v[j], q);
        }
        const float rstd = rsqrtf(warp_sum(q) * (1.f / C) + eps);
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int cc = j * 32 + lane;
            v[j] *= rstd;
            const float d = ld_as_float(dy + (long long)f * C + cc);
            ab[j] += d;
            ag[j] += d * v[j];
            if constexpr (!PGRAD_ONLY) {
                g[j] = d * gamma[cc];
                s1 += g[j];
                s2 += g[j] * v[j];
            }
        }
        if constexpr (PGRAD_ONLY) continue;
        s1 = warp_sum(s1) * (1.f / C);
        s2 = warp_sum(s2) * (1.f / C);
        float* d0 = din + ((long long)b * S + i0) * C;
        float* d1 = din + ((long long)b * S + i1) * C;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int cc = j * 32 + lane;
            const float dv = rstd * (g[j] - s1 - v[j] * s2);
            atomicAdd(d0 + cc, l0 * dv);
            if (l1 != 0.f) atomicAdd(d1 + cc, l1 * dv);
        }
    }
    __shared__ float sh[8][C];
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PER; ++j) sh[warp][j * 32 + lane] = ag[j];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += sh[w][c];
        atomicAdd(dgamma + c, t);
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PER; ++j) sh[warp][j * 32 + lane] = ab[j];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += sh[w][c];
        atomicAdd(dbeta + c, t);
    }
}

// ------------------------------------------------------------------------------------------------ conv0 backward
// y = conv(xhat, w)  (k10, s5), zhat = (y - mu)*rstd, z = zhat*gamma + beta, a = gelu(z)   per (utterance, channel).
// pass A:  S1 = sum_t dz, S2 = sum_t dz*zhat   with dz = da * gelu'(z)        -> atomics into S[b][c][2]
// pass B:  dy = gamma*rstd*(dz - S1/L - zhat*S2/L);  dw[c][k] += sum_t dy*xhat[5t+k];  (chunk 0: dgamma += S2, dbeta += S1)
constexpr int C0B_TCH = 256;

template <typename TD, int PASS>
__global__ void __launch_bounds__(256) conv0_bwd_kernel(const float* __restrict__ audio, const float* __restrict__ stats,
                                                        const float* __restrict__ w, const float2* __restrict__ gn,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        const TD* __restrict__ da, long long N, int L0,
                                                        float* __restrict__ S, float* __restrict__ dw,
                                                        float* __restrict__ dgamma, float* __restrict__ dbeta) {
    const int b = blockIdx.y, t0 = blockIdx.x * C0B_TCH;
    __shared__ float xs[5 * C0B_TCH + 8];
    const float* x = audio + (long long)b * N;
    const float mean = stats[2 * b], rstd_a = stats[2 * b + 1];
    for (int i = threadIdx.x; i < 5 * C0B_TCH + 8; i += blockDim.x) {
        const long long gi = 5LL * t0 + i;
        xs[i] = (gi < N) ? (x[gi] - mean) * rstd_a : 0.f;
    }
    const int c = threadIdx.x * 2;
    float w0[10], w1[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) {
        w0[k] = w[c * 10 + k];
        w1[k] = w[(c + 1) * 10 + k];
    }
    const float2 g0 = gn[b * 512 + c], g1 = gn[b * 512 + c + 1];
    const float ga0 = gamma[c], ga1 = gamma[c + 1], be0 = beta[c], be1 = beta[c + 1];
    float m1a = 0.f, m2a = 0.f, m1b = 0.f, m2b = 0.f;
    float S1a = 0.f, S2a = 0.f, S1b = 0.f, S2b = 0.f;
    const float invL = 1.f / (float)L0;
    if (PASS == 1) {
        S1a = S[(b * 512 + c) * 2] * invL; S2a = S[(b * 512 + c) * 2 + 1] * invL;
        S1b = S[(b * 512 + c + 1) * 2] * invL; S2b = S[(b * 512 + c + 1) * 2 + 1] * invL;
    }
    float dwa[10], dwb[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) dwa[k] = dwb[k] = 0.f;
    __syncthreads();
    const TD* dab = da + (long long)b * L0 * 512;
    const int tn = min(C0B_TCH, L0 - t0);
    for (int t = 0; t < tn; ++t) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            a0 = fmaf(w0[k], xs[5 * t + k], a0);
            a1 = fmaf(w1[k], xs[5 * t + k], a1);
        }
        const float zh0 = (a0 - g0.x) * g0.y, zh1 = (a1 - g1.x) * g1.y;
        const float z0 = zh0 * ga0 + be0, z1 = zh1 * ga1 + be1;
        const TD* dp = dab + (long long)(t0 + t) * 512 + c;
        // bf16 path: MUFU-based GELU' (same tanh-form Phi as the forward's gelu_fast); fp32 path: exact erf form
        const float dz0 = ld_as_float(dp) * (sizeof(TD) == 2 ? gelu_grad_fast(z0) : act_grad(z0, A2F_ACT_GELU));
        const float dz1 = ld_as_float(dp + 1) * (sizeof(TD) == 2 ? gelu_grad_fast(z1) : act_grad(z1, A2F_ACT_GELU));
        if (PASS == 0) {
            m1a += dz0; m2a = fmaf(dz0, zh0, m2a);
            m1b += dz1; m2b = fmaf(dz1, zh1, m2b);
        } else {
            const float dy0 = ga0 * g0.y * (dz0 - S1a - zh0 * S2a);
            const float dy1 = ga1 * g1.y * (dz1 - S1b - zh1 * S2b);
#pragma unroll
            for (int k = 0; k < 10; ++k) {
                dwa[k] = fmaf(dy0, xs[5 * t + k], dwa[k]);
                dwb[k] = fmaf(dy1, xs[5 * t + k], dwb[k]);
            }
        }
    }
    if (PASS == 0) {
        atomicAdd(S + (b * 512 + c) * 2, m1a);
        atomicAdd(S + (b * 512 + c) * 2 + 1, m2a);
        atomicAdd(S + (b * 512 + c + 1) * 2, m1b);
        atomicAdd(S + (b * 512 + c + 1) * 2 + 1, m2b);
    } else {
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            atomicAdd(dw + c * 10 + k, dwa[k]);
            atomicAdd(dw + (c + 1) * 10 + k, dwb[k]);
        }
        if (blockIdx.x == 0) {
            atomicAdd(dbeta + c, S1a * (float)L0);
            atomicAdd(dgamma + c, S2a * (float)L0);
            atomicAdd(dbeta + c + 1, S1b * (float)L0);
            atomicAdd(dgamma + c + 1, S2b * (float)L0);
        }
    }
}

// ------------------------------------------------------------------------------------------------ weight norm backward
// w[o,c,tap] = v[o,c,tap] * g[tap] / n[tap],  n[tap] = ||v[:,:,tap]||.   dWp is in the packed layout
// [16 groups][48 out][128 taps][48 in] (the layout a2f_gemm_wgrad writes).
//   dot[tap] = sum_{o,c} dW*v ;  dg[tap] += dot/n ;  dv += (g/n) * (dW - v*dot/n^2)
__global__ void __launch_bounds__(256) wn_dot_kernel(const float* __restrict__ dWp, const float* __restrict__ v,
                                                     double* __restrict__ dot, double* __restrict__ nrm2) {
    const int tap = blockIdx.x;
    double s = 0.0, n2 = 0.0;
    for (int i = threadIdx.x; i < 768 * 48; i += blockDim.x) {
        const int o = i / 48, c = i - o * 48;
        const double vv = v[(long long)i * 128 + tap];
        const double dw = dWp[((long long)o * 128 + tap) * 48 + c];
        s += dw * vv;
        n2 += vv * vv;
    }
    __shared__ double sh[2][8];
    s = warp_sum_d(s);
    n2 = warp_sum_d(n2);
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = n2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, bq = 0.0;
        for (int i = 0; i < 8; ++i) { a += sh[0][i]; bq += sh[1][i]; }
        dot[tap] = a;
        nrm2[tap] = bq;
    }
}
__global__ void __launch_bounds__(256) wn_apply_kernel(const float* __restrict__ dWp, const float* __restrict__ v,
                                                       const float* __restrict__ g, const double* __restrict__ dot,
                                                       const double* __restrict__ nrm2, float* __restrict__ dv,
                                                       float* __restrict__ dg) {
    const long long n = (long long)768 * 48 * 128;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (i < 128) dg[i] += (float)(dot[i] / sqrt(nrm2[i]));
    for (; i < n; i += stride) {
        const int tap = (int)(i % 128);
        const long long oc = i / 128;
        const int c = (int)(oc % 48);
        const long long o = oc / 48;
        const double nn = sqrt(nrm2[tap]);
        const double dw = dWp[(o * 128 + tap) * 48 + c];
        dv[i] += (float)(((double)g[tap] / nn) * (dw - (double)v[i] * dot[tap] / nrm2[tap]));
    }
}

// Data-gradient weight of the positional conv: Wd[g][ci(48)][tap'(128)][co (kpad)] = w_eff[g*48+co, ci, 127-tap']
// so that the forward grouped-conv kernel run on the output gradient with a time shift of 63 gives the input gradient.
template <typename TO>
__global__ void posconv_pack_dgrad_kernel(const float* __restrict__ gw, const float* __restrict__ v,
                                          const float* __restrict__ norm, TO* __restrict__ out, int kpad) {
    const int kp = kpad == 8 ? 48 : kpad;      // kpad 8: chunked layout of posconv_tc.cu
    const long long n = (long long)768 * 128 * kp;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int co = (int)(i % kp);
        long long r = i / kp;
        const int tapp = (int)(r % 128);
        r /= 128;                    // g*48 + ci
        const int ci = (int)(r % 48), grp = (int)(r / 48);
        float val = 0.f;
        if (co < 48) {
            const int tap = 127 - tapp;
            val = v[((long long)(grp * 48 + co) * 48 + ci) * 128 + tap] * (gw[tap] / norm[tap]);
        }
        st_from_float(out + (kpad == 8 ? posconv_chunked_index(grp, ci, tapp, co) : i), val);
    }
}

// ------------------------------------------------------------------------------------------------ Adam
// torch.optim.Adam(lr, weight_decay) semantics (L2 added to the gradient), bias-corrected; grad pre-scaled by gscale.
// G = float: the local (or fp32 all-reduced) gradient; G = bf16: the gradient as it came off the wire of the bf16
// all-reduce (trainer.FlatBuffers wire="bf16").  Four parameters per thread and iteration (every flat-buffer entry
// starts on a 256-byte boundary and the buffers are padded to multiples of 64 floats).
template <typename G>
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const G* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, long long n, float lr, float b1, float b2,
                                                   float eps, float wd, float bc1, float bc2_sqrt, float gscale,
                                                   const int* __restrict__ step_dev) {
    if (step_dev != nullptr) {
        // step count kept on the device (a captured CUDA graph replays the same launch for every step): bias corrections
        // 1 - beta^t are evaluated here instead of on the host
        const float t = (float)__ldg(step_dev);
        bc1 = 1.f - powf(b1, t);
        bc2_sqrt = sqrtf(1.f - powf(b2, t));
    }
    const float step = lr / bc1;
    const long long n4 = n >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 pi = reinterpret_cast<const float4*>(p)[i];
        float4 mi = reinterpret_cast<const float4*>(m)[i];
        float4 vi = reinterpret_cast<const float4*>(v)[i];
        float gi[4];
        if (sizeof(G) == 4) {
            const float4 t = reinterpret_cast<const float4*>(g)[i];
            gi[0] = t.x; gi[1] = t.y; gi[2] = t.z; gi[3] = t.w;
        } else {
            const uint2 t = reinterpret_cast<const uint2*>(g)[i];
            const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
            const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
            gi[0] = a.x; gi[1] = a.y; gi[2] = b.x; gi[3] = b.y;
        }
        float* pp = &pi.x; float* mp = &mi.x; float* vp = &vi.x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float gj = fmaf(wd, pp[j], gi[j] * gscale);
            mp[j] = fmaf(b1, mp[j], (1.f - b1) * gj);
            vp[j] = fmaf(b2, vp[j], (1.f - b2) * gj * gj);
            pp[j] = pp[j] - step * (mp[j] / (sqrtf(vp[j]) / bc2_sqrt + eps));
        }
        reinterpret_cast<float4*>(m)[i] = mi;
        reinterpret_cast<float4*>(v)[i] = vi;
        reinterpret_cast<float4*>(p)[i] = pi;
    }
    // tail (n not a multiple of 4): one thread
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (long long i = n4 << 2; i < n; ++i) {
            const float pi = p[i];
            const float gi = fmaf(wd, pi, ld_as_float(g + i) * gscale);
            const float mi = fmaf(b1, m[i], (1.f - b1) * gi);
            const float vi = fmaf(b2, v[i], (1.f - b2) * gi * gi);
            m[i] = mi;
            v[i] = vi;
            p[i] = pi - step * (mi / (sqrtf(vi) / bc2_sqrt + eps));
        }
    }
}

static int ew_grid(long long n, int per_thread = 1) {
    long long blocks = (n / per_thread + 255) / 256;
    const long long cap = 16LL * sm_count();
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}


// ------------------------------------------------------------------------------------------------ SpecAugment
// ref:src/model/wav2vec.py:149-162: hidden_states[mask_time_indices] = masked_spec_embed (training only).
// mask: one byte per row of the [rows, cols] activation, non-zero = replaced.  One warp per row.
template <typename T>
__global__ void __launch_bounds__(256) spec_mask_fwd_kernel(T* __restrict__ h, const unsigned char* __restrict__ mask,
                                                            const float* __restrict__ embed, long long rows, int cols) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows || mask[row] == 0) return;
    T* dst = h + row * cols;
    for (int c = threadIdx.x & 31; c < cols; c += 32) st_from_float(dst + c, embed[c]);
}
// backward: dembed[c] += sum over masked rows of dh[row, c]; the masked rows of dh become zero (the projection below
// them received no signal).  One thread per column walks the rows in order: deterministic, and the walk only touches
// the ~5-10 % masked rows.
template <typename T>
__global__ void __launch_bounds__(128) spec_mask_bwd_kernel(T* __restrict__ dh, const unsigned char* __restrict__ mask,
                                                            float* __restrict__ dembed, long long rows, int cols) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    float acc = 0.f;
    for (long long r = 0; r < rows; ++r) {
        if (mask[r] == 0) continue;
        acc += ld_as_float(dh + r * cols + c);
        st_from_float(dh + r * cols + c, 0.f);
    }
    dembed[c] += acc;
}

}  // namespace a2f

using namespace a2f;

extern "C" {

int a2f_act_fwd(const void* z, int z_dtype, const void* resid, void* y, int y_dtype, long long n, int act, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(z && y && n >= 0, "a2f_act_fwd: bad arguments");
    if (n == 0) return A2F_OK;
    cudaStream_t s = as_stream(stream);
    const int grid = ew_grid(n, 4);
    const bool zi = z_dtype == A2F_BF16, yi = y_dtype == A2F_BF16;
    // bf16 path: same MUFU.TANH GELU as the inference epilogues; fp32 path: exact erf
    if (!zi && !yi) act_fwd_kernel<float, float><<<grid, 256, 0, s>>>((const float*)z, (const float*)resid, (float*)y, n, act, 0);
    else if (zi && yi && n % 8 == 0 &&
             ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(resid)) & 15) == 0)
        act_fwd_bf16x8_kernel<<<ew_grid(n / 8), 256, 0, s>>>((const bf16*)z, (const bf16*)resid, (bf16*)y, n / 8, act);
    else if (zi && yi) act_fwd_kernel<bf16, bf16><<<grid, 256, 0, s>>>((const bf16*)z, (const bf16*)resid, (bf16*)y, n, act, 1);
    else if (!zi && yi) act_fwd_kernel<float, bf16><<<grid, 256, 0, s>>>((const float*)z, (const bf16*)resid, (bf16*)y, n, act, 1);
    else act_fwd_kernel<bf16, float><<<grid, 256, 0, s>>>((const bf16*)z, (const float*)resid, (float*)y, n, act, 0);
    A2F_CHECK_LAUNCH("act_fwd_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_act_bwd(const void* dy, int dy_dtype, const void* z, int z_dtype, void* dz, int dz_dtype, long long n, int act,
                void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dy && z && dz && n >= 0, "a2f_act_bwd: bad arguments");
    if (n == 0) return A2F_OK;
    cudaStream_t s = as_stream(stream);
    const int grid = ew_grid(n);
    const int key = (dy_dtype == A2F_BF16 ? 4 : 0) | (z_dtype == A2F_BF16 ? 2 : 0) | (dz_dtype == A2F_BF16 ? 1 : 0);
    switch (key) {
        case 0: act_bwd_kernel<float, float, float><<<grid, 256, 0, s>>>((const float*)dy, (const float*)z, (float*)dz, n, act); break;
        case 3: act_bwd_kernel<float, bf16, bf16><<<grid, 256, 0, s>>>((const float*)dy, (const bf16*)z, (bf16*)dz, n, act); break;
        case 7: act_bwd_kernel<bf16, bf16, bf16><<<grid, 256, 0, s>>>((const bf16*)dy, (const bf16*)z, (bf16*)dz, n, act); break;
        case 1: act_bwd_kernel<float, float, bf16><<<grid, 256, 0, s>>>((const float*)dy, (const float*)z, (bf16*)dz, n, act); break;
        default: return set_error(A2F_EINVAL, "a2f_act_bwd: unsupported dtype combination");
    }
    A2F_CHECK_LAUNCH("act_bwd_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_cast_rows(const void* in, int in_dtype, long long ld_in, void* out, int out_dtype, long long ld_out, long long rows,
                  int cols, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(in && out && rows >= 0 && cols > 0 && ld_in >= cols && ld_out >= cols, "a2f_cast_rows: bad arguments");
    if (rows == 0) return A2F_OK;
    cudaStream_t s = as_stream(stream);
    const int grid = ew_grid(rows * ld_out);
    const bool ii = in_dtype == A2F_BF16, oi = out_dtype == A2F_BF16;
    if (!ii && oi) cast_rows_kernel<float, bf16><<<grid, 256, 0, s>>>((const float*)in, ld_in, (bf16*)out, ld_out, rows, cols);
    else if (ii && !oi) cast_rows_kernel<bf16, float><<<grid, 256, 0, s>>>((const bf16*)in, ld_in, (float*)out, ld_out, rows, cols);
    else if (!ii && !oi) cast_rows_kernel<float, float><<<grid, 256, 0, s>>>((const float*)in, ld_in, (float*)out, ld_out, rows, cols);
    else cast_rows_kernel<bf16, bf16><<<grid, 256, 0, s>>>((const bf16*)in, ld_in, (bf16*)out, ld_out, rows, cols);
    A2F_CHECK_LAUNCH("cast_rows_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_transpose_cast(const float* in, long long ld_r, long long ld_c, int R, int Cc, void* out, int out_dtype,
                       long long ldo, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(in && out && R > 0 && Cc > 0 && ldo >= R, "a2f_transpose_cast: bad arguments");
    const dim3 grid((Cc + 31) / 32, (R + 31) / 32);
    cudaStream_t s = as_stream(stream);
    if (out_dtype == A2F_BF16) transpose_cast_kernel<bf16><<<grid, 256, 0, s>>>(in, ld_r, ld_c, R, Cc, (bf16*)out, ldo);
    else transpose_cast_kernel<float><<<grid, 256, 0, s>>>(in, ld_r, ld_c, R, Cc, (float*)out, ldo);
    A2F_CHECK_LAUNCH("transpose_cast_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_strided_copy_jobs(const a2f_copy_job* jobs_dev, int n_jobs, int total_tiles, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(jobs_dev && n_jobs > 0 && total_tiles > 0, "a2f_strided_copy_jobs: bad arguments");
    strided_copy_jobs_kernel<<<(total_tiles + CJ_TILES - 1) / CJ_TILES, 256, 0, as_stream(stream)>>>(jobs_dev, n_jobs, total_tiles);
    A2F_CHECK_LAUNCH("strided_copy_jobs_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_add_strided3(const float* in, float* out, int n0, int n1, int n2, long long si0, long long si1, long long si2,
                     long long so0, long long so1, long long so2, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(in && out && n0 > 0 && n1 > 0 && n2 > 0, "a2f_add_strided3: bad arguments");
    const long long n = (long long)n0 * n1 * n2;
    add_strided3_kernel<<<ew_grid(n), 256, 0, as_stream(stream)>>>(in, out, n1, n2, n, si0, si1, si2, so0, so1, so2);
    A2F_CHECK_LAUNCH("add_strided3_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_colsum(const void* x, int dtype, long long ld, long long rows, int cols, float* out, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(x && out && rows >= 0 && cols > 0 && ld >= cols, "a2f_colsum: bad arguments");
    if (rows == 0) return A2F_OK;
    cudaStream_t s = as_stream(stream);
    const int vec = dtype == A2F_BF16 ? 8 : 4;
    if (cols % vec == 0 && ld % vec == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && rows >= 64) {
        const dim3 vgrid((cols / vec + 31) / 32, (unsigned)((rows + 63) / 64));
        ColsumOuts outs;
        outs.p[0] = out; outs.p[1] = outs.p[2] = nullptr; outs.seg_cols = cols;
        if (dtype == A2F_BF16) colsum_vec_kernel<bf16><<<vgrid, 256, 0, s>>>((const bf16*)x, ld, rows, cols, outs);
        else colsum_vec_kernel<float><<<vgrid, 256, 0, s>>>((const float*)x, ld, rows, cols, outs);
        A2F_CHECK_LAUNCH("colsum_vec_kernel");
        count_launch();
        return A2F_OK;
    }
    const dim3 grid((cols + 63) / 64, (unsigned)((rows + 255) / 256));
    if (dtype == A2F_BF16) colsum_kernel<bf16><<<grid, 256, 0, s>>>((const bf16*)x, ld, rows, cols, out);
    else colsum_kernel<float><<<grid, 256, 0, s>>>((const float*)x, ld, rows, cols, out);
    A2F_CHECK_LAUNCH("colsum_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_colsum3(const void* x, int dtype, long long ld, long long rows, int seg_cols, float* out0, float* out1, float* out2,
                void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(x && out0 && out1 && out2 && rows >= 0 && seg_cols > 0 && ld >= 3 * seg_cols, "a2f_colsum3: bad arguments");
    if (rows == 0) return A2F_OK;
    const int vec = dtype == A2F_BF16 ? 8 : 4;
    if (!(seg_cols % vec == 0 && ld % vec == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && rows >= 64)) {
        // small or unaligned: three ordinary launches
        const size_t esz = dtype == A2F_BF16 ? 2 : 4;
        float* outs[3] = {out0, out1, out2};
        for (int i = 0; i < 3; ++i) {
            rc = a2f_colsum(static_cast<const char*>(x) + (size_t)i * seg_cols * esz, dtype, ld, rows, seg_cols, outs[i], stream);
            if (rc != A2F_OK) return rc;
        }
        return A2F_OK;
    }
    const int cols = 3 * seg_cols;
    const dim3 vgrid((cols / vec + 31) / 32, (unsigned)((rows + 63) / 64));
    ColsumOuts outs;
    outs.p[0] = out0; outs.p[1] = out1; outs.p[2] = out2; outs.seg_cols = seg_cols;
    cudaStream_t s = as_stream(stream);
    if (dtype == A2F_BF16) colsum_vec_kernel<bf16><<<vgrid, 256, 0, s>>>((const bf16*)x, ld, rows, cols, outs);
    else colsum_vec_kernel<float><<<vgrid, 256, 0, s>>>((const float*)x, ld, rows, cols, outs);
    A2F_CHECK_LAUNCH("colsum_vec_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* gamma, float eps, void* dx,
                      int dx_dtype, float* dgamma, float* dbeta, float* dbias, long long rows, int C, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dy && x && gamma && rows >= 0, "a2f_layernorm_bwd: bad arguments");
    A2F_REQUIRE(dx || (!dbias && (dgamma || dbeta)), "a2f_layernorm_bwd: without dx, dbias must be NULL and dgamma or dbeta set");
    A2F_REQUIRE(C == 512 || C == 768, "a2f_layernorm_bwd: C must be 512 or 768");
    A2F_REQUIRE(dy_dtype == x_dtype && x_dtype == dx_dtype, "a2f_layernorm_bwd: dy, x and dx must share a dtype");
    if (rows == 0) return A2F_OK;
    long long blocks = (rows + 7) / 8;
    if (blocks > 2LL * sm_count()) blocks = 2LL * sm_count();
    cudaStream_t s = as_stream(stream);
    const int grid = (int)blocks;
#define A2F_LNB(T, NV)                                                                                                  \
    if (dx) layernorm_bwd_kernel<T, T, T, NV><<<grid, 256, 0, s>>>((const T*)dy, (const T*)x, gamma, eps, (T*)dx, dgamma, \
                                                                    dbeta, dbias, rows);                                 \
    else layernorm_bwd_kernel<T, T, T, NV, true><<<grid, 256, 0, s>>>((const T*)dy, (const T*)x, gamma, eps, nullptr,   \
                                                                      dgamma, dbeta, nullptr, rows)
    if (x_dtype == A2F_BF16) {
        if (C == 512) { A2F_LNB(bf16, 4); } else { A2F_LNB(bf16, 6); }
    } else {
        if (C == 512) { A2F_LNB(float, 4); } else { A2F_LNB(float, 6); }
    }
#undef A2F_LNB
    A2F_CHECK_LAUNCH("layernorm_bwd_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_interp_ln_bwd(const void* in, int in_dtype, const void* dy, int dy_dtype, const float* gamma, float eps,
                      float* din, float* dgamma, float* dbeta, int B, int S, int T, int C, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(in && dy && gamma && dgamma && dbeta && B > 0 && S > 0 && T > 0, "a2f_interp_ln_bwd: bad arguments");
    A2F_REQUIRE(C == 512, "a2f_interp_ln_bwd: C must be 512");
    A2F_REQUIRE(in_dtype == dy_dtype, "a2f_interp_ln_bwd: in and dy must share a dtype");
    long long blocks = ((long long)B * T + 7) / 8;
    if (blocks > 2LL * sm_count()) blocks = 2LL * sm_count();
    cudaStream_t s = as_stream(stream);
    if (in_dtype == A2F_BF16) {
        if (din)
            interp_ln_bwd_kernel<bf16, bf16, 512><<<(int)blocks, 256, 0, s>>>((const bf16*)in, (const bf16*)dy, gamma, eps,
                                                                              din, dgamma, dbeta, B, S, T);
        else
            interp_ln_bwd_kernel<bf16, bf16, 512, true><<<(int)blocks, 256, 0, s>>>((const bf16*)in, (const bf16*)dy, gamma,
                                                                                    eps, nullptr, dgamma, dbeta, B, S, T);
    } else {
        if (din)
            interp_ln_bwd_kernel<float, float, 512><<<(int)blocks, 256, 0, s>>>((const float*)in, (const float*)dy, gamma,
                                                                                eps, din, dgamma, dbeta, B, S, T);
        else
            interp_ln_bwd_kernel<float, float, 512, true><<<(int)blocks, 256, 0, s>>>((const float*)in, (const float*)dy,
                                                                                      gamma, eps, nullptr, dgamma, dbeta,
                                                                                      B, S, T);
    }
    A2F_CHECK_LAUNCH("interp_ln_bwd_kernel");
    count_launch();
    return A2F_OK;
}

size_t a2f_conv0_bwd_workspace_bytes(int B) { return B > 0 ? (size_t)B * 512 * 2 * sizeof(float) : 0; }

int a2f_conv0_bwd(const float* audio, const float* stats, const float* w, const float* gamma, const float* beta,
                  const void* gn_stats, const void* da, int da_dtype, int B, long long N, float* dw, float* dgamma,
                  float* dbeta, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(audio && stats && w && gamma && beta && gn_stats && da && dw && dgamma && dbeta && workspace,
                "a2f_conv0_bwd: NULL argument");
    A2F_REQUIRE(B > 0 && N >= 10, "a2f_conv0_bwd: bad sizes");
    A2F_REQUIRE(workspace_bytes >= a2f_conv0_bwd_workspace_bytes(B), "a2f_conv0_bwd: workspace too small");
    const int L0 = (int)((N - 10) / 5 + 1);
    cudaStream_t s = as_stream(stream);
    float* S = static_cast<float*>(workspace);
    A2F_CHECK_CUDA(cudaMemsetAsync(S, 0, a2f_conv0_bwd_workspace_bytes(B), s));
    const dim3 grid((L0 + C0B_TCH - 1) / C0B_TCH, B);
    const float2* gn = static_cast<const float2*>(gn_stats);
    if (da_dtype == A2F_BF16) {
        conv0_bwd_kernel<bf16, 0><<<grid, 256, 0, s>>>(audio, stats, w, gn, gamma, beta, (const bf16*)da, N, L0, S, dw, dgamma, dbeta);
        conv0_bwd_kernel<bf16, 1><<<grid, 256, 0, s>>>(audio, stats, w, gn, gamma, beta, (const bf16*)da, N, L0, S, dw, dgamma, dbeta);
    } else {
        conv0_bwd_kernel<float, 0><<<grid, 256, 0, s>>>(audio, stats, w, gn, gamma, beta, (const float*)da, N, L0, S, dw, dgamma, dbeta);
        conv0_bwd_kernel<float, 1><<<grid, 256, 0, s>>>(audio, stats, w, gn, gamma, beta, (const float*)da, N, L0, S, dw, dgamma, dbeta);
    }
    A2F_CHECK_LAUNCH("conv0_bwd_kernel");
    count_launch(2);
    return A2F_OK;
}

int a2f_weight_norm_bwd(const float* dWp, const float* v, const float* g, float* dv, float* dg, void* workspace,
                        size_t workspace_bytes, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dWp && v && g && dv && dg && workspace, "a2f_weight_norm_bwd: NULL argument");
    A2F_REQUIRE(workspace_bytes >= 256 * sizeof(double) && reinterpret_cast<uintptr_t>(workspace) % 8 == 0,
                "a2f_weight_norm_bwd: workspace must hold 256 doubles");
    double* dot = static_cast<double*>(workspace);
    double* nrm2 = dot + 128;
    cudaStream_t s = as_stream(stream);
    wn_dot_kernel<<<128, 256, 0, s>>>(dWp, v, dot, nrm2);
    A2F_CHECK_LAUNCH("wn_dot_kernel");
    wn_apply_kernel<<<ew_grid(768LL * 48 * 128), 256, 0, s>>>(dWp, v, g, dot, nrm2, dv, dg);
    A2F_CHECK_LAUNCH("wn_apply_kernel");
    count_launch(2);
    return A2F_OK;
}

int a2f_pack_posconv_dgrad_weight(const float* g, const float* v, void* out, int out_dtype, int kpad, float* norm,
                                  void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(g && v && out && norm && (kpad == 48 || kpad == 64 || kpad == 8), "a2f_pack_posconv_dgrad_weight: bad arguments");
    // norm[128] must already hold ||v[:,:,tap]|| (a2f_pack_posconv_weight fills it)
    cudaStream_t s = as_stream(stream);
    const int grid = ew_grid(768LL * 128 * kpad);
    if (out_dtype == A2F_BF16) posconv_pack_dgrad_kernel<bf16><<<grid, 256, 0, s>>>(g, v, norm, (bf16*)out, kpad);
    else posconv_pack_dgrad_kernel<float><<<grid, 256, 0, s>>>(g, v, norm, (float*)out, kpad);
    A2F_CHECK_LAUNCH("posconv_pack_dgrad_kernel");
    count_launch();
    return A2F_OK;
}

static int adam_launch(float* p, const void* g, int g_bf16, float* m, float* v, long long n, float lr, float beta1, float beta2,
                       float eps, float weight_decay, int step, float grad_scale, void* stream, const int* step_dev = nullptr) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(p && g && m && v && n >= 0 && (step >= 1 || step_dev != nullptr), "a2f_adam_step: bad arguments");
    if (step < 1) step = 1;
    if (n == 0) return A2F_OK;
    A2F_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0 &&
                (reinterpret_cast<uintptr_t>(g) & (g_bf16 ? 7 : 15)) == 0, "a2f_adam_step: buffers must be 16-byte aligned");
    const float bc1 = 1.f - powf(beta1, (float)step);
    const float bc2s = sqrtf(1.f - powf(beta2, (float)step));
    if (g_bf16)
        adam_kernel<bf16><<<ew_grid(n, 4), 256, 0, as_stream(stream)>>>(p, static_cast<const bf16*>(g), m, v, n, lr, beta1, beta2, eps,
                                                                       weight_decay, bc1, bc2s, grad_scale, step_dev);
    else
        adam_kernel<float><<<ew_grid(n, 4), 256, 0, as_stream(stream)>>>(p, static_cast<const float*>(g), m, v, n, lr, beta1, beta2,
                                                                        eps, weight_decay, bc1, bc2s, grad_scale, step_dev);
    A2F_CHECK_LAUNCH("adam_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int step, float grad_scale, void* stream) {
    return adam_launch(p, g, 0, m, v, n, lr, beta1, beta2, eps, weight_decay, step, grad_scale, stream);
}

int a2f_adam_step_bf16g(float* p, const void* g_bf16, float* m, float* v, long long n, float lr, float beta1, float beta2,
                        float eps, float weight_decay, int step, float grad_scale, void* stream) {
    return adam_launch(p, g_bf16, 1, m, v, n, lr, beta1, beta2, eps, weight_decay, step, grad_scale, stream);
}

int a2f_adam_step_dev(float* p, const void* g, int g_dtype, float* m, float* v, long long n, float lr, float beta1, float beta2,
                      float eps, float weight_decay, const int* step_dev, float grad_scale, void* stream) {
    A2F_REQUIRE(step_dev != nullptr, "a2f_adam_step_dev: step_dev is NULL");
    A2F_REQUIRE(g_dtype == A2F_F32 || g_dtype == A2F_BF16, "a2f_adam_step_dev: gradient dtype must be fp32 or bf16");
    return adam_launch(p, g, g_dtype == A2F_BF16, m, v, n, lr, beta1, beta2, eps, weight_decay, 0, grad_scale, stream, step_dev);
}

int a2f_spec_mask_fwd(void* h, int dtype, const unsigned char* mask, const float* embed, long long rows, int cols,
                      void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(h && mask && embed && rows >= 0 && cols > 0, "a2f_spec_mask_fwd: bad arguments");
    A2F_REQUIRE(dtype == A2F_F32 || dtype == A2F_BF16, "a2f_spec_mask_fwd: bad dtype");
    if (rows == 0) return A2F_OK;
    const unsigned grid = (unsigned)((rows + 7) / 8);
    if (dtype == A2F_BF16) spec_mask_fwd_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>((bf16*)h, mask, embed, rows, cols);
    else spec_mask_fwd_kernel<float><<<grid, 256, 0, as_stream(stream)>>>((float*)h, mask, embed, rows, cols);
    A2F_CHECK_LAUNCH("spec_mask_fwd_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_spec_mask_bwd(void* dh, int dtype, const unsigned char* mask, float* dembed, long long rows, int cols,
                      void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(dh && mask && dembed && rows >= 0 && cols > 0, "a2f_spec_mask_bwd: bad arguments");
    A2F_REQUIRE(dtype == A2F_F32 || dtype == A2F_BF16, "a2f_spec_mask_bwd: bad dtype");
    if (rows == 0) return A2F_OK;
    const unsigned grid = (unsigned)((cols + 127) / 128);
    if (dtype == A2F_BF16) spec_mask_bwd_kernel<bf16><<<grid, 128, 0, as_stream(stream)>>>((bf16*)dh, mask, dembed, rows, cols);
    else spec_mask_bwd_kernel<float><<<grid, 128, 0, as_stream(stream)>>>((float*)dh, mask, dembed, rows, cols);
    A2F_CHECK_LAUNCH("spec_mask_bwd_kernel");
    count_launch();
    return A2F_OK;
}

}  // extern "C"
