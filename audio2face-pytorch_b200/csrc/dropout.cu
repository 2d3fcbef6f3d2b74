// Train-mode dropout of the wav2vec2 encoder (HF modeling_wav2vec2.py, p = 0.1 at the hidden / activation sites):
//   a2f_dropout_mask    the keep mask of one site as bytes (tests, debugging)
//   a2f_dropout_apply   y = drop(x) [+ resid]; with the same arguments it is also the backward of the site (dx = drop(dy))
// The mask of an element is a function of (seed, offset, site, linear index) only -- see the RNG contract in
// include/a2f.h -- so every launch that applies a site, here or elsewhere, drops the same elements.
#include "a2f_common.cuh"

namespace a2f {

struct DropoutState {
    unsigned long long seed;
    uint32_t offset, site, threshold;
    float scale;
};

// seed / offset come from device memory (a2f_dropout_args.seed_offset_dev), so that a captured CUDA graph draws new
// masks every replay: the caller advances the offset on the stream between steps
A2F_D DropoutState load_dropout(const unsigned long long* so, uint32_t site, uint32_t threshold, float scale) {
    DropoutState d;
    d.seed = so[0];
    d.offset = (uint32_t)so[1];
    d.site = site;
    d.threshold = threshold;
    d.scale = scale;
    return d;
}

__global__ void __launch_bounds__(256) dropout_mask_kernel(const unsigned long long* __restrict__ so, uint32_t site,
                                                           uint32_t threshold, long long n, unsigned char* __restrict__ mask) {
    const DropoutState d = load_dropout(so, site, threshold, 1.f);
    const long long groups = (n + 7) / 8;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
        const uint32_t bits = dropout_keep8(d.seed, d.offset, d.site, (unsigned long long)g, d.threshold);
        const long long e0 = g * 8;
        if (e0 + 8 <= n) {
            uint2 v;
            v.x = (bits & 1u) | ((bits >> 1) & 1u) << 8 | ((bits >> 2) & 1u) << 16 | ((bits >> 3) & 1u) << 24;
            v.y = ((bits >> 4) & 1u) | ((bits >> 5) & 1u) << 8 | ((bits >> 6) & 1u) << 16 | ((bits >> 7) & 1u) << 24;
            if ((reinterpret_cast<uintptr_t>(mask + e0) & 7) == 0) {
                *reinterpret_cast<uint2*>(mask + e0) = v;
                continue;
            }
        }
        for (int i = 0; i < 8 && e0 + i < n; ++i) mask[e0 + i] = (bits >> i) & 1u;
    }
}

A2F_D void load8(const float* p, float* v) {
    const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
A2F_D void load8(const bf16* p, float* v) {
    const uint4 r = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[i]);
        const float2 f = __bfloat1622float2(h);
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
    }
}
A2F_D void store8(float* p, const float* v) {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
A2F_D void store8(bf16* p, const float* v) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                                              pack_bf16x2(v[6], v[7]));
}

// one Philox call per thread and 8 consecutive elements (n % 8 == 0, 16-byte aligned rows): HBM-bound.  y may alias
// x or resid (in-place use), hence no __restrict__
template <typename T>
__global__ void __launch_bounds__(256) dropout_apply_kernel(const T* x, const T* resid, T* y,
                                                            long long groups, const unsigned long long* __restrict__ so,
                                                            uint32_t site, uint32_t threshold, float scale) {
    const bool on = so != nullptr;
    const DropoutState d = on ? load_dropout(so, site, threshold, scale) : DropoutState{0ull, 0u, 0u, 0u, 1.f};
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
        float v[8], r[8];
        load8(x + g * 8, v);
        const uint32_t bits = on ? dropout_keep8(d.seed, d.offset, d.site, (unsigned long long)g, d.threshold) : 0xFFu;
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = ((bits >> i) & 1u) ? v[i] * d.scale : 0.f;
        if (resid != nullptr) {
            load8(resid + g * 8, r);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += r[i];
        }
        store8(y + g * 8, v);
    }
}

static int dropout_grid(long long work) {
    long long blocks = (work + 255) / 256;
    const long long cap = 16LL * sm_count();
    return (int)(blocks > cap ? cap : (blocks < 1 ? 1 : blocks));
}

// A2F_OK with `active` set when the site drops anything; args == NULL, p == 0 or a NULL pointer mean "off"
static int parse_dropout(const a2f_dropout_args* a, bool* active, uint32_t* threshold, float* scale, const char* what) {
    *active = false;
    *threshold = 0;
    *scale = 1.f;
    if (a == nullptr || a->seed_offset_dev == nullptr || a->p == 0.f) return A2F_OK;
    if (!(a->p > 0.f && a->p < 1.f)) return set_error(A2F_EINVAL, what);
    *active = true;
    *threshold = dropout_threshold(a->p);
    *scale = 1.f / (1.f - a->p);
    return A2F_OK;
}

}  // namespace a2f

using namespace a2f;

extern "C" {

int a2f_dropout_mask(const a2f_dropout_args* args, long long n, unsigned char* mask, void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(mask && n >= 0, "a2f_dropout_mask: bad arguments");
    bool on;
    uint32_t thr;
    float scale;
    rc = parse_dropout(args, &on, &thr, &scale, "a2f_dropout_mask: p must lie in [0, 1)");
    if (rc != A2F_OK) return rc;
    if (n == 0) return A2F_OK;
    cudaStream_t s = as_stream(stream);
    if (!on) {
        A2F_CHECK_CUDA(cudaMemsetAsync(mask, 1, (size_t)n, s));
        return A2F_OK;
    }
    dropout_mask_kernel<<<dropout_grid((n + 7) / 8), 256, 0, s>>>(
        static_cast<const unsigned long long*>(args->seed_offset_dev), args->site, thr, n, mask);
    A2F_CHECK_LAUNCH("dropout_mask_kernel");
    count_launch();
    return A2F_OK;
}

int a2f_dropout_apply(const void* x, const void* resid, void* y, int dtype, long long n, const a2f_dropout_args* args,
                      void* stream) {
    int rc = require_sm100();
    if (rc != A2F_OK) return rc;
    A2F_REQUIRE(x && y && n >= 0, "a2f_dropout_apply: bad arguments");
    A2F_REQUIRE(n % 8 == 0, "a2f_dropout_apply: n must be a multiple of 8");
    A2F_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(resid)) & 15) == 0,
                "a2f_dropout_apply: x, resid and y must be 16-byte aligned");
    A2F_REQUIRE(dtype == A2F_F32 || dtype == A2F_BF16, "a2f_dropout_apply: bad dtype");
    bool on;
    uint32_t thr;
    float scale;
    rc = parse_dropout(args, &on, &thr, &scale, "a2f_dropout_apply: p must lie in [0, 1)");
    if (rc != A2F_OK) return rc;
    if (n == 0) return A2F_OK;
    cudaStream_t s = as_stream(stream);
    const unsigned long long* so = on ? static_cast<const unsigned long long*>(args->seed_offset_dev) : nullptr;
    const uint32_t site = on ? args->site : 0u;
    const long long groups = n / 8;
    if (dtype == A2F_F32)
        dropout_apply_kernel<float><<<dropout_grid(groups), 256, 0, s>>>((const float*)x, (const float*)resid, (float*)y, groups,
                                                                         so, site, thr, scale);
    else
        dropout_apply_kernel<bf16><<<dropout_grid(groups), 256, 0, s>>>((const bf16*)x, (const bf16*)resid, (bf16*)y, groups,
                                                                       so, site, thr, scale);
    A2F_CHECK_LAUNCH("dropout_apply_kernel");
    count_launch();
    return A2F_OK;
}

}  // extern "C"
