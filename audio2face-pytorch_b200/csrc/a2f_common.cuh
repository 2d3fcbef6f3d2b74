// Shared device/host helpers for the sm_100a audio->mesh kernels.
// Everything here is internal to liba2f_sm100.so; the public C-ABI is include/a2f.h.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stddef.h>
#include <math.h>
#include <string.h>
#include "../../include/a2f.h"

#define A2F_HD __host__ __device__ __forceinline__
#define A2F_D __device__ __forceinline__

namespace a2f {

typedef __nv_bfloat16 bf16;

// ---- status plumbing -----------------------------------------------------------------------
int set_cuda_error(cudaError_t e, const char* where);     // records message, returns A2F_ECUDA
int set_error(int code, const char* msg);                  // records message, returns code
#define A2F_CHECK_CUDA(expr)                                                     \
    do {                                                                         \
        cudaError_t _e = (expr);                                                 \
        if (_e != cudaSuccess) return a2f::set_cuda_error(_e, #expr);            \
    } while (0)
#define A2F_CHECK_LAUNCH(name)                                                   \
    do {                                                                         \
        cudaError_t _e = cudaGetLastError();                                     \
        if (_e != cudaSuccess) return a2f::set_cuda_error(_e, name);             \
    } while (0)
#define A2F_REQUIRE(cond, msg)                                                   \
    do {                                                                         \
        if (!(cond)) return a2f::set_error(A2F_EINVAL, msg);                     \
    } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
int sm_count();   // cached multiprocessor count of the current device
void count_launch(int n = 1);   // feeds a2f_launch_count()
int require_sm100();           // A2F_OK or A2F_EARCH (cached per device)

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------
// Every kernel of the inference chain is launched with cudaLaunchAttributeProgrammaticStreamSerialization
// (launch_pdl below) and runs `pdl_sync()` after its private prologue (barrier init, TMEM allocation, descriptor
// prefetch) and BEFORE its first access to global memory.  griddepcontrol.wait blocks until the previous kernel of the
// stream has completed and flushed; griddepcontrol.launch_dependents lets the NEXT kernel's CTAs become resident (and
// run their own prologue up to their wait) as soon as SM resources free up -- so launch latency and prologues overlap
// the tail of the running kernel instead of adding ~2 us per launch to a ~100-launch step.  Without the launch
// attribute both instructions are no-ops, so the same kernels work when launched the ordinary way.
int pdl_enabled();             // 1 unless A2F_PDL=0 in the environment (debug switch)
#ifdef __CUDACC__
A2F_D void pdl_sync() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
#endif

// ---- scalar math -----------------------------------------------------------------------------
A2F_D float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
A2F_D float relu(float x) { return x > 0.f ? x : 0.f; }
// GELU for the bf16 tensor-core path: tanh form 0.5x(1+tanh(sqrt(2/pi)(x+0.044715x^3))) on MUFU.TANH, 6 instructions
// instead of erff's ~30 (the epilogues of the GELU GEMMs and conv0 are instruction-issue bound, profiles/r1_*).
// |tanh-form - erf-form| <= 4.7e-4; measured end-to-end effect on FaceFormer vertices (oracle experiment, DESIGN.md):
// 4.8e-6 m, ~1% of the bf16 tolerance.  The fp32 path always uses the exact erf form (gelu_erf).
A2F_D float gelu_fast(float x) {
    const float u = x * fmaf(0.0356774081f, x * x, 0.7978845608f);
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
    const float hx = 0.5f * x;
    return fmaf(hx, t, hx);
}

// Packed fp32 arithmetic (sm_100: FFMA2 / FMUL2 -- two fp32 lanes per instruction).  The 3-register FFMA issues at
// one warp-instruction per 2 cycles per SM sub-partition (B300_MICROARCH.md "pipe rates"), so instruction-issue-bound
// fp32 loops (conv0, GELU epilogues) run up to twice as fast in the packed form with bit-identical results.
A2F_D float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}
A2F_D float2 fmul2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
A2F_D float2 fadd2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
// gelu_fast on two lanes: same operation order as the scalar form (results are bit-identical)
A2F_D float2 gelu_fast2(float2 x) {
    const float2 u = fmul2(x, ffma2(make_float2(0.0356774081f, 0.0356774081f), fmul2(x, x),
                                    make_float2(0.7978845608f, 0.7978845608f)));
    float2 t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t.x) : "f"(u.x));
    asm("tanh.approx.f32 %0, %1;" : "=f"(t.y) : "f"(u.y));
    const float2 hx = fmul2(x, make_float2(0.5f, 0.5f));
    return ffma2(hx, t, hx);
}

template <int ACT> A2F_D float apply_act(float x) {
    if (ACT == A2F_ACT_RELU) return relu(x);
    if (ACT == A2F_ACT_GELU) return gelu_erf(x);
    if (ACT == A2F_ACT_TANH) return tanhf(x);
    return x;
}
A2F_D float apply_act_rt(float x, int act) {
    switch (act) {
        case A2F_ACT_RELU: return relu(x);
        case A2F_ACT_GELU: return gelu_erf(x);
        case A2F_ACT_TANH: return tanhf(x);
        default: return x;
    }
}

A2F_D float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
A2F_D float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// warp-wide float max in ONE instruction: map floats to order-preserving signed integers, REDUX.MAX.S32, map back
// (five dependent shuffles, ~130 cycles, sat on the critical path of every decoder step).  -inf stays -inf; NaN-free input.
A2F_D float warp_max_redux(float v) {
    int x = __float_as_int(v);
    x ^= (x >> 31) & 0x7fffffff;
    x = __reduce_max_sync(0xffffffffu, x);
    x ^= (x >> 31) & 0x7fffffff;
    return __int_as_float(x);
}
A2F_D double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// typed load/store helpers (fp32 <-> bf16 storage)
A2F_D float ld_as_float(const float* p) { return *p; }
A2F_D float ld_as_float(const bf16* p) { return __bfloat162float(*p); }
A2F_D void st_from_float(float* p, float v) { *p = v; }
A2F_D void st_from_float(bf16* p, float v) { *p = __float2bfloat16_rn(v); }

// ---- dropout RNG (the contract is written down in include/a2f.h, "Encoder dropout") -----------------------------
// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants): counter c[4], key k[2].
A2F_D uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    }
    return c;
}

// keep threshold: an element survives iff its 16-bit uniform is >= round(p * 65536)
A2F_HD uint32_t dropout_threshold(float p) {
    const float t = rintf(p * 65536.f);
    return t <= 0.f ? 0u : (t >= 65536.f ? 65536u : (uint32_t)t);
}

// keep bits of the eight elements e = 8g .. 8g+7 of one site (bit i = element 8g+i); seed / offset as read from
// a2f_dropout_args.seed_offset_dev.  Half-word i of the Philox output word i/2 (low half first) decides element 8g+i.
A2F_D uint32_t dropout_keep8(unsigned long long seed, uint32_t offset, uint32_t site, unsigned long long g,
                             uint32_t threshold) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), site, offset),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const uint32_t u = (w[i >> 1] >> ((i & 1) * 16)) & 0xFFFFu;
        bits |= (u >= threshold ? 1u : 0u) << i;
    }
    return bits;
}

A2F_D uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

// ---- PTX wrappers: shared addresses, mbarrier, TMA, tcgen05 ---------------------------------
A2F_D uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

A2F_D void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
A2F_D void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
A2F_D void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

A2F_D void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
A2F_D void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
A2F_D bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug becomes a trap (launch error) instead of a hung GPU box.
A2F_D void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 26)) __trap();
    }
}

A2F_D void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
A2F_D void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
A2F_D void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "r"(c2)
        : "memory");
}

A2F_D void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
A2F_D void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int NCOLS> A2F_D void tmem_alloc(uint32_t* smem_result) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "n"(NCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS> A2F_D void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate.
A2F_D void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread have completed.
A2F_D void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = TMEM lane = tile row).
A2F_D void tmem_ld_32x32(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
          "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
// registers -> 32 lanes x 32 consecutive fp32 columns (inverse of tmem_ld_32x32)
A2F_D void tmem_st_32x32(uint32_t taddr, const float* v) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
          "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
          "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
A2F_D void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
A2F_D void tmem_ld_32x16(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
A2F_D void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
A2F_D void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
A2F_D void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
A2F_D void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the most recent bulk store have finished READING their shared-memory source (double-buffered staging)
A2F_D void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
A2F_D void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
A2F_D void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

A2F_D void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA-pair (cta_group::2) variants: two SMs of one TPC execute one 256-row UMMA; the leader (even rank) issues --
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;   // clears the pair-rank bit of a shared::cluster address -> the leader CTA
A2F_D uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
A2F_D uint32_t cluster_id_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
A2F_D uint32_t cluster_count_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
    return r;
}
A2F_D void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load issued by either CTA of the pair; the transaction bytes complete on the LEADER's barrier
A2F_D void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1)
        : "memory");
}
A2F_D void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1),
        "r"(c2)
        : "memory");
}
template <int NCOLS> A2F_D void tmem_alloc_2sm(uint32_t* smem_result) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "n"(NCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS> A2F_D void tmem_dealloc_2sm(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
A2F_D void umma_f16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once the issued MMAs retire) on the barrier at this smem offset in BOTH CTAs of the pair
A2F_D void umma_commit_2sm(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}
A2F_D void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_MASK) : "memory");
}

A2F_D bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---- host: TMA descriptor encoding (driver entry point fetched through the runtime, no -lcuda) ----
// dims/strides innermost first; strides_bytes[i] is the byte stride of dim i+1 (dim 0 is contiguous).
int encode_tmap(CUtensorMap* out, const void* base, int elem_bytes /*2=bf16, 4=f32*/, int rank, const uint64_t* dims,
                const uint64_t* strides_bytes, const uint32_t* box, int swizzle128);
inline int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                            const uint64_t* strides_bytes, const uint32_t* box, int swizzle128) {
    return encode_tmap(out, base, 2, rank, dims, strides_bytes, box, swizzle128);
}

}  // namespace a2f
