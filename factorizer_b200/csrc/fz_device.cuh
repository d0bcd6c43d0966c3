// Device primitives shared by the kernel families (sm_100a): packed FP32 pairs, MUFU reciprocals and exponentials,
// mbarriers, proxy fences, TMA and bulk copies, cp.async, a transposing warp reduction and the exact-erf GELU.  One copy of
// each: a fix to a wait loop or a fence lands in every kernel.  All of it is __forceinline__, so where a helper lives does
// not change the machine code of its callers.  What only the tensor-core kernels use (descriptors, MMA issue, TMEM) is in
// fz_tc.cuh.
#pragma once
#include <cuda.h>

#include "fz_common.cuh"

namespace fz {

// ---- packed FP32 pairs (FFMA2 / FMUL2 / FADD2) ---------------------------------------------------------------------
typedef float2 f2;
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ f2 dup(float a) { return make_float2(a, a); }

// ---- MUFU ----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// 1 / d for d >= eps > 0: MUFU.RCP (1 ulp) + one Newton step
__device__ __forceinline__ float rcp_nr(float d) {
    const float r = rcp_approx(d);
    return fmaf(r, fmaf(-d, r, 1.f), r);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarriers: `bar` is the shared-memory address; the uint64_t* forms take the barrier object itself ------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// expect `bytes` more without arriving
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// arrival that fires once every cp.async this thread has issued so far has landed
__device__ __forceinline__ void mbar_arrive_after_cp_async(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) { while (!mbar_try_wait(bar, parity)) {} }

__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) { mbar_init(smem_u32(b), count); }
__device__ __forceinline__ void mbar_arrive(uint64_t* b) { mbar_arrive(smem_u32(b)); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* b, uint32_t bytes) { mbar_arrive_expect_tx(smem_u32(b), bytes); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) { mbar_expect_tx(smem_u32(b), bytes); }
__device__ __forceinline__ void mbar_arrive_after_cp_async(uint64_t* b) { mbar_arrive_after_cp_async(smem_u32(b)); }
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) { mbar_wait(smem_u32(b), parity); }

// ---- fences --------------------------------------------------------------------------------------------------------
// initialised mbarriers -> visible to the async proxy (TMA, tcgen05.commit) before the CTA-wide barrier that follows
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy accesses to shared memory (all memory) ordered with later async-proxy ones (TMA, bulk copies, tcgen05.mma)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ---- TMA tile copies, completion counted in bytes on an mbarrier --------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 :: "r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// 5-D box of an NCDHW volume at (W, H, D, C, B)
__device__ __forceinline__ void tma_load_tile(void* dst, const CUtensorMap* m, uint64_t* bar, int cw, int ch, int cd, int cc, int cb) {
    asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(m), "r"(smem_u32(bar)), "r"(cw), "r"(ch), "r"(cd), "r"(cc), "r"(cb) : "memory");
}
// the same load with an L2 eviction-priority hint (createpolicy value)
__device__ __forceinline__ void tma_load_tile_hint(void* dst, const CUtensorMap* m, uint64_t* bar, int cw, int ch, int cd, int cc,
                                                   int cb, uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6, %7}], [%2], %8;"
                 ::"r"(smem_u32(dst)), "l"(m), "r"(smem_u32(bar)), "r"(cw), "r"(ch), "r"(cd), "r"(cc), "r"(cb), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_store_tile(const CUtensorMap* m, const void* src, int cw, int ch, int cd, int cc, int cb) {
    asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
                 ::"l"(m), "r"(smem_u32(src)), "r"(cw), "r"(ch), "r"(cd), "r"(cc), "r"(cb) : "memory");
}

// ---- contiguous bulk copies (bytes: multiple of 16) -----------------------------------------------------------------
// global -> shared, completion counted on an mbarrier
__device__ __forceinline__ void bulk_copy(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// shared -> global, completion through the bulk async-group
__device__ __forceinline__ void bulk_store_1d(void* dst, const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ---- cp.async ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
// 16 bytes from `src`, or 16 zero bytes (src is not read) when !real
__device__ __forceinline__ void cp_async16_zfill(void* dst, const void* src, bool real) {
    const int n = real ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// until at most N of this thread's committed groups are still in flight
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- warp reductions -----------------------------------------------------------------------------------------------
// Transposing warp reduction: every lane passes N values; returns, in every lane, the warp-wide total of
// element (lane / (32 / N)).  N = 32: 31 shuffles.
template <int N>
__device__ __forceinline__ float warp_vec_sum(float (&v)[N], int lane) {
    static_assert(N == 32 || N == 16 || N == 8 || N == 4, "N");
    int off = 16;
#pragma unroll
    for (int n = N; n > 1; n >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
            const float keep = up ? v[i + n / 2] : v[i];
            const float send = up ? v[i] : v[i + n / 2];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
        off >>= 1;
    }
    float r = v[0];
    for (; off > 0; off >>= 1) r += __shfl_xor_sync(0xffffffffu, r, off);
    return r;
}

// ---- exact (erf) GELU ----------------------------------------------------------------------------------------------
// Abramowitz-Stegun 7.1.26: erf(z) = 1 - (a1 t + ... + a5 t^5) exp(-z^2), t = 1/(1 + p z), |error| <= 1.5e-7 for z >= 0,
// odd extension below.  With z = |h|/sqrt(2) the exponential is exp(-h^2/2), which is also the density the derivative
// needs; two MUFU ops (RCP, EX2) and ~12 FP32 ops instead of erff + expf (~45).
// gauss_cdf2 returns Phi(h) = (1 + erf(h/sqrt 2))/2 and e = exp(-h^2/2), two values at a time: the polynomial in packed
// FFMA2, one MUFU.RCP + one MUFU.EX2 per value.
__device__ __forceinline__ f2 gauss_cdf2(f2 h, f2& e) {
    const f2 z = make_float2(fabsf(h.x) * 0.70710678118654752f, fabsf(h.y) * 0.70710678118654752f);
    const f2 d = fma2(dup(0.3275911f), z, dup(1.f));
    const f2 t = make_float2(rcp_approx(d.x), rcp_approx(d.y));
    const f2 hh = __fmul2_rn(h, h);
    e = make_float2(ex2_approx(hh.x * -0.72134752044448170f), ex2_approx(hh.y * -0.72134752044448170f));   // exp(-h^2/2)
    f2 p = fma2(t, dup(1.061405429f), dup(-1.453152027f));
    p = fma2(t, p, dup(1.421413741f));
    p = fma2(t, p, dup(-0.284496736f));
    p = fma2(t, p, dup(0.254829592f));
    const f2 pt = __fmul2_rn(p, t);
    const f2 erf_abs = fma2(make_float2(-pt.x, -pt.y), e, dup(1.f));
    return fma2(make_float2(copysignf(0.5f, h.x), copysignf(0.5f, h.y)), erf_abs, dup(0.5f));
}
__device__ __forceinline__ f2 gelu2(f2 h) {
    f2 e;
    return __fmul2_rn(h, gauss_cdf2(h, e));
}
// gelu(h) and its derivative Phi(h) + h phi(h)  (torch: GeluBackward, approximate='none')
__device__ __forceinline__ void gelu_grad2(f2 h, f2& g, f2& gp) {
    f2 e;
    const f2 cdf = gauss_cdf2(h, e);
    g = __fmul2_rn(h, cdf);
    gp = fma2(__fmul2_rn(h, dup(0.39894228040143268f)), e, cdf);
}

}  // namespace fz
