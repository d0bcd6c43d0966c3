// tcgen05 / TMEM building blocks shared by the tensor-core kernels (sm_100a): shared-memory matrix descriptors,
// kind::tf32 MMA issue and commit, TMEM allocation, loads and stores, and the 3xTF32 split.  The primitives that are not
// specific to tcgen05 (mbarriers, TMA, fences, the exact-erf GELU) are in fz_device.cuh.
//
// Operand forms used by these kernels (all pinned on B200 by bench_probes/tcgen05_*probe.cu; kind::tf32):
//   * A in TENSOR MEMORY (per-voxel GEMMs, M = 128 voxels = TMEM lanes): column c of lane v = A(v, k = c); every thread
//     writes its own voxel's row with tcgen05.st, no shared memory, no swizzle.  The tensor core reads the top 19 bits.
//   * MN-major, SWIZZLE_128B_BASE32B (descriptor layout type 1; the only swizzle 32-bit MN-major operands accept, and
//     K-major operands reject it): element (mn, k) at
//         LBO (mn / 32) + SBO (k / 4) + 128 (k % 4) + 32 (((mn % 32) / 8) ^ (k % 4)) + 4 (mn % 8).
//     For a contraction over voxels (k = voxel) with SBO = 512 this is "voxel rows": the 32 values of a voxel are one
//     128-byte row whose 32-byte chunks are XOR-ed with (voxel % 4) -- a thread stores its voxel's row with STS.128.
//   * K-major without swizzle (layout type 0; the weights): 8 x 16-byte core matrices, LBO along K, SBO along M / N.
#pragma once
#include "fz_device.cuh"

namespace fz {
namespace tc {

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;                       // descriptor version (Blackwell)
    d |= (uint64_t)(layout_type & 7) << 61;
    return d;
}
// the same matrix `bytes` further on in shared memory (the 14-bit start field cannot overflow below 256 KiB)
__device__ __forceinline__ uint64_t desc_at(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }

// instruction descriptor: D = F32, A = B = TF32
__device__ __forceinline__ uint32_t make_idesc(int m, int n, bool a_mn_major, bool b_mn_major) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// kind::f16 with A = B = BF16 and D = F32 (bench_probes/tcgen05_bf16_layout_probe.cu): one MMA per 16 values of K.  16-bit
// operands use the plain SWIZZLE_128B layout (type 2) in both majors -- K-major: 128-byte rows of 64 K values, SBO = 1024
// between groups of 8 rows, a K step of 16 is +32 bytes; MN-major: 128-byte rows of 64 MN values, one row per K, SBO = 1024
// between groups of 8 K, LBO between groups of 64 MN, a K step of 16 is +2048 bytes.  fp16 operands are the same MMA with
// A / B format 0 in bits 7-12 (bf16: 1), pinned by the same probe; the layouts are those of any 2-byte type.
__device__ __forceinline__ uint32_t make_idesc_16bit(int m, int n, bool a_mn_major, bool b_mn_major, uint32_t ab_format) {
    return (1u << 4) | (ab_format << 7) | (ab_format << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ uint32_t make_idesc_bf16(int m, int n, bool a_mn_major, bool b_mn_major) {
    return make_idesc_16bit(m, n, a_mn_major, b_mn_major, 1u);
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// UTCHMMA takes its operands from UNIFORM registers.  Issued under `if (threadIdx.x == 0)` the compiler wraps every MMA in
// an ELECT / R2UR.BROADCAST / BRA.U.ANY loop (~70 cycles per MMA, measured); issued from warp-uniform control flow on
// warp-uniform values (uniform_u32) under elect_one() it is a single predicated instruction.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
// tells the compiler that a value is the same in every lane of the (converged) warp
__device__ __forceinline__ uint32_t uniform_u32(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }

__device__ __forceinline__ void commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
// TMEM allocation by one warp: COLS columns (a power of two, 32 .. 512), their address written to the shared-memory word at
// `slot`; the allocating warp then gives up the permit to allocate more, and frees the same COLS columns at the end
template <uint32_t COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t slot) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(slot), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_alloc_permit() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 / 16 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 3xTF32: the tensor core reads the top 19 bits of an fp32 word, so the word itself is the "hi" operand and
// lo = x - hi (exact, representable in TF32 up to its own rounding) the correction
__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xffffe000u); }
__device__ __forceinline__ float tf32_lo(float v) { return v - tf32_hi(v); }

// K-major, no swizzle: element (n, k) of a matrix with KC columns (SBO = 32 KC, LBO = 128, 256 bytes per K step of 8)
__device__ __forceinline__ uint32_t kmajor_off(int n, int k, int KC) {
    return (uint32_t)((n >> 3) * (KC * 32) + (k >> 2) * 128 + (n & 7) * 16 + (k & 3) * 4);
}

__device__ __forceinline__ void mma_tf32_ta(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// 16 / 32 consecutive TMEM columns of this thread's lane <- registers
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
           "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// One 32-byte chunk (8 consecutive values) of a thread's voxel row, as two STS.128 (forced: left to itself the compiler
// turns the select into predicated scalar stores, which conflict 8-way).  `chunk`: shared-memory address of the chunk;
// lanes whose voxel has bit 2 set (swap) store the upper half first, so that a quarter-warp's STS.128 covers all 32 banks.
__device__ __forceinline__ void st_row_chunk(uint32_t chunk, bool swap, const float (&a)[8]) {
    const uint32_t first = chunk + (swap ? 16u : 0u), second = chunk + (swap ? 0u : 16u);
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};"
                 :: "r"(first), "f"(swap ? a[4] : a[0]), "f"(swap ? a[5] : a[1]), "f"(swap ? a[6] : a[2]), "f"(swap ? a[7] : a[3]) : "memory");
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};"
                 :: "r"(second), "f"(swap ? a[0] : a[4]), "f"(swap ? a[1] : a[5]), "f"(swap ? a[2] : a[6]), "f"(swap ? a[3] : a[7]) : "memory");
}

// Sums of two values over the TWO threads that share a voxel (warps w and w + 4 of a 256-thread CTA: same lane, same TMEM
// lane quarter).  `slots`: 2 x 2 x 128 float2 of shared memory ([call parity][half][voxel]); `turn` counts the calls (two
// buffers: the partner is at most one exchange behind); named barrier 1 + quarter, 64 threads.
__device__ __forceinline__ float2 pair_sum2(float2 mine, float2* slots, uint32_t& turn, int hh, int vq, int v) {
    float2* s = slots + (turn & 1u) * 256;
    s[hh * 128 + v] = mine;
    asm volatile("bar.sync %0, 64;" :: "r"(1 + vq) : "memory");
    const float2 other = s[(hh ^ 1) * 128 + v];
    ++turn;
    return make_float2(mine.x + other.x, mine.y + other.y);
}

}  // namespace tc
}  // namespace fz
