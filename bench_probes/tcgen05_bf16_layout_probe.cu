// Pins the shared-memory layouts of the bf16 and fp16 tensor-core kernels (csrc/fz_bf16_block.cu) before they are built on:
// tcgen05.mma kind::f16 with BF16 or FP16 A and B (instruction-descriptor A / B format 1 or 0), an F32 accumulator, the 128-byte swizzle (descriptor layout type 2) that TMA
// writes for 16-bit boxes whose rows are 128 bytes, and the K steps of 16 values.  Two configurations, each four MMAs
// (K = 64) into one accumulator:
//   fwd:   A MN-major (128 voxels x 64 channels, two 64-voxel atoms LBO = 8192 apart, SBO = 1024, K step +2048 bytes),
//          B K-major (64 outputs x 64 channels, SBO = 1024, K step +32 bytes), N = 64   -- the channel map
//   wgrad: A K-major (128 rows), B K-major (144 rows), N = 144                              -- the weight gradient
// The operands are small integers (every product and sum exact in fp32); the result is compared with the host product
// element by element.  The fp16 operands go up to +-511, which bf16 cannot hold, so a wrong format field shows.  Each
// configuration runs for both types.  Not part of the product.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t lt) {
    return (uint64_t)((saddr >> 4) & 0x3fff) | (uint64_t)((lbo >> 4) & 0x3fff) << 16 | (uint64_t)((sbo >> 4) & 0x3fff) << 32 | (uint64_t)1 << 46 | (uint64_t)(lt & 7) << 61;
}
// byte offset of element (row r, column c) of a region of 128-byte rows (64 bf16) in the 128-byte swizzle
__host__ __device__ inline uint32_t sw128(int r, int c) { return r * 128 + (((c >> 3) ^ (r & 7)) << 4) + (c & 7) * 2; }

constexpr int M = 128, K = 64, NMAX = 144;
constexpr uint32_t kA = 16384, kB = NMAX * 128;

// mode 0: A MN-major (fwd), N = 64; mode 1: A K-major (wgrad), N = 144.  a: [M][K], b: [N][K] as 16-bit patterns of the
// format `fmt` (1 = bf16, 0 = fp16)
__global__ void __launch_bounds__(128) probe(int mode, uint32_t fmt, const uint16_t* __restrict__ a, const uint16_t* __restrict__ b,
                                             float* __restrict__ D) {
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* sa = smem;
    unsigned char* sb = smem + kA;
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int N = mode ? 144 : 64;
    for (int i = tid; i < M * K; i += 128) {
        const int m = i / K, k = i % K;
        const uint32_t off = mode ? sw128(m, k) : (m >> 6) * 8192 + sw128(k, m & 63);
        *reinterpret_cast<uint16_t*>(sa + off) = a[i];
    }
    for (int i = tid; i < N * K; i += 128) *reinterpret_cast<uint16_t*>(sb + sw128(i / K, i % K)) = b[i];
    if (tid == 0) { asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&bar))); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" :: "r"(smem_u32(&tmem_base)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(mode ? 0 : 1) << 15) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
    if (tid == 0) {
        const uint64_t ad = mode ? make_desc(smem_u32(sa), 16, 1024, 2) : make_desc(smem_u32(sa), 8192, 1024, 2);
        const uint64_t bd = make_desc(smem_u32(sb), 16, 1024, 2);
        for (int k = 0; k < K / 16; ++k) {
            const uint64_t a_k = ad + ((mode ? 32u * k : 2048u * k) >> 4), b_k = bd + ((32u * k) >> 4);
            asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                         :: "r"(tmem), "l"(a_k), "l"(b_k), "r"(idesc), "r"((uint32_t)(k > 0)) : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(&bar)) : "memory");
    }
    uint32_t ok = 0;
    while (!ok) asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(smem_u32(&bar)), "r"(0u) : "memory");
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    for (int c0 = 0; c0 < N; c0 += 16) {
        uint32_t r[16];
        const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + c0;
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                       "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                     : "r"(taddr) : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        for (int n = 0; n < 16; ++n) D[tid * NMAX + c0 + n] = __uint_as_float(r[n]);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" :: "r"(tmem) : "memory");
}

static uint16_t bf16_bits(float v) { __nv_bfloat16 h = __float2bfloat16(v); uint16_t u; memcpy(&u, &h, 2); return u; }
static uint16_t f16_bits(float v) { __half h = __float2half(v); uint16_t u; memcpy(&u, &h, 2); return u; }

int main() {
    uint16_t *dA, *dB;
    float* dD;
    CK(cudaMalloc(&dA, M * K * 2));
    CK(cudaMalloc(&dB, NMAX * K * 2));
    CK(cudaMalloc(&dD, M * NMAX * 4));
    const int smem = kA + kB + 1024;
    CK(cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int bad_total = 0;
    for (uint32_t fmt = 1; fmt != ~0u; --fmt) {                      // bf16, then fp16
        const int range = fmt ? 3 : 511;                             // |operand| <= range: 64 products sum exactly in fp32
        std::vector<float> A(M * K), B(NMAX * K);
        std::vector<uint16_t> Ab(M * K), Bb(NMAX * K);
        srand(12345);
        for (int i = 0; i < M * K; ++i) { A[i] = (float)(rand() % (2 * range + 1) - range); Ab[i] = fmt ? bf16_bits(A[i]) : f16_bits(A[i]); }
        for (int i = 0; i < NMAX * K; ++i) { B[i] = (float)(rand() % (2 * range + 1) - range); Bb[i] = fmt ? bf16_bits(B[i]) : f16_bits(B[i]); }
        CK(cudaMemcpy(dA, Ab.data(), Ab.size() * 2, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dB, Bb.data(), Bb.size() * 2, cudaMemcpyHostToDevice));
        for (int mode = 0; mode < 2; ++mode) {
            const int N = mode ? 144 : 64;
            CK(cudaMemset(dD, 0, M * NMAX * 4));
            probe<<<1, 128, smem>>>(mode, fmt, dA, dB, dD);
            CK(cudaDeviceSynchronize());
            std::vector<float> D(M * NMAX);
            CK(cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost));
            int bad = 0;
            for (int m = 0; m < M; ++m)
                for (int n = 0; n < N; ++n) {
                    float ref = 0.f;
                    for (int k = 0; k < K; ++k) ref += A[m * K + k] * B[n * K + k];
                    if (D[m * NMAX + n] != ref) {
                        if (bad < 8) printf("  %s mode %d: D[%d][%d] = %g, expected %g\n", fmt ? "bf16" : "fp16", mode, m, n, D[m * NMAX + n], ref);
                        ++bad;
                    }
                }
            printf("%s %s (A %s, N = %d): %d of %d entries differ -> %s\n", fmt ? "bf16" : "fp16", mode ? "wgrad" : "fwd",
                   mode ? "K-major" : "MN-major", N, bad, M * N, bad ? "FAIL" : "PASS");
            bad_total += bad;
        }
    }
    return bad_total ? 1 : 0;
}
