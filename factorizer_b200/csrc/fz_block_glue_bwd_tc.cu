// Tensor-core (tcgen05 / TMEM, 3xTF32) backward of the MLP half of a 32-channel FactorizerBlock with hidden width 64:
//     out = x1 + W2 gelu(W1 LN(x1) + b1) + b2      (reference factorizer/factorizer.py:76, layers/mlp.py:54-60,
//                                                   layers/norm.py:29-34)
// given x1 and d(out): d(x1) and the gradients of LN's gamma / beta, W1, b1, W2, b2.
//
// Per tile of 96 voxels (voxel = TMEM lane; lanes 96..127 idle), with xh = the normalised (pre-affine) input and
// W1g = W1 diag(gamma):
//   GEMM1  h      = xh  W1g^T (+ b1 + W1 beta)      N = 64, K = 32      per-voxel GEMMs, M = 128: the A operand is written
//   GEMM2  dg     = dOut W2                         N = 64, K = 32      by its voxel's thread straight into TENSOR MEMORY
//          g = gelu(h),  dh = dg gelu'(h)           (FP32 pipe, thread = voxel x half of the hidden units)
//   GEMM3  d(xh)  = dh W1g                          N = 32, K = 64
//   WG1    [g ; g_lo]   (128 rows) x [dOut | dOut_lo] (64 columns), contraction over the 96 voxels  -> dW2^T
//   WG2    [dh ; dh_lo] (128 rows) x [xh | xh_lo]     (64 columns)                                  -> Q = sum_v dh xh^T
//          dx1    = dOut + rstd (d(xh) - mean(d(xh)) - xh mean(d(xh) xh))
// The contraction operands live in shared memory as "voxel rows" (MN-major SWIZZLE_128B_BASE32B, fz_tc.cuh): a thread
// stores the 32 values of its voxel as one 128-byte row with STS.128.  3xTF32: every operand is staged as the fp32 word
// (hi: the tensor core drops the low 13 bits) and its remainder (lo); a per-voxel GEMM issues a_lo b_hi + a_hi b_lo +
// a_hi b_hi, a contraction computes all four hi / lo blocks in ONE MMA and the flush adds them.  WG1 / WG2 accumulate in
// TMEM over ALL tiles of the CTA.  No per-voxel reductions for the small gradients:
//   db1 = sum_v dh and db2 = sum_v dOut accumulate in registers (thread-private, reduced once per CTA),
//   dW1 = Q diag(gamma) + db1 beta^T,  d(gamma)_c = sum_j W1[j][c] Q[j][c],  d(beta)_c = sum_j W1[j][c] db1[j].
// One CTA per SM, 16 warps: the twelve warps with w % 4 != 3 are the workers (warp w: voxels 32 (w % 4) .. + 31 = the TMEM
// lanes it may touch; quarter w / 4 of the hidden units and of the channels), warp 3 issues the MMAs (7, 11 and 15 idle); mbarriers hand the phases over, and every wait of a worker has independent work scheduled before it
// (dOut staging behind GEMM1, gelu behind GEMM2, the next tile's LayerNorm behind GEMM3, P3 behind WG1 / WG2).  Layouts and the TMEM A operand were pinned by bench_probes/tcgen05_layout_probe.cu and tcgen05_tmem_a_probe.cu.
#include "fz_tc.cuh"

namespace fz {
namespace {

using namespace tc;

constexpr int kC = 32;
constexpr int kH = 64;
constexpr int kTV = 96;                   // voxels per tile
constexpr int kWorkers = 384;
constexpr int kThreads = 512;
constexpr int kMmaWarp = 3;

// shared memory map (bytes).  A voxel-row atom = 96 rows x 128 bytes.
constexpr uint32_t kAtom = kTV * 128;     // 12 KiB
constexpr uint32_t oXH = 0;               // xh   atoms [hi | lo]
constexpr uint32_t oDO = 2 * kAtom;       // dOut atoms [hi | lo]
constexpr uint32_t oG = 4 * kAtom;        // g    atoms [hi 0..31 | hi 32..63 | lo 0..31 | lo 32..63]
constexpr uint32_t oDH = 8 * kAtom;       // dh   same
constexpr uint32_t oW1 = 12 * kAtom;      // W1g  as B(n = j, k = c), K-major: hi 8 KiB | lo 8 KiB       (GEMM1)
constexpr uint32_t oW2 = oW1 + 16384;     // W2   as B(n = j, k = o)                                     (GEMM2)
constexpr uint32_t oW3 = oW2 + 16384;     // W1g  as B(n = c, k = j)                                     (GEMM3)
constexpr uint32_t oPar = oW3 + 16384;    // b1f[64] | db1 of the CTA [64] | db2 [32]
constexpr uint32_t oEx = oPar + 160 * 4;  // exchange slots of the LayerNorm partial sums: 4 x [3 lane quarters][4][32]
constexpr uint32_t oBar = oEx + 4 * 384 * 4;   // 8 mbarriers
constexpr uint32_t oTmem = oBar + 8 * 8;
constexpr uint32_t kSmem = oTmem + 8;

// TMEM columns: A operands (xh hi / lo, dOut hi / lo; later dh hi / lo) | h | dg | d(xh) | WG1 | WG2
constexpr uint32_t cA = 0, cH = 128, cDG = 192, cDX = 256, cWG1 = 288, cWG2 = 352, kTmemCols = 512;

#ifdef FZ_TUNING
// experiment builds only: clock stamps of CTA 0 (worker warp 0 and the MMA thread), 16 slots per tile, first 16 tiles
__device__ long long* g_mlp_bwd_trace = nullptr;
#define FZ_TR(slot) do { if (trace_buf && lane == 0 && it < 16) trace_buf[it * 16 + (slot)] = clock64(); } while (0)
#else
#define FZ_TR(slot) do { } while (0)
#endif

__global__ void __launch_bounds__(kThreads, 1)
mlp_bwd_tc(const float* __restrict__ x1, const float* __restrict__ dout, const float* __restrict__ gamma,
           const float* __restrict__ beta, const float* __restrict__ W1, const float* __restrict__ b1,
           const float* __restrict__ W2, float* __restrict__ dx1, float* __restrict__ dgamma, float* __restrict__ dbeta,
           float* __restrict__ dW1, float* __restrict__ db1, float* __restrict__ dW2, float* __restrict__ db2, int ldw2,
           int accumulate, long long vox, int tiles_per_sample, long long total_tiles, float eps) {
    // One launch covers 64 hidden units; wider MLPs run slice by slice (the backward is additive over hidden units): W1 / b1 /
    // dW1 / db1 point at the slice's first row, W2 / dW2 at its first column (rows ldw2 apart), and with `accumulate` dx1
    // already holds dOut + the other slices' contributions.
    extern __shared__ __align__(1024) unsigned char smem[];
    float* par = reinterpret_cast<float*>(smem + oPar);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar_p1a = sbase + oBar, bar_p1b = bar_p1a + 8, bar_g1 = bar_p1a + 16, bar_g2 = bar_p1a + 24, bar_p2 = bar_p1a + 32,
                   bar_g3 = bar_p1a + 40, bar_wg = bar_p1a + 48;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#ifdef FZ_TUNING
    long long* const trace_buf = blockIdx.x == 0 ? g_mlp_bwd_trace : nullptr;     // read once: a stamp must not cost a global load
#endif

    // ---- once per CTA: weights (3xTF32 halves), folded bias, barriers, TMEM ----
    for (int e = tid; e < kH * kC; e += kThreads) {
        {
            const int j = e >> 5, c = e & 31;                 // W1 (64, 32)
            const float w = W1[e] * (gamma ? gamma[c] : 1.f);
            const uint32_t o1 = oW1 + kmajor_off(j, c, kC), o3 = oW3 + kmajor_off(c, j, kH);
            *reinterpret_cast<float*>(smem + o1) = w;
            *reinterpret_cast<float*>(smem + o1 + 8192) = tf32_lo(w);
            *reinterpret_cast<float*>(smem + o3) = w;
            *reinterpret_cast<float*>(smem + o3 + 8192) = tf32_lo(w);
        }
        {
            const int o_ = e >> 6, j = e & 63;                // W2 (32, 64): B(n = j, k = o)
            const float w = W2[o_ * ldw2 + j];
            const uint32_t o = oW2 + kmajor_off(j, o_, kC);
            *reinterpret_cast<float*>(smem + o) = w;
            *reinterpret_cast<float*>(smem + o + 8192) = tf32_lo(w);
        }
    }
    for (int j = tid; j < kH; j += kThreads) {
        float s = b1 ? b1[j] : 0.f;
        if (beta)
            for (int c = 0; c < kC; ++c) s = fmaf(W1[j * kC + c], beta[c], s);
        par[j] = s;
    }
    if (tid == 0) {
        mbar_init(bar_p1a, kWorkers); mbar_init(bar_p1b, kWorkers); mbar_init(bar_g1, 1); mbar_init(bar_g2, 1); mbar_init(bar_p2, kWorkers);
        mbar_init(bar_g3, 1); mbar_init(bar_wg, 1);
        fence_mbarrier_init();
    }
    if (warp == kMmaWarp) {
        tmem_alloc<kTmemCols>(sbase + oTmem);
        tmem_relinquish_alloc_permit();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<const uint32_t*>(smem + oTmem);
    const long long my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    const int warp_u = (int)uniform_u32((uint32_t)warp);
    if ((warp_u & 3) == 3) {
        // =============================== MMA issue: the four warps that own no voxels ===============================
        // Warp 3 issues every MMA, in the order the workers need the results: GEMM1 | GEMM2 | GEMM3, then the two
        // contractions (the tensor pipe runs in issue order).  Warp-uniform code, the MMAs themselves under elect_one()
        // (see fz_tc.cuh); warps 7, 11 and 15 idle.
        if (my_tiles > 0 && warp_u == kMmaWarp) {
            const uint32_t tm = uniform_u32(tmem);
            const uint32_t id_g12 = make_idesc(128, kH, false, false);
            const uint32_t id_g3 = make_idesc(128, kC, false, false);
            const uint32_t id_wg = make_idesc(128, 64, true, true);
            const uint64_t b_w1 = make_desc(sbase + oW1, 128, 1024, 0);
            const uint64_t b_w2 = make_desc(sbase + oW2, 128, 1024, 0);
            const uint64_t b_w3 = make_desc(sbase + oW3, 128, 2048, 0);
            const uint64_t k_g = make_desc(sbase + oG, kAtom, 512, 1);            // voxel rows: 4 atoms of 32 rows (M = 128)
            const uint64_t k_dh = make_desc(sbase + oDH, kAtom, 512, 1);
            const uint64_t k_do = make_desc(sbase + oDO, kAtom, 512, 1);          //             2 atoms of 32 columns (N = 64)
            const uint64_t k_xh = make_desc(sbase + oXH, kAtom, 512, 1);
            for (long long it = 0; it < my_tiles; ++it) {
                const uint32_t ph = (uint32_t)(it & 1);
                mbar_wait(bar_p1a, ph);
                tc_fence_after();
                FZ_TR(8);
                if (elect_one()) {
#pragma unroll
                    for (int s = 0; s < kC / 8; ++s) {    // GEMM1: h = xh W1g^T   (A: hi columns cA .. + 31, lo + 32 ..)
                        mma_tf32_ta(tm + cH, tm + cA + 32 + s * 8, desc_at(b_w1, s * 256), id_g12, s > 0);
                        mma_tf32_ta(tm + cH, tm + cA + s * 8, desc_at(b_w1, 8192 + s * 256), id_g12, 1);
                        mma_tf32_ta(tm + cH, tm + cA + s * 8, desc_at(b_w1, s * 256), id_g12, 1);
                    }
                    commit(bar_g1);
                }
                __syncwarp();
                FZ_TR(9);
                mbar_wait(bar_p1b, ph);
                tc_fence_after();
                FZ_TR(14);
                if (elect_one()) {
#pragma unroll
                    for (int s = 0; s < kC / 8; ++s) {    // GEMM2: dg = dOut W2   (A: hi columns cA + 64 .., lo + 96 ..)
                        mma_tf32_ta(tm + cDG, tm + cA + 96 + s * 8, desc_at(b_w2, s * 256), id_g12, s > 0);
                        mma_tf32_ta(tm + cDG, tm + cA + 64 + s * 8, desc_at(b_w2, 8192 + s * 256), id_g12, 1);
                        mma_tf32_ta(tm + cDG, tm + cA + 64 + s * 8, desc_at(b_w2, s * 256), id_g12, 1);
                    }
                    commit(bar_g2);
                }
                __syncwarp();
                FZ_TR(15);
                mbar_wait(bar_p2, ph);
                tc_fence_after();
                FZ_TR(10);
                if (elect_one()) {
#pragma unroll
                    for (int s = 0; s < kH / 8; ++s) {    // GEMM3: d(xh) = dh W1g (A: hi columns cA .. + 63, lo + 64 ..)
                        mma_tf32_ta(tm + cDX, tm + cA + 64 + s * 8, desc_at(b_w3, s * 256), id_g3, s > 0);
                        mma_tf32_ta(tm + cDX, tm + cA + s * 8, desc_at(b_w3, 8192 + s * 256), id_g3, 1);
                        mma_tf32_ta(tm + cDX, tm + cA + s * 8, desc_at(b_w3, s * 256), id_g3, 1);
                    }
                    commit(bar_g3);
                    // WG1 = [g ; g_lo] x [dOut | dOut_lo], WG2 = [dh ; dh_lo] x [xh | xh_lo] over the tile's 12 groups of 8 voxels
                    mma_tf32(tm + cWG1, k_g, k_do, id_wg, it > 0);
                    mma_tf32(tm + cWG2, k_dh, k_xh, id_wg, it > 0);
#pragma unroll
                    for (int s = 1; s < kTV / 8; ++s) {
                        mma_tf32(tm + cWG1, desc_at(k_g, s * 1024), desc_at(k_do, s * 1024), id_wg, 1);
                        mma_tf32(tm + cWG2, desc_at(k_dh, s * 1024), desc_at(k_xh, s * 1024), id_wg, 1);
                    }
                    commit(bar_wg);
                }
                __syncwarp();
                FZ_TR(11);
            }
        }
    } else {
        // =============================== workers: thread = (voxel, quarter) ===============================
        const int vq = warp & 3, qq = warp >> 2;                         // TMEM lane quarter; quarter of the channels / hidden units
        const int v = vq * 32 + lane;                                    // voxel of the tile = TMEM lane
        const uint32_t lane_addr = tmem + ((uint32_t)(vq * 32) << 16);
        const bool swap = (v & 4) != 0;
        // voxel row addressing: chunk q of this voxel's row sits at row + 32 (q ^ (v % 4)); the thread owns chunk qq of the
        // 32-channel rows (xh, dOut) and chunks 2 (qq % 2), + 1 of the 32-hidden-unit rows of atom qq / 2 (g, dh)
        const uint32_t row = (uint32_t)v * 128;
        const uint32_t cx = row + (uint32_t)((qq ^ (v & 3)) << 5);
        const uint32_t cg0 = row + (uint32_t)(((2 * (qq & 1)) ^ (v & 3)) << 5) + (uint32_t)(qq >> 1) * kAtom;
        const uint32_t cg1 = row + (uint32_t)(((2 * (qq & 1) + 1) ^ (v & 3)) << 5) + (uint32_t)(qq >> 1) * kAtom;
        float* const ex = reinterpret_cast<float*>(smem + oEx) + vq * 128 + lane;     // [vq][quarter][lane] exchange slots
        const uint32_t pair_bar = 1 + vq;
        const float* const b1f = par + qq * 16;
        float acc_db1[16], acc_db2[8];
#pragma unroll
        for (int i = 0; i < 16; ++i) acc_db1[i] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc_db2[i] = 0.f;

        float xr[8], dr[8];                                              // the next tile's x1 and dOut, this thread's 8 channels
        float rstd_next = 0.f;
        bool valid = false;
        long long base = 0;
        // (sample, tile of the sample) of the next fetch, advanced by the grid size without a 64-bit division per tile
        long long nb = (long long)blockIdx.x / tiles_per_sample;
        int nt = (int)((long long)blockIdx.x - nb * tiles_per_sample);
        auto fetch = [&]() {
            const long long v0 = (long long)nt * kTV + v;
            valid = v0 < vox;
            base = (nb * kC + qq * 8) * vox + v0;
            nt += (int)gridDim.x;
            while (nt >= tiles_per_sample) { nt -= tiles_per_sample; ++nb; }
            const float* px = x1 + base;
            const float* pd = dout + base;
#pragma unroll
            for (int c = 0; c < 8; ++c) { xr[c] = valid ? __ldg(px) : 0.f; px += vox; }
#pragma unroll
            for (int c = 0; c < 8; ++c) { dr[c] = valid ? __ldg(pd) : 0.f; pd += vox; }
        };
        // LayerNorm of the fetched x1 (partial sums meet in shared memory): xr <- xh
        auto normalise = [&]() {
            float s = 0.f;
#pragma unroll
            for (int c = 0; c < 8; ++c) s += xr[c];
            ex[qq * 32] = s;
            asm volatile("bar.sync %0, 128;" :: "r"(pair_bar) : "memory");
            const float mean = ((ex[0] + ex[32]) + (ex[64] + ex[96])) * (1.f / kC);
            float ss = 0.f;
#pragma unroll
            for (int c = 0; c < 8; ++c) { xr[c] -= mean; ss = fmaf(xr[c], xr[c], ss); }
            ex[384 + qq * 32] = ss;
            asm volatile("bar.sync %0, 128;" :: "r"(pair_bar) : "memory");
            const float var = ((ex[384] + ex[416]) + (ex[448] + ex[480])) * (1.f / kC);
            rstd_next = rsqrtf(var + eps);
#pragma unroll
            for (int c = 0; c < 8; ++c) xr[c] *= rstd_next;
        };
        if (my_tiles > 0) { fetch(); normalise(); }
        for (long long it = 0; it < my_tiles; ++it) {
            const uint32_t ph = (uint32_t)(it & 1), pph = ph ^ 1u;
            const bool cur_valid = valid;
            const long long cur_base = base;
            const float rstd = rstd_next;
            if (warp == 0) FZ_TR(0);
            // ---- P1: xh and dOut -> TMEM (A of GEMM1 / GEMM2) and voxel rows (B of WG2 / WG1) ----
            float xh[8], go[8];
            {
                float l8[8];
                uint32_t th[8], tl[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    xh[i] = xr[i]; go[i] = dr[i];
                    l8[i] = tf32_lo(xh[i]); th[i] = __float_as_uint(xh[i]); tl[i] = __float_as_uint(l8[i]);
                }
                if (it > 0) mbar_wait(bar_wg, pph);                       // the previous tile's contractions have read their operands
                tc_fence_after();
                if (warp == 0) FZ_TR(1);
                st_row_chunk(sbase + oXH + cx, swap, xh);
                st_row_chunk(sbase + oXH + kAtom + cx, swap, l8);
                tmem_st8(lane_addr + cA + qq * 8, th);
                tmem_st8(lane_addr + cA + 32 + qq * 8, tl);
                tmem_st_wait();
                tc_fence_before();
                fence_proxy_async_smem();
                mbar_arrive(bar_p1a);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    l8[i] = tf32_lo(go[i]); th[i] = __float_as_uint(go[i]); tl[i] = __float_as_uint(l8[i]);
                    acc_db2[i] += go[i];
                }
                if (warp == 0) FZ_TR(2);
                st_row_chunk(sbase + oDO + cx, swap, go);
                st_row_chunk(sbase + oDO + kAtom + cx, swap, l8);
                tmem_st8(lane_addr + cA + 64 + qq * 8, th);
                tmem_st8(lane_addr + cA + 96 + qq * 8, tl);
                tmem_st_wait();
                tc_fence_before();
                fence_proxy_async_smem();
                mbar_arrive(bar_p1b);
            }
            if (warp == 0) FZ_TR(3);
            // next tile's loads: in flight during this tile's GELU phase
            if (it + 1 < my_tiles) fetch();
            if (warp == 0) FZ_TR(13);
            // ---- P2: g = gelu(h) as soon as GEMM1 is done, then dh = dg gelu'(h) for this thread's 16 hidden units ----
            {
                uint32_t hr[16], dh_hi[16], dh_lo[16];
                float gp[16];
                mbar_wait(bar_g1, ph);
                tc_fence_after();
                if (warp == 0) FZ_TR(4);
                tmem_ld16_nowait(lane_addr + cH + qq * 16, hr);
                tmem_ld_wait();
#pragma unroll
                for (int o = 0; o < 2; ++o) {                            // one 32-byte chunk (8 hidden units) at a time
                    float g8[8], gl8[8];
#pragma unroll
                    for (int p = 0; p < 8; p += 2) {
                        const int i = o * 8 + p;
                        const float2 bj = *reinterpret_cast<const float2*>(b1f + i);
                        float2 g, gpp;
                        gelu_grad2(make_float2(__uint_as_float(hr[i]) + bj.x, __uint_as_float(hr[i + 1]) + bj.y), g, gpp);
                        gp[i] = gpp.x; gp[i + 1] = gpp.y;
                        g8[p] = g.x; g8[p + 1] = g.y; gl8[p] = tf32_lo(g.x); gl8[p + 1] = tf32_lo(g.y);
                    }
                    const uint32_t cg = o ? cg1 : cg0;
                    st_row_chunk(sbase + oG + cg, swap, g8);
                    st_row_chunk(sbase + oG + 2 * kAtom + cg, swap, gl8);
                }
                mbar_wait(bar_g2, ph);
                tc_fence_after();
                tmem_ld16_nowait(lane_addr + cDG + qq * 16, hr);
                tmem_ld_wait();
#pragma unroll
                for (int o = 0; o < 2; ++o) {
                    float d8[8], dl8[8];
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        const int i = o * 8 + p;
                        const float dh = __uint_as_float(hr[i]) * gp[i];
                        acc_db1[i] += dh;
                        d8[p] = dh; dl8[p] = tf32_lo(dh);
                        dh_hi[i] = __float_as_uint(dh); dh_lo[i] = __float_as_uint(dl8[p]);
                    }
                    const uint32_t cg = o ? cg1 : cg0;
                    st_row_chunk(sbase + oDH + cg, swap, d8);
                    st_row_chunk(sbase + oDH + 2 * kAtom + cg, swap, dl8);
                }
                tmem_st16(lane_addr + cA + qq * 16, dh_hi);
                tmem_st16(lane_addr + cA + 64 + qq * 16, dh_lo);
                tmem_st_wait();
            }
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(bar_p2);
            if (warp == 0) FZ_TR(5);
            // the next tile's LayerNorm while GEMM3 runs
            if (it + 1 < my_tiles) normalise();
            mbar_wait(bar_g3, ph);
            tc_fence_after();
            if (warp == 0) FZ_TR(6);
            // ---- P3: through LayerNorm, plus the residual branch ----
            {
                uint32_t dxa[8];
                tmem_ld8(lane_addr + cDX + qq * 8, dxa);
                float dx[8];
                float m1 = 0.f, m2 = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    dx[i] = __uint_as_float(dxa[i]);
                    m1 += dx[i];
                    m2 = fmaf(dx[i], xh[i], m2);
                }
                ex[768 + qq * 32] = m1;
                ex[1152 + qq * 32] = m2;
                asm volatile("bar.sync %0, 128;" :: "r"(pair_bar) : "memory");
                m1 = ((ex[768] + ex[800]) + (ex[832] + ex[864])) * (1.f / kC);
                m2 = ((ex[1152] + ex[1184]) + (ex[1216] + ex[1248])) * (1.f / kC);
                if (cur_valid) {
                    float* po = dx1 + cur_base;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        *po = (accumulate ? *po : go[i]) + rstd * (dx[i] - m1 - xh[i] * m2);
                        po += vox;
                    }
                }
            }
            tc_fence_before();
            if (warp == 0) FZ_TR(7);
        }
        if (my_tiles > 0) mbar_wait(bar_wg, (uint32_t)((my_tiles - 1) & 1));
        tc_fence_after();
        // ---- per-CTA totals of the register accumulators ----
        {
            const float t1 = warp_vec_sum<16>(acc_db1, lane);            // hidden unit 16 qq + lane / 2
            const float t2 = warp_vec_sum<8>(acc_db2, lane);             // channel 8 qq + lane / 4
            float* scr = reinterpret_cast<float*>(smem + oW1);           // [warp][24]; every MMA has completed: the weights are dead
            if ((lane & 1) == 0) scr[warp * 24 + (lane >> 1)] = t1;
            if ((lane & 3) == 0) scr[warp * 24 + 16 + (lane >> 2)] = t2;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (my_tiles > 0) {
        // ---- flush.  Accumulator row r (TMEM lane r): hidden unit r % 64, hi block for r < 64, lo block above;
        //      column n: channel n % 32 against the hi (n < 32) or lo operand.  The four blocks add up. ----
        float* scr = reinterpret_cast<float*>(smem + oW1);
        float* S1 = reinterpret_cast<float*>(smem + oG);                 // [128][65] dW2^T blocks
        float* S2 = S1 + 128 * 65;                                       // [128][65] Q blocks
        float* cdb1 = par + 64;
        float* cdb2 = par + 128;
        if (tid >= 128 && tid < 192) {
            const int j = tid - 128, q4 = j >> 4;
            float s = 0.f;
            for (int w = 0; w < 3; ++w) s += scr[(q4 * 4 + w) * 24 + (j & 15)];
            cdb1[j] = s;
        } else if (tid >= 192 && tid < 224) {
            const int c = tid - 192, q4 = c >> 3;
            float s = 0.f;
            for (int w = 0; w < 3; ++w) s += scr[(q4 * 4 + w) * 24 + 16 + (c & 7)];
            cdb2[c] = s;
        }
        if (warp < 4) {
            const uint32_t row_addr = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                float d[32];
                tmem_ld32(row_addr + cWG1 + half * 32, d);
#pragma unroll
                for (int c = 0; c < 32; ++c) S1[tid * 65 + half * 32 + c] = d[c];
                tmem_ld32(row_addr + cWG2 + half * 32, d);
#pragma unroll
                for (int c = 0; c < 32; ++c) S2[tid * 65 + half * 32 + c] = d[c];
            }
        }
        tc_fence_before();
        __syncthreads();
        // thread t: column c = t % 32 of rows j = t / 32, + 16, ...
        const int c = tid & 31;
        const float gm = gamma ? gamma[c] : 1.f, bt = beta ? beta[c] : 0.f;
        float dgp = 0.f, dbp = 0.f;
        for (int j = tid >> 5; j < kH; j += kThreads / 32) {
            const float w2g = (S1[j * 65 + c] + S1[j * 65 + 32 + c]) + (S1[(64 + j) * 65 + c] + S1[(64 + j) * 65 + 32 + c]);   // dW2[o = c][j]
            const float q = (S2[j * 65 + c] + S2[j * 65 + 32 + c]) + (S2[(64 + j) * 65 + c] + S2[(64 + j) * 65 + 32 + c]);     // Q[j][c]
            atomicAdd(dW2 + c * ldw2 + j, w2g);
            atomicAdd(dW1 + j * kC + c, fmaf(gm, q, bt * cdb1[j]));
            const float w = W1[j * kC + c];
            dgp = fmaf(w, q, dgp);
            dbp = fmaf(w, cdb1[j], dbp);
        }
        if (dgamma) atomicAdd(dgamma + c, dgp);
        if (dbeta) atomicAdd(dbeta + c, dbp);
        if (db1 && tid < kH) atomicAdd(db1 + tid, cdb1[tid]);
        if (db2 && tid >= 64 && tid < 96) atomicAdd(db2 + tid - 64, cdb2[tid - 64]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        __syncwarp();
        tmem_dealloc<kTmemCols>(tmem);
    }
}

}  // namespace

#ifdef FZ_TUNING
extern "C" int fz_debug_mlp_bwd_trace(long long* buf) {
    FZ_CUDA_CHECK(cudaMemcpyToSymbol(g_mlp_bwd_trace, &buf, sizeof(buf)));
    return FZ_OK;
}
#endif

bool mlp_bwd_tc_supported(int hidden) { return hidden >= kH && hidden % kH == 0; }

// gradients must be zeroed by the caller (the kernel adds its CTA totals with atomics)
int mlp_bwd_tc_launch(const float* x1, const float* dout, const float* gamma, const float* beta, const float* W1, const float* b1,
                      const float* W2, float* dx1, float* dgamma, float* dbeta, float* dW1, float* db1, float* dW2, float* db2,
                      long long batch, int hidden, long long voxels, float eps, cudaStream_t st) {
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(mlp_bwd_tc, kSmem));
    const int tps = (int)((voxels + kTV - 1) / kTV);
    const long long tiles = batch * tps;
    // one persistent CTA per SM; beyond 192 tiles per CTA more CTAs instead: the tensor core accumulates with truncation, so the
    // error of the weight gradients' TMEM accumulation chains grows with their length (fz_linear_tc.cu)
    long long nblk = tiles < num_sms() ? tiles : num_sms();
    if (nblk * 192 < tiles) nblk = (tiles + 191) / 192;
    const unsigned blocks = (unsigned)nblk;
    for (int h0 = 0; h0 < hidden; h0 += kH) {
        mlp_bwd_tc<<<blocks, kThreads, kSmem, st>>>(x1, dout, gamma, beta, W1 + (size_t)h0 * kC, b1 ? b1 + h0 : nullptr, W2 + h0, dx1,
                                                    dgamma, dbeta, dW1 + (size_t)h0 * kC, db1 ? db1 + h0 : nullptr, dW2 + h0,
                                                    h0 == 0 ? db2 : nullptr, hidden, h0 > 0, voxels, tps, tiles, eps);
        FZ_LAUNCH_CHECK();
    }
    return FZ_OK;
}

}  // namespace fz
