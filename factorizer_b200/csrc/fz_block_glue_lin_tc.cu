// Tensor-core (tcgen05 / TMEM, 3xTF32) backward of the two channel projections of a 32-channel FactorizerBlock
// (reference factorizer/layers/linear.py:53-58, layers/norm.py:29-34; factorizer.py:38,53):
//   LN = false (out_proj):            y = W a + b        ->  da = W^T dy,  dW = sum_v dy a^T,  db = sum_v dy
//   LN = true  (norm1 + in_proj):     y = W LN(a)        ->  da = LN'(W^T dy) + resid,  dW,  d(gamma),  d(beta)
// Per tile of 128 voxels (voxel = TMEM lane), with xh = the normalised (pre-affine) a (LN) or a itself, Wg = W diag(gamma):
//   GEMM   d(xh) = dy Wg              M = 128, N = 32, K = 32; A = dy written by its voxel's thread into TENSOR MEMORY
//   WG     Q    += [dy ; dy_lo] (64 rows) x [xh | xh_lo] (64 columns), contraction over the tile's voxels, operands in
//                  shared memory as voxel rows (fz_tc.cuh), accumulated in TMEM over ALL tiles of the CTA
//   da           = rstd (d(xh) - mean(d(xh)) - xh mean(d(xh) xh)) + resid                      (LN)
// and, once per CTA:  dW = Q diag(gamma) + S beta^T,  d(gamma)_c = sum_o W[o][c] Q[o][c],  d(beta)_c = sum_o W[o][c] S[o],
// db = S, with S = sum_v dy accumulated in registers.
// 8 warps per CTA: warp w owns the voxels 32 (w % 4) .. + 31 and half w / 4 of the channels; warp 0 also issues the MMAs
// (warp-uniform code under elect.sync).  72 KB of shared memory and 256 TMEM columns: two CTAs per SM.
#include "fz_tc.cuh"

namespace fz {
namespace {

using namespace tc;

constexpr int kC = 32;
constexpr int kTM = 128;
constexpr int kThreads = 256;
constexpr uint32_t kAtom = kTM * 128;         // a voxel-row atom: 128 rows x 128 bytes = 16 KiB
constexpr uint32_t oDY = 0;                   // dy atoms [hi | lo]
constexpr uint32_t oXH = 2 * kAtom;           // xh atoms [hi | lo]
constexpr uint32_t oW = 4 * kAtom;            // Wg as B(n = c, k = o), K-major: hi 4 KiB | lo 4 KiB
constexpr uint32_t oPar = oW + 8192;          // gamma | beta | S of the CTA
constexpr uint32_t oEx = oPar + 3 * kC * 4;   // pair_sum2 slots: 2 x [half][128] float2
constexpr uint32_t oBar = oEx + 2 * 256 * 8;  // bar_g | bar_wg
constexpr uint32_t oTmem = oBar + 16;
constexpr uint32_t kSmem = oTmem + 8;
// TMEM columns: A = dy hi | lo, D = d(xh), contraction accumulator (64 rows x 64 columns)
constexpr uint32_t cA = 0, cD = 64, cWG = 96, kTmemCols = 256;

template <bool LN>
__global__ void __launch_bounds__(kThreads, 2)
linear_bwd_tc2(const float* __restrict__ dy, const float* __restrict__ a, const float* __restrict__ gamma,
               const float* __restrict__ beta, const float* __restrict__ W, const float* __restrict__ resid,
               float* __restrict__ da, float* __restrict__ dW, float* __restrict__ db, float* __restrict__ dgamma,
               float* __restrict__ dbeta, long long vox, int tiles_per_sample, long long total_tiles, float eps) {
    extern __shared__ __align__(1024) unsigned char smem[];
    float* par = reinterpret_cast<float*>(smem + oPar);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar_g = sbase + oBar, bar_wg = bar_g + 8;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool issuer = uniform_u32((uint32_t)warp) == 0;

    for (int e = tid; e < kC * kC; e += kThreads) {
        const int o = e >> 5, c = e & 31;
        const float w = W[e] * (LN && gamma ? gamma[c] : 1.f);
        const uint32_t off = oW + kmajor_off(c, o, kC);
        *reinterpret_cast<float*>(smem + off) = w;
        *reinterpret_cast<float*>(smem + off + 4096) = tf32_lo(w);
    }
    for (int c = tid; c < kC; c += kThreads) {
        par[c] = LN && gamma ? gamma[c] : 1.f;
        par[kC + c] = LN && beta ? beta[c] : 0.f;
    }
    if (tid == 0) {
        mbar_init(bar_g, 1); mbar_init(bar_wg, 1);
        fence_mbarrier_init();
    }
    if (warp == 0) {
        tmem_alloc<kTmemCols>(sbase + oTmem);
        tmem_relinquish_alloc_permit();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + oTmem));
    const int vq = warp & 3, hh = warp >> 2;
    const int v = vq * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(vq * 32) << 16);
    const bool swap = (v & 4) != 0;
    // this thread's two 32-byte chunks (channels 16 hh .. + 15) of its voxel row
    const uint32_t c0 = (uint32_t)v * 128 + (uint32_t)(((2 * hh) ^ (v & 3)) << 5);
    const uint32_t c1 = (uint32_t)v * 128 + (uint32_t)(((2 * hh + 1) ^ (v & 3)) << 5);
    const uint32_t id_g = make_idesc(128, kC, false, false), id_wg = make_idesc(64, 64, true, true);
    const uint64_t b_w = make_desc(sbase + oW, 128, kC * 32, 0);
    const uint64_t k_dy = make_desc(sbase + oDY, kAtom, 512, 1), k_xh = make_desc(sbase + oXH, kAtom, 512, 1);

    long long nb = (long long)blockIdx.x / tiles_per_sample;
    int nt = (int)((long long)blockIdx.x - nb * tiles_per_sample);
    const long long my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    float gr[16], ar[16];                     // the next tile's dy and a (own 16 channels)
    float2* const slots = reinterpret_cast<float2*>(smem + oEx);
    uint32_t turn = 0;
    float acc_s[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc_s[i] = 0.f;
    bool valid = false;
    long long base = 0;
    auto fetch = [&]() {
        const long long v0 = (long long)nt * kTM + v;
        valid = v0 < vox;
        base = nb * kC * vox + v0;
        nt += (int)gridDim.x;
        while (nt >= tiles_per_sample) { nt -= tiles_per_sample; ++nb; }
        const long long own = base + (long long)(hh * 16) * vox;
        const float* pg = dy + own;
        const float* pa = a + own;
#pragma unroll
        for (int c = 0; c < 16; ++c) { gr[c] = valid ? __ldg(pg) : 0.f; pg += vox; }
#pragma unroll
        for (int c = 0; c < 16; ++c) { ar[c] = valid ? __ldg(pa) : 0.f; pa += vox; }
    };
    if (my_tiles > 0) fetch();
    uint32_t ph = 0;
    for (long long it = 0; it < my_tiles; ++it, ph ^= 1) {
        const bool cur_valid = valid;
        const long long cur_base = base;
        // ---- LayerNorm statistics (the two threads of a voxel exchange their partial sums), own channels of xh ----
        float xh[16];
        float rstd = 1.f;
        if (LN) {
            float sm = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) sm += ar[c];
            const float mean = pair_sum2(make_float2(sm, 0.f), slots, turn, hh, vq, v).x * (1.f / kC);
            float ss = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) { xh[c] = ar[c] - mean; ss = fmaf(xh[c], xh[c], ss); }
            rstd = rsqrtf(pair_sum2(make_float2(ss, 0.f), slots, turn, hh, vq, v).x * (1.f / kC) + eps);
#pragma unroll
            for (int c = 0; c < 16; ++c) xh[c] *= rstd;
        } else {
#pragma unroll
            for (int c = 0; c < 16; ++c) xh[c] = ar[c];
        }
        // ---- dy -> TMEM (A of the GEMM) and voxel rows; xh -> voxel rows ----
        if (it > 0) mbar_wait(bar_wg, ph ^ 1);                // the previous tile's contraction has read the rows
        tc_fence_after();
        {
            uint32_t th[16], tl[16];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                float h8[8], l8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float g = gr[q * 8 + i];
                    h8[i] = g; l8[i] = tf32_lo(g);
                    th[q * 8 + i] = __float_as_uint(g); tl[q * 8 + i] = __float_as_uint(l8[i]);
                    acc_s[q * 8 + i] += g;
                }
                st_row_chunk(sbase + oDY + (q ? c1 : c0), swap, h8);
                st_row_chunk(sbase + oDY + kAtom + (q ? c1 : c0), swap, l8);
#pragma unroll
                for (int i = 0; i < 8; ++i) { h8[i] = xh[q * 8 + i]; l8[i] = tf32_lo(h8[i]); }
                st_row_chunk(sbase + oXH + (q ? c1 : c0), swap, h8);
                st_row_chunk(sbase + oXH + kAtom + (q ? c1 : c0), swap, l8);
            }
            tmem_st16(lane_addr + cA + hh * 16, th);
            tmem_st16(lane_addr + cA + 32 + hh * 16, tl);
            tmem_st_wait();
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncthreads();
        if (issuer) {
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int s = 0; s < kC / 8; ++s) {        // d(xh) = dy Wg
                    mma_tf32_ta(tmem + cD, tmem + cA + 32 + s * 8, desc_at(b_w, s * 256), id_g, s > 0);
                    mma_tf32_ta(tmem + cD, tmem + cA + s * 8, desc_at(b_w, 4096 + s * 256), id_g, 1);
                    mma_tf32_ta(tmem + cD, tmem + cA + s * 8, desc_at(b_w, s * 256), id_g, 1);
                }
                commit(bar_g);
                mma_tf32(tmem + cWG, k_dy, k_xh, id_wg, it > 0);
#pragma unroll
                for (int s = 1; s < kTM / 8; ++s) mma_tf32(tmem + cWG, desc_at(k_dy, s * 1024), desc_at(k_xh, s * 1024), id_wg, 1);
                commit(bar_wg);
            }
            __syncwarp();
        }
        // this tile's residual gradient and the next tile's loads: in flight while the GEMM runs
        float rs[16];
        if (LN) {
            const float* pr = resid + cur_base + (long long)(hh * 16) * vox;
#pragma unroll
            for (int c = 0; c < 16; ++c) { rs[c] = (resid && cur_valid) ? __ldg(pr) : 0.f; pr += vox; }
        }
        if (it + 1 < my_tiles) fetch();
        mbar_wait(bar_g, ph);
        tc_fence_after();
        // ---- da ----
        if (LN) {
            uint32_t du[16];
            tmem_ld16_nowait(lane_addr + cD + hh * 16, du);
            tmem_ld_wait();
            float m1 = 0.f, m2 = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) { m1 += __uint_as_float(du[c]); m2 = fmaf(__uint_as_float(du[c]), xh[c], m2); }
            const float2 m = pair_sum2(make_float2(m1, m2), slots, turn, hh, vq, v);
            m1 = m.x * (1.f / kC); m2 = m.y * (1.f / kC);
            if (cur_valid) {
                float* po = da + cur_base + (long long)(hh * 16) * vox;
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    *po = rstd * (__uint_as_float(du[c]) - m1 - xh[c] * m2) + rs[c];
                    po += vox;
                }
            }
        } else {
            uint32_t d[16];
            tmem_ld16_nowait(lane_addr + cD + hh * 16, d);
            tmem_ld_wait();
            if (cur_valid) {
                float* po = da + cur_base + (long long)(hh * 16) * vox;
#pragma unroll
                for (int c = 0; c < 16; ++c) { *po = __uint_as_float(d[c]); po += vox; }
            }
        }
        tc_fence_before();
    }
    if (my_tiles > 0) mbar_wait(bar_wg, ph ^ 1);
    tc_fence_after();
    // ---- per-CTA totals ----
    {
        const float t = warp_vec_sum<16>(acc_s, lane);       // channel 16 hh + lane / 2
        float* scr = reinterpret_cast<float*>(smem + oW);    // [warp][16]; the weights are dead
        if ((lane & 1) == 0) scr[warp * 16 + (lane >> 1)] = t;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (my_tiles > 0) {
        // accumulator row r (dy channel r % 32: hi block for r < 32, lo block above) sits in TMEM lane 32 (r / 16) + r % 16;
        // column n: channel n % 32 of xh (hi for n < 32).  The four blocks add up to Q.
        const float* scr = reinterpret_cast<const float*>(smem + oW);
        float* S = reinterpret_cast<float*>(smem + oDY);      // [64][65]
        float* cs = par + 2 * kC;
        if (tid >= 128 && tid < 160) {
            const int o = tid - 128, h2 = o >> 4;
            float s = 0.f;
            for (int w = 0; w < 4; ++w) s += scr[(h2 * 4 + w) * 16 + (o & 15)];
            cs[o] = s;
        }
        if (warp < 4) {
            const uint32_t row_addr = tmem + ((uint32_t)(warp * 32) << 16);
            const int r = warp * 16 + lane;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                float d[32];
                tmem_ld32(row_addr + cWG + half * 32, d);        // warp-collective: lanes 16 .. 31 read idle TMEM lanes
                if (lane < 16) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) S[r * 65 + half * 32 + c] = d[c];
                }
            }
        }
        tc_fence_before();
        __syncthreads();
        const int c = tid & 31;
        const float gm = par[c], bt = par[kC + c];
        float dgp = 0.f, dbp = 0.f;
        for (int o = tid >> 5; o < kC; o += kThreads / 32) {
            const float q = (S[o * 65 + c] + S[o * 65 + 32 + c]) + (S[(32 + o) * 65 + c] + S[(32 + o) * 65 + 32 + c]);
            atomicAdd(dW + o * kC + c, fmaf(gm, q, bt * cs[o]));
            if (LN) {
                const float w = W[o * kC + c];
                dgp = fmaf(w, q, dgp);
                dbp = fmaf(w, cs[o], dbp);
            }
        }
        if (LN && dgamma) atomicAdd(dgamma + c, dgp);
        if (LN && dbeta) atomicAdd(dbeta + c, dbp);
        if (db && tid < kC) atomicAdd(db + tid, cs[tid]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<kTmemCols>(tmem);
}

}  // namespace

// gradients must be zeroed by the caller (the kernel adds its CTA totals with atomics)
int linear_bwd_tc2_launch(const float* dy, const float* a, const float* gamma, const float* beta, const float* W, const float* resid,
                          float* da, float* dW, float* db, float* dgamma, float* dbeta, long long batch, long long voxels, float eps,
                          int layernorm, cudaStream_t st) {
    static SmemConfig cfg_ln, cfg_plain;
    FZ_CUDA_CHECK(cfg_ln.ensure(linear_bwd_tc2<true>, kSmem));
    FZ_CUDA_CHECK(cfg_plain.ensure(linear_bwd_tc2<false>, kSmem));
    const int tps = (int)((voxels + kTM - 1) / kTM);
    const long long tiles = batch * tps;
    // two persistent CTAs per SM; beyond 128 tiles per CTA more CTAs instead (length of the TMEM accumulation chain of the
    // weight gradient: fz_linear_tc.cu)
    long long nblk = tiles < 2LL * num_sms() ? tiles : 2LL * num_sms();
    if (nblk * 128 < tiles) nblk = (tiles + 127) / 128;
    const unsigned blocks = (unsigned)nblk;
    if (layernorm)
        linear_bwd_tc2<true><<<blocks, kThreads, kSmem, st>>>(dy, a, gamma, beta, W, resid, da, dW, db, dgamma, dbeta, voxels, tps, tiles, eps);
    else
        linear_bwd_tc2<false><<<blocks, kThreads, kSmem, st>>>(dy, a, nullptr, nullptr, W, nullptr, da, dW, db, nullptr, nullptr, voxels, tps, tiles, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // namespace fz
