// Tensor-core (tcgen05 / TMEM, 3xTF32) forward of the second half of a 32-channel FactorizerBlock:
//     x1 = x + W_out m + b_out ;  out = x1 + W2 gelu(W1 LN(x1) + b1) + b2
// (reference factorizer/factorizer.py:53,75-76, layers/mlp.py:54-60, layers/norm.py:29-34).
//
// The three projections are per-voxel GEMMs with M = 128 voxels = TMEM lanes.  Their A operands (m, LN(x1), gelu(h)) never
// touch shared memory: the thread that owns a voxel writes the operand row straight into TENSOR MEMORY (tcgen05.st), as
// the fp32 word (hi: the tensor core reads the top 19 bits) and its remainder (lo); a GEMM issues a_lo b_hi + a_hi b_lo +
// a_hi b_hi (3xTF32, measured 5e-7 relative).  The weights are the B operands, staged once per CTA, K-major without
// swizzle.  D comes back through tcgen05.ld (32x32b: a thread reads ITS voxel's row), so bias / residual / LayerNorm /
// GELU run per thread in registers.
// A CTA has 8 warps: warp w owns the voxels 32 (w % 4) .. + 31 (the TMEM lanes it may touch) and half w / 4 of the channels
// and hidden units; the two threads of a voxel exchange their partial sums for the LayerNorm statistics.  Warp 0 issues the MMAs from warp-uniform code under elect.sync.  40 KB of shared memory and 256 TMEM
// columns per CTA: two CTAs per SM overlap each other's MMA round trips.
#include "fz_tc.cuh"

namespace fz {
namespace {

using namespace tc;

constexpr int kC = 32;
constexpr int kTM = 128;                  // voxels per tile
constexpr int kThreads = 256;
constexpr int kSlice = 64;                // hidden units per GEMM pair; wider MLPs run slice by slice inside a tile

// shared memory (bytes): weights hi | lo
template <int HID>
struct FwdSmem {
    static constexpr uint32_t oWo = 0;                               // W_out (32, 32) as B(n = o, k = c)
    static constexpr uint32_t oW1 = oWo + 2 * kC * kC * 4;           // W1 (HID, 32)   as B(n = j, k = c)
    static constexpr uint32_t oW2 = oW1 + 2 * HID * kC * 4;          // W2 (32, HID)   as B(n = o, k = j)
    static constexpr uint32_t oPar = oW2 + 2 * kC * HID * 4;         // bout | b2 | gamma | beta | b1
    static constexpr uint32_t oEx = oPar + (4 * kC + HID) * 4;       // pair_sum2 slots: 2 x [half][128] float2
    static constexpr uint32_t oBar = oEx + 2 * 256 * 8;
    static constexpr uint32_t oTmem = oBar + 8;
    static constexpr uint32_t bytes = oTmem + 8;
};

// TMEM columns: D of out_proj, later of the output projection | hidden pre-activation of a slice, later its gelu hi |
// A operand (m, then LN(x1): hi 32 | lo 32) | gelu lo of the slice
constexpr uint32_t cD = 0, cHid = 32, cA = 96, cGlo = 160, kTmemCols = 256;

template <int HID>
__global__ void __launch_bounds__(kThreads, 2)
mixer_mlp_fwd_tc2(const float* __restrict__ x, const float* __restrict__ m, const float* __restrict__ Wout,
                  const float* __restrict__ bout, const float* __restrict__ gamma, const float* __restrict__ beta,
                  const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
                  const float* __restrict__ b2, float* __restrict__ x1_out, float* __restrict__ out, long long vox,
                  int tiles_per_sample, long long total_tiles, float eps) {
    using L = FwdSmem<HID>;
    constexpr int NS = HID > kSlice ? kSlice : HID;      // hidden units per slice
    extern __shared__ __align__(1024) unsigned char smem[];
    float* par = reinterpret_cast<float*>(smem + L::oPar);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar = sbase + L::oBar;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool issuer = uniform_u32((uint32_t)warp) == 0;

    for (int e = tid; e < kC * kC; e += kThreads) {
        const float w = Wout[e];
        const uint32_t o = L::oWo + kmajor_off(e >> 5, e & 31, kC);
        *reinterpret_cast<float*>(smem + o) = w;
        *reinterpret_cast<float*>(smem + o + kC * kC * 4) = tf32_lo(w);
    }
    for (int e = tid; e < HID * kC; e += kThreads) {
        {
            const float w = W1[e];                            // (HID, 32)
            const uint32_t o = L::oW1 + kmajor_off(e >> 5, e & 31, kC);
            *reinterpret_cast<float*>(smem + o) = w;
            *reinterpret_cast<float*>(smem + o + HID * kC * 4) = tf32_lo(w);
        }
        {
            const float w = W2[e];                            // (32, HID)
            const uint32_t o = L::oW2 + kmajor_off(e / HID, e % HID, HID);
            *reinterpret_cast<float*>(smem + o) = w;
            *reinterpret_cast<float*>(smem + o + kC * HID * 4) = tf32_lo(w);
        }
    }
    for (int c = tid; c < kC; c += kThreads) {
        par[c] = bout ? bout[c] : 0.f; par[kC + c] = b2 ? b2[c] : 0.f;
        par[2 * kC + c] = gamma ? gamma[c] : 1.f; par[3 * kC + c] = beta ? beta[c] : 0.f;
    }
    for (int j = tid; j < HID; j += kThreads) par[4 * kC + j] = b1 ? b1[j] : 0.f;
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbarrier_init();
    }
    if (warp == 0) {
        tmem_alloc<kTmemCols>(sbase + L::oTmem);
        tmem_relinquish_alloc_permit();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + L::oTmem));
    const int vq = warp & 3, hh = warp >> 2;
    const int v = vq * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(vq * 32) << 16);
    const uint32_t id32 = make_idesc(128, kC, false, false), idH = make_idesc(128, NS, false, false);
    const uint64_t b_wo = make_desc(sbase + L::oWo, 128, kC * 32, 0);
    const uint64_t b_w1 = make_desc(sbase + L::oW1, 128, kC * 32, 0);
    const uint64_t b_w2 = make_desc(sbase + L::oW2, 128, HID * 32, 0);
    uint32_t parity = 0;

    // (sample, tile of the sample) of the next fetch, advanced by the grid size
    long long nb = (long long)blockIdx.x / tiles_per_sample;
    int nt = (int)((long long)blockIdx.x - nb * tiles_per_sample);
    const long long my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    float mr[16], xr[16];                     // the next tile's m and x (own 16 channels)
    float2* const slots = reinterpret_cast<float2*>(smem + L::oEx);
    uint32_t turn = 0;
    bool valid = false;
    long long base = 0;
    auto fetch = [&]() {
        const long long v0 = (long long)nt * kTM + v;
        valid = v0 < vox;
        base = (nb * kC + hh * 16) * vox + v0;
        nt += (int)gridDim.x;
        while (nt >= tiles_per_sample) { nt -= tiles_per_sample; ++nb; }
        const float* pm = m + base;
        const float* px = x + base;
#pragma unroll
        for (int c = 0; c < 16; ++c) { mr[c] = valid ? __ldg(pm) : 0.f; pm += vox; }
#pragma unroll
        for (int c = 0; c < 16; ++c) { xr[c] = valid ? __ldg(px) : 0.f; px += vox; }
    };
    // one GEMM D[cols d ..) = A[128 x K] W^T, A hi at TMEM columns a_hi .., lo at a_lo ..; issued by warp 0 once every thread has
    // published its part of A; every thread then waits for the result
    auto gemm = [&](uint32_t d, uint32_t a_hi, uint32_t a_lo, uint64_t b, uint32_t b_lo_off, int K, uint32_t idesc, bool acc0) {
        tmem_st_wait();
        tc_fence_before();
        __syncthreads();
        if (issuer) {
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int s = 0; s < K / 8; ++s) {
                    mma_tf32_ta(tmem + d, tmem + a_lo + s * 8, desc_at(b, s * 256), idesc, acc0 || s > 0);
                    mma_tf32_ta(tmem + d, tmem + a_hi + s * 8, desc_at(b, b_lo_off + s * 256), idesc, 1);
                    mma_tf32_ta(tmem + d, tmem + a_hi + s * 8, desc_at(b, s * 256), idesc, 1);
                }
                commit(bar);
            }
            __syncwarp();
        }
    };
    auto wait_gemm = [&]() {
        mbar_wait(bar, parity);
        parity ^= 1;
        tc_fence_after();
    };

    if (my_tiles > 0) fetch();
    for (long long it = 0; it < my_tiles; ++it) {
        const bool cur_valid = valid;
        const long long cur_base = base;
        // ---- A <- m (own 16 channels) ----
        {
            uint32_t th[16], tl[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) { th[c] = __float_as_uint(mr[c]); tl[c] = __float_as_uint(tf32_lo(mr[c])); }
            tmem_st16(lane_addr + cA + hh * 16, th);
            tmem_st16(lane_addr + cA + 32 + hh * 16, tl);
        }
        gemm(cD, cA, cA + 32, b_wo, kC * kC * 4, kC, id32, false);
        float x1o[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) x1o[c] = xr[c];
        wait_gemm();
        // ---- x1 = x + out_proj(m) + b, LayerNorm (the two threads of a voxel exchange partial sums), A <- LN(x1): own 16 channels ----
        {
            uint32_t d[16];
            tmem_ld16_nowait(lane_addr + cD + hh * 16, d);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 16; ++c) x1o[c] += __uint_as_float(d[c]) + par[hh * 16 + c];
        }
        if (x1_out && cur_valid) {
            float* po = x1_out + cur_base;
#pragma unroll
            for (int c = 0; c < 16; ++c) { *po = x1o[c]; po += vox; }
        }
        {
            float sm = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) sm += x1o[c];
            const float mean = pair_sum2(make_float2(sm, 0.f), slots, turn, hh, vq, v).x * (1.f / kC);
            float ss = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) { const float dlt = x1o[c] - mean; ss = fmaf(dlt, dlt, ss); }
            const float rstd = rsqrtf(pair_sum2(make_float2(ss, 0.f), slots, turn, hh, vq, v).x * (1.f / kC) + eps);
            uint32_t th[16], tl[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const float n = fmaf((x1o[c] - mean) * rstd, par[2 * kC + hh * 16 + c], par[3 * kC + hh * 16 + c]);
                th[c] = __float_as_uint(n); tl[c] = __float_as_uint(tf32_lo(n));
            }
            tmem_st16(lane_addr + cA + hh * 16, th);
            tmem_st16(lane_addr + cA + 32 + hh * 16, tl);
        }
#pragma unroll 1
        for (int sl = 0; sl < HID / NS; ++sl) {
            // hidden units NS sl .. + NS - 1: h = W1 LN(x1), then the output projection accumulates over the slices
            gemm(cHid, cA, cA + 32, desc_at(b_w1, sl * NS * 128), HID * kC * 4, kC, idH, false);
            // fetch the next tile's m and x: in flight during the GELU and output phases
            if (sl == 0 && it + 1 < my_tiles) fetch();
            wait_gemm();
            // ---- A <- gelu(h) (own NS / 2 hidden units): hi over the pre-activation's columns, lo in its own columns ----
#pragma unroll
            for (int q = 0; q < NS / 32; ++q) {
                uint32_t hr[16], gh[16], gl[16];
                tmem_ld16_nowait(lane_addr + cHid + hh * (NS / 2) + q * 16, hr);
                tmem_ld_wait();
#pragma unroll
                for (int p = 0; p < 16; p += 2) {
                    const float2 bj = *reinterpret_cast<const float2*>(par + 4 * kC + sl * NS + hh * (NS / 2) + q * 16 + p);
                    float2 e;
                    const float2 h2 = make_float2(__uint_as_float(hr[p]) + bj.x, __uint_as_float(hr[p + 1]) + bj.y);
                    const float2 g = __fmul2_rn(h2, gauss_cdf2(h2, e));
                    gh[p] = __float_as_uint(g.x); gh[p + 1] = __float_as_uint(g.y);
                    gl[p] = __float_as_uint(tf32_lo(g.x)); gl[p + 1] = __float_as_uint(tf32_lo(g.y));
                }
                tmem_st16(lane_addr + cHid + hh * (NS / 2) + q * 16, gh);
                tmem_st16(lane_addr + cGlo + hh * (NS / 2) + q * 16, gl);
            }
            gemm(cD, cHid, cGlo, desc_at(b_w2, sl * (NS / 4) * 128), kC * HID * 4, NS, id32, sl > 0);
            wait_gemm();                 // before the next slice's pre-activation overwrites the gelu columns
        }
        {
            uint32_t d[16];
            tmem_ld16_nowait(lane_addr + cD + hh * 16, d);
            tmem_ld_wait();
            if (cur_valid) {
                float* po = out + cur_base;
#pragma unroll
                for (int c = 0; c < 16; ++c) { *po = x1o[c] + __uint_as_float(d[c]) + par[kC + hh * 16 + c]; po += vox; }
            }
        }
        // the next tile's tcgen05.st / MMAs reuse these TMEM columns: every thread is past its loads at the next __syncthreads
        tc_fence_before();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<kTmemCols>(tmem);
}

// --------------------------------------------------------------------------------------------------------------------
// z = W LN(x)   (norm1 + in_proj; reference factorizer/factorizer.py:38, layers/norm.py:29-34, layers/linear.py:53-58)
// Same scheme: the normalised input is written into tensor memory by its voxel's two threads (16 channels each; they
// exchange their partial sums for the statistics), one 3xTF32 GEMM per 128-voxel tile with W diag(gamma) as B (the beta term is a bias W beta),
// 12 KB of shared memory and 128 TMEM columns per CTA: four CTAs per SM keep the two HBM passes busy.
// --------------------------------------------------------------------------------------------------------------------
constexpr uint32_t lW = 0, lPar = 8192, lEx = lPar + kC * 4, lBar = lEx + 2 * 256 * 8, lTmem = lBar + 8, kSmemLn = lTmem + 8;

__global__ void __launch_bounds__(kThreads, 4)
ln_linear_fwd_tc(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                 const float* __restrict__ W, float* __restrict__ y, long long vox, int tiles_per_sample, long long total_tiles,
                 float eps) {
    extern __shared__ __align__(1024) unsigned char smem[];
    float* wb = reinterpret_cast<float*>(smem + lPar);        // (W beta)[o]
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar = sbase + lBar;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool issuer = uniform_u32((uint32_t)warp) == 0;
    for (int e = tid; e < kC * kC; e += kThreads) {
        const int o = e >> 5, c = e & 31;
        const float w = W[e] * (gamma ? gamma[c] : 1.f);
        const uint32_t off = lW + kmajor_off(o, c, kC);
        *reinterpret_cast<float*>(smem + off) = w;
        *reinterpret_cast<float*>(smem + off + 4096) = tf32_lo(w);
    }
    for (int o = tid; o < kC; o += kThreads) {
        float s = 0.f;
        if (beta)
            for (int c = 0; c < kC; ++c) s = fmaf(W[o * kC + c], beta[c], s);
        wb[o] = s;
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbarrier_init();
    }
    if (warp == 0) {
        tmem_alloc<128>(sbase + lTmem);
        tmem_relinquish_alloc_permit();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + lTmem));
    const int vq = warp & 3, hh = warp >> 2;
    const int v = vq * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(vq * 32) << 16);
    const uint32_t idesc = make_idesc(128, kC, false, false);
    const uint64_t b_w = make_desc(sbase + lW, 128, kC * 32, 0);
    uint32_t parity = 0;
    long long nb = (long long)blockIdx.x / tiles_per_sample;
    int nt = (int)((long long)blockIdx.x - nb * tiles_per_sample);
    const long long my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    float xr[16];                             // this thread's 16 channels of the next tile
    float2* const slots = reinterpret_cast<float2*>(smem + lEx);
    uint32_t turn = 0;
    bool valid = false;
    long long base = 0;
    auto fetch = [&]() {
        const long long v0 = (long long)nt * kTM + v;
        valid = v0 < vox;
        base = (nb * kC + hh * 16) * vox + v0;
        nt += (int)gridDim.x;
        while (nt >= tiles_per_sample) { nt -= tiles_per_sample; ++nb; }
        const float* px = x + base;
#pragma unroll
        for (int c = 0; c < 16; ++c) { xr[c] = valid ? __ldg(px) : 0.f; px += vox; }
    };
    if (my_tiles > 0) fetch();
    for (long long it = 0; it < my_tiles; ++it) {
        const bool cur_valid = valid;
        const long long cur_base = base;
        {
            // LayerNorm statistics: the two threads of a voxel own 16 channels each and exchange their partial sums
            float s = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) s += xr[c];
            const float mean = pair_sum2(make_float2(s, 0.f), slots, turn, hh, vq, v).x * (1.f / kC);
            float ss = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) { xr[c] -= mean; ss = fmaf(xr[c], xr[c], ss); }
            const float rstd = rsqrtf(pair_sum2(make_float2(ss, 0.f), slots, turn, hh, vq, v).x * (1.f / kC) + eps);
            uint32_t th[16], tl[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const float xh = xr[c] * rstd;
                th[c] = __float_as_uint(xh); tl[c] = __float_as_uint(tf32_lo(xh));
            }
            tmem_st16(lane_addr + hh * 16, th);               // A: hi columns 0 .. 31, lo 32 .. 63; D: 64 .. 95
            tmem_st16(lane_addr + 32 + hh * 16, tl);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncthreads();
        if (issuer) {
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int s = 0; s < kC / 8; ++s) {
                    mma_tf32_ta(tmem + 64, tmem + 32 + s * 8, desc_at(b_w, s * 256), idesc, s > 0);
                    mma_tf32_ta(tmem + 64, tmem + s * 8, desc_at(b_w, 4096 + s * 256), idesc, 1);
                    mma_tf32_ta(tmem + 64, tmem + s * 8, desc_at(b_w, s * 256), idesc, 1);
                }
                commit(bar);
            }
            __syncwarp();
        }
        if (it + 1 < my_tiles) fetch();
        mbar_wait(bar, parity);
        parity ^= 1;
        tc_fence_after();
        {
            uint32_t d[16];
            tmem_ld16_nowait(lane_addr + 64 + hh * 16, d);
            tmem_ld_wait();
            if (cur_valid) {
                float* po = y + cur_base;
#pragma unroll
                for (int c = 0; c < 16; ++c) { *po = __uint_as_float(d[c]) + wb[hh * 16 + c]; po += vox; }
            }
        }
        tc_fence_before();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<128>(tmem);
}

}  // namespace

// hidden width 32, 64, 128 or 256 (mlp_ratio 1, 2, 4, 8 at 32 channels)
bool mixer_mlp_tc_supported(int hidden) { return hidden == 32 || hidden == 64 || hidden == 128 || hidden == 256; }

template <int HID>
static int launch_fwd(const float* x, const float* m, const float* Wout, const float* bout, const float* gamma, const float* beta,
                      const float* W1, const float* b1, const float* W2, const float* b2, float* x1, float* out, long long batch,
                      long long voxels, float eps, cudaStream_t st) {
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(mixer_mlp_fwd_tc2<HID>, FwdSmem<HID>::bytes));
    const int tps = (int)((voxels + kTM - 1) / kTM);
    const long long tiles = batch * tps;
    const long long cap = (FwdSmem<HID>::bytes > 110 * 1024 ? 1LL : 2LL) * num_sms();
    const unsigned blocks = (unsigned)(tiles < cap ? tiles : cap);
    mixer_mlp_fwd_tc2<HID><<<blocks, kThreads, FwdSmem<HID>::bytes, st>>>(x, m, Wout, bout, gamma, beta, W1, b1, W2, b2, x1, out, voxels,
                                                                          tps, tiles, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int mixer_mlp_tc_launch(const float* x, const float* m, const float* Wout, const float* bout, const float* gamma, const float* beta,
                        const float* W1, const float* b1, const float* W2, const float* b2, float* x1, float* out, long long batch,
                        int hidden, long long voxels, float eps, cudaStream_t st) {
    switch (hidden) {
        case 32: return launch_fwd<32>(x, m, Wout, bout, gamma, beta, W1, b1, W2, b2, x1, out, batch, voxels, eps, st);
        case 64: return launch_fwd<64>(x, m, Wout, bout, gamma, beta, W1, b1, W2, b2, x1, out, batch, voxels, eps, st);
        case 128: return launch_fwd<128>(x, m, Wout, bout, gamma, beta, W1, b1, W2, b2, x1, out, batch, voxels, eps, st);
        case 256: return launch_fwd<256>(x, m, Wout, bout, gamma, beta, W1, b1, W2, b2, x1, out, batch, voxels, eps, st);
    }
    return fail(FZ_ERR_UNSUPPORTED, "tensor-core MLP forward: hidden width %d", hidden);
}

}  // namespace fz

namespace fz {
int ln_linear_tc_launch(const float* x, const float* gamma, const float* beta, const float* W, float* y, long long batch,
                        long long voxels, float eps, cudaStream_t st) {
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(ln_linear_fwd_tc, kSmemLn));
    const int tps = (int)((voxels + kTM - 1) / kTM);
    const long long tiles = batch * tps;
    const long long cap = 4LL * num_sms();
    const unsigned blocks = (unsigned)(tiles < cap ? tiles : cap);
    ln_linear_fwd_tc<<<blocks, kThreads, kSmemLn, st>>>(x, gamma, beta, W, y, voxels, tps, tiles, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}
}  // namespace fz
