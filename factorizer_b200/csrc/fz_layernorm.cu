// LayerNorm over the channel axis of a channels-first (B, C, voxels) fp32 tensor, forward and backward,
// without the movedim + contiguous round trips the reference's wrapper makes
// (factorizer/layers/norm.py:25-34 permutes to channels-last, calls nn.LayerNorm, permutes back: on a
// (1,32,128^3) activation that is 6 full-tensor copies and two 3 ms LayerNorm kernels per block step).
//
// One thread owns two neighbouring voxels (float2 per channel, so a warp reads 256 contiguous bytes per
// channel), keeps all C values in registers, and loops over voxel pairs grid-stride; the backward
// accumulates d(gamma), d(beta) per thread across its voxels, reduces them per CTA in shared memory and
// issues one atomicAdd per channel and CTA.  HBM-bound: forward reads x and writes y once, backward reads
// x and dy once and writes dx once.
//
// The kernels are templated on the element type T of x, y, dy, add and dx: float, or bf16 / fp16 (the 16-bit FactorizerBlocks),
// which is read and written as pairs and computed in fp32; gamma, beta, their gradients and the statistics stay fp32.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "fz_common.cuh"

namespace fz {
namespace {

template <typename T> struct Pair2;
template <> struct Pair2<float> { typedef float2 type; };
template <> struct Pair2<__nv_bfloat16> { typedef __nv_bfloat162 type; };
template <> struct Pair2<__half> { typedef __half2 type; };
template <typename T> using pair_t = typename Pair2<T>::type;   // two neighbouring voxels of one channel

__device__ __forceinline__ float2 ld2(const float2* p) { return __ldg(p); }
__device__ __forceinline__ float2 ld2(const __nv_bfloat162* p) { return __bfloat1622float2(__ldg(p)); }
__device__ __forceinline__ float2 ld2(const __half2* p) { return __half22float2(__ldg(p)); }
__device__ __forceinline__ float2 ld2cs(const float2* p) { return __ldcs(p); }
__device__ __forceinline__ float2 ld2cs(const __nv_bfloat162* p) { return __bfloat1622float2(__ldcs(p)); }
// fp16 streaming loads as one 32-bit word and two scalar conversions: in the 32-channel backward this keeps 256 bytes fewer
// of spills than __half22float2 (sm_100a, -Xptxas -v)
__device__ __forceinline__ float2 ld2cs(const __half2* p) {
    const unsigned u = __ldcs(reinterpret_cast<const unsigned*>(p));
    return make_float2(__half2float(__ushort_as_half((unsigned short)(u & 0xffffu))), __half2float(__ushort_as_half((unsigned short)(u >> 16))));
}
__device__ __forceinline__ void st2(float2* p, float2 v) { *p = v; }
__device__ __forceinline__ void st2(__nv_bfloat162* p, float2 v) { *p = __float22bfloat162_rn(v); }
__device__ __forceinline__ void st2(__half2* p, float2 v) { *p = __float22half2_rn(v); }

constexpr int kLnThreads = 256;

template <int C, typename T>
__global__ void __launch_bounds__(kLnThreads) layernorm_cf_fwd(const T* __restrict__ x, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, T* __restrict__ y,
                                                               long long pairs_per_sample, long long total_pairs, float eps) {
    __shared__ float gs[C], bs[C];
    for (int c = threadIdx.x; c < C; c += blockDim.x) { gs[c] = gamma ? gamma[c] : 1.f; bs[c] = beta ? beta[c] : 0.f; }
    __syncthreads();
    const long long vox = 2 * pairs_per_sample;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total_pairs; p += (long long)gridDim.x * blockDim.x) {
        const long long b = p / pairs_per_sample, v = p - b * pairs_per_sample;
        const pair_t<T>* xp = reinterpret_cast<const pair_t<T>*>(x + b * C * vox) + v;
        float2 val[C];
        float2 sum = make_float2(0.f, 0.f);
#pragma unroll
        for (int c = 0; c < C; ++c) { val[c] = ld2cs(xp + (long long)c * pairs_per_sample); sum.x += val[c].x; sum.y += val[c].y; }
        const float2 mean = make_float2(sum.x * (1.f / C), sum.y * (1.f / C));
        float2 var = make_float2(0.f, 0.f);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float dx = val[c].x - mean.x, dy = val[c].y - mean.y;
            var.x = fmaf(dx, dx, var.x); var.y = fmaf(dy, dy, var.y);
        }
        const float2 rstd = make_float2(rsqrtf(var.x * (1.f / C) + eps), rsqrtf(var.y * (1.f / C) + eps));
        pair_t<T>* yp = reinterpret_cast<pair_t<T>*>(y + b * C * vox) + v;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            float2 o;
            o.x = fmaf((val[c].x - mean.x) * rstd.x, gs[c], bs[c]);
            o.y = fmaf((val[c].y - mean.y) * rstd.y, gs[c], bs[c]);
            st2(yp + (long long)c * pairs_per_sample, o);
        }
    }
}

template <int C, typename T>
__global__ void __launch_bounds__(kLnThreads) layernorm_cf_bwd(const T* __restrict__ x, const float* __restrict__ gamma,
                                                               const T* __restrict__ dy, const T* __restrict__ add,
                                                               T* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                               long long pairs_per_sample, long long total_pairs, float eps) {
    __shared__ float gs[C];
    __shared__ float red[2][C][kLnThreads / 32];
    for (int c = threadIdx.x; c < C; c += blockDim.x) gs[c] = gamma ? gamma[c] : 1.f;
    __syncthreads();
    const long long vox = 2 * pairs_per_sample;
    float dg[C], db[C];
#pragma unroll
    for (int c = 0; c < C; ++c) { dg[c] = 0.f; db[c] = 0.f; }
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total_pairs; p += (long long)gridDim.x * blockDim.x) {
        const long long b = p / pairs_per_sample, v = p - b * pairs_per_sample;
        const pair_t<T>* xp = reinterpret_cast<const pair_t<T>*>(x + b * C * vox) + v;
        const pair_t<T>* gp = reinterpret_cast<const pair_t<T>*>(dy + b * C * vox) + v;
        float2 xh[C], g[C];
        float2 sum = make_float2(0.f, 0.f);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            xh[c] = ld2cs(xp + (long long)c * pairs_per_sample);
            g[c] = ld2cs(gp + (long long)c * pairs_per_sample);
            sum.x += xh[c].x; sum.y += xh[c].y;
        }
        const float2 mean = make_float2(sum.x * (1.f / C), sum.y * (1.f / C));
        float2 var = make_float2(0.f, 0.f);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            xh[c].x -= mean.x; xh[c].y -= mean.y;
            var.x = fmaf(xh[c].x, xh[c].x, var.x); var.y = fmaf(xh[c].y, xh[c].y, var.y);
        }
        const float2 rstd = make_float2(rsqrtf(var.x * (1.f / C) + eps), rsqrtf(var.y * (1.f / C) + eps));
        // xh = normalised input; parameter gradients; g <- dy * gamma
        float2 m1 = make_float2(0.f, 0.f), m2 = make_float2(0.f, 0.f);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            xh[c].x *= rstd.x; xh[c].y *= rstd.y;
            dg[c] = fmaf(g[c].x, xh[c].x, fmaf(g[c].y, xh[c].y, dg[c]));
            db[c] += g[c].x + g[c].y;
            g[c].x *= gs[c]; g[c].y *= gs[c];
            m1.x += g[c].x; m1.y += g[c].y;
            m2.x = fmaf(g[c].x, xh[c].x, m2.x); m2.y = fmaf(g[c].y, xh[c].y, m2.y);
        }
        m1.x *= (1.f / C); m1.y *= (1.f / C); m2.x *= (1.f / C); m2.y *= (1.f / C);
        pair_t<T>* op = reinterpret_cast<pair_t<T>*>(dx + b * C * vox) + v;
        const pair_t<T>* ap = add ? reinterpret_cast<const pair_t<T>*>(add + b * C * vox) + v : nullptr;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            float2 o;
            o.x = rstd.x * (g[c].x - m1.x - xh[c].x * m2.x);
            o.y = rstd.y * (g[c].y - m1.y - xh[c].y * m2.y);
            if (ap) { const float2 r = ld2cs(ap + (long long)c * pairs_per_sample); o.x += r.x; o.y += r.y; }
            st2(op + (long long)c * pairs_per_sample, o);
        }
    }
    if (dgamma || dbeta) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float a = warp_sum(dg[c]), b = warp_sum(db[c]);
            if (lane == 0) { red[0][c][warp] = a; red[1][c][warp] = b; }
        }
        __syncthreads();
        for (int q = threadIdx.x; q < 2 * C; q += blockDim.x) {
            const int which = q / C, c = q - which * C;
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kLnThreads / 32; ++w) s += red[which][c][w];
            float* dst = which ? dbeta : dgamma;
            if (dst) atomicAdd(dst + c, s);
        }
    }
}

// ---- any channel count up to kLnMaxC: channels are looped, not held in registers ------------------------------------
// Statistics come from shifted sums (shift = the voxel's first channel), so x is read twice (the second time from
// L1 / L2) instead of three times; the backward keeps per-warp rows of d(gamma), d(beta) partials in shared memory.
constexpr int kLnMaxC = 512;

template <typename P>
__device__ __forceinline__ void ln_stats(const P* __restrict__ xp, long long pps, int C, float eps, float2& mean, float2& rstd) {
    const float2 k = ld2(xp);
    float2 s1 = make_float2(0.f, 0.f), s2 = make_float2(0.f, 0.f);
#pragma unroll 8
    for (int c = 0; c < C; ++c) {
        const float2 v = ld2(xp + (long long)c * pps);
        const float dx = v.x - k.x, dy = v.y - k.y;
        s1.x += dx; s1.y += dy;
        s2.x = fmaf(dx, dx, s2.x); s2.y = fmaf(dy, dy, s2.y);
    }
    const float inv = 1.f / (float)C;
    const float mx = s1.x * inv, my = s1.y * inv;
    mean = make_float2(k.x + mx, k.y + my);
    rstd = make_float2(rsqrtf(fmaxf(s2.x * inv - mx * mx, 0.f) + eps), rsqrtf(fmaxf(s2.y * inv - my * my, 0.f) + eps));
}

template <typename T>
__global__ void __launch_bounds__(kLnThreads) layernorm_cf_fwd_any(const T* __restrict__ x, const float* __restrict__ gamma,
                                                                   const float* __restrict__ beta, T* __restrict__ y, int C,
                                                                   long long pairs_per_sample, long long total_pairs, float eps) {
    __shared__ float gs[kLnMaxC], bs[kLnMaxC];
    for (int c = threadIdx.x; c < C; c += blockDim.x) { gs[c] = gamma ? gamma[c] : 1.f; bs[c] = beta ? beta[c] : 0.f; }
    __syncthreads();
    const long long vox = 2 * pairs_per_sample;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total_pairs; p += (long long)gridDim.x * blockDim.x) {
        const long long b = p / pairs_per_sample, v = p - b * pairs_per_sample;
        const pair_t<T>* xp = reinterpret_cast<const pair_t<T>*>(x + b * C * vox) + v;
        pair_t<T>* yp = reinterpret_cast<pair_t<T>*>(y + b * C * vox) + v;
        float2 mean, rstd;
        ln_stats(xp, pairs_per_sample, C, eps, mean, rstd);
#pragma unroll 8
        for (int c = 0; c < C; ++c) {
            const float2 val = ld2(xp + (long long)c * pairs_per_sample);
            st2(yp + (long long)c * pairs_per_sample, make_float2(fmaf((val.x - mean.x) * rstd.x, gs[c], bs[c]),
                                                              fmaf((val.y - mean.y) * rstd.y, gs[c], bs[c])));
        }
    }
}

// Transposing warp reduction of 32 values per lane: lane l ends up with the warp-wide total of element l (31 shuffles
// instead of 160 for 32 separate butterfly sums).
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
    int off = 16;
#pragma unroll
    for (int n = 32; n > 1; n >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
            const float keep = up ? v[i + n / 2] : v[i];
            const float send = up ? v[i] : v[i + n / 2];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
        off >>= 1;
    }
    return v[0];
}

template <typename T>
__global__ void __launch_bounds__(kLnThreads) layernorm_cf_bwd_any(const T* __restrict__ x, const float* __restrict__ gamma,
                                                                   const T* __restrict__ dy, const T* __restrict__ add,
                                                                   T* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta, int C,
                                                                   long long pairs_per_sample, long long total_pairs, float eps) {
    extern __shared__ float lsm[];
    const int CP = (C + 31) & ~31;                     // channels rounded up to whole chunks of 32
    float* gs = lsm;                                   // [CP]
    float* part = lsm + CP;                            // [warps][2 CP]: d(gamma) | d(beta) partials of each warp
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    for (int c = threadIdx.x; c < CP; c += blockDim.x) gs[c] = (c < C && gamma) ? gamma[c] : (c < C ? 1.f : 0.f);
    for (int i = threadIdx.x; i < warps * 2 * CP; i += blockDim.x) part[i] = 0.f;
    __syncthreads();
    float* mine = part + warp * 2 * CP;
    const long long vox = 2 * pairs_per_sample;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // whole warps iterate together (the per-channel sums over voxels are warp reductions)
    for (long long p0 = first - lane; p0 < total_pairs; p0 += stride) {
        const long long p = p0 + lane;
        const bool valid = p < total_pairs;
        const long long pc = valid ? p : 0;
        const long long b = pc / pairs_per_sample, v = pc - b * pairs_per_sample;
        const pair_t<T>* xp = reinterpret_cast<const pair_t<T>*>(x + b * C * vox) + v;
        const pair_t<T>* gp = reinterpret_cast<const pair_t<T>*>(dy + b * C * vox) + v;
        pair_t<T>* op = reinterpret_cast<pair_t<T>*>(dx + b * C * vox) + v;
        float2 mean, rstd;
        ln_stats(xp, pairs_per_sample, C, eps, mean, rstd);
        float2 m1 = make_float2(0.f, 0.f), m2 = make_float2(0.f, 0.f);
        for (int c0 = 0; c0 < C; c0 += 32) {
            float sg[32], sb[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int c = min(c0 + j, C - 1);                  // the tail chunk re-reads the last channel, weighted 0
                const float2 xv = ld2(xp + (long long)c * pairs_per_sample);
                float2 g = ld2(gp + (long long)c * pairs_per_sample);
                if (!valid || c0 + j >= C) g = make_float2(0.f, 0.f);
                const float hx = (xv.x - mean.x) * rstd.x, hy = (xv.y - mean.y) * rstd.y;
                sg[j] = fmaf(g.x, hx, g.y * hy);
                sb[j] = g.x + g.y;
                const float w = gs[c0 + j];
                const float tx = g.x * w, ty = g.y * w;
                m1.x += tx; m1.y += ty;
                m2.x = fmaf(tx, hx, m2.x); m2.y = fmaf(ty, hy, m2.y);
            }
            if (dgamma || dbeta) {
                mine[c0 + lane] += warp_transpose_sum32(sg, lane);
                mine[CP + c0 + lane] += warp_transpose_sum32(sb, lane);
            }
        }
        const float inv = 1.f / (float)C;
        m1.x *= inv; m1.y *= inv; m2.x *= inv; m2.y *= inv;
        if (valid) {
#pragma unroll 8
            for (int c = 0; c < C; ++c) {
                const float2 xv = ld2(xp + (long long)c * pairs_per_sample);
                const float2 g = ld2(gp + (long long)c * pairs_per_sample);
                const float hx = (xv.x - mean.x) * rstd.x, hy = (xv.y - mean.y) * rstd.y;
                float2 o = make_float2(rstd.x * (g.x * gs[c] - m1.x - hx * m2.x), rstd.y * (g.y * gs[c] - m1.y - hy * m2.y));
                if (add) {
                    const float2 r = ld2(reinterpret_cast<const pair_t<T>*>(add + b * C * vox) + v + (long long)c * pairs_per_sample);
                    o.x += r.x; o.y += r.y;
                }
                st2(op + (long long)c * pairs_per_sample, o);
            }
        }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < 2 * CP; q += blockDim.x) {
        const int c = q < CP ? q : q - CP;
        if (c >= C) continue;
        float t = 0.f;
        for (int w = 0; w < warps; ++w) t += part[w * 2 * CP + q];
        float* dst = q < CP ? dgamma : dbeta;
        if (dst) atomicAdd(dst + c, t);
    }
}

// ---- few voxels, many channels (the deep stages: 128 ch at 32^3 ... 512 ch at 8^3) -------------------------------------
// A thread walking all C channels of its voxel pair is one long latency chain there and the grid is a handful of CTAs.
// Sliced form: blockDim = (32 voxel pairs, SL channel slices); every warp owns C / SL channels of the CTA's 32 pairs,
// the per-voxel statistics are combined across slices through shared memory.
constexpr int kLnMaxSlices = 8;

__device__ __forceinline__ void slice_range(int C, int& cbeg, int& cend) {
    const int per = (C + blockDim.y - 1) / blockDim.y;
    cbeg = min((int)threadIdx.y * per, C);
    cend = min(cbeg + per, C);
}

// partial shifted sums of this slice -> totals over all slices (every thread of a pair column gets the same values)
template <typename P>
__device__ __forceinline__ void sliced_stats(const P* __restrict__ xp, long long pps, int C, int cbeg, int cend, float eps,
                                             float2 (*sa)[32], float2 (*sb)[32], float2& mean, float2& rstd) {
    const int lane = threadIdx.x;
    const float2 k = ld2(xp);
    float2 s1 = make_float2(0.f, 0.f), s2 = make_float2(0.f, 0.f);
#pragma unroll 8
    for (int c = cbeg; c < cend; ++c) {
        const float2 v = ld2(xp + (long long)c * pps);
        const float dx = v.x - k.x, dy = v.y - k.y;
        s1.x += dx; s1.y += dy;
        s2.x = fmaf(dx, dx, s2.x); s2.y = fmaf(dy, dy, s2.y);
    }
    sa[threadIdx.y][lane] = s1;
    sb[threadIdx.y][lane] = s2;
    __syncthreads();
    s1 = make_float2(0.f, 0.f); s2 = make_float2(0.f, 0.f);
    for (int w = 0; w < (int)blockDim.y; ++w) {
        const float2 a = sa[w][lane], b = sb[w][lane];
        s1.x += a.x; s1.y += a.y; s2.x += b.x; s2.y += b.y;
    }
    const float inv = 1.f / (float)C;
    const float mx = s1.x * inv, my = s1.y * inv;
    mean = make_float2(k.x + mx, k.y + my);
    rstd = make_float2(rsqrtf(fmaxf(s2.x * inv - mx * mx, 0.f) + eps), rsqrtf(fmaxf(s2.y * inv - my * my, 0.f) + eps));
}

template <typename T>
__global__ void __launch_bounds__(32 * kLnMaxSlices) layernorm_cf_fwd_sliced(const T* __restrict__ x, const float* __restrict__ gamma,
                                                                             const float* __restrict__ beta, T* __restrict__ y, int C,
                                                                             long long pairs_per_sample, long long total_pairs, float eps) {
    __shared__ float2 sa[kLnMaxSlices][32], sb[kLnMaxSlices][32];
    const int lane = threadIdx.x;
    int cbeg, cend;
    slice_range(C, cbeg, cend);
    const long long vox = 2 * pairs_per_sample;
    for (long long p0 = 32LL * blockIdx.x; p0 < total_pairs; p0 += 32LL * gridDim.x) {
        const long long p = p0 + lane;
        const bool valid = p < total_pairs;
        const long long pc = valid ? p : 0;
        const long long b = pc / pairs_per_sample, v = pc - b * pairs_per_sample;
        const pair_t<T>* xp = reinterpret_cast<const pair_t<T>*>(x + b * C * vox) + v;
        pair_t<T>* yp = reinterpret_cast<pair_t<T>*>(y + b * C * vox) + v;
        float2 mean, rstd;
        sliced_stats(xp, pairs_per_sample, C, cbeg, cend, eps, sa, sb, mean, rstd);
        if (valid) {
#pragma unroll 8
            for (int c = cbeg; c < cend; ++c) {
                const float2 val = ld2(xp + (long long)c * pairs_per_sample);
                const float g = gamma ? __ldg(gamma + c) : 1.f, bb = beta ? __ldg(beta + c) : 0.f;
                st2(yp + (long long)c * pairs_per_sample, make_float2(fmaf((val.x - mean.x) * rstd.x, g, bb), fmaf((val.y - mean.y) * rstd.y, g, bb)));
            }
        }
        __syncthreads();          // sa / sb are rewritten by the next group
    }
}

template <typename T>
__global__ void __launch_bounds__(32 * kLnMaxSlices, 2) layernorm_cf_bwd_sliced(const T* __restrict__ x, const float* __restrict__ gamma,
                                                                             const T* __restrict__ dy, const T* __restrict__ add,
                                                                             T* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta, int C,
                                                                             long long pairs_per_sample, long long total_pairs, float eps) {
    extern __shared__ float lsm[];
    __shared__ float2 sa[kLnMaxSlices][32], sb[kLnMaxSlices][32];
    float* part = lsm;                                 // d(gamma) [C] | d(beta) [C]; every slice touches its own channels only
    float* gs = lsm + 2 * C;                           // gamma [C]
    const int lane = threadIdx.x, tid = threadIdx.y * 32 + lane, nthr = 32 * blockDim.y;
    for (int i = tid; i < 2 * C; i += nthr) part[i] = 0.f;
    for (int i = tid; i < C; i += nthr) gs[i] = gamma ? gamma[i] : 1.f;
    __syncthreads();
    int cbeg, cend;
    slice_range(C, cbeg, cend);
    const long long vox = 2 * pairs_per_sample;
    for (long long p0 = 32LL * blockIdx.x; p0 < total_pairs; p0 += 32LL * gridDim.x) {
        const long long p = p0 + lane;
        const bool valid = p < total_pairs;
        const long long pc = valid ? p : 0;
        const long long b = pc / pairs_per_sample, v = pc - b * pairs_per_sample;
        const pair_t<T>* xp = reinterpret_cast<const pair_t<T>*>(x + b * C * vox) + v;
        const pair_t<T>* gp = reinterpret_cast<const pair_t<T>*>(dy + b * C * vox) + v;
        pair_t<T>* op = reinterpret_cast<pair_t<T>*>(dx + b * C * vox) + v;
        float2 mean, rstd;
        sliced_stats(xp, pairs_per_sample, C, cbeg, cend, eps, sa, sb, mean, rstd);
        float2 m1 = make_float2(0.f, 0.f), m2 = make_float2(0.f, 0.f);
        for (int c0 = cbeg; c0 < cend; c0 += 32) {
            float sg[32], sbv[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const bool live = c0 + j < cend;
                const int c = live ? c0 + j : cend - 1;            // the tail chunk re-reads the last channel, weighted 0
                const float2 xv = ld2(xp + (long long)c * pairs_per_sample);
                float2 g = ld2(gp + (long long)c * pairs_per_sample);
                if (!valid || !live) g = make_float2(0.f, 0.f);
                const float hx = (xv.x - mean.x) * rstd.x, hy = (xv.y - mean.y) * rstd.y;
                sg[j] = fmaf(g.x, hx, g.y * hy);
                sbv[j] = g.x + g.y;
                const float w = gs[c];
                const float tx = g.x * w, ty = g.y * w;
                m1.x += tx; m1.y += ty;
                m2.x = fmaf(tx, hx, m2.x); m2.y = fmaf(ty, hy, m2.y);
            }
            if (dgamma || dbeta) {
                const float rg = warp_transpose_sum32(sg, lane), rb = warp_transpose_sum32(sbv, lane);
                if (c0 + lane < cend) { part[c0 + lane] += rg; part[C + c0 + lane] += rb; }
            }
        }
        __syncthreads();          // everyone has read the statistics partials
        sa[threadIdx.y][lane] = m1;
        sb[threadIdx.y][lane] = m2;
        __syncthreads();
        m1 = make_float2(0.f, 0.f); m2 = make_float2(0.f, 0.f);
        for (int w = 0; w < (int)blockDim.y; ++w) {
            const float2 a = sa[w][lane], bq = sb[w][lane];
            m1.x += a.x; m1.y += a.y; m2.x += bq.x; m2.y += bq.y;
        }
        const float inv = 1.f / (float)C;
        m1.x *= inv; m1.y *= inv; m2.x *= inv; m2.y *= inv;
        if (valid) {
#pragma unroll 8
            for (int c = cbeg; c < cend; ++c) {
                const float2 xv = ld2(xp + (long long)c * pairs_per_sample);
                const float2 g = ld2(gp + (long long)c * pairs_per_sample);
                const float w = gs[c];
                const float hx = (xv.x - mean.x) * rstd.x, hy = (xv.y - mean.y) * rstd.y;
                float2 o = make_float2(rstd.x * (g.x * w - m1.x - hx * m2.x), rstd.y * (g.y * w - m1.y - hy * m2.y));
                if (add) {
                    const float2 r = ld2(reinterpret_cast<const pair_t<T>*>(add + b * C * vox) + v + (long long)c * pairs_per_sample);
                    o.x += r.x; o.y += r.y;
                }
                st2(op + (long long)c * pairs_per_sample, o);
            }
        }
        __syncthreads();          // sa / sb are rewritten by the next group
    }
    __syncthreads();
    for (int q = tid; q < 2 * C; q += nthr) {
        float* dst = q < C ? dgamma : dbeta;
        if (dst) atomicAdd(dst + (q < C ? q : q - C), part[q]);
    }
}

// slices for the sliced kernels: 0 = use the one-thread-per-voxel-pair kernels
int ln_slices(int channels, long long total_pairs) {
    if (channels < 64 || total_pairs >= 256LL * num_sms()) return 0;
    return channels >= 256 ? 8 : (channels >= 128 ? 4 : 2);
}

template <int C, typename T>
int launch_fwd(const T* x, const float* gamma, const float* beta, T* y, long long batch, long long voxels, float eps, cudaStream_t st) {
    const long long pps = voxels / 2, total = batch * pps;
    long long blocks = (total + kLnThreads - 1) / kLnThreads;
    const long long cap = 8LL * num_sms();
    if (blocks > cap) blocks = cap;
    layernorm_cf_fwd<C><<<(unsigned)blocks, kLnThreads, 0, st>>>(x, gamma, beta, y, pps, total, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}
template <int C, typename T>
int launch_bwd(const T* x, const float* gamma, const T* dy, const T* add, T* dx, float* dgamma, float* dbeta, long long batch,
               long long voxels, float eps, cudaStream_t st) {
    const long long pps = voxels / 2, total = batch * pps;
    long long blocks = (total + kLnThreads - 1) / kLnThreads;
    const long long cap = 2LL * num_sms();
    if (blocks > cap) blocks = cap;
    if (dgamma) FZ_CUDA_CHECK(cudaMemsetAsync(dgamma, 0, C * sizeof(float), st));
    if (dbeta) FZ_CUDA_CHECK(cudaMemsetAsync(dbeta, 0, C * sizeof(float), st));
    layernorm_cf_bwd<C><<<(unsigned)blocks, kLnThreads, 0, st>>>(x, gamma, dy, add, dx, dgamma, dbeta, pps, total, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

// `align`: the byte alignment of a voxel pair of the element type
int check_args(const void* a, const void* b, long long batch, int channels, long long voxels, uintptr_t align) {
    if (!a || !b) return fail(FZ_ERR_INVALID, "null buffer");
    if (batch < 0 || voxels < 0) return fail(FZ_ERR_INVALID, "negative size");
    if (channels < 1 || channels > kLnMaxC)
        return fail(FZ_ERR_UNSUPPORTED, "channels-first LayerNorm kernel handles 1..%d channels, got %d", kLnMaxC, channels);
    if (voxels % 2) return fail(FZ_ERR_UNSUPPORTED, "channels-first LayerNorm kernel needs an even number of voxels, got %lld", voxels);
    if ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & (align - 1))
        return fail(FZ_ERR_INVALID, "buffers must be %d-byte aligned", (int)align);
    return FZ_OK;
}

template <typename T>
int ln_forward(const T* x, const float* gamma, const float* beta, T* y, int64_t batch, int32_t channels, int64_t voxels, float eps,
               void* stream) {
    tls().launches = 0;
    if (batch == 0 || voxels == 0) return FZ_OK;          // empty tensors carry null data pointers
    if (int e = check_args(x, y, batch, channels, voxels, sizeof(pair_t<T>))) return e;
    cudaStream_t st = (cudaStream_t)stream;
    switch (channels) {
        case 8: return launch_fwd<8>(x, gamma, beta, y, batch, voxels, eps, st);
        case 16: return launch_fwd<16>(x, gamma, beta, y, batch, voxels, eps, st);
        case 32: return launch_fwd<32>(x, gamma, beta, y, batch, voxels, eps, st);
        default: break;
    }
    {
        const long long pps = voxels / 2, total = batch * pps;
        if (const int sl = ln_slices(channels, total)) {
            long long groups = (total + 31) / 32;
            if (groups > 8LL * num_sms()) groups = 8LL * num_sms();
            layernorm_cf_fwd_sliced<<<(unsigned)groups, dim3(32, sl), 0, st>>>(x, gamma, beta, y, channels, pps, total, eps);
            FZ_LAUNCH_CHECK();
            return FZ_OK;
        }
        const int threads = total >= 256LL * num_sms() ? kLnThreads : 64;   // few voxels: spread them over more SMs
        long long blocks = (total + threads - 1) / threads;
        const long long cap = 8LL * num_sms();
        if (blocks > cap) blocks = cap;
        layernorm_cf_fwd_any<<<(unsigned)blocks, threads, 0, st>>>(x, gamma, beta, y, channels, pps, total, eps);
        FZ_LAUNCH_CHECK();
        return FZ_OK;
    }
}

template <typename T>
int ln_backward_add(const T* x, const float* gamma, const T* dy, const T* add, T* dx, float* dgamma, float* dbeta, int64_t batch,
                    int32_t channels, int64_t voxels, float eps, void* stream) {
    tls().launches = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (batch == 0 || voxels == 0) {
        if (dgamma) FZ_CUDA_CHECK(cudaMemsetAsync(dgamma, 0, channels * sizeof(float), st));
        if (dbeta) FZ_CUDA_CHECK(cudaMemsetAsync(dbeta, 0, channels * sizeof(float), st));
        return FZ_OK;
    }
    if (int e = check_args(x, dx, batch, channels, voxels, sizeof(pair_t<T>))) return e;
    if (!dy) return fail(FZ_ERR_INVALID, "null buffer");
    switch (channels) {
        case 8: return launch_bwd<8>(x, gamma, dy, add, dx, dgamma, dbeta, batch, voxels, eps, st);
        case 16: return launch_bwd<16>(x, gamma, dy, add, dx, dgamma, dbeta, batch, voxels, eps, st);
        case 32: return launch_bwd<32>(x, gamma, dy, add, dx, dgamma, dbeta, batch, voxels, eps, st);
        default: break;
    }
    {
        const long long pps = voxels / 2, total = batch * pps;
        const int threads = total >= 256LL * num_sms() ? kLnThreads : 64;
        long long blocks = (total + threads - 1) / threads;
        const long long cap = 4LL * num_sms();
        if (blocks > cap) blocks = cap;
        if (dgamma) FZ_CUDA_CHECK(cudaMemsetAsync(dgamma, 0, channels * sizeof(float), st));
        if (dbeta) FZ_CUDA_CHECK(cudaMemsetAsync(dbeta, 0, channels * sizeof(float), st));
        if (const int sl = ln_slices(channels, total)) {
            long long groups = (total + 31) / 32;
            if (groups > 4LL * num_sms()) groups = 4LL * num_sms();
            layernorm_cf_bwd_sliced<<<(unsigned)groups, dim3(32, sl), sizeof(float) * 3 * channels, st>>>(x, gamma, dy, add, dx, dgamma, dbeta,
                                                                                                         channels, pps, total, eps);
            FZ_LAUNCH_CHECK();
            return FZ_OK;
        }
        const size_t cp = ((size_t)channels + 31) & ~(size_t)31;
        const size_t smem = sizeof(float) * (cp + (threads / 32) * 2 * cp);
        static SmemConfig cfg;
        FZ_CUDA_CHECK(cfg.ensure(layernorm_cf_bwd_any<T>, sizeof(float) * (kLnMaxC + (kLnThreads / 32) * 2 * kLnMaxC)));
        layernorm_cf_bwd_any<<<(unsigned)blocks, threads, smem, st>>>(x, gamma, dy, add, dx, dgamma, dbeta, channels, pps, total, eps);
        FZ_LAUNCH_CHECK();
        return FZ_OK;
    }
}

}  // namespace
}  // namespace fz

using namespace fz;

extern "C" {

int fz_layernorm_cf_supported(int32_t channels, int64_t voxels) {
    return channels >= 1 && channels <= kLnMaxC && voxels % 2 == 0;
}

int fz_layernorm_cf_forward(const float* x, const float* gamma, const float* beta, float* y, int64_t batch,
                            int32_t channels, int64_t voxels, float eps, void* stream) {
    return ln_forward(x, gamma, beta, y, batch, channels, voxels, eps, stream);
}

int fz_layernorm_cf_backward(const float* x, const float* gamma, const float* dy, float* dx, float* dgamma,
                             float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps, void* stream) {
    return fz_layernorm_cf_backward_add(x, gamma, dy, nullptr, dx, dgamma, dbeta, batch, channels, voxels, eps, stream);
}

int fz_layernorm_cf_backward_add(const float* x, const float* gamma, const float* dy, const float* add, float* dx, float* dgamma,
                                 float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps, void* stream) {
    return ln_backward_add(x, gamma, dy, add, dx, dgamma, dbeta, batch, channels, voxels, eps, stream);
}

int fz_layernorm_cf_bf16_supported(int32_t channels, int64_t voxels) { return fz_layernorm_cf_supported(channels, voxels); }

int fz_layernorm_cf_forward_bf16(const void* x, const float* gamma, const float* beta, void* y, int64_t batch, int32_t channels,
                                 int64_t voxels, float eps, void* stream) {
    return ln_forward(static_cast<const __nv_bfloat16*>(x), gamma, beta, static_cast<__nv_bfloat16*>(y), batch, channels, voxels, eps,
                      stream);
}

int fz_layernorm_cf_backward_add_bf16(const void* x, const float* gamma, const void* dy, const void* add, void* dx, float* dgamma,
                                      float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps, void* stream) {
    typedef __nv_bfloat16 bf16;
    return ln_backward_add(static_cast<const bf16*>(x), gamma, static_cast<const bf16*>(dy), static_cast<const bf16*>(add),
                           static_cast<bf16*>(dx), dgamma, dbeta, batch, channels, voxels, eps, stream);
}

int fz_layernorm_cf_f16_supported(int32_t channels, int64_t voxels) { return fz_layernorm_cf_supported(channels, voxels); }

int fz_layernorm_cf_forward_f16(const void* x, const float* gamma, const float* beta, void* y, int64_t batch, int32_t channels,
                                int64_t voxels, float eps, void* stream) {
    return ln_forward(static_cast<const __half*>(x), gamma, beta, static_cast<__half*>(y), batch, channels, voxels, eps, stream);
}

int fz_layernorm_cf_backward_add_f16(const void* x, const float* gamma, const void* dy, const void* add, void* dx, float* dgamma,
                                     float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps, void* stream) {
    return ln_backward_add(static_cast<const __half*>(x), gamma, static_cast<const __half*>(dy), static_cast<const __half*>(add),
                           static_cast<__half*>(dx), dgamma, dbeta, batch, channels, voxels, eps, stream);
}

}  // extern "C"
