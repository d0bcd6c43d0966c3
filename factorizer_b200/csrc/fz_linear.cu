// Channel maps around the Factorizer blocks: the pieces of the reference's pointwise Linear (factorizer/layers/linear.py:53-58),
// of its U-Net scaffold's patch convolutions (factorizer/unet.py:53, 97-99, 247) and of its stem (factorizer/factorizer.py:
// 139-140) that the libraries handle badly at these shapes.  Four groups of kernels, each behind its own C entry point:
//
//   fz_linear_wgrad          dW[o][i] = sum_{b,v} dy[b][o][v] x[b][i][v],  db[o] = sum_{b,v} dy[b][o][v]
//   fz_space_depth2          (B,C,D,H,W) <-> (B,8C,DHW/8): the view on which a 2x2x2 stride-2 (transposed) convolution is a channel map
//                            (fz_space_depth2_bf16: the same on bf16)
//   fz_conv3d_stem_forward   3x3x3, padding 1, 1..4 -> 32 channels (fz_conv3d_stem_forward_bf16: fp32 or bf16 x, bf16 y)
//
// Weight gradient: the Swin Factorizer's wider stages give it a 64..1024 x 64..512 result over 512..262144 voxels, a shape
// library SGEMMs handle badly (sgemm_largek: 340 us for 64 x 64 x 262144, 10 % of the FP32 pipe; cuDNN's fp32 wgrad of the
// patch convolutions: 1.7-4.4 ms).  linear_wgrad: a CTA owns one 32 x 32 block of dW and a share of the voxel tiles, stages
// 256 voxels of its 32 + 32 rows in shared memory, keeps the partial sums in registers (a warp takes every 4th float4 column,
// a lane an 8 x 4 sub-block read with broadcast LDS.128) and adds them to dW once at the end.  linear_wgrad64 (further down):
// 64 x 64 or 32 x 128 blocks, cp.async double buffering, 8 x 8 register tiles.  FP32 pipe, exact fp32 products.
#include <cuda_bf16.h>

#include "fz_channel_map.cuh"
#include "fz_device.cuh"
#include "fz_internal.cuh"

namespace fz {
namespace {

typedef __nv_bfloat16 bf16;

constexpr int kWT = 128;            // threads
constexpr int kWV = 256;            // voxels per tile
constexpr int kWRS = kWV + 4;       // staged row stride (floats), = 4 mod 32: conflict-free row-broadcast reads
constexpr int kWWarps = kWT / 32;

// rows [r0, r0+32) x voxels [v0, v0+256) of a (rows_total, vox) matrix -> S[32][kWRS]; past-the-end voxels and rows
// (rows_left = rows_total - r0 may be below 32) read as 0
__device__ __forceinline__ void stage_rows(const float* __restrict__ g, long long vox, long long v0, int rows_left, float* __restrict__ S,
                                           int tid, float (&rowsum)[16], bool want_sums) {
    const int col4 = tid & 63, rbase = tid >> 6;
    const long long v = v0 + 4 * col4;
    const bool in_v = v < vox;                    // vox % 4 == 0: a float4 is wholly inside or outside
#pragma unroll
    for (int h = 0; h < 2; ++h) {                 // 8 rows in flight at a time (register budget of 3 CTAs per SM)
        float4 val[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
            val[i] = (in_v && rbase + 2 * (8 * h + i) < rows_left)
                         ? __ldg(reinterpret_cast<const float4*>(g + (long long)(rbase + 2 * (8 * h + i)) * vox + v))
                         : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            *reinterpret_cast<float4*>(S + (rbase + 2 * (8 * h + i)) * kWRS + 4 * col4) = val[i];
            if (want_sums) rowsum[8 * h + i] += (val[i].x + val[i].y) + (val[i].z + val[i].w);
        }
    }
}

__global__ void __launch_bounds__(kWT, 3) linear_wgrad(const float* __restrict__ dy, const float* __restrict__ x, float* __restrict__ dW,
                                                       float* __restrict__ db, int cout, int cin, long long vox, int tiles_per_sample,
                                                       long long total_tiles) {
    extern __shared__ __align__(16) float sm[];
    float* SA = sm;                     // dy rows [32][kWRS]
    float* SB = sm + 32 * kWRS;         // x rows  [32][kWRS]
    const int tid = threadIdx.x, lane = tid & 31, grp = tid >> 5, ro = lane & 3, co = lane >> 2;
    const int o0 = blockIdx.y * 32, i0 = blockIdx.z * 32;
    const bool sums = db != nullptr && blockIdx.z == 0;
    float2 acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[i][k] = make_float2(0.f, 0.f);
    float rowsum[16], unused[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) rowsum[i] = 0.f;
    for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const long long b = tile / tiles_per_sample;
        const long long v0 = (tile - b * tiles_per_sample) * kWV;
        __syncthreads();                // the previous tile has been consumed
        stage_rows(dy + (b * cout + o0) * vox, vox, v0, cout - o0, SA, tid, rowsum, sums);
        stage_rows(x + (b * cin + i0) * vox, vox, v0, cin - i0, SB, tid, unused, false);
        __syncthreads();
#pragma unroll 2
        for (int it = 0; it < kWV / 4 / kWWarps; ++it) {
            const int v = (it * kWWarps + grp) * 4;
            float4 B[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) B[k] = *reinterpret_cast<const float4*>(SB + (co + 8 * k) * kWRS + v);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 A = *reinterpret_cast<const float4*>(SA + (ro + 4 * i) * kWRS + v);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    acc[i][k] = fma2(make_float2(A.x, A.y), make_float2(B[k].x, B[k].y), acc[i][k]);
                    acc[i][k] = fma2(make_float2(A.z, A.w), make_float2(B[k].z, B[k].w), acc[i][k]);
                }
            }
        }
    }
    __syncthreads();
    // per-warp partial blocks -> shared memory (the staging area is free now) -> one atomicAdd per element and CTA
    float* scr = sm;                    // [warp][32*32]
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) scr[grp * 1024 + (ro + 4 * i) * 32 + co + 8 * k] = acc[i][k].x + acc[i][k].y;
    float* rs = sm + kWWarps * 1024;    // [32] row sums of dy
    if (tid < 32) rs[tid] = 0.f;
    __syncthreads();
    for (int e = tid; e < 1024; e += kWT) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kWWarps; ++w) t += scr[w * 1024 + e];
        if (o0 + (e >> 5) < cout && i0 + (e & 31) < cin) atomicAdd(dW + (long long)(o0 + (e >> 5)) * cin + i0 + (e & 31), t);
    }
    if (sums) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float t = warp_sum(rowsum[i]);
            if (lane == 0) atomicAdd(rs + (tid >> 6) + 2 * i, t);      // once per kernel: the CAS loop does not matter here
        }
        __syncthreads();
        if (tid < 32 && o0 + tid < cout) atomicAdd(db + o0 + tid, rs[tid]);
    }
}


// ---- both channel counts >= 64: 64 x 64 blocks, cp.async double buffering -------------------------------------------
// The 32 x 32 kernel above re-reads dy cin/32 times and x cout/32 times and exposes the load latency of every tile; for
// the wide layers (64 x 256 over 262144 voxels moves 1.07 GB that way) this one halves the re-reads and overlaps them:
// 256 threads, stages of 128 voxels x (64 dy rows + 64 x rows) filled by cp.async (zero-filled past the end), warp w
// owns 32 dy rows (w & 1) x all 64 x rows of every fourth float4 column (w >> 1).
constexpr int kW2T = 256, kW2V = 128, kW2RS = kW2V + 4;

// RB x CB = 2 x 1: a 64 x 64 block (warp halves split the dy rows); 1 x 2: a 32 x 128 block for layers with at most 32
// outputs (the stem's unfolded 32 x 108 gradient, the decoder adapters), where the warp halves split the x rows.
template <int RB, int CB>
__global__ void __launch_bounds__(kW2T, 1) linear_wgrad64(const float* __restrict__ dy, const float* __restrict__ x, float* __restrict__ dW,
                                                          float* __restrict__ db, int cout, int cin, long long vox, int tiles_per_sample,
                                                          long long total_tiles) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, ro = lane & 3, co = lane >> 2;
    static_assert((RB == 2 && CB == 1) || (RB == 1 && CB == 2), "block shape");
    constexpr int NA = 32 * RB, NR = NA + 64 * CB, kW2Stage = NR * kW2RS;
    const int kq = w >> 1, sr = RB == 2 ? (w & 1) : 0, sc = CB == 2 ? (w & 1) : 0;   // warp: float4 columns kq, kq+4, ... of 32 dy rows x 64 x rows
    const int o0 = blockIdx.y * NA, i0 = blockIdx.z * 64 * CB;
    const bool sums = db != nullptr && blockIdx.z == 0 && sc == 0;
    // an 8 x 8 register tile per lane: 16 LDS.128 per 128 FFMA2 (a 128-bit shared load holds the LSU for four cycles
    // whatever the broadcast, so the 8 x 4 tile of the kernel above is LSU-bound at two thirds of the FP32 pipe)
    float2 acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[i][k] = make_float2(0.f, 0.f);
    float rs[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) rs[i] = 0.f;

    auto issue = [&](long long tile, int stage) {
        const long long b = tile / tiles_per_sample;
        const long long v = (tile - b * tiles_per_sample) * kW2V + 4 * (tid & 31);
        const bool in_v = v < vox;
        float* S = sm + stage * kW2Stage + 4 * (tid & 31);
        const float* gdy = dy + b * cout * vox;
        const float* gx = x + b * cin * vox;
#pragma unroll
        for (int i = 0; i < NR / 8; ++i) {
            const int r = (tid >> 5) + 8 * i;              // dy rows, then x rows
            const bool isx = r >= NA;
            const int ch = isx ? i0 + r - NA : o0 + r;
            const bool real = in_v && ch < (isx ? cin : cout);
            const float* src = real ? (isx ? gx : gdy) + (long long)ch * vox + v : dy;
            cp_async16_zfill(S + r * kW2RS, src, real);
        }
        cp_async_commit();
    };

    long long tile = blockIdx.x;
    int stage = 0;
    if (tile < total_tiles) issue(tile, 0);
    for (; tile < total_tiles; tile += gridDim.x, stage ^= 1) {
        if (tile + gridDim.x < total_tiles) {
            issue(tile + gridDim.x, stage ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const float* SA = sm + stage * kW2Stage + (32 * sr) * kW2RS;
        const float* SB = sm + stage * kW2Stage + (NA + 64 * sc) * kW2RS;
#pragma unroll 1
        for (int it = 0; it < kW2V / 4 / 4; ++it) {
            const int v = (4 * it + kq) * 4;
            float4 B[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) B[k] = *reinterpret_cast<const float4*>(SB + (co + 8 * k) * kW2RS + v);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 A = *reinterpret_cast<const float4*>(SA + (ro + 4 * i) * kW2RS + v);
                if (sums) rs[i] += (A.x + A.y) + (A.z + A.w);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    acc[i][k] = fma2(make_float2(A.x, A.y), make_float2(B[k].x, B[k].y), acc[i][k]);
                    acc[i][k] = fma2(make_float2(A.z, A.w), make_float2(B[k].z, B[k].w), acc[i][k]);
                }
            }
        }
        __syncthreads();            // the stage is rewritten by the copy issued in the next iteration
    }
    // partial blocks of the 8 warps -> shared memory -> one atomicAdd per element and CTA
    float* scr = sm;                // [warp][32 * 64]
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int k = 0; k < 8; ++k) scr[w * 2048 + (ro + 4 * i) * 64 + co + 8 * k] = acc[i][k].x + acc[i][k].y;
    float* rsum = sm + 8 * 2048;    // [NA] row sums of dy
    if (tid < NA) rsum[tid] = 0.f;
    __syncthreads();
    for (int e = tid; e < 4096; e += kW2T) {
        const int half = e >> 11, q = e & 2047;                   // half = the warp pair's sr (2 x 1) or sc (1 x 2)
        float t = 0.f;
#pragma unroll
        for (int g = 0; g < 4; ++g) t += scr[(2 * g + half) * 2048 + q];
        const int o = o0 + (RB == 2 ? 32 * half : 0) + (q >> 6), c = i0 + (CB == 2 ? 64 * half : 0) + (q & 63);
        if (o < cout && c < cin) atomicAdd(dW + (long long)o * cin + c, t);
    }
    if (db != nullptr && blockIdx.z == 0) {                       // uniform over the CTA
        if (sums && co == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) atomicAdd(rsum + 32 * sr + ro + 4 * i, rs[i]);   // once per kernel
        }
        __syncthreads();
        if (tid < NA && o0 + tid < cout) atomicAdd(db + o0 + tid, rsum[tid]);
    }
}


// ---- space-to-depth / depth-to-space for 2x2x2 patches ---------------------------------------------------------------
// (B, C, D, H, W) <-> (B, C*8, D/2 * H/2 * W/2), rows ordered (c, kd, kh, kw): the view on which a kernel-2 stride-2
// convolution (or its transpose) is a channel map.  A thread moves one float4 of the full-resolution tensor = two
// float2 of the patch rows kw = 0 and kw = 1, so both sides are coalesced (torch's strided permute copy gathers 4-byte
// elements at stride 2).  On bf16 the same thread moves 8 bytes and two 4-byte pairs.
template <typename T> struct Quad;          // 4 consecutive elements along W, split into the pairs (0, 2) and (1, 3)
template <> struct Quad<float> {
    typedef float4 V4;
    typedef float2 V2;
    static __device__ __forceinline__ V2 even(V4 v) { return make_float2(v.x, v.z); }
    static __device__ __forceinline__ V2 odd(V4 v) { return make_float2(v.y, v.w); }
    static __device__ __forceinline__ V4 join(V2 a, V2 b) { return make_float4(a.x, b.x, a.y, b.y); }
};
template <> struct Quad<bf16> {
    typedef uint2 V4;                       // (e0 | e1 << 16, e2 | e3 << 16)
    typedef unsigned int V2;
    static __device__ __forceinline__ V2 even(V4 v) { return __byte_perm(v.x, v.y, 0x5410); }
    static __device__ __forceinline__ V2 odd(V4 v) { return __byte_perm(v.x, v.y, 0x7632); }
    static __device__ __forceinline__ V4 join(V2 a, V2 b) { return make_uint2(__byte_perm(a, b, 0x5410), __byte_perm(a, b, 0x7632)); }
};

template <typename T, bool TO_DEPTH>
__global__ void __launch_bounds__(256) space_depth2(const T* __restrict__ in, T* __restrict__ out, long long total4, int C, int D,
                                                    int H, int W4) {
    typedef Quad<T> Q;
    const int Hh = H >> 1, Wh = 2 * W4;                         // half-resolution height / width
    const long long Vh = (long long)(D >> 1) * Hh * Wh;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (long long)gridDim.x * blockDim.x) {
        long long t = q;
        const int j = (int)(t % W4); t /= W4;
        const int h = (int)(t % H); t /= H;
        const int d = (int)(t % D); t /= D;                     // t = b * C + c
        const long long row = t * 8 + (d & 1) * 4 + (h & 1) * 2;
        const long long off = row * Vh + ((long long)(d >> 1) * Hh + (h >> 1)) * Wh + 2 * j;
        if (TO_DEPTH) {
            const typename Q::V4 v = __ldcs(reinterpret_cast<const typename Q::V4*>(in) + q);
            *reinterpret_cast<typename Q::V2*>(out + off) = Q::even(v);
            *reinterpret_cast<typename Q::V2*>(out + off + Vh) = Q::odd(v);
        } else {
            const typename Q::V2 a = __ldcs(reinterpret_cast<const typename Q::V2*>(in + off)),
                                 b = __ldcs(reinterpret_cast<const typename Q::V2*>(in + off + Vh));
            reinterpret_cast<typename Q::V4*>(out)[q] = Q::join(a, b);
        }
    }
}


// ---- 3x3x3 stem convolution, few input channels -> 32 output channels, padding 1 ---------------------------------------
// (the Swin Factorizer's stem, reference factorizer/factorizer.py:139-140: 4 -> 32 channels at full resolution; the
// library's fp32 implicit-GEMM kernel takes 0.98 ms at 128^3 for 7.2 GFMA).  A thread owns 4 consecutive voxels along W
// and all 32 outputs (64 float2 accumulators); per input row it loads one float4 and its two neighbours, per tap it
// reads the 32 weights as 8 broadcast LDS.128 and issues 64 FFMA2 (weight broadcast x voxel pair).  x (TI) and y (TO) are
// fp32 or bf16; weights, bias and sums are fp32, and a bf16 y is the one rounding of the sum.
__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld4(const bf16* p) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xffff0000u));
}
__device__ __forceinline__ float ld1(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld1(const bf16* p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(bf16* p, float4 v) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const unsigned int*>(&a), *reinterpret_cast<const unsigned int*>(&b));
}

template <int CIN, typename TI, typename TO>
__global__ void __launch_bounds__(128, 2) conv3_stem_fwd(const TI* __restrict__ x, const float* __restrict__ wgt, const float* __restrict__ bias,
                                                         TO* __restrict__ y, int D, int H, int W, long long total4) {
    constexpr int CO = 32;
    __shared__ __align__(16) float ws[CIN * 27 * CO];          // [(ci, kd, kh, kw)][o]
    __shared__ float bs[CO];
    for (int i = threadIdx.x; i < CIN * 27 * CO; i += blockDim.x) {
        const int o = i % CO, tap = i / CO;
        ws[i] = wgt[o * CIN * 27 + tap];
    }
    for (int o = threadIdx.x; o < CO; o += blockDim.x) bs[o] = bias ? bias[o] : 0.f;
    __syncthreads();
    const int W4 = W >> 2;
    const long long vox = (long long)D * H * W;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (long long)gridDim.x * blockDim.x) {
        long long t = q;
        const int j = (int)(t % W4); t /= W4;
        const int h = (int)(t % H); t /= H;
        const int d = (int)(t % D); t /= D;                     // t = batch index
        const int w0 = 4 * j;
        float2 acc[CO][2];
#pragma unroll
        for (int o = 0; o < CO; ++o) acc[o][0] = acc[o][1] = make_float2(bs[o], bs[o]);
        const TI* xb = x + t * CIN * vox;
        // input row r = (ci, kd, kh): float4 of the thread's 4 voxels and the two neighbours; rows outside the volume are zero.
        // The next row is fetched before the current one is used (the loop is not unrolled: 192 FFMA2 per row).
        auto fetch = [&](int r, float4& c, float& lft, float& rgt) {
            const int ci = r / 9, kd = (r % 9) / 3, kh = r % 3;
            const int dd = d + kd - 1, hh = h + kh - 1;
            if (r >= CIN * 9 || dd < 0 || dd >= D || hh < 0 || hh >= H) {
                c = make_float4(0.f, 0.f, 0.f, 0.f); lft = rgt = 0.f;
                return;
            }
            const TI* row = xb + ci * vox + ((long long)dd * H + hh) * W + w0;
            c = ld4(row);
            lft = w0 > 0 ? ld1(row - 1) : 0.f;
            rgt = w0 + 4 < W ? ld1(row + 4) : 0.f;
        };
        float4 c, cn;
        float lft, rgt, lftn, rgtn;
        fetch(0, c, lft, rgt);
#pragma unroll 1
        for (int r = 0; r < CIN * 9; ++r) {
            fetch(r + 1, cn, lftn, rgtn);
            const float2 p[3][2] = {{make_float2(lft, c.x), make_float2(c.y, c.z)},
                                    {make_float2(c.x, c.y), make_float2(c.z, c.w)},
                                    {make_float2(c.y, c.z), make_float2(c.w, rgt)}};
            const float4* wr = reinterpret_cast<const float4*>(ws + r * 3 * CO);
#pragma unroll
            for (int kw = 0; kw < 3; ++kw)
#pragma unroll
                for (int o4 = 0; o4 < CO / 4; ++o4) {
                    const float4 wv = wr[kw * (CO / 4) + o4];
                    const float wa[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        acc[4 * o4 + e][0] = fma2(make_float2(wa[e], wa[e]), p[kw][0], acc[4 * o4 + e][0]);
                        acc[4 * o4 + e][1] = fma2(make_float2(wa[e], wa[e]), p[kw][1], acc[4 * o4 + e][1]);
                    }
                }
            c = cn; lft = lftn; rgt = rgtn;
        }
        TO* yo = y + t * CO * vox + ((long long)d * H + h) * W + w0;
#pragma unroll
        for (int o = 0; o < CO; ++o) st4(yo + o * vox, make_float4(acc[o][0].x, acc[o][0].y, acc[o][1].x, acc[o][1].y));
    }
}

// the kernels above move float4 (and cp.async 16-byte) words of the caller's buffers
bool unaligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) != 0; }

template <typename T>
int space_depth2_launch(const void* in, void* out, int64_t batch, int32_t channels, int32_t D, int32_t H, int32_t W, int32_t to_depth,
                        void* stream) {
    if (batch < 0 || channels <= 0) return fail(FZ_ERR_INVALID, "space/depth: bad sizes");
    if (!fz_space_depth2_supported(D, H, W))
        return fail(FZ_ERR_UNSUPPORTED, "space/depth kernel needs even D, H and W divisible by 4 (got %d x %d x %d)", D, H, W);
    if (batch == 0) return FZ_OK;
    if (!in || !out) return fail(FZ_ERR_INVALID, "space/depth: null buffer");
    if (unaligned16(in) || unaligned16(out)) return fail(FZ_ERR_UNSUPPORTED, "space/depth kernel needs 16-byte aligned buffers");
    const long long total4 = (long long)batch * channels * D * H * (W / 4);
    const int sms = num_sms();
    long long blocks = (total4 + 255) / 256;
    if (blocks > 16LL * sms) blocks = 16LL * sms;
    cudaStream_t st = (cudaStream_t)stream;
    const T* i = static_cast<const T*>(in);
    T* o = static_cast<T*>(out);
    if (to_depth) space_depth2<T, true><<<(unsigned)blocks, 256, 0, st>>>(i, o, total4, channels, D, H, W / 4);
    else space_depth2<T, false><<<(unsigned)blocks, 256, 0, st>>>(i, o, total4, channels, D, H, W / 4);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

template <typename TI, typename TO>
int stem_forward_launch(const void* x, const float* weight, const float* bias, void* y, int64_t batch, int32_t cin, int32_t cout, int32_t D,
                        int32_t H, int32_t W, void* stream) {
    if (batch < 0) return fail(FZ_ERR_INVALID, "stem convolution: bad batch");
    if (!fz_conv3d_stem_supported(cin, cout, D, H, W))
        return fail(FZ_ERR_UNSUPPORTED, "stem convolution kernel handles 1..4 -> 32 channels, W divisible by 4 (got %d -> %d, W = %d)", cin, cout, W);
    if (batch == 0) return FZ_OK;
    if (!x || !weight || !y) return fail(FZ_ERR_INVALID, "stem convolution: null buffer");
    if (unaligned16(x) || unaligned16(y)) return fail(FZ_ERR_UNSUPPORTED, "stem convolution kernel needs 16-byte aligned x and y");
    const long long total4 = (long long)batch * D * H * (W / 4);
    const int sms = num_sms();
    long long blocks = (total4 + 127) / 128;
    if (blocks > 16LL * sms) blocks = 16LL * sms;
    cudaStream_t st = (cudaStream_t)stream;
    const TI* xi = static_cast<const TI*>(x);
    TO* yo = static_cast<TO*>(y);
    switch (cin) {
        case 1: conv3_stem_fwd<1, TI, TO><<<(unsigned)blocks, 128, 0, st>>>(xi, weight, bias, yo, D, H, W, total4); break;
        case 2: conv3_stem_fwd<2, TI, TO><<<(unsigned)blocks, 128, 0, st>>>(xi, weight, bias, yo, D, H, W, total4); break;
        case 3: conv3_stem_fwd<3, TI, TO><<<(unsigned)blocks, 128, 0, st>>>(xi, weight, bias, yo, D, H, W, total4); break;
        default: conv3_stem_fwd<4, TI, TO><<<(unsigned)blocks, 128, 0, st>>>(xi, weight, bias, yo, D, H, W, total4); break;
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // namespace
}  // namespace fz

using namespace fz;

extern "C" {

int fz_linear_wgrad_supported(int32_t cout, int32_t cin, int64_t voxels) {
    return cout > 0 && cin > 0 && cout <= 32 * 65535 && cin <= 32 * 65535 && voxels > 0 && voxels % 4 == 0;
}

int fz_linear_wgrad(const float* dy, const float* x, float* dW, float* db, int64_t batch, int32_t cout, int32_t cin, int64_t voxels,
                    void* stream) {
    if (batch < 0 || cout <= 0 || cin <= 0 || voxels <= 0) return fail(FZ_ERR_INVALID, "linear wgrad: bad sizes");
    if (!fz_linear_wgrad_supported(cout, cin, voxels))
        return fail(FZ_ERR_UNSUPPORTED, "linear wgrad kernel needs a voxel count divisible by 4 (got %d x %d x %lld)", cout, cin,
                    (long long)voxels);
    if (!dW) return fail(FZ_ERR_INVALID, "linear wgrad: null dW");
    if (unaligned16(dy) || unaligned16(x)) return fail(FZ_ERR_UNSUPPORTED, "linear wgrad kernels need 16-byte aligned dy and x");
    cudaStream_t st = (cudaStream_t)stream;
    FZ_CUDA_CHECK(cudaMemsetAsync(dW, 0, sizeof(float) * (size_t)cout * cin, st));
    if (db) FZ_CUDA_CHECK(cudaMemsetAsync(db, 0, sizeof(float) * (size_t)cout, st));
    if (batch == 0) return FZ_OK;
    if (!dy || !x) return fail(FZ_ERR_INVALID, "linear wgrad: null buffer");
    // tensor-core path (csrc/fz_linear_tc.cu: TMA-fed K-major operands, 3xTF32) unless the calling thread asked for the FP32 pipe
    if ((tls().glue_mode & 2) && batch * voxels >= 4096 && linear_wgrad_tc_supported(dy, x, batch, cout, cin, voxels))
        return linear_wgrad_tc_launch(dy, x, dW, db, batch, cout, cin, voxels, st);
    const int sms = num_sms();
    // fewer voxels: the smaller CTAs of the 32 x 32 kernel spread better; a 32 x 128 block pays from 65 input rows on
    if ((cout >= 64 ? cin >= 64 : cin > 64) && batch * voxels >= 32768) {
        const int tps = (int)((voxels + kW2V - 1) / kW2V);
        const long long tiles = batch * tps;
        const bool wide = cout >= 64;                 // 64 x 64 blocks, else 32 x 128
        const int bo = wide ? (cout + 63) / 64 : (cout + 31) / 32, bi = wide ? (cin + 63) / 64 : (cin + 127) / 128;
        long long gx = (2LL * sms + bo * bi - 1) / (bo * bi);
        if (gx > tiles) gx = tiles;
        if (gx < 1) gx = 1;
        // two cp.async stages; the epilogue scratch (64.3 KB) aliases them
        const size_t smem = sizeof(float) * 2 * (wide ? 128 : 160) * kW2RS;
        static SmemConfig cfg21, cfg12;
        if (wide) {
            FZ_CUDA_CHECK(cfg21.ensure(linear_wgrad64<2, 1>, smem));
            linear_wgrad64<2, 1><<<dim3((unsigned)gx, bo, bi), kW2T, smem, st>>>(dy, x, dW, db, cout, cin, voxels, tps, tiles);
        } else {
            FZ_CUDA_CHECK(cfg12.ensure(linear_wgrad64<1, 2>, smem));
            linear_wgrad64<1, 2><<<dim3((unsigned)gx, bo, bi), kW2T, smem, st>>>(dy, x, dW, db, cout, cin, voxels, tps, tiles);
        }
        FZ_LAUNCH_CHECK();
        return FZ_OK;
    }
    const int tps = (int)((voxels + kWV - 1) / kWV);
    const long long tiles = batch * tps;
    const int bo = (cout + 31) / 32, bi = (cin + 31) / 32;       // channel counts are padded with zero rows inside the kernel
    const int blocks = bo * bi;
    long long gx = (3LL * sms + blocks - 1) / blocks;
    if (gx > tiles) gx = tiles;
    if (gx < 1) gx = 1;
    const size_t smem = sizeof(float) * 2 * 32 * kWRS;          // 66.5 KB >= the 16.1 KB epilogue scratch
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(linear_wgrad, smem));
    linear_wgrad<<<dim3((unsigned)gx, bo, bi), kWT, smem, st>>>(dy, x, dW, db, cout, cin, voxels, tps, tiles);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int fz_linear_forward_supported(int32_t cout, int32_t cin, int64_t voxels) {
    return cout > 0 && cin > 0 && cin % 4 == 0 && voxels > 0 && voxels % 4 == 0 && voxels < (1LL << 31);
}

int fz_linear_forward(const float* x, const float* W, const float* bias, float* y, int64_t batch, int32_t cin, int32_t cout,
                      int64_t voxels, void* stream) {
    return fz_linear_forward_ex(x, W, bias, y, batch, cin, cout, voxels, FZ_EPILOGUE_NONE, 0, nullptr, nullptr, stream);
}

int fz_linear_forward_ex(const float* x, const float* W, const float* bias, float* y, int64_t batch, int32_t cin, int32_t cout,
                         int64_t voxels, int32_t epilogue, int32_t w_transposed, const float* aux, float* y2, void* stream) {
    tls().launches = 0;
    if (batch < 0 || cout <= 0 || cin <= 0 || voxels <= 0) return fail(FZ_ERR_INVALID, "linear forward: bad sizes");
    if (epilogue < FZ_EPILOGUE_NONE || epilogue > FZ_EPILOGUE_GELU_ONLY) return fail(FZ_ERR_INVALID, "linear forward: unknown epilogue %d", epilogue);
    if (batch == 0) return FZ_OK;
    if (!x || !W || !y) return fail(FZ_ERR_INVALID, "linear forward: null buffer");
    if (int e = cmap::check_epilogue("linear forward", epilogue, aux, y2)) return e;
    if (!fz_linear_forward_supported(cout, cin, voxels) || !linear_fwd_tc_supported(x, W, batch, cout, cin, voxels) ||
        (w_transposed && cout % 4))
        return fail(FZ_ERR_UNSUPPORTED, "linear forward kernel needs voxels and input channels (with a transposed weight: output "
                                        "channels too) divisible by 4 and 16-byte aligned buffers (got %d x %d x %lld)", cout, cin,
                    (long long)voxels);
    return linear_fwd_tc_launch(x, W, bias, y, aux, y2, epilogue, w_transposed != 0, batch, cout, cin, voxels, (cudaStream_t)stream);
}

int fz_space_depth2_supported(int32_t D, int32_t H, int32_t W) {
    return D > 0 && H > 0 && W > 0 && D % 2 == 0 && H % 2 == 0 && W % 4 == 0;
}

int fz_space_depth2(const float* in, float* out, int64_t batch, int32_t channels, int32_t D, int32_t H, int32_t W, int32_t to_depth,
                    void* stream) {
    return space_depth2_launch<float>(in, out, batch, channels, D, H, W, to_depth, stream);
}

int fz_space_depth2_bf16_supported(int32_t D, int32_t H, int32_t W) { return fz_space_depth2_supported(D, H, W); }

int fz_space_depth2_bf16(const void* in, void* out, int64_t batch, int32_t channels, int32_t D, int32_t H, int32_t W, int32_t to_depth,
                         void* stream) {
    return space_depth2_launch<bf16>(in, out, batch, channels, D, H, W, to_depth, stream);
}

int fz_conv3d_stem_supported(int32_t cin, int32_t cout, int32_t D, int32_t H, int32_t W) {
    return cin >= 1 && cin <= 4 && cout == 32 && D > 0 && H > 0 && W > 0 && W % 4 == 0;
}

int fz_conv3d_stem_forward(const float* x, const float* weight, const float* bias, float* y, int64_t batch, int32_t cin, int32_t cout,
                           int32_t D, int32_t H, int32_t W, void* stream) {
    return stem_forward_launch<float, float>(x, weight, bias, y, batch, cin, cout, D, H, W, stream);
}

int fz_conv3d_stem_forward_bf16(const void* x, int32_t x_dtype, const float* weight, const float* bias, void* y, int64_t batch, int32_t cin,
                                int32_t cout, int32_t D, int32_t H, int32_t W, void* stream) {
    if (x_dtype == FZ_DTYPE_F32) return stem_forward_launch<float, bf16>(x, weight, bias, y, batch, cin, cout, D, H, W, stream);
    if (x_dtype == FZ_DTYPE_BF16) return stem_forward_launch<bf16, bf16>(x, weight, bias, y, batch, cin, cout, D, H, W, stream);
    return fail(FZ_ERR_INVALID, "stem convolution: unknown x dtype %d", x_dtype);
}

}  // extern "C"
