// Pointwise glue of FactMixer / FactorizerBlock around the matricize+NMF core, for 32-channel blocks
// (SURVEY.md section 8(f) row 1; reference factorizer/factorizer.py:38,53,75-76, layers/norm.py:29-34,
// layers/linear.py:53-58, layers/mlp.py:54-60).  Four kernels, all fp32 on the FP32 pipe:
//
//   ln_linear_fwd     z   = W_in  LN1(x)                                  (norm1 + in_proj)
//   mixer_mlp_fwd     x1  = x + W_out m + b_out ;  out = x1 + W2 gelu(W1 LN2(x1) + b1) + b2
//                                                                         (out_proj + residual + norm2 + MLP + residual)
//   mlp_bwd           dx1 = dout + LN2'( W1^T (gelu'(h) . W2^T dout) ) and the gradients of LN2 / W1 / b1 / W2 / b2
//   linear_bwd<LN>    da  = W^T dy  [then through LN, plus a residual gradient], dW = dy a^T, db, d(gamma), d(beta)
//                                                                         (out_proj backward, and in_proj + norm1 backward)
//
// Layout: activations stay NCDHW = (batch, 32, voxels); one thread owns two neighbouring voxels and all 32
// channels of them in registers (float2 per channel: a warp reads 256 contiguous bytes per channel row).
// The small matrix-vector products read the weights from shared memory as broadcast LDS.128 (4 weights
// per load, stored input-major so 4 consecutive OUTPUTS are contiguous) and issue packed FFMA2 on output
// pairs: 8 LDS.128 + 32 FFMA2 per input channel and voxel pair, i.e. FP32-pipe bound, not LDS bound.
// Weight gradients are contractions over voxels: the two operands of a 512-voxel (256 for linear_bwd) tile are staged in
// shared memory as [row][voxel] (row stride 516 / 260 floats, so consecutive rows start 4 banks apart), every thread then
// accumulates a small register tile of dW over a slice of the voxels and writes it to its warp's scratch slice; owner
// threads add the slices into the per-CTA accumulator (fp32 atomics on shared memory are CAS loops on sm_100a), and the
// CTA adds its total to the global gradient once at the end (global fp32 atomics).
// Per-channel sums (bias / LayerNorm parameter gradients) use a transposing warp reduction (31 shuffles for 32 values).
// Every kernel here has a tensor-core twin (tcgen05 / TMEM, 3xTF32: fz_block_glue_fwd_tc.cu, fz_block_glue_lin_tc.cu,
// fz_block_glue_bwd_tc.cu), which is the default where its shape restrictions hold (hidden width 64 for the MLP backward,
// 32 or 64 for the forward); these FP32-pipe kernels take every other hidden width and fz_set_glue_mode(0).
#include "fz_device.cuh"
#include "fz_internal.cuh"

namespace fz {
namespace {

constexpr int kC = 32;            // channels the kernels are written for
constexpr int kMaxHidden = 64;    // hidden units per launch of the backward kernel (shared memory); wider MLPs go slice by slice
constexpr int kTT = 256;          // threads per CTA of the tiled (staging) kernels
constexpr int kTV = 2 * kTT;      // voxels per tile
constexpr int kRS = kTV + 4;      // staged row stride in floats: = 4 (mod 32)

// acc{0,1}[k] += sum_c W[c][2k..2k+1] * in[c].{x,y}: NOUT outputs for the two voxels of a thread.
// Wt points at the first of the NOUT outputs of input row 0; rows are ldw floats apart (shared memory,
// 16-byte aligned).
template <int CIN, int NOUT>
__device__ __forceinline__ void matvec(const float* __restrict__ Wt, int ldw, const f2 (&in)[CIN], f2 (&acc0)[NOUT / 2],
                                       f2 (&acc1)[NOUT / 2]) {
#pragma unroll
    for (int c = 0; c < CIN; ++c) {
        const f2 x0 = dup(in[c].x), x1 = dup(in[c].y);
#pragma unroll
        for (int q = 0; q < NOUT / 4; ++q) {
            const float4 w = *reinterpret_cast<const float4*>(Wt + c * ldw + 4 * q);
            const f2 wa = make_float2(w.x, w.y), wb = make_float2(w.z, w.w);
            acc0[2 * q] = fma2(wa, x0, acc0[2 * q]);
            acc0[2 * q + 1] = fma2(wb, x0, acc0[2 * q + 1]);
            acc1[2 * q] = fma2(wa, x1, acc1[2 * q]);
            acc1[2 * q + 1] = fma2(wb, x1, acc1[2 * q + 1]);
        }
    }
}

// same with the input read from the thread's own column of a staged tile (rows kRS apart)
template <int CIN, int NOUT>
__device__ __forceinline__ void matvec_staged(const float* __restrict__ Wt, int ldw, const float* __restrict__ col,
                                              f2 (&acc0)[NOUT / 2], f2 (&acc1)[NOUT / 2]) {
#pragma unroll
    for (int c = 0; c < CIN; ++c) {
        const f2 in = *reinterpret_cast<const f2*>(col + c * kRS);
        const f2 x0 = dup(in.x), x1 = dup(in.y);
#pragma unroll
        for (int q = 0; q < NOUT / 4; ++q) {
            const float4 w = *reinterpret_cast<const float4*>(Wt + c * ldw + 4 * q);
            const f2 wa = make_float2(w.x, w.y), wb = make_float2(w.z, w.w);
            acc0[2 * q] = fma2(wa, x0, acc0[2 * q]);
            acc0[2 * q + 1] = fma2(wb, x0, acc0[2 * q + 1]);
            acc1[2 * q] = fma2(wa, x1, acc1[2 * q]);
            acc1[2 * q + 1] = fma2(wb, x1, acc1[2 * q + 1]);
        }
    }
}

// value of output c for (voxel 0, voxel 1) from the pair-of-outputs accumulators
template <int N>
__device__ __forceinline__ f2 unpair(const f2 (&a0)[N / 2], const f2 (&a1)[N / 2], int c) {
    return (c & 1) ? make_float2(a0[c >> 1].y, a1[c >> 1].y) : make_float2(a0[c >> 1].x, a1[c >> 1].x);
}

// v <- (v - mean) * rstd over the channel axis, separately for the two voxels; returns rstd
template <int C>
__device__ __forceinline__ f2 normalize(f2 (&v)[C], float eps) {
    f2 sum = make_float2(0.f, 0.f);
#pragma unroll
    for (int c = 0; c < C; ++c) { sum.x += v[c].x; sum.y += v[c].y; }
    const f2 mean = make_float2(sum.x * (1.f / C), sum.y * (1.f / C));
    f2 var = make_float2(0.f, 0.f);
#pragma unroll
    for (int c = 0; c < C; ++c) {
        v[c].x -= mean.x; v[c].y -= mean.y;
        var.x = fmaf(v[c].x, v[c].x, var.x); var.y = fmaf(v[c].y, v[c].y, var.y);
    }
    const f2 rstd = make_float2(rsqrtf(var.x * (1.f / C) + eps), rsqrtf(var.y * (1.f / C) + eps));
#pragma unroll
    for (int c = 0; c < C; ++c) { v[c].x *= rstd.x; v[c].y *= rstd.y; }
    return rstd;
}

template <int C>
__device__ __forceinline__ void load_cols(const float* __restrict__ p, long long cstride, bool valid, f2 (&r)[C]) {
#pragma unroll
    for (int c = 0; c < C; ++c) r[c] = valid ? __ldg(reinterpret_cast<const f2*>(p + c * cstride)) : make_float2(0.f, 0.f);
}

// ------------------------------------------------------------------------------------------------
// z = W LN(x)   (norm1 + in_proj; bias-free projection, factorizer.py:26)
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(128, 3) ln_linear_fwd(const float* __restrict__ x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, const float* __restrict__ W,
                                                        float* __restrict__ y, long long pps, long long total_pairs, float eps) {
    __shared__ __align__(16) float Wt[C * C];  // [c][o]
    __shared__ float gs[C], bs[C];
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) Wt[(i % C) * C + i / C] = W[i];
    for (int c = threadIdx.x; c < C; c += blockDim.x) { gs[c] = gamma ? gamma[c] : 1.f; bs[c] = beta ? beta[c] : 0.f; }
    __syncthreads();
    const long long vox = 2 * pps;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total_pairs; p += (long long)gridDim.x * blockDim.x) {
        const long long b = p / pps, v = p - b * pps;
        const long long base = b * C * vox + 2 * v;
        f2 n[C];
        load_cols<C>(x + base, vox, true, n);
        normalize<C>(n, eps);
#pragma unroll
        for (int c = 0; c < C; ++c) { n[c].x = fmaf(n[c].x, gs[c], bs[c]); n[c].y = fmaf(n[c].y, gs[c], bs[c]); }
        f2 a0[C / 2], a1[C / 2];
#pragma unroll
        for (int k = 0; k < C / 2; ++k) a0[k] = a1[k] = make_float2(0.f, 0.f);
        matvec<C, C>(Wt, C, n, a0, a1);
#pragma unroll
        for (int o = 0; o < C; ++o) *reinterpret_cast<f2*>(y + base + o * vox) = unpair<C>(a0, a1, o);
    }
}

// ------------------------------------------------------------------------------------------------
// x1 = x + W_out m + b_out ; out = x1 + W2 gelu(W1 LN(x1) + b1) + b2
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(128, 2) mixer_mlp_fwd(const float* __restrict__ x, const float* __restrict__ m,
                                                        const float* __restrict__ Wout, const float* __restrict__ bout,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        const float* __restrict__ W1, const float* __restrict__ b1,
                                                        const float* __restrict__ W2, const float* __restrict__ b2,
                                                        float* __restrict__ x1_out, float* __restrict__ out, int HID,
                                                        long long pps, long long total_pairs, float eps) {
    extern __shared__ __align__(16) float sm[];
    float* WoT = sm;                 // [c][o]
    float* W1T = WoT + C * C;        // [c][j]
    float* W2T = W1T + C * HID;      // [j][o]
    float* b1s = W2T + HID * C;      // [j]
    float* bos = b1s + HID;          // [o]
    float* b2s = bos + C;
    float* gs = b2s + C;
    float* bs = gs + C;
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) WoT[(i % C) * C + i / C] = Wout[i];
    for (int i = threadIdx.x; i < HID * C; i += blockDim.x) {
        W1T[(i % C) * HID + i / C] = W1[i];      // W1 [j][c]
        W2T[(i % HID) * C + i / HID] = W2[i];    // W2 [o][j]
    }
    for (int j = threadIdx.x; j < HID; j += blockDim.x) b1s[j] = b1 ? b1[j] : 0.f;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        bos[c] = bout ? bout[c] : 0.f; b2s[c] = b2 ? b2[c] : 0.f;
        gs[c] = gamma ? gamma[c] : 1.f; bs[c] = beta ? beta[c] : 0.f;
    }
    __syncthreads();
    const long long vox = 2 * pps;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total_pairs; p += (long long)gridDim.x * blockDim.x) {
        const long long b = p / pps, v = p - b * pps;
        const long long base = b * C * vox + 2 * v;
        f2 n[C];
        f2 o0[C / 2], o1[C / 2];
        {
            f2 mm[C];
            load_cols<C>(m + base, vox, true, mm);
#pragma unroll
            for (int k = 0; k < C / 2; ++k) { o0[k] = o1[k] = make_float2(bos[2 * k], bos[2 * k + 1]); }
            matvec<C, C>(WoT, C, mm, o0, o1);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const f2 xv = __ldg(reinterpret_cast<const f2*>(x + base + c * vox));
            const f2 pr = unpair<C>(o0, o1, c);
            n[c] = make_float2(xv.x + pr.x, xv.y + pr.y);
            if (x1_out) *reinterpret_cast<f2*>(x1_out + base + c * vox) = n[c];
        }
        // second residual accumulators start from x1 + b2
#pragma unroll
        for (int k = 0; k < C / 2; ++k) {
            o0[k] = make_float2(n[2 * k].x + b2s[2 * k], n[2 * k + 1].x + b2s[2 * k + 1]);
            o1[k] = make_float2(n[2 * k].y + b2s[2 * k], n[2 * k + 1].y + b2s[2 * k + 1]);
        }
        normalize<C>(n, eps);
#pragma unroll
        for (int c = 0; c < C; ++c) { n[c].x = fmaf(n[c].x, gs[c], bs[c]); n[c].y = fmaf(n[c].y, gs[c], bs[c]); }
#pragma unroll 1
        for (int j0 = 0; j0 < HID; j0 += 8) {
            f2 h0[4], h1[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) h0[k] = h1[k] = make_float2(b1s[j0 + 2 * k], b1s[j0 + 2 * k + 1]);
            matvec<C, 8>(W1T + j0, HID, n, h0, h1);
            f2 g[8];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const f2 ga = gelu2(h0[k]), gb = gelu2(h1[k]);          // (hidden 2k, 2k+1) of voxel 0 / voxel 1
                g[2 * k] = make_float2(ga.x, gb.x);
                g[2 * k + 1] = make_float2(ga.y, gb.y);
            }
            matvec<8, C>(W2T + j0 * C, C, g, o0, o1);
        }
#pragma unroll
        for (int o = 0; o < C; ++o) *reinterpret_cast<f2*>(out + base + o * vox) = unpair<C>(o0, o1, o);
    }
}

// ------------------------------------------------------------------------------------------------
// weight-gradient tiles
// ------------------------------------------------------------------------------------------------
// scr[(i*4+k)*32 + lane] = this warp's share of sum_v SA[ro+4i][v] * SB[co+8k][v], ro = lane&3, co = lane>>2:
// a 32x32 outer-product sum; warp w takes every NW-th float4 column and writes to its own scratch slice (fp32
// atomics on shared memory are compare-and-swap loops on this architecture, hence the two-step reduction).
template <int TV, int NW>
__device__ __forceinline__ void wgrad_32x32(const float* __restrict__ SA, const float* __restrict__ SB, float* __restrict__ scr, int tid) {
    constexpr int RS = TV + 4;
    const int lane = tid & 31, grp = tid >> 5, ro = lane & 3, co = lane >> 2;
    f2 a[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) a[i][k] = make_float2(0.f, 0.f);
#pragma unroll 1
    for (int it = 0; it < TV / 4 / NW; ++it) {
        const int v = (it * NW + grp) * 4;
        float4 B[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) B[k] = *reinterpret_cast<const float4*>(SB + (co + 8 * k) * RS + v);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 A = *reinterpret_cast<const float4*>(SA + (ro + 4 * i) * RS + v);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                a[i][k] = fma2(make_float2(A.x, A.y), make_float2(B[k].x, B[k].y), a[i][k]);
                a[i][k] = fma2(make_float2(A.z, A.w), make_float2(B[k].z, B[k].w), a[i][k]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) scr[(i * 4 + k) * 32 + lane] = a[i][k].x + a[i][k].y;
}

// scr[(i*4+k)*16 + tt] = this warp's share of sum_v SA[jh*4+i][v] * SB[rt+8k][v], tt = lane&15, jh = tt>>3,
// rt = tt&7: an 8x32 outer-product sum; 16 half-warps each take every 16th float4 column.
__device__ __forceinline__ void wgrad_8x32(const float* __restrict__ SA, const float* __restrict__ SB, float* __restrict__ scr, int tid) {
    const int lane = tid & 31, tt = lane & 15, jh = tt >> 3, rt = tt & 7, grp = (tid >> 5) * 2 + (lane >> 4);
    f2 a[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) a[i][k] = make_float2(0.f, 0.f);
#pragma unroll 2
    for (int it = 0; it < kTV / 4 / 16; ++it) {
        const int v = (it * 16 + grp) * 4;
        float4 B[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) B[k] = *reinterpret_cast<const float4*>(SB + (rt + 8 * k) * kRS + v);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 A = *reinterpret_cast<const float4*>(SA + (jh * 4 + i) * kRS + v);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                a[i][k] = fma2(make_float2(A.x, A.y), make_float2(B[k].x, B[k].y), a[i][k]);
                a[i][k] = fma2(make_float2(A.z, A.w), make_float2(B[k].z, B[k].w), a[i][k]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float s = a[i][k].x + a[i][k].y;
            s += __shfl_xor_sync(0xffffffffu, s, 16);
            if (lane < 16) scr[(i * 4 + k) * 16 + tt] = s;
        }
}

constexpr int kWarps = kTT / 32;
constexpr int kScrLin = kC * kC + 3 * kC;   // per-warp scratch of linear_bwd: dW partials | db | dgamma | dbeta
constexpr int kScrMlp = 2 * 256 + 8;        // per-warp scratch of mlp_bwd per 8 hidden units: dW2 | Q | db1
constexpr int kScrMlpV = 3 * kC;            // ... and per tile: db2 | dgamma | dbeta

// ------------------------------------------------------------------------------------------------
// backward of y = W n(a) (+ b), n = LayerNorm or identity:
//   da = W^T dy            (LN: dx = resid + LN'(da))
//   dW = sum_v dy n(a)^T,  db = sum_v dy,  d(gamma) = sum_v da . a_hat,  d(beta) = sum_v da
// ------------------------------------------------------------------------------------------------
// 128 threads / 256-voxel tiles, two CTAs per SM: one loads its tile while the other computes
constexpr int kLT = 128, kLV = 2 * kLT, kLRS = kLV + 4, kLWarps = kLT / 32;

template <int C, bool LN>
__global__ void __launch_bounds__(kLT, 2) linear_bwd(const float* __restrict__ dy, const float* __restrict__ a,
                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     const float* __restrict__ W, const float* __restrict__ resid,
                                                     float* __restrict__ da, float* __restrict__ dW, float* __restrict__ db,
                                                     float* __restrict__ dgamma, float* __restrict__ dbeta, long long vox,
                                                     int tiles_per_sample, long long total_tiles, float eps) {
    extern __shared__ __align__(16) float sm[];
    float* Ws = sm;                    // [o][c] as stored: input o, outputs c
    float* gs = Ws + C * C;
    float* bs = gs + C;
    float* accW = bs + C;              // [(i*4+k)][lane]
    float* accv = accW + C * C;        // db | dgamma | dbeta
    float* scr = accv + 3 * C;         // [warp][kScrLin]
    float* SA = scr + kLWarps * kScrLin;  // dy  [o][v]
    float* SB = SA + C * kLRS;          // n(a) [c][v]
    const int tid = threadIdx.x, lane = tid & 31;
    float* scr_w = scr + (tid >> 5) * kScrLin;
    for (int i = tid; i < C * C; i += kLT) { Ws[i] = W[i]; accW[i] = 0.f; }
    for (int c = tid; c < C; c += kLT) { gs[c] = gamma ? gamma[c] : 1.f; bs[c] = beta ? beta[c] : 0.f; }
    for (int c = tid; c < 3 * C; c += kLT) accv[c] = 0.f;
    __syncthreads();
    for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const long long b = tile / tiles_per_sample;
        const long long pv = (tile - b * tiles_per_sample) * kLT + tid;
        const bool valid = 2 * pv < vox;
        const long long base = b * C * vox + 2 * pv;
        f2 d0[C / 2], d1[C / 2];
        float r_db, r_dg = 0.f, r_dbeta = 0.f;
        {
            f2 g[C];
            load_cols<C>(dy + base, vox, valid, g);
#pragma unroll
            for (int o = 0; o < C; ++o) *reinterpret_cast<f2*>(SA + o * kLRS + 2 * tid) = g[o];
            {
                float s[C];
#pragma unroll
                for (int o = 0; o < C; ++o) s[o] = g[o].x + g[o].y;
                r_db = warp_vec_sum<C>(s, lane);
            }
#pragma unroll
            for (int k = 0; k < C / 2; ++k) d0[k] = d1[k] = make_float2(0.f, 0.f);
            matvec<C, C>(Ws, C, g, d0, d1);
        }
        f2 av[C];
        load_cols<C>(a + base, vox, valid, av);
        if (LN) {
            const f2 rstd = normalize<C>(av, eps);
            f2 m1 = make_float2(0.f, 0.f), m2 = make_float2(0.f, 0.f);
            float sg[C], sb[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                *reinterpret_cast<f2*>(SB + c * kLRS + 2 * tid) = make_float2(fmaf(av[c].x, gs[c], bs[c]), fmaf(av[c].y, gs[c], bs[c]));
                const f2 d = unpair<C>(d0, d1, c);
                sg[c] = fmaf(d.x, av[c].x, d.y * av[c].y);
                sb[c] = d.x + d.y;
                const f2 t = make_float2(d.x * gs[c], d.y * gs[c]);
                m1.x += t.x; m1.y += t.y;
                m2.x = fmaf(t.x, av[c].x, m2.x); m2.y = fmaf(t.y, av[c].y, m2.y);
            }
            m1.x *= (1.f / C); m1.y *= (1.f / C); m2.x *= (1.f / C); m2.y *= (1.f / C);
            if (valid) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const f2 d = unpair<C>(d0, d1, c);
                    f2 o;
                    o.x = rstd.x * (d.x * gs[c] - m1.x - av[c].x * m2.x);
                    o.y = rstd.y * (d.y * gs[c] - m1.y - av[c].y * m2.y);
                    if (resid) { const f2 r = __ldg(reinterpret_cast<const f2*>(resid + base + c * vox)); o.x += r.x; o.y += r.y; }
                    *reinterpret_cast<f2*>(da + base + c * vox) = o;
                }
            }
            r_dg = warp_vec_sum<C>(sg, lane);
            r_dbeta = warp_vec_sum<C>(sb, lane);
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                *reinterpret_cast<f2*>(SB + c * kLRS + 2 * tid) = av[c];
                if (valid) *reinterpret_cast<f2*>(da + base + c * vox) = unpair<C>(d0, d1, c);
            }
        }
        __syncthreads();   // tile staged; the previous tile's scratch has been consumed
        wgrad_32x32<kLV, kLWarps>(SA, SB, scr_w, tid);
        scr_w[C * C + lane] = r_db;
        scr_w[C * C + C + lane] = r_dg;
        scr_w[C * C + 2 * C + lane] = r_dbeta;
        __syncthreads();
        for (int o = tid; o < kScrLin; o += kLT) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < kLWarps; ++w) t += scr[w * kScrLin + o];
            accW[o] += t;      // accv follows accW in shared memory
        }
    }
    __syncthreads();
    // accW[(i*4+k)*32 + lane] is dW[(lane&3) + 4i][(lane>>2) + 8k]
    for (int i = tid; i < C * C; i += kLT) {
        const int e = i >> 5, l = i & 31;
        atomicAdd(dW + ((l & 3) + 4 * (e >> 2)) * C + (l >> 2) + 8 * (e & 3), accW[i]);
    }
    for (int c = tid; c < C; c += kLT) {
        if (db) atomicAdd(db + c, accv[c]);
        if (LN && dgamma) atomicAdd(dgamma + c, accv[C + c]);
        if (LN && dbeta) atomicAdd(dbeta + c, accv[2 * C + c]);
    }
}

// ------------------------------------------------------------------------------------------------
// backward of out = x1 + W2 gelu(W1 LN(x1) + b1) + b2 with respect to x1 and every parameter
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(kTT, 1) mlp_bwd(const float* __restrict__ x1, const float* __restrict__ dout,
                                                  const float* __restrict__ gamma, const float* __restrict__ beta,
                                                  const float* __restrict__ W1, const float* __restrict__ b1,
                                                  const float* __restrict__ W2, float* __restrict__ dx1,
                                                  float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ dW1,
                                                  float* __restrict__ db1, float* __restrict__ dW2, float* __restrict__ db2, int HID,
                                                  int ldw2, int accumulate, long long vox, int tiles_per_sample,
                                                  long long total_tiles, float eps) {
    // HID: the hidden units this launch covers (a slice of at most kMaxHidden; W1 / b1 / dW1 / db1 point at the
    // slice's first row, W2 / dW2 at its first column, rows ldw2 apart).  accumulate: dx1 already holds
    // dout + the other slices' contributions (the backward is additive over hidden units).
    extern __shared__ __align__(16) float sm[];
    // weights: W1T has gamma folded in ([c][j] = W1[j][c] gamma[c]) and b1f = b1 + W1 beta, so the hidden
    // pre-activation is W1T^T a_hat + b1f with a_hat the normalised (pre-affine) input kept in registers
    float* W1T = sm;                    // [c][j]
    float* W1s = W1T + C * HID;         // [j][c] as stored (input j, outputs c)
    float* W2s = W1s + HID * C;         // [o][j] as stored (input o, outputs j)
    float* b1f = W2s + C * HID;         // [j]
    float* gs = b1f + HID;
    float* bs = gs + C;
    float* accQ = bs + C;               // sum_v dh a_hat^T, [j/8][(i*4+k)*16 + tt]
    float* accW2 = accQ + HID * C;      // sum_v g dout^T, same tiling
    float* accb1 = accW2 + HID * C;     // [j]
    float* accv = accb1 + HID;          // db2 | dgamma | dbeta
    float* scr = accv + 3 * C;          // [warp][kScrMlp + kScrMlpV]
    float* Snh = scr + kWarps * (kScrMlp + kScrMlpV);   // a_hat [c][v]
    float* Sdo = Snh + C * kRS;         // dout  [o][v]
    float* Sg = Sdo + C * kRS;          // gelu(h) of the current 8 hidden units [j][v]
    float* Sdh = Sg + 8 * kRS;          // dh of the current 8 hidden units
    const int tid = threadIdx.x, lane = tid & 31;
    float* scr_w = scr + (tid >> 5) * (kScrMlp + kScrMlpV);
    for (int c = tid; c < C; c += kTT) { gs[c] = gamma ? gamma[c] : 1.f; bs[c] = beta ? beta[c] : 0.f; }
    for (int c = tid; c < 3 * C; c += kTT) accv[c] = 0.f;
    for (int j = tid; j < HID; j += kTT) accb1[j] = 0.f;
    __syncthreads();
    for (int i = tid; i < HID * C; i += kTT) {
        const int j = i / C, c = i - j * C;
        const float w = W1[i];
        W1s[i] = w;
        W1T[c * HID + j] = w * gs[c];
        W2s[i] = W2[(i / HID) * ldw2 + i % HID];
        accQ[i] = 0.f;
        accW2[i] = 0.f;
    }
    for (int j = tid; j < HID; j += kTT) {
        float s = b1 ? b1[j] : 0.f;
        for (int c = 0; c < C; ++c) s = fmaf(W1[j * C + c], bs[c], s);
        b1f[j] = s;
    }
    __syncthreads();
    for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const long long b = tile / tiles_per_sample;
        const long long pv = (tile - b * tiles_per_sample) * kTT + tid;
        const bool valid = 2 * pv < vox;
        const long long base = b * C * vox + 2 * pv;
        const float* mycol_do = Sdo + 2 * tid;
        f2 nh[C];
        load_cols<C>(x1 + base, vox, valid, nh);
        const f2 rstd = normalize<C>(nh, eps);
#pragma unroll
        for (int c = 0; c < C; ++c) *reinterpret_cast<f2*>(Snh + c * kRS + 2 * tid) = nh[c];
#pragma unroll
        for (int o = 0; o < C; ++o)
            *reinterpret_cast<f2*>(Sdo + o * kRS + 2 * tid) =
                valid ? __ldg(reinterpret_cast<const f2*>(dout + base + o * vox)) : make_float2(0.f, 0.f);
        f2 dn0[C / 2], dn1[C / 2];   // d(LN output) = W1^T dh
#pragma unroll
        for (int k = 0; k < C / 2; ++k) dn0[k] = dn1[k] = make_float2(0.f, 0.f);
#pragma unroll 1
        for (int j0 = 0; j0 < HID; j0 += 8) {
            f2 h0[4], h1[4], q0[4], q1[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                h0[k] = h1[k] = make_float2(b1f[j0 + 2 * k], b1f[j0 + 2 * k + 1]);
                q0[k] = q1[k] = make_float2(0.f, 0.f);
            }
            matvec<C, 8>(W1T + j0, HID, nh, h0, h1);                      // h  = W1 LN(x1) + b1
            matvec_staged<C, 8>(W2s + j0, HID, mycol_do, q0, q1);         // dg = W2^T dout
            f2 dh[8];
            float sb[8];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                f2 g0, gp0, g1, gp1;                                     // (hidden 2k, 2k+1) of voxel 0 / voxel 1
                gelu_grad2(h0[k], g0, gp0);
                gelu_grad2(h1[k], g1, gp1);
                const f2 ga = make_float2(g0.x, g1.x), gb = make_float2(g0.y, g1.y);
                dh[2 * k] = make_float2(q0[k].x * gp0.x, q1[k].x * gp1.x);
                dh[2 * k + 1] = make_float2(q0[k].y * gp0.y, q1[k].y * gp1.y);
                *reinterpret_cast<f2*>(Sg + (2 * k) * kRS + 2 * tid) = ga;
                *reinterpret_cast<f2*>(Sg + (2 * k + 1) * kRS + 2 * tid) = gb;
                *reinterpret_cast<f2*>(Sdh + (2 * k) * kRS + 2 * tid) = dh[2 * k];
                *reinterpret_cast<f2*>(Sdh + (2 * k + 1) * kRS + 2 * tid) = dh[2 * k + 1];
                sb[2 * k] = dh[2 * k].x + dh[2 * k].y;
                sb[2 * k + 1] = dh[2 * k + 1].x + dh[2 * k + 1].y;
            }
            const float r = warp_vec_sum<8>(sb, lane);
            matvec<8, C>(W1s + j0 * C, C, dh, dn0, dn1);
            __syncthreads();   // the 8 hidden units are staged; the previous scratch has been consumed
            wgrad_8x32(Sg, Sdo, scr_w, tid);
            wgrad_8x32(Sdh, Snh, scr_w + 256, tid);
            if ((lane & 3) == 0) scr_w[512 + (lane >> 2)] = r;
            __syncthreads();
            for (int o = tid; o < kScrMlp; o += kTT) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < kWarps; ++w) t += scr[w * (kScrMlp + kScrMlpV) + o];
                if (o < 256) accW2[(j0 >> 3) * 256 + o] += t;
                else if (o < 512) accQ[(j0 >> 3) * 256 + o - 256] += t;
                else accb1[j0 + o - 512] += t;
            }
        }
        // through LayerNorm, plus the residual branch
        {
            f2 m1 = make_float2(0.f, 0.f), m2 = make_float2(0.f, 0.f);
            float sg[C], sb[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const f2 d = unpair<C>(dn0, dn1, c);
                sg[c] = fmaf(d.x, nh[c].x, d.y * nh[c].y);
                sb[c] = d.x + d.y;
                const f2 t = make_float2(d.x * gs[c], d.y * gs[c]);
                m1.x += t.x; m1.y += t.y;
                m2.x = fmaf(t.x, nh[c].x, m2.x); m2.y = fmaf(t.y, nh[c].y, m2.y);
            }
            m1.x *= (1.f / C); m1.y *= (1.f / C); m2.x *= (1.f / C); m2.y *= (1.f / C);
            scr_w[kScrMlp + C + lane] = warp_vec_sum<C>(sg, lane);
            scr_w[kScrMlp + 2 * C + lane] = warp_vec_sum<C>(sb, lane);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const f2 d = unpair<C>(dn0, dn1, c);
                const f2 g = *reinterpret_cast<const f2*>(mycol_do + c * kRS);
                sb[c] = g.x + g.y;
                f2 o;
                o.x = rstd.x * (d.x * gs[c] - m1.x - nh[c].x * m2.x);
                o.y = rstd.y * (d.y * gs[c] - m1.y - nh[c].y * m2.y);
                if (valid) {
                    f2* dp = reinterpret_cast<f2*>(dx1 + base + c * vox);
                    const f2 prev = accumulate ? *dp : g;
                    *dp = make_float2(prev.x + o.x, prev.y + o.y);
                }
            }
            scr_w[kScrMlp + lane] = warp_vec_sum<C>(sb, lane);
        }
        __syncthreads();   // per-tile sums are in the scratch; the next tile may restage Snh / Sdo
        if (tid < kScrMlpV) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) t += scr[w * (kScrMlp + kScrMlpV) + kScrMlp + tid];
            accv[tid] += t;
        }
    }
    __syncthreads();
    // flush: acc[(j0/8)*256 + (i*4+k)*16 + tt] is the (j, r) entry with j = j0 + (tt>>3)*4 + i, r = (tt&7) + 8k
    for (int idx = tid; idx < HID * C; idx += kTT) {
        const int blk = idx >> 8, e = (idx >> 4) & 15, tt = idx & 15;
        const int j = blk * 8 + (tt >> 3) * 4 + (e >> 2), r = (tt & 7) + 8 * (e & 3);
        atomicAdd(dW2 + r * ldw2 + j, accW2[idx]);
        // dW1[j][c] = sum_v dh[j] (gamma[c] a_hat[c] + beta[c])
        atomicAdd(dW1 + j * C + r, fmaf(gs[r], accQ[idx], bs[r] * accb1[j]));
    }
    for (int j = tid; j < HID; j += kTT) if (db1) atomicAdd(db1 + j, accb1[j]);
    for (int c = tid; c < C; c += kTT) {
        if (db2) atomicAdd(db2 + c, accv[c]);
        if (dgamma) atomicAdd(dgamma + c, accv[C + c]);
        if (dbeta) atomicAdd(dbeta + c, accv[2 * C + c]);
    }
}

// ------------------------------------------------------------------------------------------------
// Per calling thread (no process-wide state): bit 0 = the forward kernels on tcgen05, bit 1 = linear_bwd, bit 2 = the MLP
// backward; all on by default.  fz_set_glue_mode() exists for the parity tests and the benchmark's FP32-pipe comparison.
int glue_mode() { return tls().glue_mode; }

int check_common(long long batch, int channels, long long voxels) {
    if (batch < 0 || voxels < 0) return fail(FZ_ERR_INVALID, "negative size");
    if (channels != kC) return fail(FZ_ERR_UNSUPPORTED, "block glue kernels are built for %d channels, got %d", kC, channels);
    if (voxels % 2) return fail(FZ_ERR_UNSUPPORTED, "block glue kernels need an even number of voxels, got %lld", voxels);
    if (voxels >= (1LL << 40)) return fail(FZ_ERR_UNSUPPORTED, "too many voxels");
    return FZ_OK;
}

bool misaligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7) != 0; }

size_t linear_bwd_smem() { return sizeof(float) * (2 * kC * kC + 2 * kC + 3 * kC + kLWarps * kScrLin + 2 * kC * kLRS); }
size_t mlp_fwd_smem(int hid) { return sizeof(float) * (kC * kC + 2 * kC * hid + hid + 4 * kC); }
size_t mlp_bwd_smem(int hid) { return sizeof(float) * (5 * kC * hid + 2 * hid + 2 * kC + 3 * kC + kWarps * (kScrMlp + kScrMlpV) + (2 * kC + 16) * kRS); }

}  // namespace
}  // namespace fz

using namespace fz;

extern "C" {

void fz_set_glue_mode(int32_t mode) { tls().glue_mode = mode & 7; }
int fz_get_glue_mode(void) { return glue_mode(); }

int fz_glue_supported(int32_t channels, int32_t hidden, int64_t voxels) {
    return channels == kC && voxels > 0 && voxels % 2 == 0 && hidden >= 8 && hidden % 8 == 0 && hidden <= 256;
}

int fz_ln_linear_forward(const float* x, const float* gamma, const float* beta, const float* W, float* y, int64_t batch,
                         int32_t channels, int64_t voxels, float eps, void* stream) {
    tls().launches = 0;
    if (int e = check_common(batch, channels, voxels)) return e;
    if (batch == 0 || voxels == 0) return FZ_OK;          // empty tensors carry null data pointers
    if (!x || !W || !y) return fail(FZ_ERR_INVALID, "null buffer");
    if (misaligned(x) || misaligned(y)) return fail(FZ_ERR_INVALID, "buffers must be 8-byte aligned");
    if (glue_mode() & 1) return ln_linear_tc_launch(x, gamma, beta, W, y, batch, voxels, eps, (cudaStream_t)stream);
    const long long pps = voxels / 2, total = batch * pps;
    long long blocks = (total + 127) / 128;
    const long long cap = 3LL * num_sms();
    if (blocks > cap) blocks = cap;
    ln_linear_fwd<kC><<<(unsigned)blocks, 128, 0, (cudaStream_t)stream>>>(x, gamma, beta, W, y, pps, total, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int fz_mixer_mlp_forward(const float* x, const float* m, const float* Wout, const float* bout, const float* gamma,
                         const float* beta, const float* W1, const float* b1, const float* W2, const float* b2, float* x1,
                         float* out, int64_t batch, int32_t channels, int32_t hidden, int64_t voxels, float eps, void* stream) {
    tls().launches = 0;
    if (int e = check_common(batch, channels, voxels)) return e;
    if (hidden < 8 || hidden % 8 || hidden > 256) return fail(FZ_ERR_UNSUPPORTED, "hidden width %d: need a multiple of 8 up to 256", hidden);
    if (batch == 0 || voxels == 0) return FZ_OK;
    if (!x || !m || !Wout || !W1 || !W2 || !out) return fail(FZ_ERR_INVALID, "null buffer");
    if (misaligned(x) || misaligned(m) || misaligned(out) || misaligned(x1)) return fail(FZ_ERR_INVALID, "buffers must be 8-byte aligned");
    {
        // tensor-core path (tcgen05, 3xTF32) unless the glue mode asks for the FP32-pipe kernel
        if ((glue_mode() & 1) && mixer_mlp_tc_supported(hidden))
            return mixer_mlp_tc_launch(x, m, Wout, bout, gamma, beta, W1, b1, W2, b2, x1, out, batch, hidden, voxels, eps,
                                       (cudaStream_t)stream);
    }
    const size_t smem = mlp_fwd_smem(hidden);
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(mixer_mlp_fwd<kC>, smem));
    const long long pps = voxels / 2, total = batch * pps;
    long long blocks = (total + 127) / 128;
    const long long cap = 2LL * num_sms();
    if (blocks > cap) blocks = cap;
    mixer_mlp_fwd<kC><<<(unsigned)blocks, 128, smem, (cudaStream_t)stream>>>(x, m, Wout, bout, gamma, beta, W1, b1, W2, b2, x1, out,
                                                                             hidden, pps, total, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int fz_linear_backward(const float* dy, const float* a, const float* gamma, const float* beta, const float* W,
                       const float* resid, float* da, float* dW, float* db, float* dgamma, float* dbeta, int64_t batch,
                       int32_t channels, int64_t voxels, float eps, int32_t layernorm, void* stream) {
    tls().launches = 0;
    if (int e = check_common(batch, channels, voxels)) return e;
    const bool empty = batch == 0 || voxels == 0;
    if (!W || !dW || (!empty && (!dy || !a || !da))) return fail(FZ_ERR_INVALID, "null buffer");
    if (misaligned(dy) || misaligned(a) || misaligned(da) || misaligned(resid)) return fail(FZ_ERR_INVALID, "buffers must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    FZ_CUDA_CHECK(cudaMemsetAsync(dW, 0, kC * kC * sizeof(float), st));
    if (db) FZ_CUDA_CHECK(cudaMemsetAsync(db, 0, kC * sizeof(float), st));
    if (dgamma) FZ_CUDA_CHECK(cudaMemsetAsync(dgamma, 0, kC * sizeof(float), st));
    if (dbeta) FZ_CUDA_CHECK(cudaMemsetAsync(dbeta, 0, kC * sizeof(float), st));
    if (batch == 0 || voxels == 0) return FZ_OK;
    {
        // tensor-core path (tcgen05, 3xTF32): dgrad with its A operand in tensor memory, weight gradient as a contraction over
        // voxel rows (csrc/fz_block_glue_lin_tc.cu)
        if (glue_mode() & 2)
            return linear_bwd_tc2_launch(dy, a, gamma, beta, W, resid, da, dW, db, dgamma, dbeta, batch, voxels, eps, layernorm, st);
    }
    const size_t smem = linear_bwd_smem();
    static SmemConfig cfg_ln, cfg_plain;
    FZ_CUDA_CHECK(cfg_ln.ensure(linear_bwd<kC, true>, smem));
    FZ_CUDA_CHECK(cfg_plain.ensure(linear_bwd<kC, false>, smem));
    const int tps = (int)((voxels + kLV - 1) / kLV);
    const long long tiles = batch * tps;
    const unsigned blocks = (unsigned)(tiles < 2LL * num_sms() ? tiles : 2LL * num_sms());
    if (layernorm)
        linear_bwd<kC, true><<<blocks, kLT, smem, st>>>(dy, a, gamma, beta, W, resid, da, dW, db, dgamma, dbeta, voxels, tps, tiles, eps);
    else
        linear_bwd<kC, false><<<blocks, kLT, smem, st>>>(dy, a, nullptr, nullptr, W, nullptr, da, dW, db, nullptr, nullptr, voxels, tps, tiles, eps);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int fz_mlp_backward(const float* x1, const float* dout, const float* gamma, const float* beta, const float* W1,
                    const float* b1, const float* W2, float* dx1, float* dgamma, float* dbeta, float* dW1, float* db1,
                    float* dW2, float* db2, int64_t batch, int32_t channels, int32_t hidden, int64_t voxels, float eps,
                    void* stream) {
    tls().launches = 0;
    if (int e = check_common(batch, channels, voxels)) return e;
    if (hidden < 8 || hidden % 8 || hidden > 256)
        return fail(FZ_ERR_UNSUPPORTED, "hidden width %d: need a multiple of 8 up to 256", hidden);
    const bool empty = batch == 0 || voxels == 0;
    if (!W1 || !W2 || !dW1 || !dW2 || (!empty && (!x1 || !dout || !dx1))) return fail(FZ_ERR_INVALID, "null buffer");
    if (misaligned(x1) || misaligned(dout) || misaligned(dx1)) return fail(FZ_ERR_INVALID, "buffers must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    FZ_CUDA_CHECK(cudaMemsetAsync(dW1, 0, (size_t)hidden * kC * sizeof(float), st));
    FZ_CUDA_CHECK(cudaMemsetAsync(dW2, 0, (size_t)hidden * kC * sizeof(float), st));
    if (db1) FZ_CUDA_CHECK(cudaMemsetAsync(db1, 0, hidden * sizeof(float), st));
    if (db2) FZ_CUDA_CHECK(cudaMemsetAsync(db2, 0, kC * sizeof(float), st));
    if (dgamma) FZ_CUDA_CHECK(cudaMemsetAsync(dgamma, 0, kC * sizeof(float), st));
    if (dbeta) FZ_CUDA_CHECK(cudaMemsetAsync(dbeta, 0, kC * sizeof(float), st));
    if (batch == 0 || voxels == 0) return FZ_OK;
    // tensor-core path (tcgen05, 3xTF32) for hidden widths that are multiples of 64 unless the glue mode asks for the FP32-pipe kernel
    if ((glue_mode() & 4) && mlp_bwd_tc_supported(hidden))
        return mlp_bwd_tc_launch(x1, dout, gamma, beta, W1, b1, W2, dx1, dgamma, dbeta, dW1, db1, dW2, db2, batch, hidden, voxels, eps, st);
    const int tps = (int)((voxels + kTV - 1) / kTV);
    const long long tiles = batch * tps;
    const unsigned blocks = (unsigned)(tiles < num_sms() ? tiles : num_sms());
    // the kernel holds the weights and weight-gradient accumulators of at most kMaxHidden hidden units in shared
    // memory; wider MLPs (mlp_ratio 4: model_zoo/factorizer_brats23/configs/train.yaml) run slice by slice
    for (int h0 = 0; h0 < hidden; h0 += kMaxHidden) {
        const int hs = hidden - h0 < kMaxHidden ? hidden - h0 : kMaxHidden;
        const size_t smem = mlp_bwd_smem(hs);
        static SmemConfig cfg;
        FZ_CUDA_CHECK(cfg.ensure(mlp_bwd<kC>, smem));
        mlp_bwd<kC><<<blocks, kTT, smem, st>>>(x1, dout, gamma, beta, W1 + (size_t)h0 * kC, b1 ? b1 + h0 : nullptr, W2 + h0, dx1,
                                               dgamma, dbeta, dW1 + (size_t)h0 * kC, db1 ? db1 + h0 : nullptr, dW2 + h0,
                                               h0 == 0 ? db2 : nullptr, hs, hidden, h0 > 0, voxels, tps, tiles, eps);
        FZ_LAUNCH_CHECK();
    }
    return FZ_OK;
}

}  // extern "C"
