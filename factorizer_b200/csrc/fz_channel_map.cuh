// What the channel maps linear_fwd_tc (fz_linear_tc.cu, fp32, 3xTF32) and linear_fwd_bf16_tc (fz_bf16_block.cu, bf16) share:
// persistent CTAs of kThreads threads (warp 0 = TMA producer, warp 1 = MMA issue, warps 2-9 = workers) walk items of kM
// voxels x kN outputs summed in fp32 in TMEM; a worker owns one voxel of every item (= its TMEM lane) and 32 of its outputs,
// and Epilogue is what it does with their running sums.  And the host side of both launchers and of the weight gradients.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "fz_device.cuh"

namespace fz {
namespace cmap {

constexpr int kM = 128, kN = 64;                      // voxels x outputs per item
constexpr int kThreads = 320;

// load as float, store from float (bf16, fp16: rounded to nearest once; an fp16 value beyond 65504 becomes +-inf)
__device__ __forceinline__ float ldg_f(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg_f(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float ldg_f(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ void st_f(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_f(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void st_f(__half* p, float v) { *p = __float2half_rn(v); }

// A worker's epilogue: y, aux and y2 hold T (bias is fp32); FZ_EPILOGUE_*: + residual | y = r, y2 = gelu(r) |
// y = r * gelu'(aux) | y = gelu(r)
template <typename T>
struct Epilogue {
    const float* bias;
    T* y;
    const T* aux;
    T* y2;
    int epi, cout, otiles, vtiles_per_sample;
    long long vox;
    int wq, wh, lane;                                 // TMEM lane quarter (warp % 4) and lane: the voxel; half of the columns

    // where this thread's 32 outputs of item `it` live: output o0 + o (if below cout) at off + o * vox; false when the voxel
    // is past the end of the sample (32-bit index arithmetic: the launcher keeps the item count below 2^31)
    __device__ __forceinline__ bool at(long long it, long long& off, int& o0) const {
        const unsigned item = blockIdx.x + (unsigned)it * gridDim.x;
        const unsigned vt_all = item / (unsigned)otiles, ot = item - vt_all * (unsigned)otiles;
        const unsigned b = vt_all / (unsigned)vtiles_per_sample;
        const long long v = (long long)(vt_all - b * (unsigned)vtiles_per_sample) * kM + wq * 32 + lane;
        o0 = (int)ot * kN + wh * 32;
        off = ((long long)b * cout + o0) * vox + v;
        return v < vox;
    }

    // the running sums of item `it` (zeroed by the caller) start from the bias -- or from the residual (FZ_EPILOGUE_RESIDUAL;
    // the bias is added at the end then).  `ahead`: they are started an item ahead of their first use, and
    // FZ_EPILOGUE_GELU_GRAD pulls its aux values into L2 meanwhile
    __device__ __forceinline__ void start(float (&sum)[32], long long it, bool ahead) const {
        long long off;
        int o0;
        const bool live = at(it, off, o0);
        if (epi != FZ_EPILOGUE_RESIDUAL) {
            if (bias) {
#pragma unroll
                for (int o = 0; o < 32; ++o)
                    if (o0 + o < cout) sum[o] = __ldg(bias + o0 + o);
            }
            if (ahead && epi == FZ_EPILOGUE_GELU_GRAD && live) {
                const T* pa = aux + off;
#pragma unroll
                for (int o = 0; o < 32; ++o) {
                    if (o0 + o < cout) asm volatile("prefetch.global.L2 [%0];" :: "l"(pa));
                    pa += vox;
                }
            }
        } else if (live) {
            const T* pa = aux + off;
#pragma unroll
            for (int o = 0; o < 32; ++o) {
                if (o0 + o < cout) sum[o] = ldg_f(pa);
                pa += vox;
            }
        }
    }

    // the end of item `it`: bias after the residual, GELU / GELU' on the fp32 sums, and the stores along the voxel axis
    // (coalesced: neighbouring lanes are neighbouring voxels)
    __device__ __forceinline__ void finish(float (&sum)[32], long long it) const {
        long long off;
        int o0;
        if (!at(it, off, o0)) return;
        const bool full = o0 + 32 <= cout;            // no channel predicates on whole groups of 32
        if (epi == FZ_EPILOGUE_RESIDUAL && bias) {
#pragma unroll
            for (int o = 0; o < 32; ++o)
                if (full || o0 + o < cout) sum[o] += __ldg(bias + o0 + o);
        }
        T* py = y + off;
        if (epi == FZ_EPILOGUE_GELU) {
            T* pg = y2 + off;
#pragma unroll
            for (int o = 0; o < 32; o += 2) {
                float2 e;
                const float2 r = make_float2(sum[o], sum[o + 1]);
                const float2 gl = __fmul2_rn(r, gauss_cdf2(r, e));
                if (full || o0 + o < cout) { st_f(py, r.x); st_f(pg, gl.x); }
                py += vox; pg += vox;
                if (full || o0 + o + 1 < cout) { st_f(py, r.y); st_f(pg, gl.y); }
                py += vox; pg += vox;
            }
            return;
        }
        if (epi == FZ_EPILOGUE_GELU_ONLY) {
#pragma unroll
            for (int o = 0; o < 32; o += 2) {
                float2 e;
                const float2 r = make_float2(sum[o], sum[o + 1]);
                const float2 gl = __fmul2_rn(r, gauss_cdf2(r, e));
                sum[o] = gl.x;
                sum[o + 1] = gl.y;
            }
        }
        if (epi == FZ_EPILOGUE_GELU_GRAD) {
            float h[32];
            const T* pa = aux + off;
#pragma unroll
            for (int o = 0; o < 32; ++o) {
                h[o] = (full || o0 + o < cout) ? ldg_f(pa) : 0.f;
                pa += vox;
            }
#pragma unroll
            for (int o = 0; o < 32; o += 2) {
                float2 gl, gp;
                gelu_grad2(make_float2(h[o], h[o + 1]), gl, gp);
                sum[o] *= gp.x;
                sum[o + 1] *= gp.y;
            }
        }
        if (full) {
#pragma unroll
            for (int o = 0; o < 32; ++o) { st_f(py, sum[o]); py += vox; }
        } else {
#pragma unroll
            for (int o = 0; o < 32; ++o) {
                if (o0 + o < cout) st_f(py, sum[o]);
                py += vox;
            }
        }
    }
};

// ---- host ----------------------------------------------------------------------------------------------------------------
// The epilogue arguments of a channel-map call: a known FZ_EPILOGUE_*, `aux` where it reads one, `y2` where it writes one
inline int check_epilogue(const char* what, int epi, const void* aux, const void* y2) {
    if (epi < FZ_EPILOGUE_NONE || epi > FZ_EPILOGUE_GELU_ONLY) return fail(FZ_ERR_INVALID, "%s: unknown epilogue %d", what, epi);
    if ((epi == FZ_EPILOGUE_RESIDUAL || epi == FZ_EPILOGUE_GELU_GRAD) && !aux)
        return fail(FZ_ERR_INVALID, "%s: epilogue %d reads `aux`", what, epi);
    if (epi == FZ_EPILOGUE_GELU && !y2) return fail(FZ_ERR_INVALID, "%s: the GELU epilogue writes `y2`", what);
    return FZ_OK;
}

// Pipeline depth and grid of a channel-map launch over `items` items of `kchunks` K chunks each.  Two stages, two CTAs per SM
// for the streaming shapes; four stages, one CTA per item and SM when there are fewer items than SMs and more than two K
// chunks (the 8^3 / 16^3 stages: few voxel tiles, long K), which are bound by the chunk hand-over latency.
struct Launch {
    int stages;
    unsigned blocks;
};
inline Launch launch_shape(long long items, int kchunks) {
    if (items <= num_sms() && kchunks > 2) return {4, (unsigned)items};
    const long long cap = 2LL * num_sms();
    return {2, (unsigned)(items < cap ? items : cap)};
}

// CTAs along the voxel axis of a tensor-core weight gradient over `tiles` stages: `ctas`, or more so that no CTA's chain is
// longer than kMaxChain stages (4 MMAs each), but at most one CTA per stage.  The tensor core adds into its fp32 accumulator
// with truncation, so the error of a TMEM accumulation chain grows linearly with its length: on same-sign operands about
// 2^-24 S per MMA, S = sum |dy| |x| (B200: 1.7e-5 S after 64 stages, 9.8e-5 S after 443; the FP32-pipe kernels stay below
// 1.1e-6 S).  32 stages keep it at 0.8-1.04e-5 S (tests/test_gpu_channel_map_scale.py holds it to 2e-5 S).
inline long long wgrad_ctas(long long ctas, long long tiles) {
    constexpr long long kMaxChain = 32;
    if (ctas * kMaxChain < tiles) ctas = (tiles + kMaxChain - 1) / kMaxChain;
    if (ctas > tiles) ctas = tiles;
    return ctas < 1 ? 1 : ctas;
}

}  // namespace cmap
}  // namespace fz
