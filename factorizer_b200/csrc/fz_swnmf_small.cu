// Rank-1 NMF (HALS or MU) on SMALL matrices, a sub-warp per matrix, everything in registers.
//
// Serves the window geometries of the reference's model-zoo bundles and tests whose matrices are tiny
// (patch 4x4x4 or 8x8 -> 64 columns; head_dim 4..32: model_zoo/factorizer_isles22/configs/train.yaml:49-53,
// tests/test_factorizer.py:112-165) and ft.NMF on small pre-matricised batches.  The generic kernels
// (fz_nmf_generic.cu) give such a matrix a whole CTA and a dozen block barriers per sweep; here L lanes of a warp
// own one M x N matrix (N = L * CPL columns, column pair j/2 lives in lane (j/2) % L), hold it in M*CPL = 64 registers
// per lane (float2 pairs, packed FFMA2), and run the reference's updates literally (no Gram reformulation, so any act / sign of X works):
//   HALS  u <- relu((X v + eps) / (v.v + eps)),  v <- relu((X^T u + eps) / (u.u + eps))
//         (factorizer/factorization/matrix_factorization.py:210-229 with R = 1, project = ReLU :609)
//   MU    u <- (u . X v + eps) / (u (v.v) + eps), v likewise                                  (:241-247)
// X v needs one sub-warp all-reduce of M values per sweep; X^T u is lane-local.  The backward recomputes the
// iterates (u_t, v_t parked in shared memory, T <= 5) and runs the hand-derived adjoint of the unrolled loop (same
// math as oracle/factorizer_oracle.py::_half_bwd), truncated to the last K sweeps (num_grad_steps, :506-512).
// Window mode gathers straight from the NCDHW volume with the roll folded into the index math
// (operations.py:266-272) and accumulates the window sets in shift order, the last one dividing by S
// (operations.py:426-433); consecutive sub-warps take windows that are neighbours along W, so a warp-wide
// load still covers whole 32-byte sectors.  Division is reciprocal (MUFU + one Newton step) times numerator,
// <= 1 ulp from the reference's true division (same deviation as the 8x512 kernels, DESIGN.md section 2).
// Window mode also takes bf16 and fp16 volumes (x, dL/dy in, y, dL/dx out; u, v, the iterates, the history and every sum stay
// fp32).  Their elements are read and written 2 bytes at a time: shifts 1 and 3 put window origins at odd W indices, where a
// column pair is not 4-byte aligned.  The window sets then sum in an fp32 accumulator volume in the caller's workspace: set 0
// writes it, later sets read-add-store it, and the last set writes the finished sum to the 16-bit output, rounded once.  So
// y / dL/dx are the fp32 kernels' results on the same (16-bit-representable) inputs, rounded to the volume's type.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "fz_device.cuh"
#include "fz_internal.cuh"

namespace fz {
namespace {

constexpr int kTMax = 5;          // iterates kept (in shared memory) by the backward
constexpr int kSmallThreads = 128;

template <typename E>     // element type of the volumes: float, or __nv_bfloat16 / __half in window mode
struct SmallParams {
    const E* x;           // window mode: volume; direct mode: (n, M, N)
    const E* gy;          // backward: dL/dy, same layout as x
    E* out;               // forward: y; backward: dL/dx
    const float* u0;      // (M)
    const float* v0;      // (N)
    long long n;          // matrices in this launch (windows of ONE set in window mode)
    int T, K, kind, relu, set, S, window;
    float eps;
    DevGeom G;
    float* acc;           // 16-bit volume, S >= 2: the fp32 sum over the window sets, laid out as the volume
};

// one rounding of an fp32 sum to the volume's 16-bit type
__device__ __forceinline__ __nv_bfloat16 round_to(float v, const __nv_bfloat16*) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ __half round_to(float v, const __half*) { return __float2half_rn(v); }

// Where a window set's sums go.  `acc` is where a set > 0 reads the sums so far.  An fp32 volume read-add-stores in `out`.  A
// 16-bit volume at S >= 2 sums in the fp32 accumulator, and its last set writes `out`, rounded once; at S == 1, set 0 writes
// `out` directly.
template <typename E>
struct SetSums;
template <>
struct SetSums<float> {
    float* acc;
    __device__ __forceinline__ SetSums(const SmallParams<float>& P, long long base) : acc(P.out + base) {}
    // v before i: the evaluation order of `acc[i] = v`, which keeps the fp32 kernels' code as it was
    __device__ __forceinline__ void store(float v, int i) const { acc[i] = v; }
};
template <typename E>                         // E = __nv_bfloat16 or __half
struct SetSums {
    const SmallParams<E>& P;                  // `out` is addressed from P at each store: two more live pointers spill
    long long base;
    float* acc;
    __device__ __forceinline__ SetSums(const SmallParams<E>& P_, long long base_) : P(P_), base(base_), acc(P_.acc + base_) {}
    __device__ __forceinline__ void store(float v, int i) const {
        if (P.set < P.S - 1) acc[i] = v;
        else P.out[base + i] = round_to(v, P.out);
    }
};

// element i of a volume, as float; the unsigned 16-bit index gives one IMAD.WIDE.U32 per address (a signed one takes three
// instructions and a register more)
__device__ __forceinline__ float ld_at(const float* p, int i) { return __ldg(p + i); }
__device__ __forceinline__ float ld_at(const __nv_bfloat16* p, int i) { return __bfloat162float(__ldg(p + (unsigned)i)); }
__device__ __forceinline__ float ld_at(const __half* p, int i) { return __half2float(__ldg(p + (unsigned)i)); }

template <int L>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// element offsets (relative to the (batch, head) base) of this lane's CPL columns of matrix `mid`
template <typename E, int M, int CPL, int L>
struct Locator {
    int rel[CPL];     // offset of column 2 ((k >> 1) L + lane) + (k & 1) relative to the window origin (no wrap)
    int lane_;
    __device__ __forceinline__ void init(const SmallParams<E>& P, int lane) {
        lane_ = lane;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
            const int j = 2 * ((k >> 1) * L + lane) + (k & 1);
            if (P.window) {
                const int q2 = j % P.G.p[2];
                const int t = j / P.G.p[2];
                const int q1 = t % P.G.p[1], q0 = t / P.G.p[1];
                rel[k] = (q0 * P.G.n[1] + q1) * P.G.n[2] + q2;
            } else {
                rel[k] = j;
            }
        }
    }
    // returns the base offset (channel row 0) and fills off[]
    __device__ __forceinline__ long long locate(const SmallParams<E>& P, long long mid, int (&off)[CPL]) const {
        if (!P.window) {
#pragma unroll
            for (int k = 0; k < CPL; ++k) off[k] = rel[k];
            return mid * (long long)(M * CPL * L);
        }
        const DevGeom& G = P.G;
        const int w = (int)(mid % G.G);
        const long long t = mid / G.G;
        const int h = (int)(t % G.heads), b = (int)(t / G.heads);
        const int g2 = w % G.g[2];
        const int tt = w / G.g[2];
        const int g1 = tt % G.g[1], g0 = tt / G.g[1];
        const int o0 = g0 * G.p[0] - G.sh[P.set][0], o1 = g1 * G.p[1] - G.sh[P.set][1], o2 = g2 * G.p[2] - G.sh[P.set][2];
        if ((o0 | o1 | o2) >= 0) {
            const int org = (o0 * G.n[1] + o1) * G.n[2] + o2;
#pragma unroll
            for (int k = 0; k < CPL; ++k) off[k] = org + rel[k];
        } else {
#pragma unroll
            for (int k = 0; k < CPL; ++k) {       // a window that wraps around the volume: rare, index math redone
                const int j = 2 * ((k >> 1) * L + lane_) + (k & 1);
                const int q2 = j % G.p[2], tq = j / G.p[2];
                int i0 = o0 + tq / G.p[1], i1 = o1 + tq % G.p[1], i2 = o2 + q2;
                if (i0 < 0) i0 += G.n[0];
                if (i1 < 0) i1 += G.n[1];
                if (i2 < 0) i2 += G.n[2];
                off[k] = (i0 * G.n[1] + i1) * G.n[2] + i2;
            }
        }
        return ((long long)b * G.C + (long long)h * G.d) * G.vox;
    }
};

// Columns come in pairs (float2, packed FFMA2): pair kp of a lane = columns 2 (kp L + lane), +1.
// one half-step for the M side: a = X v (all-reduced), b = v.v;  u <- update
template <int M, int H, int L>
__device__ __forceinline__ void step_u(const f2 (&x)[M][H], const f2 (&v)[H], float (&u)[M], float (&a)[M], float& b,
                                       int kind, float eps) {
    f2 b2 = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < H; ++k) b2 = fma2(v[k], v[k], b2);
    float bb = b2.x + b2.y;
#pragma unroll
    for (int i = 0; i < M; ++i) {
        f2 s = make_float2(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < H; ++k) s = fma2(x[i][k], v[k], s);
        a[i] = s.x + s.y;
    }
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) {
        bb += __shfl_xor_sync(0xffffffffu, bb, o);
#pragma unroll
        for (int i = 0; i < M; ++i) a[i] += __shfl_xor_sync(0xffffffffu, a[i], o);
    }
    b = bb;
    if (kind == FZ_SOLVER_HALS) {
        const float r = rcp_nr(bb + eps);
#pragma unroll
        for (int i = 0; i < M; ++i) u[i] = fmaxf((a[i] + eps) * r, 0.f);
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) u[i] = fmaf(u[i], a[i], eps) * rcp_nr(fmaf(u[i], bb, eps));
    }
}

// ... and for the N side: c = X^T u (lane-local), d = u.u;  v <- update
template <int M, int H>
__device__ __forceinline__ void step_v(const f2 (&x)[M][H], const float (&u)[M], f2 (&v)[H], f2 (&c)[H], float& d,
                                       int kind, float eps) {
    float dd = 0.f;
#pragma unroll
    for (int i = 0; i < M; ++i) dd = fmaf(u[i], u[i], dd);
#pragma unroll
    for (int k = 0; k < H; ++k) c[k] = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < M; ++i) {
        const f2 ui = dup(u[i]);
#pragma unroll
        for (int k = 0; k < H; ++k) c[k] = fma2(x[i][k], ui, c[k]);
    }
    d = dd;
    if (kind == FZ_SOLVER_HALS) {
        const float r = rcp_nr(dd + eps);
#pragma unroll
        for (int k = 0; k < H; ++k) v[k] = make_float2(fmaxf((c[k].x + eps) * r, 0.f), fmaxf((c[k].y + eps) * r, 0.f));
    } else {
#pragma unroll
        for (int k = 0; k < H; ++k)
            v[k] = make_float2(fmaf(v[k].x, c[k].x, eps) * rcp_nr(fmaf(v[k].x, dd, eps)),
                               fmaf(v[k].y, c[k].y, eps) * rcp_nr(fmaf(v[k].y, dd, eps)));
    }
}

template <typename E, int M, int CPL, int L>
__global__ void __launch_bounds__(kSmallThreads, 3) small_fwd(const SmallParams<E> P) {
    constexpr int H = CPL / 2;
    const int lane = threadIdx.x & (L - 1);
    const long long groups = (long long)gridDim.x * (kSmallThreads / L);
    const long long g0 = ((long long)blockIdx.x * kSmallThreads + threadIdx.x) / L;
    Locator<E, M, CPL, L> loc;
    loc.init(P, lane);
    const int istride = P.window ? (int)P.G.vox : CPL * L;
    const float invS = 1.f / (float)P.S;
    const float lo = P.relu ? 0.f : -__int_as_float(0x7f800000);
    for (long long first = 0; first < P.n; first += groups) {      // trip count is uniform across the warp
        const long long mid = first + g0;
        const bool valid = mid < P.n;
        int off[CPL];
        const long long base = loc.locate(P, valid ? mid : 0, off);
        // every load is issued unconditionally (an idle sub-warp re-reads matrix 0) and back to back: the kernel lives
        // on memory-level parallelism; 32-bit element offsets, one IMAD.WIDE per address
        const E* src = P.x + base;
        f2 x[M][H];
        constexpr int RB = 16 / CPL > 0 ? 16 / CPL : 1;      // rows per batch of 16 loads
#pragma unroll
        for (int ib = 0; ib < M; ib += RB) {
#pragma unroll
            for (int i = ib; i < ib + RB; ++i)
#pragma unroll
                for (int k = 0; k < H; ++k)
                    x[i][k] = make_float2(ld_at(src, i * istride + off[2 * k]), ld_at(src, i * istride + off[2 * k + 1]));
            asm volatile("" ::: "memory");              // keep the batches (and their 64-bit addresses) apart
        }
#pragma unroll
        for (int i = 0; i < M; ++i)
#pragma unroll
            for (int k = 0; k < H; ++k) x[i][k] = make_float2(fmaxf(x[i][k].x, lo), fmaxf(x[i][k].y, lo));
        float u[M], a[M], b, d;
        f2 v[H], c[H];
#pragma unroll
        for (int i = 0; i < M; ++i) u[i] = __ldg(P.u0 + i);          // L1-resident; not worth 16 registers for the whole kernel
#pragma unroll
        for (int k = 0; k < H; ++k) v[k] = __ldg(reinterpret_cast<const f2*>(P.v0) + k * L + lane);
        for (int t = 0; t < P.T; ++t) {
            step_u<M, H, L>(x, v, u, a, b, P.kind, P.eps);
            step_v<M, H>(x, u, v, c, d, P.kind, P.eps);
        }
        if (valid) {
            const bool add = P.window && P.set > 0, last = P.window && P.set == P.S - 1 && P.S > 1;
            const SetSums<E> dst(P, base);
            const float fin = last ? ((P.S & (P.S - 1)) ? 0.f : invS) : 1.f;    // 0: true division below
            int is2 = istride;
            asm volatile("" : "+r"(is2));                 // recompute the 64 offsets here instead of carrying them in registers
#pragma unroll
            for (int i = 0; i < M; ++i) {                 // one channel row at a time: read-add-store
                f2 y[H];
#pragma unroll
                for (int k = 0; k < H; ++k) y[k] = make_float2(0.f, 0.f);
                if (add) {
#pragma unroll
                    for (int k = 0; k < H; ++k) y[k] = make_float2(dst.acc[i * is2 + off[2 * k]], dst.acc[i * is2 + off[2 * k + 1]]);
                }
#pragma unroll
                for (int k = 0; k < H; ++k) {
                    float y0 = __fadd_rn(y[k].x, u[i] * v[k].x), y1 = __fadd_rn(y[k].y, u[i] * v[k].y);
                    if (fin == 0.f) { y0 = __fdiv_rn(y0, (float)P.S); y1 = __fdiv_rn(y1, (float)P.S); }
                    else { y0 *= fin; y1 *= fin; }
                    dst.store(y0, i * is2 + off[2 * k]);
                    dst.store(y1, i * is2 + off[2 * k + 1]);
                }
            }
        }
    }
}

// floats of history per sub-warp: (T_max + 1) x (M + N), padded so that the sub-warps of a warp start L banks apart
template <int M, int CPL, int L>
struct Hist {
    static constexpr int raw = (kTMax + 1) * (M + CPL * L);
    static constexpr int floats = L < 32 ? raw + ((L - raw % 32) + 32) % 32 : raw;
};

template <typename E, int M, int CPL, int L>
__global__ void __launch_bounds__(kSmallThreads) small_bwd(const SmallParams<E> P) {
    extern __shared__ __align__(8) float hist_all[];
    constexpr int H = CPL / 2;
    constexpr int kHS = M + CPL * L;
    float* hist = hist_all + (threadIdx.x / L) * Hist<M, CPL, L>::floats;
    const int lane = threadIdx.x & (L - 1);
    const long long groups = (long long)gridDim.x * (kSmallThreads / L);
    const long long g0 = ((long long)blockIdx.x * kSmallThreads + threadIdx.x) / L;
    Locator<E, M, CPL, L> loc;
    loc.init(P, lane);
    float u0r[M];
    f2 v0r[H];
#pragma unroll
    for (int i = 0; i < M; ++i) u0r[i] = __ldg(P.u0 + i);
#pragma unroll
    for (int k = 0; k < H; ++k) v0r[k] = __ldg(reinterpret_cast<const f2*>(P.v0) + k * L + lane);
    const int istride = P.window ? (int)P.G.vox : CPL * L;
    const float lo = P.relu ? 0.f : -__int_as_float(0x7f800000);
    const float eps = P.eps;
    const int T = P.T, K = P.K;
    const float invS = 1.f / (float)P.S;
    // v_t of this lane: pair k at hist[t * kHS + M + 2 (k L + lane)]
    auto vh = [&](int t, int k) -> f2& { return *reinterpret_cast<f2*>(hist + t * kHS + M + 2 * (k * L + lane)); };
    for (long long first = 0; first < P.n; first += groups) {
        const long long mid = first + g0;
        const bool valid = mid < P.n;
        int off[CPL];
        const long long base = loc.locate(P, valid ? mid : 0, off);
        const E* src = P.x + base;
        f2 x[M][H];
        constexpr int RB = 16 / CPL > 0 ? 16 / CPL : 1;      // rows per batch of 16 loads
#pragma unroll
        for (int ib = 0; ib < M; ib += RB) {
#pragma unroll
            for (int i = ib; i < ib + RB; ++i)
#pragma unroll
                for (int k = 0; k < H; ++k)
                    x[i][k] = make_float2(ld_at(src, i * istride + off[2 * k]), ld_at(src, i * istride + off[2 * k + 1]));
            asm volatile("" ::: "memory");              // keep the batches (and their 64-bit addresses) apart
        }
        unsigned long long mask = 0;       // x > 0 before the ReLU (M*CPL = 64 bits)
#pragma unroll
        for (int i = 0; i < M; ++i)
#pragma unroll
            for (int k = 0; k < H; ++k) {
                if (x[i][k].x > 0.f) mask |= 1ULL << (i * CPL + 2 * k);
                if (x[i][k].y > 0.f) mask |= 1ULL << (i * CPL + 2 * k + 1);
                x[i][k] = make_float2(fmaxf(x[i][k].x, lo), fmaxf(x[i][k].y, lo));
            }
        if (!P.relu) mask = ~0ULL;
        // ---- recompute the iterates; u_t, v_t (t = 0..T) go to this sub-warp's slice of shared memory ----
        {
            float u[M];
            f2 v[H];
#pragma unroll
            for (int i = 0; i < M; ++i) u[i] = u0r[i];
#pragma unroll
            for (int k = 0; k < H; ++k) v[k] = v0r[k];
            __syncwarp();                      // the previous matrix's history is no longer read
            for (int t = 0;; ++t) {
                if (lane == 0) {
#pragma unroll
                    for (int i = 0; i < M; ++i) hist[t * kHS + i] = u[i];
                }
#pragma unroll
                for (int k = 0; k < H; ++k) vh(t, k) = v[k];
                if (t == T) break;
                float a[M], b, d;
                f2 c[H];
                step_u<M, H, L>(x, v, u, a, b, P.kind, eps);
                step_v<M, H>(x, u, v, c, d, P.kind, eps);
            }
            __syncwarp();
        }
        // ---- seed: y = u_T v_T^T ----
        f2 xb[M][H];                       // dL/dx accumulator; first holds dL/dy
        {
            const E* gsrc = P.gy + base;
            int is3 = istride;
            asm volatile("" : "+r"(is3));
#pragma unroll
            for (int ib = 0; ib < M; ib += RB) {
#pragma unroll
                for (int i = ib; i < ib + RB; ++i)
#pragma unroll
                    for (int k = 0; k < H; ++k)
                        xb[i][k] = make_float2(ld_at(gsrc, i * is3 + off[2 * k]), ld_at(gsrc, i * is3 + off[2 * k + 1]));
                asm volatile("" ::: "memory");
            }
            if (P.window) {
                const bool pow2 = !(P.S & (P.S - 1));
#pragma unroll
                for (int i = 0; i < M; ++i)
#pragma unroll
                    for (int k = 0; k < H; ++k)
                        xb[i][k] = pow2 ? make_float2(xb[i][k].x * invS, xb[i][k].y * invS)
                                        : make_float2(__fdiv_rn(xb[i][k].x, (float)P.S), __fdiv_rn(xb[i][k].y, (float)P.S));
            }
        }
        float ub[M];
        f2 vb[H];
        {
#pragma unroll
            for (int i = 0; i < M; ++i) {
                f2 s = make_float2(0.f, 0.f);
#pragma unroll
                for (int k = 0; k < H; ++k) s = fma2(xb[i][k], vh(T, k), s);
                ub[i] = group_sum<L>(s.x + s.y);
            }
#pragma unroll
            for (int k = 0; k < H; ++k) vb[k] = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < M; ++i) {
                const f2 ui = dup(hist[T * kHS + i]);
#pragma unroll
                for (int k = 0; k < H; ++k) { vb[k] = fma2(xb[i][k], ui, vb[k]); }
            }
#pragma unroll
            for (int i = 0; i < M; ++i)
#pragma unroll
                for (int k = 0; k < H; ++k) xb[i][k] = make_float2(0.f, 0.f);
        }
        for (int t = T; t > T - K; --t) {
            float ut[M], up[M];
            f2 vt[H], vp[H];
#pragma unroll
            for (int i = 0; i < M; ++i) { ut[i] = hist[t * kHS + i]; up[i] = hist[(t - 1) * kHS + i]; }
#pragma unroll
            for (int k = 0; k < H; ++k) { vt[k] = vh(t, k); vp[k] = vh(t - 1, k); }
            // ---- adjoint of the v half-step ----
            float d = 0.f;
#pragma unroll
            for (int i = 0; i < M; ++i) d = fmaf(ut[i], ut[i], d);
            f2 cb[H];
            float dbar = 0.f;
            if (P.kind == FZ_SOLVER_HALS) {
                const float rd = rcp_nr(d + eps);
#pragma unroll
                for (int k = 0; k < H; ++k) {
                    const f2 qb = make_float2(vt[k].x > 0.f ? vb[k].x : 0.f, vt[k].y > 0.f ? vb[k].y : 0.f);
                    cb[k] = make_float2(qb.x * rd, qb.y * rd);
                    dbar = fmaf(qb.x, vt[k].x, fmaf(qb.y, vt[k].y, dbar));
                    vb[k] = make_float2(0.f, 0.f);     // v_{t-1} enters only through the u half-step
                }
                dbar = -rd * group_sum<L>(dbar);
            } else {
                f2 c[H];
#pragma unroll
                for (int k = 0; k < H; ++k) c[k] = make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    const f2 ui = dup(ut[i]);
#pragma unroll
                    for (int k = 0; k < H; ++k) c[k] = fma2(x[i][k], ui, c[k]);
                }
#pragma unroll
                for (int k = 0; k < H; ++k) {
                    const float r0 = rcp_nr(fmaf(vp[k].x, d, eps)), r1 = rcp_nr(fmaf(vp[k].y, d, eps));
                    const float n0 = vb[k].x * r0, n1 = vb[k].y * r1;
                    const float e0 = -n0 * vt[k].x, e1 = -n1 * vt[k].y;
                    cb[k] = make_float2(n0 * vp[k].x, n1 * vp[k].y);
                    dbar = fmaf(e0, vp[k].x, fmaf(e1, vp[k].y, dbar));
                    vb[k] = make_float2(fmaf(n0, c[k].x, e0 * d), fmaf(n1, c[k].y, e1 * d));
                }
                dbar = group_sum<L>(dbar);
            }
            float un[M];                               // dL/du_t
#pragma unroll
            for (int i = 0; i < M; ++i) {
                f2 s = make_float2(0.f, 0.f);
                const f2 ui = dup(ut[i]);
#pragma unroll
                for (int k = 0; k < H; ++k) { s = fma2(x[i][k], cb[k], s); xb[i][k] = fma2(ui, cb[k], xb[i][k]); }
                un[i] = s.x + s.y;
            }
#pragma unroll
            for (int o = L / 2; o > 0; o >>= 1)
#pragma unroll
                for (int i = 0; i < M; ++i) un[i] += __shfl_xor_sync(0xffffffffu, un[i], o);
#pragma unroll
            for (int i = 0; i < M; ++i) un[i] = ub[i] + fmaf(2.f * dbar, ut[i], un[i]);
            // ---- adjoint of the u half-step ----
            f2 b2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < H; ++k) b2 = fma2(vp[k], vp[k], b2);
            const float b = group_sum<L>(b2.x + b2.y);
            float ab[M], bbar = 0.f;
            if (P.kind == FZ_SOLVER_HALS) {
                const float rb = rcp_nr(b + eps);
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    const float pb = ut[i] > 0.f ? un[i] : 0.f;
                    ab[i] = pb * rb;
                    bbar = fmaf(pb, ut[i], bbar);
                    ub[i] = 0.f;
                }
                bbar *= -rb;
            } else {
                float a[M];
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    f2 s = make_float2(0.f, 0.f);
#pragma unroll
                    for (int k = 0; k < H; ++k) s = fma2(x[i][k], vp[k], s);
                    a[i] = s.x + s.y;
                }
#pragma unroll
                for (int o = L / 2; o > 0; o >>= 1)
#pragma unroll
                    for (int i = 0; i < M; ++i) a[i] += __shfl_xor_sync(0xffffffffu, a[i], o);
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    const float rden = rcp_nr(fmaf(up[i], b, eps));
                    const float nb = un[i] * rden, db = -nb * ut[i];
                    ab[i] = nb * up[i];
                    bbar = fmaf(db, up[i], bbar);
                    ub[i] = fmaf(nb, a[i], db * b);
                }
            }
            {
                f2 s[H];
#pragma unroll
                for (int k = 0; k < H; ++k) s[k] = make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    const f2 ai = dup(ab[i]);
#pragma unroll
                    for (int k = 0; k < H; ++k) { s[k] = fma2(x[i][k], ai, s[k]); xb[i][k] = fma2(ai, vp[k], xb[i][k]); }
                }
                const f2 tb = dup(2.f * bbar);
#pragma unroll
                for (int k = 0; k < H; ++k) {
                    const f2 w = fma2(tb, vp[k], s[k]);
                    vb[k] = make_float2(vb[k].x + w.x, vb[k].y + w.y);
                }
            }
        }
        if (valid) {
            const bool add = P.window && P.set > 0;
            const SetSums<E> dst(P, base);
            int is2 = istride;
            asm volatile("" : "+r"(is2));
#pragma unroll
            for (int i = 0; i < M; ++i) {
                f2 o[H];
#pragma unroll
                for (int k = 0; k < H; ++k) o[k] = make_float2(0.f, 0.f);
                if (add) {
#pragma unroll
                    for (int k = 0; k < H; ++k) o[k] = make_float2(dst.acc[i * is2 + off[2 * k]], dst.acc[i * is2 + off[2 * k + 1]]);
                }
#pragma unroll
                for (int k = 0; k < H; ++k) {
                    const float g0v = ((mask >> (i * CPL + 2 * k)) & 1ULL) ? xb[i][k].x : 0.f;
                    const float g1v = ((mask >> (i * CPL + 2 * k + 1)) & 1ULL) ? xb[i][k].y : 0.f;
                    dst.store(__fadd_rn(o[k].x, g0v), i * is2 + off[2 * k]);
                    dst.store(__fadd_rn(o[k].y, g1v), i * is2 + off[2 * k + 1]);
                }
            }
        }
    }
}

template <typename E, int M, int CPL, int L>
int launch_small(const SmallParams<E>& P, bool bwd, cudaStream_t st) {
    const long long per_cta = kSmallThreads / L;
    long long ctas = (P.n + per_cta - 1) / per_cta;
    const long long cap = 8LL * num_sms();
    if (ctas > cap) ctas = cap;
    if (bwd) {
        const size_t smem = sizeof(float) * Hist<M, CPL, L>::floats * (kSmallThreads / L);
        static SmemConfig cfg;
        FZ_CUDA_CHECK(cfg.ensure(small_bwd<E, M, CPL, L>, smem));
        small_bwd<E, M, CPL, L><<<(unsigned)ctas, kSmallThreads, smem, st>>>(P);
    } else {
        small_fwd<E, M, CPL, L><<<(unsigned)ctas, kSmallThreads, 0, st>>>(P);
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

template <typename E>
int dispatch_small(const SmallParams<E>& P, int M, int N, bool bwd, cudaStream_t st) {
    if (N == 64) {
        switch (M) {
            case 4: return launch_small<E, 4, 16, 4>(P, bwd, st);
            case 8: return launch_small<E, 8, 8, 8>(P, bwd, st);
            case 16: return launch_small<E, 16, 4, 16>(P, bwd, st);
            case 32: return launch_small<E, 32, 2, 32>(P, bwd, st);
        }
    }
    if (N == 128 && M == 8) return launch_small<E, 8, 8, 16>(P, bwd, st);
    if (N == 256 && M == 8) return launch_small<E, 8, 8, 32>(P, bwd, st);
    if (N == 16 && M == 8) return launch_small<E, 8, 4, 4>(P, bwd, st);
    return fail(FZ_ERR_UNSUPPORTED, "no small-matrix kernel for %dx%d", M, N);
}

}  // namespace

bool small_supported(int M, int N, const fz_solver& s) {
    if (s.rank != 1 || s.num_iters < 1 || s.num_iters > kTMax) return false;
    if (s.kind != FZ_SOLVER_HALS && s.kind != FZ_SOLVER_MU) return false;
    if (N == 64) return M == 4 || M == 8 || M == 16 || M == 32;
    return M == 8 && (N == 128 || N == 256 || N == 16);
}

bool small_window_supported(const DevGeom& G, const fz_solver& s) {
    if (!small_supported(G.d, G.P, s)) return false;
    for (int k = 0; k < 3; ++k)
        if (G.p[k] > 1023 || G.n[k] > (1 << 20)) return false;
    if ((long long)G.d * G.vox >= (1LL << 31)) return false;      // 32-bit element offsets inside a (batch, head) slab
    return G.mats_per_shift > 0;
}

size_t small_workspace_bytes(const DevGeom& G) {
    if (G.dtype == FZ_DTYPE_F32 || G.S < 2) return 0;
    return ((size_t)G.B * G.C * G.vox * sizeof(float) + 255) / 256 * 256;
}

int small_direct(const float* x, const float* u0, const float* v0, const float* gy, float* out, long long n, int M, int N,
                 const fz_solver& s, int K, bool bwd, cudaStream_t st) {
    SmallParams<float> P;
    memset(&P, 0, sizeof(P));
    P.x = x; P.gy = gy; P.out = out; P.u0 = u0; P.v0 = v0; P.n = n;
    P.T = s.num_iters; P.K = K; P.kind = s.kind; P.eps = s.eps; P.S = 1;
    if (n == 0) return FZ_OK;
    return dispatch_small(P, M, N, bwd, st);
}

namespace {
template <typename E>
int small_window_sets(const E* x, const float* u0, const float* v0, const E* gy, E* out, float* acc, const DevGeom& G,
                      const fz_solver& s, int K, int relu, bool bwd, cudaStream_t st) {
    SmallParams<E> P;
    memset(&P, 0, sizeof(P));
    P.x = x; P.gy = gy; P.out = out; P.u0 = u0; P.v0 = v0; P.n = G.mats_per_shift; P.acc = acc;
    P.T = s.num_iters; P.K = K; P.kind = s.kind; P.eps = s.eps; P.S = G.S; P.window = 1; P.relu = relu;
    P.G = G;
    for (int q = 0; q < G.S; ++q)       // torch.roll semantics: any integer shift, reduced to [0, n)
        for (int k = 0; k < 3; ++k) {
            int v = G.sh[q][k] % G.n[k];
            if (v < 0) v += G.n[k];
            P.G.sh[q][k] = v;
        }
    if (P.n == 0) return FZ_OK;
    for (int q = 0; q < G.S; ++q) {
        P.set = q;
        if (int e = dispatch_small(P, G.d, G.P, bwd, st)) return e;
    }
    return FZ_OK;
}
}  // namespace

int small_window(const float* x, const float* u0, const float* v0, const float* gy, float* out, void* workspace,
                 const DevGeom& G, const fz_solver& s, int K, int relu, bool bwd, cudaStream_t st) {
    if (G.dtype == FZ_DTYPE_F32) return small_window_sets(x, u0, v0, gy, out, nullptr, G, s, K, relu, bwd, st);
    if (small_workspace_bytes(G) && !workspace)
        return fail(FZ_ERR_INVALID, "%s: workspace of %zu bytes required", bwd ? "fz_swnmf_backward" : "fz_swnmf_forward",
                    small_workspace_bytes(G));
    if (G.dtype == FZ_DTYPE_F16)
        return small_window_sets(reinterpret_cast<const __half*>(x), u0, v0, reinterpret_cast<const __half*>(gy),
                                 reinterpret_cast<__half*>(out), static_cast<float*>(workspace), G, s, K, relu, bwd, st);
    typedef __nv_bfloat16 bf;
    return small_window_sets(reinterpret_cast<const bf*>(x), u0, v0, reinterpret_cast<const bf*>(gy), reinterpret_cast<bf*>(out),
                             static_cast<float*>(workspace), G, s, K, relu, bwd, st);
}

}  // namespace fz
