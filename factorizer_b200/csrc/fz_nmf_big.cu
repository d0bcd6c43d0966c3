// Rank-1 NMF (MU or HALS) on matrices that are far too large for one CTA: M rows (channels) x N columns with N up to
// the whole volume -- the reference's DEFAULT FactMixer reshape, Matricize(num_heads=1, grid_size=1)
// (factorizer/factorizer.py:17; tests/test_factorizer.py:14-110 run it at 16..256 x 64^3).  With grid_size 1 and no roll the
// matrix of (sample, head) is the contiguous block x[b, h*M:(h+1)*M, :], so this is also "direct" NMF on (n, M, N).
//
// At rank 1 a sweep needs X only through  a = X v (M sums over the columns),  b = v.v  and, per column,
// c_j = x_j . u (matrix_factorization.py:210-229, :241-247).  Every sweep is therefore ONE pass over the columns
// (thread per column, rows looped, coalesced along the row) that (1) rebuilds u_t from the previous pass's sums
// -- every CTA redundantly, M is tiny --, (2) updates its columns of v, stores them, and (3) accumulates the next
// a, b (warp shuffle -> shared -> one global atomicAdd per row and CTA); the last pass writes y = u_T v_T^T instead.
// T + 1 launches forward.  X (16 MiB for 16 x 64^3) stays in L2 across the passes.
//
// The backward walks the sweeps in reverse with the same structure: per column the lane-local parts of the adjoint
// (c_bar, v_bar, the rank-1 updates of dX), per matrix the M-vector parts (u_bar, a_bar, b_bar) rebuilt in the
// prologue of the next pass from the sums the previous pass accumulated.  K + 1 launches for K differentiated sweeps.
// Same math as csrc/fz_swnmf_small.cu (and oracle/factorizer_oracle.py::_half_bwd), spread over the grid.
#include "fz_device.cuh"
#include "fz_internal.cuh"

namespace fz {
namespace {

constexpr int kBT = 256;          // threads per CTA
constexpr int kCPT = 4;           // columns per thread
constexpr int kChunk = kBT * kCPT;
constexpr int kBigMaxM = 256;
constexpr int kBigMaxT = 8;

struct BigParams {
    const float* x;      // (n, M, N)
    const float* gy;     // (n, M, N)  backward
    float* out;          // y or dX, (n, M, N)
    const float* u0;     // (M)
    const float* v0;     // (N)
    float* vh;           // (n, T, N): v_1 .. v_T
    float* uh;           // (n, T + 1, M): u_0 .. u_T
    float* ab;           // (n, T, M + 1): a_t = X v_t, b_t = v_t . v_t for t = 0 .. T-1
    float* vbar;         // (n, N)  backward: dL/dv_{t-1} part carried between passes
    float* bacc;         // (n, passes, 2M + 1)  backward sums: U (M) | S (M) | D
    float* bst;          // (n, passes, 2M + 1)  backward per-matrix state: abar (M) | ucarry (M) | bbar
    long long N;
    int M, n, T, K, kind, relu, t, pass;
    float eps;
};

// red[warp][i] <- warp sums; then rows 0..count-1 are added to dst[] with one atomic per row
__device__ __forceinline__ void flush_rows(float* red, int count, float* dst) {
    __syncthreads();
    for (int i = threadIdx.x; i < count; i += kBT) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kBT / 32; ++w) s += red[w * (2 * kBigMaxM + 2) + i];
        atomicAdd(dst + i, s);
    }
    __syncthreads();
}

// u_t from (a_{t-1}, b_{t-1}, u_{t-1}) into shared memory; returns d = u_t . u_t (every thread)
__device__ __forceinline__ void make_u(const BigParams& P, int mat, int t, float* us) {
    const float* a = P.ab + ((size_t)mat * P.T + (t - 1)) * (P.M + 1);
    const float* up = P.uh + ((size_t)mat * (P.T + 1) + (t - 1)) * P.M;
    const float b = a[P.M];
    for (int i = threadIdx.x; i < P.M; i += kBT) {
        float u;
        if (P.kind == FZ_SOLVER_HALS) u = fmaxf((a[i] + P.eps) * rcp_nr(b + P.eps), 0.f);
        else u = fmaf(up[i], a[i], P.eps) * rcp_nr(fmaf(up[i], b, P.eps));
        us[i] = u;
    }
    __syncthreads();
}

__device__ __forceinline__ float dot_self(const float* us, int M) {
    float d = 0.f;
    for (int i = 0; i < M; ++i) d = fmaf(us[i], us[i], d);
    return d;
}

// a_0 = X v_0, b_0 = v_0 . v_0; also u_0 into the history
__global__ void __launch_bounds__(kBT) big_init(const BigParams P) {
    __shared__ float red[(kBT / 32) * (2 * kBigMaxM + 2)];
    const int mat = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* X = P.x + (size_t)mat * P.M * P.N;
    const long long j0 = (long long)blockIdx.x * kChunk + threadIdx.x;
    float v[kCPT];
#pragma unroll
    for (int q = 0; q < kCPT; ++q) { const long long j = j0 + q * kBT; v[q] = j < P.N ? __ldg(P.v0 + j) : 0.f; }
    float* r = red + warp * (2 * kBigMaxM + 2);
    for (int i = 0; i < P.M; ++i) {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < kCPT; ++q) {
            const long long j = j0 + q * kBT;
            float xv = j < P.N ? __ldg(X + (size_t)i * P.N + j) : 0.f;
            if (P.relu) xv = fmaxf(xv, 0.f);
            s = fmaf(xv, v[q], s);
        }
        s = warp_sum(s);
        if (lane == 0) r[i] = s;
    }
    float b = 0.f;
#pragma unroll
    for (int q = 0; q < kCPT; ++q) b = fmaf(v[q], v[q], b);
    b = warp_sum(b);
    if (lane == 0) r[P.M] = b;
    flush_rows(red, P.M + 1, P.ab + (size_t)mat * P.T * (P.M + 1));
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < P.M; i += kBT) P.uh[(size_t)mat * (P.T + 1) * P.M + i] = P.u0[i];
}

// sweep t (1..T): u_t, then per column v_t; accumulates a_t, b_t (t < T) or writes y (t == T)
__global__ void __launch_bounds__(kBT) big_sweep(const BigParams P) {
    __shared__ float red[(kBT / 32) * (2 * kBigMaxM + 2)];
    __shared__ float us[kBigMaxM];
    const int mat = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, t = P.t;
    const float* X = P.x + (size_t)mat * P.M * P.N;
    make_u(P, mat, t, us);
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < P.M; i += kBT) P.uh[((size_t)mat * (P.T + 1) + t) * P.M + i] = us[i];
    const float d = dot_self(us, P.M);
    const long long j0 = (long long)blockIdx.x * kChunk + threadIdx.x;
    float c[kCPT], v[kCPT];
#pragma unroll
    for (int q = 0; q < kCPT; ++q) c[q] = 0.f;
    for (int i = 0; i < P.M; ++i) {
        const float ui = us[i];
#pragma unroll
        for (int q = 0; q < kCPT; ++q) {
            const long long j = j0 + q * kBT;
            float xv = j < P.N ? __ldg(X + (size_t)i * P.N + j) : 0.f;
            if (P.relu) xv = fmaxf(xv, 0.f);
            c[q] = fmaf(xv, ui, c[q]);
        }
    }
    const float* vprev = t == 1 ? P.v0 : P.vh + ((size_t)mat * P.T + (t - 2)) * P.N;
    float* vout = P.vh + ((size_t)mat * P.T + (t - 1)) * P.N;
    const float rd = rcp_nr(d + P.eps);
#pragma unroll
    for (int q = 0; q < kCPT; ++q) {
        const long long j = j0 + q * kBT;
        if (j < P.N) {
            if (P.kind == FZ_SOLVER_HALS) v[q] = fmaxf((c[q] + P.eps) * rd, 0.f);
            else { const float vp = __ldg(vprev + j); v[q] = fmaf(vp, c[q], P.eps) * rcp_nr(fmaf(vp, d, P.eps)); }
            vout[j] = v[q];
        } else {
            v[q] = 0.f;
        }
    }
    if (t == P.T) {
        float* Y = P.out + (size_t)mat * P.M * P.N;
        for (int i = 0; i < P.M; ++i) {
            const float ui = us[i];
#pragma unroll
            for (int q = 0; q < kCPT; ++q) {
                const long long j = j0 + q * kBT;
                if (j < P.N) Y[(size_t)i * P.N + j] = ui * v[q];
            }
        }
        return;
    }
    float* r = red + warp * (2 * kBigMaxM + 2);
    for (int i = 0; i < P.M; ++i) {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < kCPT; ++q) {
            const long long j = j0 + q * kBT;
            float xv = j < P.N ? __ldg(X + (size_t)i * P.N + j) : 0.f;
            if (P.relu) xv = fmaxf(xv, 0.f);
            s = fmaf(xv, v[q], s);
        }
        s = warp_sum(s);
        if (lane == 0) r[i] = s;
    }
    float b = 0.f;
#pragma unroll
    for (int q = 0; q < kCPT; ++q) b = fmaf(v[q], v[q], b);
    b = warp_sum(b);
    if (lane == 0) r[P.M] = b;
    flush_rows(red, P.M + 1, P.ab + ((size_t)mat * P.T + t) * (P.M + 1));
}

// Backward pass number `pass` (0 .. K): iteration tA = T - pass gets the adjoint of its v half-step ("A" part, if
// pass < K), iteration tB = T - pass + 1 the column part of the adjoint of its u half-step ("B" part, if pass > 0).
// Per-matrix quantities of tB (abar, bbar, carried u_bar) are rebuilt here from the sums of pass - 1.
__global__ void __launch_bounds__(kBT) big_bwd(const BigParams P) {
    __shared__ float red[(kBT / 32) * (2 * kBigMaxM + 2)];
    __shared__ float ut[kBigMaxM], abar[kBigMaxM], ucar[kBigMaxM];
    __shared__ float sc[4];
    const int mat = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, pass = P.pass, M = P.M, T = P.T;
    const int tA = T - pass, tB = tA + 1;
    const bool doA = pass < P.K, doB = pass > 0;
    const float* X = P.x + (size_t)mat * M * P.N;
    const float eps = P.eps;
    const size_t accw = 2 * (size_t)M + 1;
    float bbar = 0.f;
    // ---- per-matrix part of iteration tB: u_bar(tB) -> abar, bbar, carried u_bar(tB - 1) ----
    if (doB) {
        const float* acc = P.bacc + ((size_t)mat * (P.K + 1) + (pass - 1)) * accw;      // U | S | D of the previous pass
        const float* stp = P.bst + ((size_t)mat * (P.K + 1) + (pass - 1)) * accw;       // its carried u_bar (MU)
        const float* uB = P.uh + ((size_t)mat * (T + 1) + tB) * M;
        const float* uBp = uB - M;
        const float* ab = P.ab + ((size_t)mat * T + (tB - 1)) * (M + 1);                // a = X v_{tB-1}, b
        const float b = ab[M];
        float dB = 0.f;
        for (int i = 0; i < M; ++i) dB = fmaf(uB[i], uB[i], dB);
        const float dbar = P.kind == FZ_SOLVER_HALS ? -rcp_nr(dB + eps) * acc[2 * M] : acc[2 * M];
        float part = 0.f;
        for (int i = threadIdx.x; i < M; i += kBT) {
            const float carry = pass == 1 ? 0.f : stp[M + i];          // dL/du_tB through the u half-step of tB + 1 (MU)
            const float un = acc[i] + acc[M + i] + carry + 2.f * dbar * uB[i];
            if (P.kind == FZ_SOLVER_HALS) {
                const float pb = uB[i] > 0.f ? un : 0.f;
                abar[i] = pb * rcp_nr(b + eps);
                ucar[i] = 0.f;
                part = fmaf(pb, uB[i], part);
            } else {
                const float nb = un * rcp_nr(fmaf(uBp[i], b, eps)), db = -nb * uB[i];
                abar[i] = nb * uBp[i];
                ucar[i] = fmaf(nb, ab[i], db * b);
                part = fmaf(db, uBp[i], part);
            }
        }
        part = warp_sum(part);
        if (lane == 0) red[warp] = part;
        __syncthreads();
        if (threadIdx.x == 0) {
            float s = 0.f;
            for (int w = 0; w < kBT / 32; ++w) s += red[w];
            sc[0] = P.kind == FZ_SOLVER_HALS ? -s * rcp_nr(b + eps) : s;
        }
        __syncthreads();
        bbar = sc[0];
        if (blockIdx.x == 0) {
            float* st = P.bst + ((size_t)mat * (P.K + 1) + pass) * accw;
            for (int i = threadIdx.x; i < M; i += kBT) { st[i] = abar[i]; st[M + i] = ucar[i]; }
            if (threadIdx.x == 0) st[2 * M] = bbar;
        }
    }
    if (doA) {
        const float* uA = P.uh + ((size_t)mat * (T + 1) + tA) * M;
        for (int i = threadIdx.x; i < M; i += kBT) ut[i] = uA[i];
    }
    __syncthreads();
    float dA = 0.f;
    if (doA) dA = dot_self(ut, M);
    const float rdA = rcp_nr(dA + eps);
    const long long j0 = (long long)blockIdx.x * kChunk + threadIdx.x;
    float* DX = P.out + (size_t)mat * M * P.N;
    const float* GY = P.gy + (size_t)mat * M * P.N;
    // v of the iterations involved, at this thread's columns
    const float* vB = !doB ? nullptr : (tB == 1 ? P.v0 : P.vh + ((size_t)mat * T + (tB - 2)) * P.N);    // v_{tB-1} = v_tA
    const float* vAp = !doA ? nullptr : (tA == 1 ? P.v0 : P.vh + ((size_t)mat * T + (tA - 2)) * P.N);   // v_{tA-1}
    const float* vA = !doA ? nullptr : P.vh + ((size_t)mat * T + (tA - 1)) * P.N;                       // v_tA
    float vb[kCPT], cA[kCPT], vcur[kCPT];
#pragma unroll
    for (int q = 0; q < kCPT; ++q) { vb[q] = 0.f; cA[q] = 0.f; vcur[q] = 0.f; }
    // ---- lane-local sums over the rows: X^T abar (B part), X^T u_tA and G^T u_T (A part / seed) ----
    {
        float sB[kCPT];
#pragma unroll
        for (int q = 0; q < kCPT; ++q) sB[q] = 0.f;
        for (int i = 0; i < M; ++i) {
            const float ai = doB ? abar[i] : 0.f, ui = doA ? ut[i] : 0.f;
#pragma unroll
            for (int q = 0; q < kCPT; ++q) {
                const long long j = j0 + q * kBT;
                if (j < P.N) {
                    float xv = __ldg(X + (size_t)i * P.N + j);
                    if (P.relu) xv = fmaxf(xv, 0.f);
                    sB[q] = fmaf(xv, ai, sB[q]);
                    cA[q] = fmaf(xv, ui, cA[q]);
                    if (pass == 0) vb[q] = fmaf(__ldg(GY + (size_t)i * P.N + j), ui, vb[q]);      // seed: G^T u_T
                }
            }
        }
#pragma unroll
        for (int q = 0; q < kCPT; ++q) {
            const long long j = j0 + q * kBT;
            if (j < P.N) {
                if (doB) {
                    const float vp = __ldg(vB + j);
                    vb[q] = P.vbar[(size_t)mat * P.N + j] + fmaf(2.f * bbar, vp, sB[q]);       // dL/dv_{tB-1} complete
                    vcur[q] = vp;
                }
            }
        }
    }
    // ---- A part per column: c_bar, the carried part of dL/dv_{tA-1}, the D sum ----
    float cb[kCPT], dpart = 0.f;
#pragma unroll
    for (int q = 0; q < kCPT; ++q) cb[q] = 0.f;
    if (doA) {
#pragma unroll
        for (int q = 0; q < kCPT; ++q) {
            const long long j = j0 + q * kBT;
            if (j < P.N) {
                const float vt = __ldg(vA + j);
                float keep;
                if (P.kind == FZ_SOLVER_HALS) {
                    const float qb = vt > 0.f ? vb[q] : 0.f;
                    cb[q] = qb * rdA;
                    dpart = fmaf(qb, vt, dpart);
                    keep = 0.f;
                } else {
                    const float vp = __ldg(vAp + j);
                    const float nb = vb[q] * rcp_nr(fmaf(vp, dA, eps)), db = -nb * vt;
                    cb[q] = nb * vp;
                    dpart = fmaf(db, vp, dpart);
                    keep = fmaf(nb, cA[q], db * dA);
                }
                P.vbar[(size_t)mat * P.N + j] = keep;
            }
        }
    }
    // ---- rows again: dX updates and the U, S sums ----
    float* r = red + warp * (2 * kBigMaxM + 2);
    const bool last = pass == P.K;
    for (int i = 0; i < M; ++i) {
        const float ai = doB ? abar[i] : 0.f, ui = doA ? ut[i] : 0.f;
        float sU = 0.f, sS = 0.f;
#pragma unroll
        for (int q = 0; q < kCPT; ++q) {
            const long long j = j0 + q * kBT;
            if (j < P.N) {
                const size_t e = (size_t)i * P.N + j;
                const float xraw = __ldg(X + e);
                const float xv = P.relu ? fmaxf(xraw, 0.f) : xraw;
                float g = pass == 0 ? 0.f : DX[e];
                g = fmaf(ai, vcur[q], g);
                g = fmaf(ui, cb[q], g);
                if (last && P.relu && !(xraw > 0.f)) g = 0.f;
                DX[e] = g;
                if (pass == 0) sU = fmaf(__ldg(GY + e), __ldg(vA + j), sU);          // seed: G v_T
                sS = fmaf(xv, cb[q], sS);
            }
        }
        if (doA) {
            sU = warp_sum(sU);
            sS = warp_sum(sS);
            if (lane == 0) { r[i] = sU; r[M + i] = sS; }
        }
    }
    if (doA) {
        dpart = warp_sum(dpart);
        if (lane == 0) r[2 * M] = dpart;
        flush_rows(red, 2 * M + 1, P.bacc + ((size_t)mat * (P.K + 1) + pass) * accw);
    }
}

size_t big_saved_floats(long long n, int M, long long N, int T) {
    return (size_t)n * ((size_t)T * N + (size_t)(T + 1) * M + (size_t)T * (M + 1));
}

void big_carve(BigParams& P, void* saved) {
    float* p = static_cast<float*>(saved);
    P.vh = p; p += (size_t)P.n * P.T * P.N;
    P.uh = p; p += (size_t)P.n * (P.T + 1) * P.M;
    P.ab = p;
}

}  // namespace

bool big_supported(int M, long long N, const fz_solver& s) {
    if (s.rank != 1 || s.num_iters < 1 || s.num_iters > kBigMaxT) return false;
    if (s.kind != FZ_SOLVER_HALS && s.kind != FZ_SOLVER_MU) return false;
    return M >= 1 && M <= kBigMaxM && N >= 1 && N < (1LL << 31);
}

size_t big_saved_bytes(long long n, int M, long long N, const fz_solver& s) {
    return big_saved_floats(n, M, N, s.num_iters) * sizeof(float);
}

size_t big_workspace_bytes(long long n, int M, long long N, const fz_solver& s) {
    // backward: vbar (n N) + sums and state (2 x n (T + 1) (2M + 1)); forward without a `saved` buffer: the history
    const size_t bwd = ((size_t)n * N + 2 * (size_t)n * (s.num_iters + 1) * (2 * (size_t)M + 1)) * sizeof(float);
    const size_t fwd = big_saved_bytes(n, M, N, s);
    return bwd > fwd ? bwd : fwd;
}

int big_forward(const float* x, const float* u0, const float* v0, float* y, void* saved, void* workspace, long long n, int M,
                long long N, const fz_solver& s, int relu, cudaStream_t st) {
    void* hist = saved ? saved : workspace;
    if (!hist) return fail(FZ_ERR_INVALID, "large-matrix NMF needs a %zu-byte `saved` or `workspace` buffer", big_saved_bytes(n, M, N, s));
    if (n == 0) return FZ_OK;
    BigParams P;
    memset(&P, 0, sizeof(P));
    P.x = x; P.out = y; P.u0 = u0; P.v0 = v0; P.N = N; P.M = M; P.n = (int)n; P.T = s.num_iters; P.kind = s.kind; P.relu = relu;
    P.eps = s.eps;
    big_carve(P, hist);
    FZ_CUDA_CHECK(cudaMemsetAsync(P.ab, 0, (size_t)n * P.T * (M + 1) * sizeof(float), st));
    const dim3 grid((unsigned)((N + kChunk - 1) / kChunk), (unsigned)n);
    big_init<<<grid, kBT, 0, st>>>(P);
    FZ_LAUNCH_CHECK();
    for (int t = 1; t <= P.T; ++t) {
        P.t = t;
        big_sweep<<<grid, kBT, 0, st>>>(P);
        FZ_LAUNCH_CHECK();
    }
    return FZ_OK;
}

int big_backward(const float* x, const float* gy, const float* u0, const float* v0, const void* saved, float* gx,
                 void* workspace, long long n, int M, long long N, const fz_solver& s, int K, int relu, cudaStream_t st) {
    if (!saved || !workspace) return fail(FZ_ERR_INVALID, "large-matrix NMF backward needs the forward's `saved` buffer and a workspace");
    if (n == 0) return FZ_OK;
    BigParams P;
    memset(&P, 0, sizeof(P));
    P.x = x; P.gy = gy; P.out = gx; P.u0 = u0; P.v0 = v0; P.N = N; P.M = M; P.n = (int)n; P.T = s.num_iters; P.K = K;
    P.kind = s.kind; P.relu = relu; P.eps = s.eps;
    big_carve(P, const_cast<void*>(saved));
    float* w = static_cast<float*>(workspace);
    const size_t accw = 2 * (size_t)M + 1;
    P.vbar = w; w += (size_t)n * N;
    P.bacc = w; w += (size_t)n * (K + 1) * accw;
    P.bst = w;
    if (K == 0) {
        FZ_CUDA_CHECK(cudaMemsetAsync(gx, 0, (size_t)n * M * N * sizeof(float), st));
        return FZ_OK;
    }
    FZ_CUDA_CHECK(cudaMemsetAsync(P.bacc, 0, (size_t)n * (K + 1) * accw * sizeof(float), st));
    const dim3 grid((unsigned)((N + kChunk - 1) / kChunk), (unsigned)n);
    for (int pass = 0; pass <= K; ++pass) {
        P.pass = pass;
        big_bwd<<<grid, kBT, 0, st>>>(P);
        FZ_LAUNCH_CHECK();
    }
    return FZ_OK;
}

}  // namespace fz
