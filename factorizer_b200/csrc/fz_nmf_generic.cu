// Generic shared-memory NMF kernels: any (M, N) that fits in shared memory, rank 1..4, MU and HALS,
// forward and backward, on either already-matricised tensors (ft.NMF standalone) or on windows
// gathered straight from the NCDHW volume (the FactMixer core for geometries the specialised
// register/TMA kernel does not cover).
//
// One CTA owns one matrix at a time: X (and in backward the iterates and the dX accumulator) live in
// shared memory; the M-sided reductions are warp-per-dot-product, the N-sided updates are
// thread-per-column.  The math follows the reference line by line:
//   MU   half-step  factorizer/factorization/matrix_factorization.py:241-247
//   HALS half-step  factorizer/factorization/matrix_factorization.py:210-229 (project = ReLU, :609)
//   Gauss-Seidel order u then v with x.mT  :122-136;  decompose loop :514-530;  reconstruct :532-533
// The backward is the hand-derived adjoint of the unrolled loop (SURVEY.md App. A), restated in
// oracle/factorizer_oracle.py::_half_bwd and checked against the reference's autograd.
#include "fz_common.cuh"
#include "fz_internal.cuh"

namespace fz {

constexpr int kThreads = 256;

template <int R>
__device__ __forceinline__ void update_row(float* un, const float* uo, const float* a,
                                           const float* bm, int kind, float eps) {
    // un: out new row (R), uo: old row, a: row of A, bm: RxR gram
    if (kind == FZ_SOLVER_MU) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float den = 0.f;
#pragma unroll
            for (int s = 0; s < R; ++s) den = fmaf(uo[s], bm[s * R + r], den);
            un[r] = __fdiv_rn(fmaf(uo[r], a[r], eps), den + eps);
        }
    } else {
#pragma unroll
        for (int r = 0; r < R; ++r) un[r] = uo[r];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float dot = 0.f;
#pragma unroll
            for (int s = 0; s < R; ++s)
                if (s != r) dot = fmaf(un[s], bm[s * R + r], dot);
            float pre = __fdiv_rn((a[r] - dot) + eps, bm[r * R + r] + eps);
            un[r] = fmaxf(pre, 0.f);
        }
    }
}

// Adjoint of update_row.  g: dL/d un (R, clobbered).  Outputs gprev (dL/d uo), ga (dL/d a row),
// gbm (R*R partial of dL/d bm, *added into*).
template <int R>
__device__ __forceinline__ void update_row_bwd(float* g, const float* uo, const float* un,
                                               const float* a, const float* bm, int kind, float eps,
                                               float* gprev, float* ga, float* gbm) {
    if (kind == FZ_SOLVER_MU) {
        float gn[R], gd[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float den = 0.f;
#pragma unroll
            for (int s = 0; s < R; ++s) den = fmaf(uo[s], bm[s * R + r], den);
            den += eps;
            gn[r] = __fdiv_rn(g[r], den);
            gd[r] = -__fdiv_rn(g[r] * un[r], den);
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float acc = gn[r] * a[r];
#pragma unroll
            for (int s = 0; s < R; ++s) acc = fmaf(gd[s], bm[r * R + s], acc);
            gprev[r] = acc;
            ga[r] = gn[r] * uo[r];
#pragma unroll
            for (int s = 0; s < R; ++s) gbm[s * R + r] = fmaf(uo[s], gd[r], gbm[s * R + r]);
        }
    } else {
#pragma unroll
        for (int r = 0; r < R; ++r) { gprev[r] = 0.f; ga[r] = 0.f; }
#pragma unroll
        for (int r = R - 1; r >= 0; --r) {
            const float gg = un[r] > 0.f ? g[r] : 0.f;  // pre_r > 0  <=>  un_r > 0
            const float den = bm[r * R + r] + eps;
            const float acc = __fdiv_rn(gg, den);
            gbm[r * R + r] -= __fdiv_rn(gg * un[r], den);  // pre_r == un_r wherever gg != 0
            ga[r] += acc;
#pragma unroll
            for (int s = 0; s < R; ++s) {
                if (s == r) continue;
                const float colval = s < r ? un[s] : uo[s];
                gbm[s * R + r] = fmaf(-acc, colval, gbm[s * R + r]);
                const float contrib = -acc * bm[s * R + r];
                if (s < r) g[s] += contrib; else gprev[s] += contrib;
            }
        }
    }
}

struct Smem {
    float *X, *GX, *V, *U, *A, *Bm, *GB, *VH, *UH, *GV, *GC, *GU, *GA, *red, *rowpart;
    int* coloff;
};

// ---- cooperative phases ---------------------------------------------------------------------------
// a[i][r] = sum_j X[i][j] * V[r][j]  and  bm[r][s] = sum_j V[r][j] V[s][j];  warp per dot product.
template <int R>
__device__ __forceinline__ void phase_gram_rows(const float* X, const float* V, float* A, float* Bm,
                                                int M, int N) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int tasks = M * R + R * R;
    for (int q = warp; q < tasks; q += nw) {
        const float *p0, *p1;
        if (q < M * R) { p0 = X + (q / R) * N; p1 = V + (q % R) * N; }
        else { int e = q - M * R; p0 = V + (e / R) * N; p1 = V + (e % R) * N; }
        float acc = 0.f;
        for (int j = lane; j < N; j += 32) acc = fmaf(p0[j], p1[j], acc);
        acc = warp_sum(acc);
        if (lane == 0) { if (q < M * R) A[q] = acc; else Bm[q - M * R] = acc; }
    }
}

template <int R>
__device__ __forceinline__ void phase_gram_small(const float* U, float* Dm, int M) {
    if (threadIdx.x < R * R) {
        const int r = threadIdx.x / R, s = threadIdx.x % R;
        float acc = 0.f;
        for (int i = 0; i < M; ++i) acc = fmaf(U[i * R + r], U[i * R + s], acc);
        Dm[threadIdx.x] = acc;
    }
}

// One forward iteration on shared-memory operands: U (M,R) and V (R,N) updated in place.
template <int R>
__device__ __forceinline__ void iterate(const float* X, float* U, float* V, float* A, float* Bm,
                                        int M, int N, int kind, float eps) {
    phase_gram_rows<R>(X, V, A, Bm, M, N);
    __syncthreads();
    if (threadIdx.x < M) {
        const int i = threadIdx.x;
        float uo[R], un[R], ar[R];
#pragma unroll
        for (int r = 0; r < R; ++r) { uo[r] = U[i * R + r]; ar[r] = A[i * R + r]; }
        update_row<R>(un, uo, ar, Bm, kind, eps);
#pragma unroll
        for (int r = 0; r < R; ++r) U[i * R + r] = un[r];
    }
    __syncthreads();
    phase_gram_small<R>(U, Bm, M);  // Bm now holds d = u^T u
    __syncthreads();
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        float c[R], vo[R], vn[R];
#pragma unroll
        for (int r = 0; r < R; ++r) { c[r] = 0.f; vo[r] = V[r * N + j]; }
        for (int i = 0; i < M; ++i) {
            const float xv = X[i * N + j];
#pragma unroll
            for (int r = 0; r < R; ++r) c[r] = fmaf(xv, U[i * R + r], c[r]);
        }
        update_row<R>(vn, vo, c, Bm, kind, eps);
#pragma unroll
        for (int r = 0; r < R; ++r) V[r * N + j] = vn[r];
    }
    __syncthreads();
}

template <bool WINDOW>
__device__ __forceinline__ void locate(const NmfArgs& a, long long mid, int* coloff,
                                       long long* base) {
    if (WINDOW) {
        const DevGeom& G = a.G;
        const int w = (int)(mid % G.G);
        long long t = mid / G.G;
        const int h = (int)(t % G.heads);
        const int b = (int)(t / G.heads);
        *base = ((long long)b * G.C + (long long)h * G.d) * G.vox;
        for (int j = threadIdx.x; j < a.N; j += blockDim.x)
            coloff[j] = (int)window_col_offset(G, a.shift, w, j);
    } else {
        *base = mid * (long long)a.M * a.N;
    }
}

template <bool WINDOW>
__device__ __forceinline__ void load_tile(float* dst, const float* src, long long base,
                                          const int* coloff, int M, int N, long long vox, bool relu,
                                          float scale_div) {
    for (int e = threadIdx.x; e < M * N; e += blockDim.x) {
        float v;
        if (WINDOW) {
            const int i = e / N, j = e - i * N;
            v = __ldg(src + base + (long long)i * vox + coloff[j]);
        } else {
            v = __ldg(src + base + e);
        }
        if (relu) v = fmaxf(v, 0.f);
        if (scale_div != 1.f) v = __fdiv_rn(v, scale_div);
        dst[e] = v;
    }
}

__device__ __forceinline__ Smem carve(float* smem, int M, int N, int R, int T, bool bwd, bool window, bool spill) {
    Smem s;
    float* p = smem;
    s.X = p;
    if (!spill) p += M * N;
    s.V = p; p += R * N;
    s.U = p; p += M * R;
    s.A = p; p += M * R;
    s.Bm = p; p += R * R;
    s.GX = s.VH = s.UH = s.GV = s.GC = s.GU = s.GA = s.GB = s.red = s.rowpart = nullptr;
    if (bwd) {
        s.GX = p;
        if (!spill) p += M * N;
        s.VH = p; p += (T + 1) * R * N;
        s.UH = p; p += (T + 1) * M * R;
        s.GV = p; p += R * N;
        s.GC = p; p += R * N;
        s.GU = p; p += M * R;
        s.GA = p; p += M * R;
        s.GB = p; p += R * R;
        s.red = p; p += (kThreads / 32) * R * R;
        s.rowpart = p; p += M * R * R;
    }
    s.coloff = window ? reinterpret_cast<int*>(p) : nullptr;
    return s;
}

size_t generic_smem_bytes(int M, int N, int R, int T, bool bwd, bool window, bool spill = false) {
    const size_t mn = spill ? 0 : (size_t)M * N;
    size_t f = mn + (size_t)R * N + 2 * (size_t)M * R + (size_t)R * R;
    if (bwd)
        f += mn + (size_t)(T + 1) * R * N + (size_t)(T + 1) * M * R + 2 * (size_t)R * N +
             2 * (size_t)M * R + (size_t)R * R + (size_t)(kThreads / 32) * R * R + (size_t)M * R * R;
    if (window) f += (size_t)N;
    return f * sizeof(float);
}

// ---- forward ------------------------------------------------------------------------------------
template <int R, bool WINDOW>
__global__ void __launch_bounds__(kThreads) nmf_fwd_generic(NmfArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const int M = a.M, N = a.N;
    const bool spill = !WINDOW && a.spill;
    Smem s = carve(smem_f, M, N, R, a.T, false, WINDOW, spill);
    for (long long mid = blockIdx.x; mid < a.n; mid += gridDim.x) {
        long long base;
        locate<WINDOW>(a, mid, s.coloff, &base);
        if (WINDOW) __syncthreads();
        if (spill) s.X = const_cast<float*>(a.x) + base;        // read in place (generic addressing; L2-resident across the sweeps)
        else load_tile<WINDOW>(s.X, a.x, base, s.coloff, M, N, a.G.vox, WINDOW && a.relu, 1.f);
        for (int e = threadIdx.x; e < M * R; e += blockDim.x) s.U[e] = a.u0[e];
        for (int e = threadIdx.x; e < N * R; e += blockDim.x) s.V[(e % R) * N + e / R] = a.v0[e];
        __syncthreads();
        for (int t = 0; t < a.T; ++t) iterate<R>(s.X, s.U, s.V, s.A, s.Bm, M, N, a.kind, a.eps);
        if (a.u)
            for (int e = threadIdx.x; e < M * R; e += blockDim.x) a.u[mid * M * R + e] = s.U[e];
        if (a.v)
            for (int e = threadIdx.x; e < N * R; e += blockDim.x)
                a.v[mid * (long long)N * R + e] = s.V[(e % R) * N + e / R];
        if (a.y) {
            for (int e = threadIdx.x; e < M * N; e += blockDim.x) {
                const int i = e / N, j = e - i * N;
                float acc = 0.f;
#pragma unroll
                for (int r = 0; r < R; ++r) acc = fmaf(s.U[i * R + r], s.V[r * N + j], acc);
                if (WINDOW) {
                    // SWMatricize.inverse_forward order (operations.py:426-433): one launch per
                    // window set, out = out + inv_s, the last set divides by S.
                    float* dst = a.y + base + (long long)i * a.G.vox + s.coloff[j];
                    if (a.shift > 0) acc = __fadd_rn(*dst, acc);
                    if (a.shift == a.G.S - 1) acc = __fdiv_rn(acc, (float)a.G.S);
                    *dst = acc;
                } else {
                    a.y[base + e] = acc;
                }
            }
        }
        __syncthreads();
    }
}

// ---- backward -----------------------------------------------------------------------------------
template <int R, bool WINDOW>
__global__ void __launch_bounds__(kThreads) nmf_bwd_generic(NmfArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const int M = a.M, N = a.N, T = a.T;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const bool spill = !WINDOW && a.spill;
    Smem s = carve(smem_f, M, N, R, T, true, WINDOW, spill);
    for (long long mid = blockIdx.x; mid < a.n; mid += gridDim.x) {
        long long base;
        locate<WINDOW>(a, mid, s.coloff, &base);
        if (WINDOW) __syncthreads();
        if (spill) {                                             // X read in place, the gradient accumulated in its output buffer
            s.X = const_cast<float*>(a.x) + base;
            s.GX = a.gx + base;
        } else {
            load_tile<WINDOW>(s.X, a.x, base, s.coloff, M, N, a.G.vox, WINDOW && a.relu, 1.f);
        }
        // upstream gradient staged in GX for the two initial products
        if (a.gy) {
            load_tile<WINDOW>(s.GX, a.gy, base, s.coloff, M, N, a.G.vox, false,
                              WINDOW ? (float)a.G.S : 1.f);
        } else {
            for (int e = threadIdx.x; e < M * N; e += blockDim.x) s.GX[e] = 0.f;
        }
        for (int e = threadIdx.x; e < M * R; e += blockDim.x) s.U[e] = s.UH[e] = a.u0[e];
        for (int e = threadIdx.x; e < N * R; e += blockDim.x)
            s.V[(e % R) * N + e / R] = s.VH[(e % R) * N + e / R] = a.v0[e];
        __syncthreads();
        // recompute and keep every iterate
        for (int t = 1; t <= T; ++t) {
            iterate<R>(s.X, s.U, s.V, s.A, s.Bm, M, N, a.kind, a.eps);
            for (int e = threadIdx.x; e < M * R; e += blockDim.x) s.UH[t * M * R + e] = s.U[e];
            for (int e = threadIdx.x; e < N * R; e += blockDim.x) s.VH[t * R * N + e] = s.V[e];
        }
        __syncthreads();
        // gv = gv_in + G^T u_T ; gu = gu_in + G v_T   (matrix_factorization.py:532-533 adjoint)
        for (int j = threadIdx.x; j < N; j += blockDim.x) {
            float acc[R];
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = a.gv ? a.gv[mid * (long long)N * R + j * R + r] : 0.f;
            for (int i = 0; i < M; ++i) {
                const float gvv = s.GX[i * N + j];
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = fmaf(gvv, s.U[i * R + r], acc[r]);
            }
#pragma unroll
            for (int r = 0; r < R; ++r) s.GV[r * N + j] = acc[r];
        }
        for (int q = warp; q < M * R; q += nw) {
            const float* p0 = s.GX + (q / R) * N;
            const float* p1 = s.V + (q % R) * N;
            float acc = 0.f;
            for (int j = lane; j < N; j += 32) acc = fmaf(p0[j], p1[j], acc);
            acc = warp_sum(acc);
            if (lane == 0) s.GU[q] = acc + (a.gu ? a.gu[mid * M * R + q] : 0.f);
        }
        __syncthreads();
        for (int e = threadIdx.x; e < M * N; e += blockDim.x) s.GX[e] = 0.f;
        __syncthreads();

        for (int t = T; t > T - a.K; --t) {
            const float* Ut = s.UH + t * M * R;
            const float* Up = s.UH + (t - 1) * M * R;
            const float* Vt = s.VH + t * R * N;
            const float* Vp = s.VH + (t - 1) * R * N;
            // ---- adjoint of v_t = update(x.mT, v_{t-1}, u_t) ----
            phase_gram_small<R>(Ut, s.Bm, M);
            __syncthreads();
            float part[R * R];
#pragma unroll
            for (int q = 0; q < R * R; ++q) part[q] = 0.f;
            for (int j = threadIdx.x; j < N; j += blockDim.x) {
                float c[R], vp[R], vn[R], g[R], gprev[R], gc[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    c[r] = 0.f; vp[r] = Vp[r * N + j]; vn[r] = Vt[r * N + j]; g[r] = s.GV[r * N + j];
                }
                for (int i = 0; i < M; ++i) {
                    const float xv = s.X[i * N + j];
#pragma unroll
                    for (int r = 0; r < R; ++r) c[r] = fmaf(xv, Ut[i * R + r], c[r]);
                }
                update_row_bwd<R>(g, vp, vn, c, s.Bm, a.kind, a.eps, gprev, gc, part);
#pragma unroll
                for (int r = 0; r < R; ++r) { s.GC[r * N + j] = gc[r]; s.GV[r * N + j] = gprev[r]; }
            }
#pragma unroll
            for (int q = 0; q < R * R; ++q) {
                const float v = warp_sum(part[q]);
                if (lane == 0) s.red[warp * R * R + q] = v;
            }
            __syncthreads();
            if (threadIdx.x < R * R) {
                float acc = 0.f;
                for (int w = 0; w < nw; ++w) acc += s.red[w * R * R + threadIdx.x];
                s.GB[threadIdx.x] = acc;
            }
            __syncthreads();
            // gu_t += X gc + u_t (GB + GB^T);   GX += u_t gc^T
            for (int q = warp; q < M * R; q += nw) {
                const int i = q / R, r = q % R;
                const float* p0 = s.X + i * N;
                const float* p1 = s.GC + r * N;
                float acc = 0.f;
                for (int j = lane; j < N; j += 32) acc = fmaf(p0[j], p1[j], acc);
                acc = warp_sum(acc);
                if (lane == 0) {
#pragma unroll
                    for (int sidx = 0; sidx < R; ++sidx)
                        acc = fmaf(Ut[i * R + sidx], s.GB[sidx * R + r] + s.GB[r * R + sidx], acc);
                    s.GU[q] += acc;
                }
            }
            for (int j = threadIdx.x; j < N; j += blockDim.x) {
                float gc[R];
#pragma unroll
                for (int r = 0; r < R; ++r) gc[r] = s.GC[r * N + j];
                for (int i = 0; i < M; ++i) {
                    float acc = s.GX[i * N + j];
#pragma unroll
                    for (int r = 0; r < R; ++r) acc = fmaf(Ut[i * R + r], gc[r], acc);
                    s.GX[i * N + j] = acc;
                }
            }
            __syncthreads();
            // ---- adjoint of u_t = update(x, u_{t-1}, v_{t-1}) ----
            phase_gram_rows<R>(s.X, Vp, s.A, s.Bm, M, N);
            __syncthreads();
            if (threadIdx.x < M) {
                const int i = threadIdx.x;
                float up[R], un[R], g[R], ar[R], gprev[R], ga[R], rp[R * R];
#pragma unroll
                for (int q = 0; q < R * R; ++q) rp[q] = 0.f;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    up[r] = Up[i * R + r]; un[r] = Ut[i * R + r]; g[r] = s.GU[i * R + r]; ar[r] = s.A[i * R + r];
                }
                update_row_bwd<R>(g, up, un, ar, s.Bm, a.kind, a.eps, gprev, ga, rp);
#pragma unroll
                for (int r = 0; r < R; ++r) { s.GA[i * R + r] = ga[r]; s.GU[i * R + r] = gprev[r]; }
#pragma unroll
                for (int q = 0; q < R * R; ++q) s.rowpart[i * R * R + q] = rp[q];
            }
            __syncthreads();
            if (threadIdx.x < R * R) {
                float acc = 0.f;
                for (int i = 0; i < M; ++i) acc += s.rowpart[i * R * R + threadIdx.x];
                s.GB[threadIdx.x] = acc;
            }
            __syncthreads();
            // GX += ga v_{t-1}^T ;  gv_{t-1} += X^T ga + v_{t-1} (GB + GB^T)
            for (int j = threadIdx.x; j < N; j += blockDim.x) {
                float vp[R], acc_v[R];
#pragma unroll
                for (int r = 0; r < R; ++r) { vp[r] = Vp[r * N + j]; acc_v[r] = s.GV[r * N + j]; }
                for (int i = 0; i < M; ++i) {
                    const float xv = s.X[i * N + j];
                    float acc = s.GX[i * N + j];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const float ga = s.GA[i * R + r];
                        acc = fmaf(ga, vp[r], acc);
                        acc_v[r] = fmaf(xv, ga, acc_v[r]);
                    }
                    s.GX[i * N + j] = acc;
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float acc = acc_v[r];
#pragma unroll
                    for (int sidx = 0; sidx < R; ++sidx)
                        acc = fmaf(vp[sidx], s.GB[sidx * R + r] + s.GB[r * R + sidx], acc);
                    s.GV[r * N + j] = acc;
                }
            }
            __syncthreads();
        }
        // ---- write dX (ReLU mask folded, factorizer.py:44 adjoint) ----
        for (int e = threadIdx.x; e < M * N; e += blockDim.x) {
            float val = s.GX[e];
            if (WINDOW) {
                if (a.relu && !(s.X[e] > 0.f)) val = 0.f;
                const int i = e / N, j = e - i * N;
                float* dst = a.gx + base + (long long)i * a.G.vox + s.coloff[j];
                if (a.shift > 0) val += *dst;
                *dst = val;
            } else {
                a.gx[base + e] = val;
            }
        }
        __syncthreads();
    }
}

// ---- host launchers -------------------------------------------------------------------------------
template <int R, bool WINDOW>
static int launch_generic(const NmfArgs& a_in, bool bwd, cudaStream_t st) {
    NmfArgs a = a_in;
    a.spill = 0;
    size_t smem = generic_smem_bytes(a.M, a.N, R, a.T, bwd, WINDOW);
    if (smem > 227 * 1024 && !WINDOW) {        // standalone matrices: leave X (and dX) in global memory
        a.spill = 1;
        smem = generic_smem_bytes(a.M, a.N, R, a.T, bwd, WINDOW, true);
    }
    if (smem > 227 * 1024)
        return fail(FZ_ERR_UNSUPPORTED,
                    "matrix %dx%d (rank %d, %d iters) needs %zu B of shared memory in the generic "
                    "%s kernel; the limit is 232448 B", a.M, a.N, R, a.T, smem, bwd ? "backward" : "forward");
    if (a.n == 0) return FZ_OK;
    auto kern = bwd ? nmf_bwd_generic<R, WINDOW> : nmf_fwd_generic<R, WINDOW>;
    if (smem > 48 * 1024)
        FZ_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    FZ_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, smem));
    if (per_sm < 1) per_sm = 1;
    long long grid = (long long)num_sms() * per_sm;
    if (grid > a.n) grid = a.n;
    kern<<<(unsigned)grid, kThreads, smem, st>>>(a);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

template <bool WINDOW>
static int dispatch_rank(const NmfArgs& a, int R, bool bwd, cudaStream_t st) {
    switch (R) {
        case 1: return launch_generic<1, WINDOW>(a, bwd, st);
        case 2: return launch_generic<2, WINDOW>(a, bwd, st);
        case 3: return launch_generic<3, WINDOW>(a, bwd, st);
        case 4: return launch_generic<4, WINDOW>(a, bwd, st);
        case 5: return launch_generic<5, WINDOW>(a, bwd, st);
        case 6: return launch_generic<6, WINDOW>(a, bwd, st);
        case 7: return launch_generic<7, WINDOW>(a, bwd, st);
        case 8: return launch_generic<8, WINDOW>(a, bwd, st);
        default: return fail(FZ_ERR_UNSUPPORTED, "rank %d not supported (1..%d)", R, FZ_MAX_RANK);
    }
}

int check_solver(const fz_solver* s, int M, int N, int* K) {
    if (!s) return fail(FZ_ERR_INVALID, "null solver");
    if (s->kind != FZ_SOLVER_MU && s->kind != FZ_SOLVER_HALS)
        return fail(FZ_ERR_UNSUPPORTED, "solver kind %d not implemented (only 'mu' and 'hals')", s->kind);
    if (s->rank < 1 || s->rank > FZ_MAX_RANK)
        return fail(FZ_ERR_UNSUPPORTED, "rank %d not supported (1..%d)", s->rank, FZ_MAX_RANK);
    if (s->num_iters < 0) return fail(FZ_ERR_INVALID, "num_iters %d < 0", s->num_iters);
    if (M < 1 || N < 1) return fail(FZ_ERR_INVALID, "empty matrix %dx%d", M, N);
    if (M > kThreads) return fail(FZ_ERR_UNSUPPORTED, "M=%d > %d rows not supported", M, kThreads);
    int k = s->num_grad_steps;
    if (k < 0 || k > s->num_iters) k = s->num_iters;
    *K = k;
    return FZ_OK;
}

int generic_direct(const NmfArgs& a, int R, bool bwd, cudaStream_t st) {
    return dispatch_rank<false>(a, R, bwd, st);
}

// One launch per window set, in shift order (keeps the reference's summation order).
int generic_window(NmfArgs a, int R, bool bwd, cudaStream_t st) {
    for (int s = 0; s < a.G.S; ++s) {
        a.shift = s;
        if (int e = dispatch_rank<true>(a, R, bwd, st)) return e;
    }
    return FZ_OK;
}

}  // namespace fz
