// Gram-matrix form of the rank-1 HALS layer for non-negative windows (act = ReLU, the configuration
// of every Swin-Factorizer block).  Included at the end of fz_swnmf_fast.cu (same namespace, same
// FastParams / window order / completion counters); the kernels there remain the path for act = Identity.
//
// With X >= 0 no ReLU of the solver ever clips after the first half-step (a = X v >= 0, c = X^T u >= 0),
// so every iterate after u_1 lives in the 8-dimensional row space of X:
//     v_t = rd_t (X^T u_t + eps 1),  rd_t = 1 / (u_t.u_t + eps)
//     a_{t+1} = X v_t = rd_t (Gam u_t + eps r),            Gam = X X^T (8x8),  r = X 1
//     b_{t+1} = v_t.v_t = rd_t^2 (u_t.Gam u_t + 2 eps u_t.r + 512 eps^2)
//     u_{t+1} = relu((a_{t+1} + eps) / (b_{t+1} + eps))
// (reference matrix_factorization.py:224-227 evaluated on both half-steps, :122-136).  One pass over the
// window gives Gam, r and a_1 = X v_0; ONE cross-lane reduction replaces the T reductions of the direct
// form, the T sweeps become 8-vector arithmetic, and a second pass gives v_T and Y = u_T v_T^T.  The
// backward is the same idea applied to SURVEY App. A.3: vbar_t = X^T z_t + kappa_t 1 for t < T, so
//     X cbar_t = rd_t (Gam z_t + kappa_t r),   qbar_t.v_t = rd_t (z_t.Gam u_t + eps z_t.r + kappa_t u_t.r + 512 kappa_t eps)
//     dX = rd_T u_T gv^T + M X + m 1^T + abar_1 v_0^T,   gv = G^T u_T,
//     M = sum_{t<T} rd_t (u_t z_t^T + abar_{t+1} u_t^T),   m = sum_{t<T} rd_t (kappa_t u_t + eps abar_{t+1})
// with z_t = abar_{t+1} + 2 bbar_{t+1} rd_t u_t, kappa_t = 2 bbar_{t+1} rd_t eps: one reduction (of
// G v_T + X cbar_T and qbar_T.v_T), an 8-vector recursion, and one 8x8 by 8x512 product per window.
// fp32 error of this form against the fp64 reference is below the reference's own fp32 error
// (tests/test_oracle.py::test_gram_form_is_well_conditioned pins that on the golden vectors).
//
// Forward: ONE warp per window (lane: 16 columns of all 8 rows in registers), no block-level barrier at
// all; backward: a pair of warps per window as in the direct kernels, one named barrier per window.
#pragma once

constexpr int kGFwdWarps = 8;         // forward: 8 independent warps / CTA, 1 CTA / SM
constexpr int kGBwdPairs = 4;         // backward: 4 pairs / CTA, 1 CTA / SM
constexpr int kGramVals = 52;         // 36 (upper triangle of Gam) + 8 (r) + 8 (a_1)
constexpr int kGramFloats = 80;       // shared-memory image: full 8x8 Gam, r, a_1

// ---- one-warp-per-window addressing (forward) -------------------------------------------------------
// Lane l owns chunks r = l + 32 j (j = 0..3) of every row: q0 = (l >> 4) + 2 j, q1 = (l >> 1) & 7,
// q2 = 4 (l & 1) + e.
struct LaneAddr4 {
    int rowoff[4];   // (i0 * n1 + i1) * n2 for the four chunks
    int i2;          // W coordinate of the chunks' first column (the following ones may wrap)
};
__device__ __forceinline__ LaneAddr4 lane_addr4(const FastParams& P, const Info& it, int lane) {
    LaneAddr4 a;
    int i1 = it.c1 + ((lane >> 1) & 7); if (i1 >= P.n1) i1 -= P.n1;
    int i2 = it.c2 + 4 * (lane & 1); if (i2 >= P.n2) i2 -= P.n2;
    a.i2 = i2;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int i0 = it.c0 + (lane >> 4) + 2 * j; if (i0 >= P.n0) i0 -= P.n0;
        a.rowoff[j] = (i0 * P.n1 + i1) * P.n2;
    }
    return a;
}

// fetch window `it` into `tile` (standard layout) with the 32 lanes of one warp; one phase of `bar`
// (32 arrivals + the TMA byte count)
__device__ __forceinline__ void fetch_tile_warp(const FastParams& P, const Info& it, int lane, float* tile, uint64_t* bar) {
    if (it.flags & kInterior) {
        if (lane == 0) {
            mbar_expect_tx(bar, kTileBytes);
            tma_load_tile(tile, &P.tm_x, bar, it.c2, it.c1, it.c0, it.head * 8, it.b);
        }
        mbar_arrive(bar);
    } else {
        const LaneAddr4 a = lane_addr4(P, it, lane);
        const float* base = P.x + it.chan_base;
        if (it.flags & kAligned4) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    cp_async16(tile + i * 512 + 4 * (lane + 32 * j), base + (long long)i * P.vox + a.rowoff[j] + a.i2);
        } else {
#pragma unroll 1
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        cp_async4(tile + i * 512 + 4 * (lane + 32 * j) + e,
                                  base + (long long)i * P.vox + a.rowoff[j] + wrap2(P, a.i2 + e));
        }
        mbar_arrive_after_cp_async(bar);
    }
}

// a[row] for a register array and a run-time row (a select chain; dynamic indexing would spill the array)
__device__ __forceinline__ float pick8(const float (&a)[8], int row) {
    float v = a[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) v = (row == j) ? a[j] : v;
    return v;
}

// one level of a recursive-halving all-reduce: N values -> ceil(N/2); lanes with `hi` keep the upper half
template <int N>
__device__ __forceinline__ void halve_level(float (&v)[kGramVals], bool hi, int bit) {
    constexpr int m = (N + 1) / 2;
#pragma unroll
    for (int j = 0; j < N - m; ++j) {
        const float keep = hi ? v[j + m] : v[j], send = hi ? v[j] : v[j + m];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
    if (N & 1) v[m - 1] += __shfl_xor_sync(0xffffffffu, v[m - 1], bit);
}
template <int N>
__device__ __forceinline__ void halve_ids(int (&id)[kGramVals], bool hi) {
    constexpr int m = (N + 1) / 2;
#pragma unroll
    for (int j = 0; j < N - m; ++j) id[j] = hi ? id[j + m] : id[j];
}

// =====================================================================================================
// forward, Gram form
// =====================================================================================================
__global__ void __launch_bounds__(kGFwdWarps * 32, 1) swnmf_fwd_gram(const __grid_constant__ FastParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ __align__(16) float gram_all[kGFwdWarps][kGramFloats];
    __shared__ uint64_t full_all[kGFwdWarps];
    __shared__ int pos_tab[2][kGramVals];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* xin = reinterpret_cast<float*>(smem_raw) + (size_t)warp * 4096;
    float* stage = reinterpret_cast<float*>(smem_raw) + (size_t)kGFwdWarps * 4096 + (size_t)warp * 2048;   // half a Y tile
    float* gram = gram_all[warp];
    uint64_t* full = &full_all[warp];
    const long long G = (long long)P.NR * P.G2;
    const float eps = P.eps;

    for (int j = threadIdx.x; j < 512; j += blockDim.x) v0s[j] = P.v0[j];
    if (threadIdx.x < kGramVals) {
        // where value s of the reduction goes in the shared image: Gam(i,j) and Gam(j,i), r, a_1
        const int s = threadIdx.x;
        int a, b;
        if (s < 36) {
            int i = 0, rem = s;
            while (rem >= 8 - i) { rem -= 8 - i; ++i; }
            const int j = i + rem;
            a = i * 8 + j; b = j * 8 + i;
        } else {
            a = b = 64 + (s - 36);
        }
        pos_tab[0][s] = a; pos_tab[1][s] = b;
    }
    if (lane == 0) {
        mbar_init(full, 32);
        fence_mbarrier_init();
    }
    __syncthreads();

    // b_1 = v_0 . v_0 is the same for every window
    float b1;
    {
        float s = 0.f;
        for (int j = lane; j < 512; j += 32) s = fmaf(v0s[j], v0s[j], s);
        b1 = warp_sum(s);
    }
    // which two reduced values end up in this lane, and where they go in the shared image
    int dst[4];
    {
        int id[kGramVals];
#pragma unroll
        for (int s = 0; s < kGramVals; ++s) id[s] = s;
        halve_ids<52>(id, lane & 16); halve_ids<26>(id, lane & 8); halve_ids<13>(id, lane & 4);
        halve_ids<7>(id, lane & 2); halve_ids<4>(id, lane & 1);
        dst[0] = pos_tab[0][id[0]]; dst[1] = pos_tab[1][id[0]];
        dst[2] = pos_tab[0][id[1]]; dst[3] = pos_tab[1][id[1]];
    }

    Info it;
    {
        int first = 0;
        if (lane == 0) first = claim(P);
        first = __shfl_sync(0xffffffffu, first, 0);
        decode(P, first, &it);
        if (it.item < P.total_items) fetch_tile_warp(P, it, lane, xin, full);
    }
    int next_raw = 0;
    if (lane == 0) next_raw = claim(P);

    uint32_t parity = 0;
    Pending pend; pend.set = -1; pend.b = 0; pend.rowid = 0; pend.bulk = 1;
    while (it.item < P.total_items) {
        const bool is_final = (it.set == P.final_set);
        // ---- X tile -> registers: x[i][2j], x[i][2j+1] = chunk lane + 32 j of row i ----
        f2 x[8][8];
        mbar_wait(full, parity);
        parity ^= 1;
        {
            const float4* t4 = reinterpret_cast<const float4*>(xin);
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 a = t4[i * 128 + lane + 32 * j];
                    x[i][2 * j] = make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
                    x[i][2 * j + 1] = make_float2(fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
                }
        }
        __syncwarp();
        // the slot is free: start fetching the next window (claimed near the end of the previous one)
        Info nt;
        {
            const int next = __shfl_sync(0xffffffffu, next_raw, 0);
            decode(P, next, &nt);
            if (nt.item < P.total_items) fetch_tile_warp(P, nt, lane, xin, full);
        }
        int dc[4] = {0, 0, 0, 0};
        if (lane == 0 && is_final && P.S > 1 && !(P.debug & 1)) {
            const DepRows d = dep_rows(P, it, P.final_set == 0 ? 1 : 0);
#pragma unroll
            for (int q = 0; q < 4; ++q) dc[q] = ld_poll(d.p[q]);
        }

        // ---- pass 1: lane-partial Gam (upper triangle), r = X 1, a_1 = X v_0 ----
        float pv[kGramVals];
        {
            int s = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = i; j < 8; ++j) {
                    f2 acc = mul2(x[i][0], x[j][0]);
#pragma unroll
                    for (int kp = 1; kp < 8; ++kp) acc = fma2(x[i][kp], x[j][kp], acc);
                    pv[s++] = acc.x + acc.y;
                }
            f2 v0c[8];
            {
                const float4* v4 = reinterpret_cast<const float4*>(v0s);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 a = v4[lane + 32 * j];
                    v0c[2 * j] = make_float2(a.x, a.y); v0c[2 * j + 1] = make_float2(a.z, a.w);
                }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                f2 sum = add2(x[i][0], x[i][1]);
                f2 acc = mul2(x[i][0], v0c[0]);
#pragma unroll
                for (int kp = 1; kp < 8; ++kp) acc = fma2(x[i][kp], v0c[kp], acc);
#pragma unroll
                for (int kp = 2; kp < 8; ++kp) sum = add2(sum, x[i][kp]);
                pv[36 + i] = sum.x + sum.y;
                pv[44 + i] = acc.x + acc.y;
            }
        }
        // ---- the one all-reduce of the window: 52 values over 32 lanes, recursive halving ----
        halve_level<52>(pv, lane & 16, 16);
        halve_level<26>(pv, lane & 8, 8);
        halve_level<13>(pv, lane & 4, 4);
        halve_level<7>(pv, lane & 2, 2);
        halve_level<4>(pv, lane & 1, 1);
        __syncwarp();                      // previous window's readers of `gram` are done
        gram[dst[0]] = pv[0]; gram[dst[1]] = pv[0];
        gram[dst[2]] = pv[1]; gram[dst[3]] = pv[1];
        __syncwarp();
        // Publish the previous window's completion here: its factor stores were issued a reduction ago,
        // so the release does not wait on them, and this window has not stored anything yet.
        if (lane == 0 && pend.set >= 0) { bulk_wait_all(); signal_row_done(P, pend.set, pend.b, pend.rowid); pend.set = -1; }
        // Final-set window whose early-set rows are already complete (the usual case): start copying the
        // factors it will combine (12 x 16 bytes per lane) into the staging buffer now, so their L2
        // latency hides behind the sweeps.
        bool fac_staged = false;
        if (is_final && P.S == 2) {
            int ready = 0;
            if (lane == 0) {
                ready = (P.debug & 1) || (dc[0] >= P.TPR && dc[1] >= P.TPR && dc[2] >= P.TPR && dc[3] >= P.TPR);
                if (ready) bulk_wait_read_all();      // the previous Y half has left the staging buffer
            }
            ready = __shfl_sync(0xffffffffu, ready, 0);
            const int s = P.final_set == 0 ? 1 : 0;
            int rho2 = it.c2 + 4 * (lane & 1) + P.sh[s][2]; if (rho2 >= P.n2) rho2 -= P.n2;
            if (ready && (rho2 & 3) == 0) {
                const float* fs = P.fac + (((long long)P.fac_idx[s] * P.B + it.b) * P.heads + it.head) * G * kFacFloats;
                int i1 = it.c1 + ((lane >> 1) & 7); if (i1 >= P.n1) i1 -= P.n1;
                int rho1 = i1 + P.sh[s][1]; if (rho1 >= P.n1) rho1 -= P.n1;
                float4* st4 = reinterpret_cast<float4*>(stage);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    int i0 = it.c0 + (lane >> 4) + 2 * j; if (i0 >= P.n0) i0 -= P.n0;
                    int rho0 = i0 + P.sh[s][0]; if (rho0 >= P.n0) rho0 -= P.n0;
                    const int wrow = ((rho0 >> 3) * P.G1 + (rho1 >> 3)) * P.G2;
                    const int jrow = ((rho0 & 7) * 8 + (rho1 & 7)) * 8;
                    const float* fw = fs + (long long)(wrow + (rho2 >> 3)) * kFacFloats;
                    cp_async16(st4 + (3 * j) * 32 + lane, fw);
                    cp_async16(st4 + (3 * j + 1) * 32 + lane, fw + 4);
                    cp_async16(st4 + (3 * j + 2) * 32 + lane, fw + 8 + jrow + (rho2 & 7));
                }
                cp_async_commit();
                fac_staged = true;
            }
        }

        // ---- T sweeps on 8-vectors.  Lane l holds row (l & 7) of Gam; r, a, u in full. ----
        float grow[8], r[8], a[8], u[8];
        {
            const float4* g4 = reinterpret_cast<const float4*>(gram);
            get8(g4, 2 * (lane & 7), grow);
            get8(g4, 16, r);
            get8(g4, 18, a);
        }
        float* rec = P.saved ? P.saved + it.win_id * P.rec_floats : nullptr;
        if (rec && lane < 18) {
            // Gam (64) and r (8) for the backward
            const float4* g4 = reinterpret_cast<const float4*>(gram);
            reinterpret_cast<float4*>(rec + P.rec_head)[lane] = g4[lane];
        }
        float b = b1, rd = 0.f;
        for (int t = 0; t < P.T; ++t) {
            const float rb = rcp_nr(b + eps);
            const float erb = eps * rb;
#pragma unroll
            for (int j = 0; j < 8; ++j) u[j] = fmaxf(fmaf(a[j], rb, erb), 0.f);
            float d = u[0] * u[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) d = fmaf(u[j], u[j], d);
            rd = rcp_nr(d + eps);
            if (rec && lane == 0) {
                reinterpret_cast<float4*>(rec)[2 * t] = make_float4(u[0], u[1], u[2], u[3]);
                reinterpret_cast<float4*>(rec)[2 * t + 1] = make_float4(u[4], u[5], u[6], u[7]);
                rec[8 * P.T + t] = b;
            }
            if (t == P.T - 1) break;
            float gi = grow[0] * u[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) gi = fmaf(grow[j], u[j], gi);
            float gu[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) gu[j] = __shfl_sync(0xffffffffu, gi, (lane & 24) | j);
            float s = u[0] * gu[0], q = u[0] * r[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) { s = fmaf(u[j], gu[j], s); q = fmaf(u[j], r[j], q); }
            b = (fmaf(2.f * eps, q, s) + 512.f * eps * eps) * rd * rd;
#pragma unroll
            for (int j = 0; j < 8; ++j) a[j] = fmaf(eps, r[j], gu[j]) * rd;
        }
        if (lane == 0) next_raw = claim(P);

        // ---- pass 2: v_T = relu((X^T u_T + eps) rd_T) for the lane's 16 columns ----
        f2 v[8];
        {
            const f2 u0 = dup(u[0]);
#pragma unroll
            for (int kp = 0; kp < 8; ++kp) v[kp] = mul2(x[0][kp], u0);
#pragma unroll
            for (int i = 1; i < 8; ++i) {
                const f2 ui = dup(u[i]);
#pragma unroll
                for (int kp = 0; kp < 8; ++kp) v[kp] = fma2(x[i][kp], ui, v[kp]);
            }
            const f2 rd2 = dup(rd), e2 = dup(eps * rd);
#pragma unroll
            for (int kp = 0; kp < 8; ++kp) {
                const f2 q = fma2(v[kp], rd2, e2);
                v[kp] = make_float2(fmaxf(q.x, 0.f), fmaxf(q.y, 0.f));
            }
        }

        if (P.debug & 2) {
            if (u[0] * v[0].x == 123.456f) P.out[0] = 1.f;
        } else if (!is_final) {
            // ---- early set: publish the rank-1 factors only: [u (8) | v (512)] assembled in the staging
            // buffer and sent as ONE 2080-byte bulk store, whose completion (wait_group) tells us the
            // record is in L2 without a memory fence ----
            const long long local = it.win_id - ((long long)it.set * P.B + it.b) * P.heads * G;   // head*G + window
            float* frec = P.fac + (((long long)P.fac_idx[it.set] * P.B + it.b) * P.heads * G + local) * kFacFloats;
            if (lane == 0) bulk_wait_read_all();
            __syncwarp();
            float4* f4 = reinterpret_cast<float4*>(stage);
            if (lane == 0) { f4[0] = make_float4(u[0], u[1], u[2], u[3]); f4[1] = make_float4(u[4], u[5], u[6], u[7]); }
#pragma unroll
            for (int j = 0; j < 4; ++j)
                f4[2 + lane + 32 * j] = make_float4(v[2 * j].x, v[2 * j].y, v[2 * j + 1].x, v[2 * j + 1].y);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                bulk_store_1d(frec, stage, kFacFloats * 4);
                bulk_commit();
                pend.set = it.set; pend.b = it.b; pend.rowid = it.rowid;
            }
        } else {
            // ---- final set: Y = (u v^T + sum over early sets of their overlapping factors) / S ----
            if (P.S > 1 && !fac_staged) {
                if (lane == 0 && !(P.debug & 1)) {
                    if (pend.set >= 0) { bulk_wait_all(); signal_row_done(P, pend.set, pend.b, pend.rowid); pend.set = -1; }
                    const int first = P.final_set == 0 ? 1 : 0;
                    if (dc[0] < P.TPR || dc[1] < P.TPR || dc[2] < P.TPR || dc[3] < P.TPR) wait_rows(P, it, first);
                    for (int s = first + 1; s < P.S; ++s)
                        if (s != P.final_set) wait_rows(P, it, s);
                }
                __syncwarp();
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const f2 ui = dup(u[i] * P.inv_S);
#pragma unroll
                for (int kp = 0; kp < 8; ++kp) x[i][kp] = mul2(ui, v[kp]);      // x is dead: reuse as the accumulator
            }
            const LaneAddr4 la = lane_addr4(P, it, lane);
            int i1 = it.c1 + ((lane >> 1) & 7); if (i1 >= P.n1) i1 -= P.n1;
            if (fac_staged) {
                cp_async_wait<0>();
                const float4* st4 = reinterpret_cast<const float4*>(stage);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 ua = st4[(3 * j) * 32 + lane], ub = st4[(3 * j + 1) * 32 + lane], vv = st4[(3 * j + 2) * 32 + lane];
                    const float uu[8] = {ua.x, ua.y, ua.z, ua.w, ub.x, ub.y, ub.z, ub.w};
                    const f2 va = make_float2(vv.x * P.inv_S, vv.y * P.inv_S), vb = make_float2(vv.z * P.inv_S, vv.w * P.inv_S);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const f2 ui = dup(uu[i]);
                        x[i][2 * j] = fma2(ui, va, x[i][2 * j]);
                        x[i][2 * j + 1] = fma2(ui, vb, x[i][2 * j + 1]);
                    }
                }
            }
            for (int s = 0; s < P.S && !fac_staged; ++s) {
                if (s == P.final_set) continue;
                const float* fs = P.fac + (((long long)P.fac_idx[s] * P.B + it.b) * P.heads + it.head) * G * kFacFloats;
                // position of this lane's columns in set s's rolled coordinates
                int rho1 = i1 + P.sh[s][1]; if (rho1 >= P.n1) rho1 -= P.n1;
                int rho2 = la.i2 + P.sh[s][2]; if (rho2 >= P.n2) rho2 -= P.n2;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    int i0 = it.c0 + (lane >> 4) + 2 * j; if (i0 >= P.n0) i0 -= P.n0;
                    int rho0 = i0 + P.sh[s][0]; if (rho0 >= P.n0) rho0 -= P.n0;
                    const int wrow = ((rho0 >> 3) * P.G1 + (rho1 >> 3)) * P.G2;
                    const int jrow = ((rho0 & 7) * 8 + (rho1 & 7)) * 8;
                    if ((rho2 & 3) == 0) {
                        const float* fw = fs + (long long)(wrow + (rho2 >> 3)) * kFacFloats;
                        const float4 ua = __ldcg(reinterpret_cast<const float4*>(fw));
                        const float4 ub = __ldcg(reinterpret_cast<const float4*>(fw) + 1);
                        const float4 vv = __ldcg(reinterpret_cast<const float4*>(fw + 8 + jrow + (rho2 & 7)));
                        const float uu[8] = {ua.x, ua.y, ua.z, ua.w, ub.x, ub.y, ub.z, ub.w};
                        const f2 va = make_float2(vv.x * P.inv_S, vv.y * P.inv_S), vb = make_float2(vv.z * P.inv_S, vv.w * P.inv_S);
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const f2 ui = dup(uu[i]);
                            x[i][2 * j] = fma2(ui, va, x[i][2 * j]);
                            x[i][2 * j + 1] = fma2(ui, vb, x[i][2 * j + 1]);
                        }
                    } else {
                        float acc[8][4];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            acc[i][0] = x[i][2 * j].x; acc[i][1] = x[i][2 * j].y; acc[i][2] = x[i][2 * j + 1].x; acc[i][3] = x[i][2 * j + 1].y;
                        }
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            int r2 = rho2 + e; if (r2 >= P.n2) r2 -= P.n2;
                            const float* fw = fs + (long long)(wrow + (r2 >> 3)) * kFacFloats;
                            const float vv = __ldcg(fw + 8 + jrow + (r2 & 7)) * P.inv_S;
#pragma unroll
                            for (int i = 0; i < 8; ++i) acc[i][e] = fmaf(__ldcg(fw + i), vv, acc[i][e]);
                        }
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            x[i][2 * j] = make_float2(acc[i][0], acc[i][1]); x[i][2 * j + 1] = make_float2(acc[i][2], acc[i][3]);
                        }
                    }
                }
            }
            float* base = P.out + it.chan_base;
            if (it.flags & kInterior) {
                // Y leaves through TMA, half a window (q0 = 4h .. 4h+3) at a time: the 32-byte runs of a
                // window cost the LSU one pass per run when stored from registers
                float4* st4 = reinterpret_cast<float4*>(stage);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (lane == 0) bulk_wait_read_all();          // the previous half has left the staging buffer
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; ++i)
#pragma unroll
                        for (int jj = 0; jj < 2; ++jj) {
                            const int j = 2 * h + jj;
                            st4[i * 64 + lane + 32 * jj] = make_float4(x[i][2 * j].x, x[i][2 * j].y, x[i][2 * j + 1].x, x[i][2 * j + 1].y);
                        }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        tma_store_tile(&P.tm_out, stage, it.c2, it.c1, it.c0 + 4 * h, it.head * 8, it.b);
                        bulk_commit();
                    }
                }
            } else if (it.flags & kAligned4) {
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<float4*>(base + (long long)i * P.vox + la.rowoff[j] + la.i2) =
                            make_float4(x[i][2 * j].x, x[i][2 * j].y, x[i][2 * j + 1].x, x[i][2 * j + 1].y);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float* row = base + (long long)i * P.vox + la.rowoff[j];
                        row[wrap2(P, la.i2)] = x[i][2 * j].x;
                        row[wrap2(P, la.i2 + 1)] = x[i][2 * j].y;
                        row[wrap2(P, la.i2 + 2)] = x[i][2 * j + 1].x;
                        row[wrap2(P, la.i2 + 3)] = x[i][2 * j + 1].y;
                    }
            }
        }
        it = nt;
    }
    __syncwarp();
    if (lane == 0) {
        bulk_wait_all();
        if (pend.set >= 0) signal_row_done(P, pend.set, pend.b, pend.rowid);
    }
}

// =====================================================================================================
// backward, Gram form
// =====================================================================================================
struct alignas(16) GPairShared {      // static shared memory, one per pair
    float red[48];
    float rec[2][kRecStride];         // record of the current / next window: u_t, b_t, Gam, r
    float mm[2][80];                  // per warp: M (64), m (8), abar_1 (8) for the final product
    Info info[2];
    uint64_t xfull, gfull, ofull;
    int oready;
};

__global__ void __launch_bounds__(kGBwdPairs * 64, 1) swnmf_bwd_gram(const __grid_constant__ FastParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ __align__(16) GPairShared ps_all[kGBwdPairs];

    const PairCtx c = pair_ctx();
    float* xin = reinterpret_cast<float*>(smem_raw + (size_t)c.pair * 3 * kTileBytes);
    float* gin = xin + 4096;         // dY tile
    float* oin = gin + 4096;         // partial dX of the previous window set of the chain
    GPairShared& ps = ps_all[c.pair];
    const int rec_lanes = P.rec_floats >> 2;
    const float eps = P.eps;
    const int row = c.lane & 7;      // the row of Gam / M this lane works on in the 8-vector recursion

    for (int j = threadIdx.x; j < 512; j += blockDim.x) v0s[j] = P.v0[j];
    int claimed = 0;
    if (c.leader) {
        mbar_init(&ps.xfull, 64);
        mbar_init(&ps.gfull, 64);
        mbar_init(&ps.ofull, 64);
        ps.oready = 0;
        fence_mbarrier_init();
        decode(P, claim(P), &ps.info[0]);
        decode(P, claim(P), &ps.info[1]);
        claimed = claim(P);
    }
    __syncthreads();
    {
        const Info first = ps.info[0];
        if (first.item < P.total_items) {
            if (c.p < rec_lanes) cp_async16(ps.rec[0] + 4 * c.p, P.saved + first.win_id * P.rec_floats + 4 * c.p);
            fetch_tile(P, &P.tm_x, P.x, first, c.p, xin, &ps.xfull, c.p < rec_lanes);
            fetch_tile(P, &P.tm_g, P.gy, first, c.p, gin, &ps.gfull, false);
        }
    }

    uint32_t xparity = 0, gparity = 0, oparity = 0;
    int slot = 0;
    Pending pend; pend.set = -1; pend.b = 0; pend.rowid = 0; pend.bulk = 1;
    for (int n = 0;; ++n) {
        const Info it = ps.info[n & 1];
        if (it.item >= P.total_items) break;
        const int dep = P.dep_of[it.set];
        int dc[4] = {0, 0, 0, 0};
        if (c.second && dep >= 0 && !(P.debug & 1)) {
            const DepRows d = dep_rows(P, it, dep);
#pragma unroll
            for (int q = 0; q < 4; ++q) dc[q] = ld_poll(d.p[q]);
        }

        f2 x[8][4];
        mbar_wait(&ps.xfull, xparity);
        xparity ^= 1;
        load_rows_smem<true>(xin, c.p, x);
        const float* rec = ps.rec[n & 1];
        const float4* rec4 = reinterpret_cast<const float4*>(rec);
        const int T = P.T;

        // ---- v_T from the saved u_T ----
        float u[8], rdT;
        f2 vt[4];
        get8(rec4, 2 * (T - 1), u);
        v_from_u(x, u, eps, rdT, vt);

        // ---- gv = G^T u_T / S (lane-local), and the lane-partials of  G v_T / S + X cbar_T  and  qbar_T . v_T ----
        float w[8], e;
        f2 gv[4];
        {
            mbar_wait(&ps.gfull, gparity);
            gparity ^= 1;
            const float4* g4 = reinterpret_cast<const float4*>(gin);
            f2 gup[8];
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) gv[kp] = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 ga = g4[i * 128 + c.p], gb = g4[i * 128 + 64 + c.p];
                const f2 g0 = make_float2(ga.x, ga.y), g1 = make_float2(ga.z, ga.w);
                const f2 g2 = make_float2(gb.x, gb.y), g3 = make_float2(gb.z, gb.w);
                f2 acc = mul2(g0, vt[0]);
                acc = fma2(g1, vt[1], acc); acc = fma2(g2, vt[2], acc); acc = fma2(g3, vt[3], acc);
                gup[i] = acc;
                const f2 ui = dup(u[i]);
                gv[0] = fma2(g0, ui, gv[0]); gv[1] = fma2(g1, ui, gv[1]);
                gv[2] = fma2(g2, ui, gv[2]); gv[3] = fma2(g3, ui, gv[3]);
            }
            const f2 is2 = dup(P.inv_S), rd2 = dup(rdT);
            f2 cb[4], e2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) {
                gv[kp] = mul2(gv[kp], is2);
                cb[kp] = mul2(gv[kp], rd2);                 // cbar_T = qbar_T rd_T, qbar_T = gv (v_T > 0 wherever it matters)
                e2 = fma2(gv[kp], vt[kp], e2);
            }
            e = e2.x + e2.y;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                f2 acc = mul2(gup[i], is2);
#pragma unroll
                for (int kp = 0; kp < 4; ++kp) acc = fma2(x[i][kp], cb[kp], acc);
                w[i] = acc.x + acc.y;
            }
        }
        if (c.second)
            ps.oready = (dep >= 0) && ((P.debug & 1) || (dc[0] >= P.TPR && dc[1] >= P.TPR && dc[2] >= P.TPR && dc[3] >= P.TPR));
        // the O slot is written again in this window: the TMA store of the previous window must have
        // finished reading it before anyone passes the barrier below
        if (c.leader) bulk_wait_read_all();
        pair_reduce9(w, e, ps.red, slot, c.wip, c.lane, c.barid);
        // Both warps are past the window's only barrier: refill the slots for the next window, publish
        // the previous window's completion, decode the next-but-one item, start fetching this window's
        // partial sum.
        const bool oready = ps.oready != 0;
        {
            if (c.leader && pend.set >= 0) {
                if (pend.bulk) { bulk_wait_all(); signal_row_done(P, pend.set, pend.b, pend.rowid); }   // the dX tile is in L2
                else signal_row(P, pend.set, pend.b, pend.rowid);     // stored from registers: release
                pend.set = -1;
            }
            if (oready) {
                if (c.leader) fence_proxy_async_all();   // counters were polled through the generic proxy
                fetch_tile(P, &P.tm_out, P.out, it, c.p, oin, &ps.ofull, false);
            }
            const Info nt = ps.info[(n + 1) & 1];
            if (nt.item < P.total_items) {
                if (c.p < rec_lanes) cp_async16(ps.rec[(n + 1) & 1] + 4 * c.p, P.saved + nt.win_id * P.rec_floats + 4 * c.p);
                fetch_tile(P, &P.tm_x, P.x, nt, c.p, xin, &ps.xfull, c.p < rec_lanes);
                fetch_tile(P, &P.tm_g, P.gy, nt, c.p, gin, &ps.gfull, false);
            }
            if (c.leader) decode(P, claimed, &ps.info[n & 1]);
        }

        // ---- the 8-vector recursion t = T .. 1 (both warps, every 8-lane group redundantly) ----
        // lane (row) holds row `row` of Gam and accumulates row `row` of M
        float grow[8], r[8];
        get8(rec4, (P.rec_head >> 2) + 2 * row, grow);
        get8(rec4, (P.rec_head >> 2) + 16, r);
        float mrow[8], mi = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) mrow[j] = 0.f;
        float ab[8];           // abar_{t} of the step just finished, full vector
        float bbar;
        {
            // step T: ubar = (G v_T/S + X cbar_T) + 2 dbar u_T,  dbar = -(qbar.v_T) rd_T
            const float db = -e * rdT;
            const float rb = rcp_nr(rec[8 * T + (T - 1)] + eps);
            float bacc = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float ub = fmaf(2.f * db, u[j], w[j]);
                const float pb = (T == 1 && !(u[j] > 0.f)) ? 0.f : ub;      // only u_1 can be clipped
                ab[j] = pb * rb;
                bacc = fmaf(pb, u[j], bacc);
            }
            bbar = -bacc * rb;
        }
        float uT[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) uT[j] = u[j] * rdT;                      // rd_T u_T for dX += (rd_T u_T) gv^T
        for (int t = T - 2; t >= T - P.K; --t) {
            // u = u_{t+1} in 1-based terms: the iterate the finished step differentiated against
            get8(rec4, 2 * t, u);
            float d = u[0] * u[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) d = fmaf(u[j], u[j], d);
            const float rd = rcp_nr(d + eps);
            const float brd = 2.f * bbar * rd, kappa = brd * eps;
            float z[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) z[j] = fmaf(brd, u[j], ab[j]);
            // M += rd (u z^T + abar u^T), m += rd (kappa u + eps abar): this lane's row
            {
                const float ur = rec[8 * t + row] * rd, ar = pick8(ab, row) * rd;
#pragma unroll
                for (int j = 0; j < 8; ++j) mrow[j] = fmaf(ur, z[j], fmaf(ar, u[j], mrow[j]));
                mi = fmaf(kappa, ur, fmaf(eps, ar, mi));
            }
            // Gam z and Gam u: this lane's row, then all-gather within the 8-lane group
            float gzi = grow[0] * z[0], gui = grow[0] * u[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) { gzi = fmaf(grow[j], z[j], gzi); gui = fmaf(grow[j], u[j], gui); }
            float gz[8], gu[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                gz[j] = __shfl_sync(0xffffffffu, gzi, (c.lane & 24) | j);
                gu[j] = __shfl_sync(0xffffffffu, gui, (c.lane & 24) | j);
            }
            float zgu = z[0] * gu[0], zr = z[0] * r[0], ur = u[0] * r[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) { zgu = fmaf(z[j], gu[j], zgu); zr = fmaf(z[j], r[j], zr); ur = fmaf(u[j], r[j], ur); }
            const float qv = rd * (zgu + eps * zr + kappa * ur + 512.f * kappa * eps);
            const float db = -qv * rd;
            const float rb = rcp_nr(rec[8 * T + t] + eps);
            float bacc = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float wj = rd * fmaf(kappa, r[j], gz[j]);
                const float ub = fmaf(2.f * db, u[j], wj);
                const float pb = (t == 0 && !(u[j] > 0.f)) ? 0.f : ub;
                ab[j] = pb * rb;
                bacc = fmaf(pb, u[j], bacc);
            }
            bbar = -bacc * rb;
        }
        if (P.K < T) {
            // truncated unroll (num_grad_steps < num_iters): the last differentiated half-step still
            // reads X through a_t = X v_{t-1}; v_{t-1} = rd (X^T u_{t-1} + eps 1) is a constant there
            get8(rec4, 2 * (T - P.K - 1), u);
            float d = u[0] * u[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) d = fmaf(u[j], u[j], d);
            const float ar = pick8(ab, row) * rcp_nr(d + eps);
#pragma unroll
            for (int j = 0; j < 8; ++j) mrow[j] = fmaf(ar, u[j], mrow[j]);
            mi = fmaf(eps, ar, mi);
        }
        // share M (rows), m and abar_1 with the whole warp
        float* mm = ps.mm[c.wip];
        __syncwarp();
        if (c.lane < 8) {
            float4* m4 = reinterpret_cast<float4*>(mm);
            m4[2 * row] = make_float4(mrow[0], mrow[1], mrow[2], mrow[3]);
            m4[2 * row + 1] = make_float4(mrow[4], mrow[5], mrow[6], mrow[7]);
            mm[64 + row] = mi;
            mm[72 + row] = pick8(ab, row);
        }
        __syncwarp();
        if (c.leader) claimed = claim(P);

        // ---- dX = rd_T u_T gv^T + M X + m 1^T + abar_1 v_0^T  (the last term only if the sweep reached t = 1) ----
        f2 xb[8][4];
        {
            const float4* m4 = reinterpret_cast<const float4*>(mm);
            f2 v0c[4];
            get4x2(reinterpret_cast<const float4*>(v0s), c.p, 64 + c.p, v0c);
            const bool full_sweep = (P.K >= T);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const f2 mi2 = dup(mm[64 + i]);
                const f2 a1 = dup(full_sweep ? mm[72 + i] : 0.f);
                const f2 ut = dup(uT[i]);
                float mr[8];
                get8(m4, 2 * i, mr);
#pragma unroll
                for (int kp = 0; kp < 4; ++kp) {
                    f2 acc = fma2(a1, v0c[kp], mi2);
                    acc = fma2(ut, gv[kp], acc);
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc = fma2(dup(mr[j]), x[j][kp], acc);
                    xb[i][kp] = acc;
                }
            }
        }
        // ReLU adjoint (factorizer.py:44)
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) {
                xb[i][kp].x = x[i][kp].x > 0.f ? xb[i][kp].x : 0.f;
                xb[i][kp].y = x[i][kp].y > 0.f ? xb[i][kp].y : 0.f;
            }
        if (dep >= 0) {
            if (!oready) {
                // rare: the rows this window continues were not finished when it started
                if (c.leader) {
                    if (pend.set >= 0) {
                        if (pend.bulk) { bulk_wait_all(); signal_row_done(P, pend.set, pend.b, pend.rowid); }
                        else signal_row(P, pend.set, pend.b, pend.rowid);
                        pend.set = -1;
                    }
                    wait_rows(P, it, dep);
                    fence_proxy_async_all();
                }
                pair_bar(c.barid);
                fetch_tile(P, &P.tm_out, P.out, it, c.p, oin, &ps.ofull, false);
            }
            mbar_wait(&ps.ofull, oparity);
            oparity ^= 1;
            const float4* o4 = reinterpret_cast<const float4*>(oin);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 a = o4[i * 128 + c.p], b = o4[i * 128 + 64 + c.p];
                xb[i][0] = add2(xb[i][0], make_float2(a.x, a.y)); xb[i][1] = add2(xb[i][1], make_float2(a.z, a.w));
                xb[i][2] = add2(xb[i][2], make_float2(b.x, b.y)); xb[i][3] = add2(xb[i][3], make_float2(b.z, b.w));
            }
        }
        if (P.debug & 2) {
            if (xb[0][0].x == 123.456f) P.out[0] = 1.f;
        } else if (it.flags & kInterior) {
            // stage the tile in the O slot (each lane rewrites exactly the chunks it read) and let TMA
            // scatter its 512 32-byte runs
            float4* o4 = reinterpret_cast<float4*>(oin);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                o4[i * 128 + c.p] = make_float4(xb[i][0].x, xb[i][0].y, xb[i][1].x, xb[i][1].y);
                o4[i * 128 + 64 + c.p] = make_float4(xb[i][2].x, xb[i][2].y, xb[i][3].x, xb[i][3].y);
            }
            fence_proxy_async_smem();
            pair_bar(c.barid);
            if (c.leader) {
                tma_store_tile(&P.tm_out, oin, it.c2, it.c1, it.c0, it.head * 8, it.b);
                bulk_commit();
                if (P.signals[it.set]) { pend.set = it.set; pend.b = it.b; pend.rowid = it.rowid; pend.bulk = 1; }
            }
        } else {
            store_rows_direct(P, P.out + it.chan_base, it, c.p, xb);
            if (c.leader && P.signals[it.set]) { pend.set = it.set; pend.b = it.b; pend.rowid = it.rowid; pend.bulk = 0; }
        }
    }
    pair_bar(c.barid);
    if (c.leader) {
        bulk_wait_all();
        if (pend.set >= 0) {
            if (pend.bulk) signal_row_done(P, pend.set, pend.b, pend.rowid);
            else signal_row(P, pend.set, pend.b, pend.rowid);
        }
    }
}
