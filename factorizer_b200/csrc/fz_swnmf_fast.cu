// Specialised fused kernels for the production geometry of every Swin-Factorizer config:
// head_dim 8, patch 8x8x8 (an 8 x 512 matrix per window), rank 1, HALS, any number of window sets
// with any integer shifts.  One kernel per direction does
//     gather (roll + window partition + ReLU)  ->  T unrolled HALS sweeps  ->  U V^T  ->  scatter-mean
// (reference factorizer/factorizer.py:41-50, operations.py:266-280/417-434,
//  matrix_factorization.py:210-229/514-533), reading X once and writing Y once.
//
// Design (B200, sm_100a), third revision:
//  * work unit = one window = one 16 KiB tile; a PAIR of warps (64 lanes) owns it: lane p holds
//    columns 4p..4p+3 and 256+4p..+3 of all 8 rows in registers as packed float2, so X^T u, the V
//    update and the rank-1 reconstruction are lane-local FFMA2 streams and only the 8 row sums (X v)
//    need a 64-lane reduction (recursive-halving shuffles + one named barrier);
//  * every tile (X, dY, the partial dX of the previous window set) is fetched ASYNCHRONOUSLY one
//    window ahead into shared memory: windows that are one clean box of the volume by a single TMA
//    box load (5-D tensor map over (W,H,D,C,B), box (8,8,8,8,1), which lands the window in exactly
//    the reference's column order), windows that wrap around the volume (the roll) by per-lane
//    cp.async with modular addressing.  Both complete on the same mbarrier, so the compute path does
//    not care which one ran;
//  * the mean over window sets never round-trips a full tile through memory in the forward: the
//    early sets write only their rank-1 factors (u: 8, v: 512 floats = 13 % of a tile) and the last
//    set -- chosen to be the unshifted one -- adds the factor products of the (up to 8 per set)
//    windows it overlaps and writes Y exactly once;
//  * the backward's dX is a dense sum, so set j reads the partial sum left by set j-1 (L2-resident),
//    adds its own contribution and stores it back (plain stores, no atomics);
//  * persistent CTAs pull windows from an atomic counter in a host-built order: one (sample, head)
//    sub-volume after the other, rows of windows (g0,g1 fixed, g2 running) of the window sets
//    interleaved so that a dependent row is claimed about one generation of in-flight windows after
//    the last row it needs.  Second touches of X / dY / partial dX then hit L2 (the live footprint is
//    ~30 MB) and HBM sees each tensor once.  Per-(set,sample,head,row) completion counters guard the
//    dependencies; they are deadlock-free because a window only ever waits for windows claimed
//    earlier, and completion signals are always flushed before a pair blocks;
//  * forward saves u_t (8 floats) and b_t per sweep and window (1.2 % extra traffic); backward
//    recomputes every v_t from them with one lane-local GEMV (overlapping the reduction of the same
//    sweep), keeps X and the dX accumulator in registers and streams dY through shared memory once.
//  * arithmetic: packed FFMA2 (fma.rn.f32x2) for every GEMV / rank-1 update -- same FP32 pipe rate,
//    half the issue slots, which is what the scalar overhead (shuffles, selects, addressing) needs;
//    reciprocals are MUFU.RCP + one Newton step, (a+eps)/(b+eps) is evaluated as fma(a, r, eps*r).
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "fz_device.cuh"
#include "fz_internal.cuh"

namespace fz {

constexpr int kMaxOrder = 4096;       // rows of windows (all sets, all heads of one sample) in the ordering table
constexpr int kTileBytes = 16384;     // 8 x 512 fp32
constexpr int kMaxT = 8;
constexpr int kFwdPairs = 8;          // 16 warps / CTA, 1 CTA / SM
constexpr int kBwdPairs = 4;          // 8 warps / CTA, 1 CTA / SM
constexpr int kFacFloats = 520;       // u (8) + v (512) per early-set window
constexpr int kRecStride = 144;       // shared-memory floats reserved per window record (T <= 8: 72 + 72)

struct alignas(64) FastParams {
    CUtensorMap tm_x;     // X volume
    CUtensorMap tm_g;     // dY volume (backward)
    CUtensorMap tm_out;   // output volume: dX (backward: partial-sum load, tile store) / Y (forward: half-tile store, box (8,8,4,8,1))
    const float* x;
    const float* gy;
    float* out;
    const float* v0;
    float* saved;
    float* fac;           // forward: factors of the early sets
    int* ctr;             // [0] work counter, [2 + ((set*B + b)*heads + head)*NR + row] finished windows
    int n0, n1, n2, G0, G1, G2, heads, B, S, C;
    int sh[FZ_MAX_SHIFTS][3];   // shifts normalised into [0, n)
    int dep_of[FZ_MAX_SHIFTS];  // backward: set whose partial sum this set continues (-1: chain head)
    int fac_idx[FZ_MAX_SHIFTS]; // forward: slot of an early set in `fac` (-1: the final set)
    int signals[FZ_MAX_SHIFTS]; // does a finished window of this set bump its row counter?
    int final_set;
    long long vox;
    int NR, TPR, tpr_shift, entries, per_sample, total_items;
    int T, K, relu;
    int rec_floats;       // floats per saved window record: [u_t (8T) | b_t (T) | pad to 4 | Gam (64) | r (8)]
    int rec_head;         // offset of Gam = 9T rounded up to 4
    float eps, inv_S;
    int debug;            // FZ_DEBUG_FLAGS (timing experiments only): 1 = skip dependency waits, 2 = skip output
    unsigned order[kMaxOrder];  // (set << 29) | (head << 20) | (g0 << 10) | g1, in processing order
};

// ---- PTX helpers ------------------------------------------------------------------------------------
__device__ __forceinline__ void pair_bar(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
// Completion counters are polled with relaxed gpu-scope loads (an acquire on every poll costs an L1 invalidation,
// ~1 us, per iteration); once a poll shows "done" the observer issues ONE acquire fence, plus a proxy fence because
// the dependent reads are TMA / bulk loads in the async proxy (acquire_after_poll).  The writer publishes with a
// release reduction after its bulk stores have completed.
__device__ __forceinline__ int ld_poll(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void acquire_after_poll() {
    asm volatile("fence.acq_rel.gpu;" ::: "memory");
    fence_proxy_async_all();
}
__device__ __forceinline__ void red_release_add(int* p, int v) {
    asm volatile("red.release.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---- work decoding ----------------------------------------------------------------------------------
struct Info {             // one claimed window, decoded by the pair leader and shared through smem
    int item;             // >= total_items: no more work
    int b, set, head;
    int rowid;            // head * NR + g0 * G1 + g1: index of the completion counter within (set, b)
    int c0, c1, c2;       // first voxel of the window in the un-rolled volume
    int flags;            // 1: one contiguous, 16-byte aligned box (TMA);  2: c2 % 4 == 0 (16-byte chunks never straddle the wrap)
    int pad;
    long long win_id;     // canonical index ((set*B + b)*heads + head)*G + window
    long long chan_base;  // element offset of channel head*8 of sample b
};
constexpr int kInterior = 1, kAligned4 = 2;

__device__ __forceinline__ void decode(const FastParams& P, int item, Info* o) {
    o->item = item;
    if (item >= P.total_items) return;
    const int b = (P.B == 1) ? 0 : item / P.per_sample;
    const int rem = item - b * P.per_sample;
    const int e = (P.tpr_shift >= 0) ? (rem >> P.tpr_shift) : rem / P.TPR;
    const int g2 = rem - e * P.TPR;
    const unsigned entry = P.order[e];
    const int set = (int)(entry >> 29), head = (int)((entry >> 20) & 0x1ffu);
    const int k = (int)((entry >> 10) & 0x3ffu), g1 = (int)(entry & 0x3ffu);
    int c0 = k * 8 - P.sh[set][0]; if (c0 < 0) c0 += P.n0;
    int c1 = g1 * 8 - P.sh[set][1]; if (c1 < 0) c1 += P.n1;
    int c2 = g2 * 8 - P.sh[set][2]; if (c2 < 0) c2 += P.n2;
    const bool al = (c2 & 3) == 0;
    const bool inside = (c0 + 8 <= P.n0) && (c1 + 8 <= P.n1) && (c2 + 8 <= P.n2);
    const int row = k * P.G1 + g1;
    o->b = b; o->set = set; o->head = head; o->rowid = head * P.NR + row;
    o->c0 = c0; o->c1 = c1; o->c2 = c2;
    o->flags = ((inside && al) ? kInterior : 0) | (al ? kAligned4 : 0);
    const long long G = (long long)P.NR * P.G2;
    o->win_id = (((long long)set * P.B + b) * P.heads + head) * G + (long long)row * P.G2 + g2;
    o->chan_base = ((long long)b * P.C + (long long)head * 8) * P.vox;
}

// Lane p owns chunks r = p and p + 64 of every row; chunk r <-> (q0 = r >> 4, q1 = (r >> 1) & 7,
// q2 = 4 * (r & 1) + e), i.e. matrix columns 4r .. 4r+3 (reference column order, operations.py:321-325).
struct LaneAddr {
    int rowoff[2];   // (i0 * n1 + i1) * n2 for the two chunks
    int i2[2];       // W coordinate of the chunk's first column (the following ones may wrap)
};
__device__ __forceinline__ LaneAddr lane_addr(const FastParams& P, const Info& it, int p) {
    LaneAddr a;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int r = p + 64 * h;
        int i0 = it.c0 + (r >> 4); if (i0 >= P.n0) i0 -= P.n0;
        int i1 = it.c1 + ((r >> 1) & 7); if (i1 >= P.n1) i1 -= P.n1;
        int i2 = it.c2 + 4 * (r & 1); if (i2 >= P.n2) i2 -= P.n2;
        a.rowoff[h] = (i0 * P.n1 + i1) * P.n2;
        a.i2[h] = i2;
    }
    return a;
}
__device__ __forceinline__ int wrap2(const FastParams& P, int i2) { return i2 >= P.n2 ? i2 - P.n2 : i2; }

// Asynchronous gather of one window into a tile slot in the standard layout (row i, chunk r at float
// offset i*512 + 4r), each lane fetching the chunks it will later read.  Used when the window is not
// one clean TMA box.
__device__ __forceinline__ void gather_async(const FastParams& P, const float* base, const Info& it, int p, float* tile) {
    const LaneAddr a = lane_addr(P, it, p);
    if (it.flags & kAligned4) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h)
                cp_async16(tile + i * 512 + 4 * (p + 64 * h), base + (long long)i * P.vox + a.rowoff[h] + a.i2[h]);
    } else {
#pragma unroll 1
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    cp_async4(tile + i * 512 + 4 * (p + 64 * h) + e,
                              base + (long long)i * P.vox + a.rowoff[h] + wrap2(P, a.i2[h] + e));
    }
}

// Start fetching window `it` of volume `base` (tensor map `map`) into `tile`; completion is one phase
// of `bar` (64 arrivals + the TMA byte count).  Every lane of the pair calls this.
__device__ __forceinline__ void fetch_tile(const FastParams& P, const CUtensorMap* map, const float* base, const Info& it,
                                           int p, float* tile, uint64_t* bar, bool extra_cp_async) {
    if (it.flags & kInterior) {
        if (p == 0) {
            mbar_expect_tx(bar, kTileBytes);
            tma_load_tile(tile, map, bar, it.c2, it.c1, it.c0, it.head * 8, it.b);
        }
        if (extra_cp_async) mbar_arrive_after_cp_async(bar); else mbar_arrive(bar);
    } else {
        gather_async(P, base + it.chan_base, it, p, tile);
        mbar_arrive_after_cp_async(bar);
    }
}

// The partial dX of the previous window set was written by other SMs with plain stores; it is fetched
// with cp.async.cg (generic proxy, L2) so that no cross-proxy fence is needed after the counter poll.
__device__ __forceinline__ void fetch_partial(const FastParams& P, const Info& it, int p, float* tile, uint64_t* bar) {
    gather_async(P, P.out + it.chan_base, it, p, tile);
    mbar_arrive_after_cp_async(bar);
}

// out = val; plain stores, the caller owns these voxels.
__device__ __forceinline__ void store_rows_direct(const FastParams& P, float* base, const Info& it, int p, const f2 (&x)[8][4]) {
    const LaneAddr a = lane_addr(P, it, p);
    if (it.flags & kAligned4) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float4* dst = reinterpret_cast<float4*>(base + (long long)i * P.vox + a.rowoff[h] + a.i2[h]);
                *dst = make_float4(x[i][2 * h].x, x[i][2 * h].y, x[i][2 * h + 1].x, x[i][2 * h + 1].y);
            }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float* row = base + (long long)i * P.vox + a.rowoff[h];
                row[wrap2(P, a.i2[h])] = x[i][2 * h].x;
                row[wrap2(P, a.i2[h] + 1)] = x[i][2 * h].y;
                row[wrap2(P, a.i2[h] + 2)] = x[i][2 * h + 1].x;
                row[wrap2(P, a.i2[h] + 3)] = x[i][2 * h + 1].y;
            }
    }
}

// Completion counters of the (up to 4) rows of window set `dep` that window `it` overlaps.
struct DepRows { const int* p[4]; };
__device__ __forceinline__ DepRows dep_rows(const FastParams& P, const Info& it, int dep) {
    int r0 = it.c0 + P.sh[dep][0]; if (r0 >= P.n0) r0 -= P.n0;
    int r1 = it.c1 + P.sh[dep][1]; if (r1 >= P.n1) r1 -= P.n1;
    int r0b = r0 + 7; if (r0b >= P.n0) r0b -= P.n0;
    int r1b = r1 + 7; if (r1b >= P.n1) r1b -= P.n1;
    const int ka = r0 >> 3, kb = r0b >> 3, ga = r1 >> 3, gb = r1b >> 3;
    const int* done = P.ctr + 2 + (((long long)dep * P.B + it.b) * P.heads + it.head) * P.NR;
    DepRows d;
    d.p[0] = done + ka * P.G1 + ga; d.p[1] = done + ka * P.G1 + gb;
    d.p[2] = done + kb * P.G1 + ga; d.p[3] = done + kb * P.G1 + gb;
    return d;
}
__device__ __forceinline__ void wait_rows(const FastParams& P, const Info& it, int dep) {
    const DepRows d = dep_rows(P, it, dep);
#pragma unroll
    for (int q = 0; q < 4; ++q)
        while (ld_poll(d.p[q]) < P.TPR) __nanosleep(64);
    acquire_after_poll();
}
// Completion of a window whose output left through TMA / bulk stores that the caller has already waited
// for with cp.async.bulk.wait_group 0.  That wait alone is NOT enough to publish with a relaxed
// reduction: measured on B200, a dependent window then occasionally reads the previous contents of
// the tile (the bulk writes are complete for the issuing thread, not yet performed at gpu scope), so
// the counter is bumped with release semantics.
__device__ __forceinline__ void signal_row_done(const FastParams& P, int set, int b, int rowid) {
    red_release_add(P.ctr + 2 + ((long long)set * P.B + b) * P.heads * P.NR + rowid, 1);
}
__device__ __forceinline__ void signal_row(const FastParams& P, int set, int b, int rowid) {
    red_release_add(P.ctr + 2 + ((long long)set * P.B + b) * P.heads * P.NR + rowid, 1);
}

// 64-lane all-reduce of 8 row sums and one scalar.  red: 2 slots x 2 warps x 12 floats.  Contains the
// pair's named barrier exactly once.
__device__ __forceinline__ void pair_reduce9(float (&v)[8], float& e, float* red, int& slot, int wip, int lane, int barid) {
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
    float k4[4], k2[2], k1;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float keep = h16 ? v[j + 4] : v[j], send = h16 ? v[j] : v[j + 4];
        k4[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float keep = h8 ? k4[j + 2] : k4[j], send = h8 ? k4[j] : k4[j + 2];
        k2[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    {
        const float keep = h4 ? k2[1] : k2[0], send = h4 ? k2[0] : k2[1];
        k1 = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    k1 += __shfl_xor_sync(0xffffffffu, k1, 2);
    k1 += __shfl_xor_sync(0xffffffffu, k1, 1);
    e = warp_sum(e);
    float* mine = red + slot * 24 + wip * 12;
    if ((lane & 3) == 0) mine[lane >> 2] = k1;   // row (lane >> 2) & 7
    if (lane == 0) mine[8] = e;
    pair_bar(barid);
    const float4* r4 = reinterpret_cast<const float4*>(red + slot * 24);
    const float4 a0 = r4[0], a1 = r4[1], b0 = r4[3], b1 = r4[4];
    v[0] = a0.x + b0.x; v[1] = a0.y + b0.y; v[2] = a0.z + b0.z; v[3] = a0.w + b0.w;
    v[4] = a1.x + b1.x; v[5] = a1.y + b1.y; v[6] = a1.z + b1.z; v[7] = a1.w + b1.w;
    e = red[slot * 24 + 8] + red[slot * 24 + 20];
    slot ^= 1;
}

// X tile -> registers.  x[i][0..1] = chunk p, x[i][2..3] = chunk p+64 (packed pairs of columns).
template <bool RELU>
__device__ __forceinline__ void load_rows_smem(const float* tile, int p, f2 (&x)[8][4]) {
    const float4* t4 = reinterpret_cast<const float4*>(tile);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float4 a = t4[i * 128 + p], b = t4[i * 128 + 64 + p];
        if (RELU) {
            a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f);
            b.x = fmaxf(b.x, 0.f); b.y = fmaxf(b.y, 0.f); b.z = fmaxf(b.z, 0.f); b.w = fmaxf(b.w, 0.f);
        }
        x[i][0] = make_float2(a.x, a.y); x[i][1] = make_float2(a.z, a.w);
        x[i][2] = make_float2(b.x, b.y); x[i][3] = make_float2(b.z, b.w);
    }
}
__device__ __forceinline__ void get4x2(const float4* src, int idx_a, int idx_b, f2 (&v)[4]) {
    const float4 a = src[idx_a], b = src[idx_b];
    v[0] = make_float2(a.x, a.y); v[1] = make_float2(a.z, a.w); v[2] = make_float2(b.x, b.y); v[3] = make_float2(b.z, b.w);
}
__device__ __forceinline__ void get8(const float4* src, int idx, float (&v)[8]) {
    const float4 a = src[idx], b = src[idx + 1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// a = X v (lane-partial), bb = v . v (lane-partial)
__device__ __forceinline__ void xv_partial(const f2 (&x)[8][4], const f2 (&v)[4], float (&a)[8], float& bb) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        f2 acc = mul2(x[i][0], v[0]);
#pragma unroll
        for (int kp = 1; kp < 4; ++kp) acc = fma2(x[i][kp], v[kp], acc);
        a[i] = acc.x + acc.y;
    }
    f2 b2 = mul2(v[0], v[0]);
#pragma unroll
    for (int kp = 1; kp < 4; ++kp) b2 = fma2(v[kp], v[kp], b2);
    bb = b2.x + b2.y;
}
// c = X^T u for the lane's 8 columns
__device__ __forceinline__ void xtu(const f2 (&x)[8][4], const float (&u)[8], f2 (&c)[4]) {
    {
        const f2 u0 = dup(u[0]);
#pragma unroll
        for (int kp = 0; kp < 4; ++kp) c[kp] = mul2(x[0][kp], u0);
    }
#pragma unroll
    for (int i = 1; i < 8; ++i) {
        const f2 ui = dup(u[i]);
#pragma unroll
        for (int kp = 0; kp < 4; ++kp) c[kp] = fma2(x[i][kp], ui, c[kp]);
    }
}
// v = relu((X^T u + eps) / (d + eps)), d = u . u   (matrix_factorization.py:224-227 on the transposed problem)
__device__ __forceinline__ void v_from_u(const f2 (&x)[8][4], const float (&u)[8], float eps, float& rd, f2 (&v)[4]) {
    float d = u[0] * u[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) d = fmaf(u[i], u[i], d);
    rd = rcp_nr(d + eps);
    f2 c[4];
    xtu(x, u, c);
    const f2 rd2 = dup(rd), e2 = dup(eps * rd);
#pragma unroll
    for (int kp = 0; kp < 4; ++kp) {
        const f2 q = fma2(c[kp], rd2, e2);
        v[kp] = make_float2(fmaxf(q.x, 0.f), fmaxf(q.y, 0.f));
    }
}

struct PairCtx {
    int pair, wip, lane, p, barid;
    bool leader;   // lane 0 of the pair's first warp: claims, decodes, issues TMA
    bool second;   // lane 0 of the pair's second warp: polls dependencies, publishes completions
};
__device__ __forceinline__ PairCtx pair_ctx() {
    PairCtx c;
    const int warp = threadIdx.x >> 5;
    c.pair = warp >> 1; c.wip = warp & 1; c.lane = threadIdx.x & 31; c.p = c.wip * 32 + c.lane;
    c.barid = 1 + c.pair; c.leader = (c.p == 0); c.second = (c.p == 32);
    return c;
}

struct alignas(16) PairShared {       // static shared memory, one per pair
    float red[48];
    float rec[2][kRecStride];         // backward: iterate summaries of the current / next window
    Info info[2];
    uint64_t xfull, gfull, ofull;
    int oready;
};

// Next item of the global work queue.  Inline PTX on purpose: nvcc turns atomicAdd() under a lane
// predicate into its warp-aggregated form, which shuffles the RESULT around immediately and so stalls
// the warp for the full round trip; here the result is not looked at until the next window.
__device__ __forceinline__ int claim(const FastParams& P) {
    int v;
    asm volatile("atom.relaxed.gpu.global.add.s32 %0, [%1], 1;" : "=r"(v) : "l"(P.ctr) : "memory");
    return v;
}

struct Pending { int set, b, rowid, bulk; };   // bulk: the output left through a bulk async store   // leader: finished window whose completion is not yet published

// =====================================================================================================
// forward
// =====================================================================================================
template <bool RELU>
__global__ void __launch_bounds__(kFwdPairs * 64, 1) swnmf_fwd_fast(const __grid_constant__ FastParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ __align__(16) PairShared ps_all[kFwdPairs];

    const PairCtx c = pair_ctx();
    float* xin = reinterpret_cast<float*>(smem_raw) + (size_t)c.pair * 4096;
    PairShared& ps = ps_all[c.pair];
    const long long G = (long long)P.NR * P.G2;

    for (int j = threadIdx.x; j < 512; j += blockDim.x) v0s[j] = P.v0[j];
    int claimed = 0;     // leader: item claimed ahead, not yet decoded
    if (c.leader) {
        mbar_init(&ps.xfull, 64);
        fence_mbarrier_init();
        decode(P, claim(P), &ps.info[0]);
        decode(P, claim(P), &ps.info[1]);
        claimed = claim(P);
    }
    __syncthreads();
    {
        const Info first = ps.info[0];
        if (first.item < P.total_items) fetch_tile(P, &P.tm_x, P.x, first, c.p, xin, &ps.xfull, false);
    }

    uint32_t xparity = 0;
    int slot = 0;
    Pending pend; pend.set = -1; pend.b = 0; pend.rowid = 0;
    for (int n = 0;; ++n) {
        const Info it = ps.info[n & 1];
        if (it.item >= P.total_items) break;
        const bool is_final = (it.set == P.final_set);
        f2 x[8][4];
        mbar_wait(&ps.xfull, xparity);
        xparity ^= 1;
        load_rows_smem<RELU>(xin, c.p, x);

        // ---- T HALS sweeps, rank 1 (matrix_factorization.py:224-227 twice per sweep, :122-136) ----
        f2 v[4];
        float u[8];
        get4x2(reinterpret_cast<const float4*>(v0s), c.p, 64 + c.p, v);
        float* rec = P.saved ? P.saved + it.win_id * P.rec_floats : nullptr;
        int dc[4] = {0, 0, 0, 0};   // second: completion counters of the first early set, fetched ahead of the epilogue
        for (int t = 0; t < P.T; ++t) {
            float a[8], bb;
            xv_partial(x, v, a, bb);
            pair_reduce9(a, bb, ps.red, slot, c.wip, c.lane, c.barid);
            if (t == 0) {
                // both warps hold X in registers and their copy of `it`: refill the tile slot with the
                // next window, publish the previous window's completion, decode the item claimed a
                // window ago into the free info slot
                if (c.second && pend.set >= 0) { signal_row(P, pend.set, pend.b, pend.rowid); pend.set = -1; }
                const Info nt = ps.info[(n + 1) & 1];
                if (nt.item < P.total_items) fetch_tile(P, &P.tm_x, P.x, nt, c.p, xin, &ps.xfull, false);
                if (c.leader) decode(P, claimed, &ps.info[n & 1]);
            }
            if (t == P.T - 1) {
                if (c.leader) claimed = claim(P);
                if (c.second && is_final && P.S > 1 && !(P.debug & 1)) {
                    const DepRows d = dep_rows(P, it, P.final_set == 0 ? 1 : 0);
#pragma unroll
                    for (int q = 0; q < 4; ++q) dc[q] = ld_poll(d.p[q]);
                }
            }
            const float rb = rcp_nr(bb + P.eps);
            const float erb = P.eps * rb;
#pragma unroll
            for (int i = 0; i < 8; ++i) u[i] = fmaxf(fmaf(a[i], rb, erb), 0.f);
            float rd;
            v_from_u(x, u, P.eps, rd, v);
            if (rec && c.leader) {
                reinterpret_cast<float4*>(rec)[2 * t] = make_float4(u[0], u[1], u[2], u[3]);
                reinterpret_cast<float4*>(rec)[2 * t + 1] = make_float4(u[4], u[5], u[6], u[7]);
                rec[8 * P.T + t] = bb;
            }
        }

        if (P.debug & 2) {
            if (u[0] * v[0].x == 123.456f) P.out[0] = 1.f;
        } else if (!is_final) {
            // ---- early set: publish the rank-1 factors only ----
            const long long local = it.win_id - ((long long)it.set * P.B + it.b) * P.heads * G;   // head*G + window
            float4* f4 = reinterpret_cast<float4*>(P.fac + (((long long)P.fac_idx[it.set] * P.B + it.b) * P.heads * G + local) * kFacFloats);
            if (c.leader) { f4[0] = make_float4(u[0], u[1], u[2], u[3]); f4[1] = make_float4(u[4], u[5], u[6], u[7]); }
            f4[2 + c.p] = make_float4(v[0].x, v[0].y, v[1].x, v[1].y);
            f4[2 + 64 + c.p] = make_float4(v[2].x, v[2].y, v[3].x, v[3].y);
            if (c.second) { pend.set = it.set; pend.b = it.b; pend.rowid = it.rowid; }
        } else {
            // ---- final set: Y = (u v^T + sum over early sets of their overlapping factors) / S ----
            if (P.S > 1) {
                if (c.second && !(P.debug & 1)) {
                    // a pair never blocks while it owes a completion signal
                    if (pend.set >= 0) { signal_row(P, pend.set, pend.b, pend.rowid); pend.set = -1; }
                    const int first = P.final_set == 0 ? 1 : 0;
                    if (dc[0] < P.TPR || dc[1] < P.TPR || dc[2] < P.TPR || dc[3] < P.TPR) wait_rows(P, it, first);
                    else acquire_after_poll();
                    for (int s = first + 1; s < P.S; ++s)
                        if (s != P.final_set) wait_rows(P, it, s);
                }
                pair_bar(c.barid);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const f2 ui = dup(u[i] * P.inv_S);
#pragma unroll
                for (int kp = 0; kp < 4; ++kp) x[i][kp] = mul2(ui, v[kp]);      // x is dead: reuse as the accumulator
            }
            const LaneAddr la = lane_addr(P, it, c.p);
            const int q0v[2] = {c.p >> 4, (c.p + 64) >> 4};
            int i1 = it.c1 + ((c.p >> 1) & 7); if (i1 >= P.n1) i1 -= P.n1;
            for (int s = 0; s < P.S; ++s) {
                if (s == P.final_set) continue;
                const float* fs = P.fac + (((long long)P.fac_idx[s] * P.B + it.b) * P.heads + it.head) * G * kFacFloats;
                // position of this lane's columns in set s's rolled coordinates
                int rho1 = i1 + P.sh[s][1]; if (rho1 >= P.n1) rho1 -= P.n1;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    int i0 = it.c0 + q0v[h]; if (i0 >= P.n0) i0 -= P.n0;
                    int rho0 = i0 + P.sh[s][0]; if (rho0 >= P.n0) rho0 -= P.n0;
                    const int wrow = ((rho0 >> 3) * P.G1 + (rho1 >> 3)) * P.G2;
                    const int jrow = ((rho0 & 7) * 8 + (rho1 & 7)) * 8;
                    int rho2 = la.i2[h] + P.sh[s][2]; if (rho2 >= P.n2) rho2 -= P.n2;
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
                            x[i][2 * h] = fma2(ui, va, x[i][2 * h]);
                            x[i][2 * h + 1] = fma2(ui, vb, x[i][2 * h + 1]);
                        }
                    } else {
                        float acc[8][4];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            acc[i][0] = x[i][2 * h].x; acc[i][1] = x[i][2 * h].y; acc[i][2] = x[i][2 * h + 1].x; acc[i][3] = x[i][2 * h + 1].y;
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
                            x[i][2 * h] = make_float2(acc[i][0], acc[i][1]); x[i][2 * h + 1] = make_float2(acc[i][2], acc[i][3]);
                        }
                    }
                }
            }
            store_rows_direct(P, P.out + it.chan_base, it, c.p, x);
        }
    }
    // the last early-set window of this pair: its factor stores are ordered before the signal by the barrier
    pair_bar(c.barid);
    if (c.second && pend.set >= 0) signal_row(P, pend.set, pend.b, pend.rowid);
}

// =====================================================================================================
// backward
// =====================================================================================================
template <bool RELU>
__global__ void __launch_bounds__(kBwdPairs * 64, 1) swnmf_bwd_fast(const __grid_constant__ FastParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ __align__(16) PairShared ps_all[kBwdPairs];

    const PairCtx c = pair_ctx();
    float* xin = reinterpret_cast<float*>(smem_raw + (size_t)c.pair * 3 * kTileBytes);
    float* gin = xin + 4096;         // dY tile
    float* oin = gin + 4096;         // partial dX of the previous window set of the chain
    PairShared& ps = ps_all[c.pair];
    const int rec_lanes = P.rec_head >> 2;

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
    Pending pend; pend.set = -1; pend.b = 0; pend.rowid = 0;
    for (int n = 0;; ++n) {
        const Info it = ps.info[n & 1];
        if (it.item >= P.total_items) break;
        const int dep = P.dep_of[it.set];
        // second: completion counters of the rows whose partial sum this window continues, fetched now,
        // looked at just before the first barrier
        int dc[4] = {0, 0, 0, 0};
        if (c.second && dep >= 0 && !(P.debug & 1)) {
            const DepRows d = dep_rows(P, it, dep);
#pragma unroll
            for (int q = 0; q < 4; ++q) dc[q] = ld_poll(d.p[q]);
        }

        f2 x[8][4];
        mbar_wait(&ps.xfull, xparity);
        xparity ^= 1;
        load_rows_smem<RELU>(xin, c.p, x);
        const float* rec = ps.rec[n & 1];
        const float4* rec4 = reinterpret_cast<const float4*>(rec);

        // ---- v_T from the saved u_T (one lane-local GEMV) ----
        float u[8];
        float rd;
        f2 vt[4];
        get8(rec4, 2 * (P.T - 1), u);
        v_from_u(x, u, P.eps, rd, vt);

        // ---- gu = G v_T / S, gv = G^T u_T / S  (adjoint of u v^T and of the mean over sets) ----
        float gu[8];
        f2 gv[4];
        {
            mbar_wait(&ps.gfull, gparity);
            gparity ^= 1;
            const float4* g4 = reinterpret_cast<const float4*>(gin);
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) gv[kp] = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 ga = g4[i * 128 + c.p], gb = g4[i * 128 + 64 + c.p];
                const f2 g0 = make_float2(ga.x, ga.y), g1 = make_float2(ga.z, ga.w);
                const f2 g2 = make_float2(gb.x, gb.y), g3 = make_float2(gb.z, gb.w);
                f2 acc = mul2(g0, vt[0]);
                acc = fma2(g1, vt[1], acc); acc = fma2(g2, vt[2], acc); acc = fma2(g3, vt[3], acc);
                gu[i] = acc.x + acc.y;
                const f2 ui = dup(u[i]);
                gv[0] = fma2(g0, ui, gv[0]); gv[1] = fma2(g1, ui, gv[1]);
                gv[2] = fma2(g2, ui, gv[2]); gv[3] = fma2(g3, ui, gv[3]);
            }
            if (c.second) {
                ps.oready = (dep >= 0) && ((P.debug & 1) || (dc[0] >= P.TPR && dc[1] >= P.TPR && dc[2] >= P.TPR && dc[3] >= P.TPR));
                if (ps.oready) acquire_after_poll();      // ordered before the pair's fetch by the barrier in pair_reduce9
            }
            float dummy = 0.f;
            pair_reduce9(gu, dummy, ps.red, slot, c.wip, c.lane, c.barid);
            const f2 is2 = dup(P.inv_S);
#pragma unroll
            for (int i = 0; i < 8; ++i) gu[i] *= P.inv_S;
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) gv[kp] = mul2(gv[kp], is2);
        }
        // Both warps are past the barrier: X, dY and the previous partial tile have been consumed and
        // everyone holds its copy of `it`.  Refill the slots for the next window, publish the previous
        // window's completion, decode the next-but-one item, start fetching this window's partial sum.
        const bool oready = ps.oready != 0;
        {
            if (c.second && pend.set >= 0) { signal_row(P, pend.set, pend.b, pend.rowid); pend.set = -1; }
            if (oready) fetch_partial(P, it, c.p, oin, &ps.ofull);
            const Info nt = ps.info[(n + 1) & 1];
            if (nt.item < P.total_items) {
                if (c.p < rec_lanes) cp_async16(ps.rec[(n + 1) & 1] + 4 * c.p, P.saved + nt.win_id * P.rec_floats + 4 * c.p);
                fetch_tile(P, &P.tm_x, P.x, nt, c.p, xin, &ps.xfull, c.p < rec_lanes);
                fetch_tile(P, &P.tm_g, P.gy, nt, c.p, gin, &ps.gfull, false);
            }
            if (c.leader) decode(P, claimed, &ps.info[n & 1]);
        }

        // ---- reverse sweep (SURVEY App. A.3); dX accumulates in registers ----
        f2 xb[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) xb[i][kp] = make_float2(0.f, 0.f);
        for (int t = P.T - 1; t >= P.T - P.K; --t) {
            // u = u_t, rd = 1 / (u_t . u_t + eps), vt = v_t are live here
            const float rb = rcp_nr(rec[8 * P.T + t] + P.eps);
            // adjoint of v_t = relu((X^T u_t + eps) / (d_t + eps))
            f2 cb[4];
            float w[8], e;
            {
                const f2 rd2 = dup(rd);
                f2 e2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int kp = 0; kp < 4; ++kp) {
                    const f2 qb = make_float2(vt[kp].x > 0.f ? gv[kp].x : 0.f, vt[kp].y > 0.f ? gv[kp].y : 0.f);
                    cb[kp] = mul2(qb, rd2);
                    e2 = fma2(qb, vt[kp], e2);
                }
                e = e2.x + e2.y;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const f2 ui = dup(u[i]);
                f2 acc = mul2(x[i][0], cb[0]);
                xb[i][0] = fma2(ui, cb[0], xb[i][0]);
#pragma unroll
                for (int kp = 1; kp < 4; ++kp) {
                    xb[i][kp] = fma2(ui, cb[kp], xb[i][kp]);
                    acc = fma2(x[i][kp], cb[kp], acc);
                }
                w[i] = acc.x + acc.y;
            }
            // v_{t-1}: independent of the reduction below, so its FFMA2 stream fills the shuffle /
            // barrier latency
            float up[8], rdp = 0.f;
            f2 vp[4];
            if (t > 0) {
                get8(rec4, 2 * (t - 1), up);
                v_from_u(x, up, P.eps, rdp, vp);
            } else {
                get4x2(reinterpret_cast<const float4*>(v0s), c.p, 64 + c.p, vp);
#pragma unroll
                for (int i = 0; i < 8; ++i) up[i] = 0.f;
            }
            pair_reduce9(w, e, ps.red, slot, c.wip, c.lane, c.barid);
            const float db = -e * rd;
            // adjoint of u_t = relu((X v_{t-1} + eps) / (b_t + eps)); u_{t-1} does not feed u_t at rank 1
            float ab[8], bacc = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float ub = fmaf(2.f * db, u[i], w[i]);
                if (t == P.T - 1) ub += gu[i];
                const float pb = u[i] > 0.f ? ub : 0.f;
                ab[i] = pb * rb;
                bacc = fmaf(pb, u[i], bacc);
            }
            const f2 bbar2 = dup(-2.f * bacc * rb);
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) gv[kp] = mul2(bbar2, vp[kp]);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const f2 ai = dup(ab[i]);
#pragma unroll
                for (int kp = 0; kp < 4; ++kp) {
                    xb[i][kp] = fma2(ai, vp[kp], xb[i][kp]);
                    gv[kp] = fma2(x[i][kp], ai, gv[kp]);
                }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) u[i] = up[i];
#pragma unroll
            for (int kp = 0; kp < 4; ++kp) vt[kp] = vp[kp];
            rd = rdp;
        }
        if (c.leader) claimed = claim(P);

        // ---- dX (ReLU-masked, factorizer.py:44), added to the chain's partial sum and stored ----
        if (RELU) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int kp = 0; kp < 4; ++kp) {
                    xb[i][kp].x = x[i][kp].x > 0.f ? xb[i][kp].x : 0.f;
                    xb[i][kp].y = x[i][kp].y > 0.f ? xb[i][kp].y : 0.f;
                }
        }
        if (dep >= 0) {
            if (!oready) {
                // rare: the rows this window continues were not finished when it started
                if (c.second) {
                    if (pend.set >= 0) { signal_row(P, pend.set, pend.b, pend.rowid); pend.set = -1; }
                    wait_rows(P, it, dep);
                }
                pair_bar(c.barid);
                fetch_partial(P, it, c.p, oin, &ps.ofull);
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
        } else {
            store_rows_direct(P, P.out + it.chan_base, it, c.p, xb);
            if (c.second && P.signals[it.set]) { pend.set = it.set; pend.b = it.b; pend.rowid = it.rowid; }
        }
    }
    pair_bar(c.barid);
    if (c.second && pend.set >= 0) signal_row(P, pend.set, pend.b, pend.rowid);
}

#include "fz_swnmf_gram.cuh"

// =====================================================================================================
// host side
// =====================================================================================================
static int make_map(CUtensorMap* m, const void* ptr, const DevGeom& G, int box_d = 8) {
    if (reinterpret_cast<uintptr_t>(ptr) & 15) return fail(FZ_ERR_INVALID, "volume pointer %p is not 16-byte aligned", ptr);
    cuuint64_t dims[5] = {(cuuint64_t)G.n[2], (cuuint64_t)G.n[1], (cuuint64_t)G.n[0], (cuuint64_t)G.C, (cuuint64_t)G.B};
    cuuint64_t strides[4] = {(cuuint64_t)G.n[2] * 4, (cuuint64_t)G.n[2] * G.n[1] * 4, (cuuint64_t)G.vox * 4,
                             (cuuint64_t)G.vox * G.C * 4};
    cuuint32_t box[5] = {8, 8, (cuuint32_t)box_d, 8, 1};
    return encode_tiled_map(m, "volume", CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, ptr, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE);
}

static int rec_head_for(int T) { return ((9 * T + 3) / 4) * 4; }
static int rec_floats_for(int T) { return rec_head_for(T) + 72; }
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

bool fast_supported(const DevGeom& G, const fz_solver& s) {
    if (s.kind != FZ_SOLVER_HALS || s.rank != 1) return false;
    if (s.num_iters < 1 || s.num_iters > kMaxT) return false;
    if (G.d != 8 || G.p[0] != 8 || G.p[1] != 8 || G.p[2] != 8) return false;
    if ((long long)G.S * G.heads * G.g[0] * G.g[1] > kMaxOrder) return false;
    if (G.heads > 512 || G.g[0] > 1024 || G.g[1] > 1024) return false;
    if ((long long)G.B * G.S * G.heads * G.G >= (1LL << 30)) return false;
    if (G.mats_per_shift == 0) return false;
    return true;
}

size_t fast_saved_bytes(const DevGeom& G, const fz_solver& s) {
    if (!fast_supported(G, s)) return 0;
    return (size_t)G.S * G.mats_per_shift * rec_floats_for(s.num_iters) * sizeof(float);
}

static size_t counter_bytes(const DevGeom& G) {
    return align_up((size_t)(2 + (long long)G.S * G.B * G.heads * G.g[0] * G.g[1]) * sizeof(int), 256);
}

size_t fast_workspace_bytes(const DevGeom& G, const fz_solver& s) {
    if (!fast_supported(G, s)) return 0;
    return counter_bytes(G) + (size_t)(G.S - 1) * G.mats_per_shift * kFacFloats * sizeof(float);
}


// rows of set `dep` overlapped by row `row` of set `s`; returns the largest of `when[]` over them
static long long latest_needed(const DevGeom& G, const FastParams& P, int s, int row, int dep, const long long* when) {
    const int k = row / G.g[1], g1 = row % G.g[1];
    int c0 = k * 8 - P.sh[s][0]; if (c0 < 0) c0 += G.n[0];
    int c1 = g1 * 8 - P.sh[s][1]; if (c1 < 0) c1 += G.n[1];
    const int r0 = (c0 + P.sh[dep][0]) % G.n[0], r1 = (c1 + P.sh[dep][1]) % G.n[1];
    const int r0b = (r0 + 7) % G.n[0], r1b = (r1 + 7) % G.n[1];
    const int ks[2] = {r0 / 8, r0b / 8}, gs[2] = {r1 / 8, r1b / 8};
    long long best = 0;
    for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2; ++b) {
            const long long t = when[ks[a] * G.g[1] + gs[b]];
            if (t > best) best = t;
        }
    return best;
}

// Processing order of the rows of one sample.  Virtual time: the chain-head sets of head h run row r
// at time h*NR + r (sub-volume after sub-volume, so the live footprint is a slab of ONE head);
// a dependent row runs `lag` time units after the last row it needs, where one time unit is one row
// of every set (S * G2 windows) and `lag` covers one generation of in-flight windows: a window
// claimed that much later than its dependency starts (and needs the dependency's output only near
// its own end) when the dependency is finishing.
// forward: all early sets are heads, the final set depends on all of them.  backward: set j depends
// on set j-1.
static void build_order(const DevGeom& G, FastParams& P, bool forward, int windows_in_flight) {
    const int NR = G.g[0] * G.g[1];
    static thread_local long long when[FZ_MAX_SHIFTS][kMaxOrder];
    struct Key { long long key; unsigned entry; };
    static thread_local Key keys[kMaxOrder];
    const long long per_unit = (long long)G.g[2] * G.S;
    // `windows_in_flight`: how many windows are claimed but not finished at any time
    int lag = (int)((windows_in_flight + per_unit - 1) / per_unit) + 2;
    if (const char* env = getenv(forward ? "FZ_LAG_FWD" : "FZ_LAG_BWD")) lag = atoi(env);
    int n = 0;
    for (int h = 0; h < G.heads; ++h) {
        const long long base = (long long)h * NR;
        if (forward) {
            for (int s = 0; s < G.S; ++s)
                if (s != P.final_set)
                    for (int row = 0; row < NR; ++row) when[s][row] = base + row;
            for (int row = 0; row < NR; ++row) {
                long long t = base + row;
                for (int s = 0; s < G.S; ++s)
                    if (s != P.final_set) {
                        const long long need = latest_needed(G, P, P.final_set, row, s, when[s]) + lag;
                        if (need > t) t = need;
                    }
                when[P.final_set][row] = t;
            }
        } else {
            for (int s = 0; s < G.S; ++s)
                for (int row = 0; row < NR; ++row)
                    when[s][row] = (s == 0) ? base + row : latest_needed(G, P, s, row, s - 1, when[s - 1]) + lag;
        }
        for (int s = 0; s < G.S; ++s)
            for (int row = 0; row < NR; ++row) {
                keys[n].key = when[s][row] * FZ_MAX_SHIFTS + s;
                keys[n].entry = ((unsigned)s << 29) | ((unsigned)h << 20) | ((unsigned)(row / G.g[1]) << 10) | (unsigned)(row % G.g[1]);
                ++n;
            }
    }
    std::stable_sort(keys, keys + n, [](const Key& a, const Key& b) { return a.key < b.key; });
    for (int i = 0; i < n; ++i) P.order[i] = keys[i].entry;
    P.entries = n;
}

struct PlanKey {
    int B, C, n[3], S, sh[FZ_MAX_SHIFTS][3], T, K, relu, forward, lag_env, sms;
};

static int fill_params(FastParams& P, PlanKey& cached, const DevGeom& G, const fz_solver& s, int K, int relu, bool forward) {
    const bool gram = relu != 0;
    PlanKey key;
    memset(&key, 0, sizeof(key));
    key.B = G.B; key.C = G.C; key.S = G.S; key.T = s.num_iters; key.K = K; key.relu = relu; key.forward = forward;
    key.sms = num_sms();
    { const char* env = getenv(forward ? "FZ_LAG_FWD" : "FZ_LAG_BWD"); key.lag_env = env ? atoi(env) + 1 : 0; }
    for (int k = 0; k < 3; ++k) key.n[k] = G.n[k];
    for (int q = 0; q < G.S; ++q)
        for (int k = 0; k < 3; ++k) key.sh[q][k] = G.sh[q][k];
    { const char* env = getenv("FZ_DEBUG_FLAGS"); P.debug = env ? atoi(env) : 0; }
    P.eps = s.eps;
    if (memcmp(&key, &cached, sizeof(key)) == 0) return FZ_OK;   // same plan as the previous call on this thread

    const int debug = P.debug;
    memset(&P, 0, sizeof(P));
    P.debug = debug;
    P.n0 = G.n[0]; P.n1 = G.n[1]; P.n2 = G.n[2];
    P.G0 = G.g[0]; P.G1 = G.g[1]; P.G2 = G.g[2];
    P.heads = G.heads; P.B = G.B; P.S = G.S; P.C = G.C; P.vox = G.vox;
    for (int q = 0; q < G.S; ++q)
        for (int k = 0; k < 3; ++k) {
            int v = G.sh[q][k] % G.n[k];
            if (v < 0) v += G.n[k];
            P.sh[q][k] = v;
        }
    P.NR = G.g[0] * G.g[1];
    P.TPR = G.g[2];
    P.tpr_shift = -1;
    for (int q = 0; q < 12; ++q)
        if ((1 << q) == P.TPR) P.tpr_shift = q;
    // forward: the set that writes Y should have only clean boxes -> prefer an unshifted one
    P.final_set = G.S - 1;
    for (int q = 0; q < G.S; ++q)
        if (P.sh[q][0] % 8 == 0 && P.sh[q][1] % 8 == 0 && P.sh[q][2] % 8 == 0) { P.final_set = q; break; }
    int slot = 0;
    for (int q = 0; q < FZ_MAX_SHIFTS; ++q) {
        P.fac_idx[q] = (q < G.S && q != P.final_set) ? slot++ : -1;
        P.dep_of[q] = (q > 0 && q < G.S) ? q - 1 : -1;
        P.signals[q] = forward ? (q < G.S && q != P.final_set) : (q + 1 < G.S);
    }
    // direct kernels: a pair holds three claimed windows (current, next, next-but-one); Gram forward:
    // a warp holds two; Gram backward: a pair holds three
    int in_flight;
    if (gram) in_flight = forward ? 2 * num_sms() * kGFwdWarps : 2 * num_sms() * kGBwdPairs;
    else in_flight = 2 * num_sms() * (forward ? kFwdPairs : kBwdPairs);
    build_order(G, P, forward, in_flight);
    P.per_sample = P.entries * P.TPR;
    P.total_items = G.B * P.per_sample;
    P.T = s.num_iters; P.K = K; P.relu = relu; P.rec_floats = rec_floats_for(s.num_iters); P.rec_head = rec_head_for(s.num_iters);
    P.eps = s.eps; P.inv_S = 1.0f / (float)G.S;
    cached = key;
    return FZ_OK;
}

int fast_forward(const float* x, const float* u0, const float* v0, float* y, void* saved,
                 void* workspace, const DevGeom& G, const fz_solver& s, int relu, cudaStream_t st) {
    (void)u0;  // at rank 1 the HALS update of u does not read the previous u (matrix_factorization.py:224-227)
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_forward: workspace of %zu bytes required", fast_workspace_bytes(G, s));
    static thread_local FastParams P;
    static thread_local PlanKey cached;
    if (int e = fill_params(P, cached, G, s, 0, relu, true)) return e;
    if (int e = make_map(&P.tm_x, x, G)) return e;
    P.tm_g = P.tm_x;
    if (int e = make_map(&P.tm_out, y, G, relu ? 4 : 8)) return e;
    if (reinterpret_cast<uintptr_t>(y) & 15) return fail(FZ_ERR_INVALID, "output pointer %p is not 16-byte aligned", (void*)y);
    P.x = x; P.gy = nullptr; P.out = y; P.v0 = v0; P.saved = static_cast<float*>(saved);
    P.ctr = static_cast<int*>(workspace);
    P.fac = reinterpret_cast<float*>(static_cast<char*>(workspace) + counter_bytes(G));
    FZ_CUDA_CHECK(cudaMemsetAsync(workspace, 0, counter_bytes(G), st));
    const size_t smem = (size_t)kFwdPairs * kTileBytes;
    static SmemConfig cfg_fwd;
    FZ_CUDA_CHECK(cfg_fwd.ensure(swnmf_fwd_fast<false>, smem));
    if (relu) {
        const size_t gsmem = (size_t)kGFwdWarps * (kTileBytes + kTileBytes / 2);
        static SmemConfig cfg_gfwd;
        FZ_CUDA_CHECK(cfg_gfwd.ensure(swnmf_fwd_gram, gsmem));
        int ctas_needed = (P.total_items + kGFwdWarps - 1) / kGFwdWarps;
        int grid = num_sms();
        if (ctas_needed < grid) grid = ctas_needed;
        swnmf_fwd_gram<<<grid, kGFwdWarps * 32, gsmem, st>>>(P);
    } else {
        int ctas_needed = (P.total_items + kFwdPairs - 1) / kFwdPairs;
        int grid = num_sms();
        if (ctas_needed < grid) grid = ctas_needed;
        swnmf_fwd_fast<false><<<grid, kFwdPairs * 64, smem, st>>>(P);
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int fast_backward(const float* x, const float* gy, const float* u0, const float* v0,
                  const void* saved, float* gx, void* workspace, const DevGeom& G,
                  const fz_solver& s, int K, int relu, cudaStream_t st) {
    (void)u0;
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: workspace of %zu bytes required", fast_workspace_bytes(G, s));
    if (!saved) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: the `saved` buffer written by fz_swnmf_forward is required");
    static thread_local FastParams P;
    static thread_local PlanKey cached;
    if (int e = fill_params(P, cached, G, s, K, relu, false)) return e;
    if (int e = make_map(&P.tm_x, x, G)) return e;
    if (int e = make_map(&P.tm_g, gy, G)) return e;
    if (int e = make_map(&P.tm_out, gx, G)) return e;
    P.x = x; P.gy = gy; P.out = gx; P.v0 = v0;
    P.saved = const_cast<float*>(static_cast<const float*>(saved));
    P.ctr = static_cast<int*>(workspace);
    FZ_CUDA_CHECK(cudaMemsetAsync(workspace, 0, counter_bytes(G), st));
    const size_t smem = (size_t)kBwdPairs * 3 * kTileBytes;
    static SmemConfig cfg_bwd;
    FZ_CUDA_CHECK(cfg_bwd.ensure(swnmf_bwd_fast<false>, smem));
    if (relu) {
        const size_t gsmem = (size_t)kGBwdPairs * 3 * kTileBytes;
        static SmemConfig cfg_gbwd;
        FZ_CUDA_CHECK(cfg_gbwd.ensure(swnmf_bwd_gram, gsmem));
        int ctas_needed = (P.total_items + kGBwdPairs - 1) / kGBwdPairs;
        int grid = num_sms();
        if (ctas_needed < grid) grid = ctas_needed;
        swnmf_bwd_gram<<<grid, kGBwdPairs * 64, gsmem, st>>>(P);
    } else {
        int ctas_needed = (P.total_items + kBwdPairs - 1) / kBwdPairs;
        int grid = num_sms();
        if (ctas_needed < grid) grid = ctas_needed;
        swnmf_bwd_fast<false><<<grid, kBwdPairs * 64, smem, st>>>(P);
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // namespace fz
