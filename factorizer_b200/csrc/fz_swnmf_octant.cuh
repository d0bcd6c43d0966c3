// Device code shared by the two launch schemes of the "octant" formulation of the fused FactMixer core
// (head_dim 8, patch 8x8x8, window sets [unshifted, shifted by patch/2], act = ReLU, rank-1 HALS; reference
// factorizer/factorizer.py:41-50, operations.py:397-398 default shifts, matrix_factorization.py:210-229):
//   fz_swnmf_pipe.cu    ONE persistent launch per direction: the three passes below run as a software pipeline over
//                       planes of tiles, so that pass 3 finds in L2 what pass 1 read from HBM (production path)
//   fz_swnmf_phase.cu   three launches per direction (pass 1 | pass 2 | pass 3, each over the whole volume); small
//                       volumes, and the paired-window-set variant
//
// Why the octant form.  Measured on B200 (bench_probes/tma_l2_probe.cu): tile traffic made of 32-byte runs (one
// 8x8x8 window of an NCDHW volume) tops out near 20 B/clk/SM through TMA whether it comes from HBM or from L2.
// The Gram form (fz_swnmf_gram.cuh header) needs X only through SUMS OVER COLUMNS (Gam = X X^T, r = X 1,
// a_1 = X v_0 forward; G v_T + X cbar_T and qbar.v_T backward), and such sums split over any partition of the
// columns.  A shifted window is the union of 8 octants (4x4x4 voxels) of 8 different unshifted tiles, so:
//   pass 1 (per unshifted tile, X [and dY] read once, every access a clean TMA box):
//           per-octant partial sums, written as a 60-float (forward) / 2x12-float (backward) record;
//   pass 2 (per window of either set, tiny): add the 8 octant records, run the 8-vector recursion;
//   pass 3 (per unshifted tile, X [and dY] read again, output written once): per voxel
//           forward   y  = 1/2 sum_s u_s rd_s (u_s . x + eps)
//           backward  dx = [x > 0] sum_s ( rd_s u_s (u_s . g)/2 + M_s x + m_s + abar1_s v0[col_s] )
//           where s runs over the unshifted window of the tile and the shifted window of the voxel's octant.
// There are no wrapped or misaligned boxes and no partial-sum round trip through the volume.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <type_traits>
#include <stdlib.h>
#include <string.h>

#include "fz_device.cuh"
#include "fz_internal.cuh"

namespace fz {
namespace oct {

constexpr int kTileBytes = 16384;
constexpr int kOctFloats = 60;        // per octant: Gam upper triangle (36) | r (8) | a1 for set 0 (8) | a1 for set 1 (8)
constexpr int kTileRec = 8 * kOctFloats;   // 480 floats per tile
constexpr int kFacF = 12;             // per window: u_T (8), rd_T, pad
constexpr int kBwdOct = 12;           // per (octant, set): w (8), e, pad
constexpr int kBwdTileRec = 8 * 2 * kBwdOct;   // 192 floats per tile
constexpr int kMbF = 100;             // per window: M (64) | m (8) | abar_1 (8) | rd_T u_T (8) | u_T (8) | pad (4); 400 B keeps 8 records in distinct banks

// How the pipelined launch (fz_swnmf_pipe.cu) walks the volume: sub-volumes (sample, head) are taken `gs` at a time
// (a gang); a PLANE-GROUP is one plane t0 of tiles of every sub-volume of a gang (nA = gs * G1 * G2 tiles), and
// plane-groups are numbered J = gang * G0 + pos with pos = (t0 + 1) mod G0 (the last plane first, because the
// shifted windows of plane 0 reach back into it).
struct PipeGeom {
    int enabled;
    int gs, gs_shift;         // sub-volumes per gang (a power of two)
    int per_plane;            // G1 * G2
    int nA;                   // tiles (= windows of either set) per plane-group
    int nBset;                // ceil(nA / 4): solve items per plane-group and window set
    int NP;                   // number of plane-groups = gangs * G0
    int lead;                 // pass 1 runs at most `lead` plane-groups ahead of the completed pass 3
    int ring;                 // pass 1 records live in ring slots J mod ring (a power of two), pos 0 in slots ring, ring + 1
    int flags;                // 1: pass 1 loads ask L2 to keep the tile, 2: pass 3 loads release it, 4: streaming stores of the output
    int solve_items;
    int role_period, role_solve, role_gram;   // CTA roles by blockIdx % role_period: [0, role_solve) pass 2, then role_gram pass 1, rest pass 3
    int* ctr;                 // queue heads and per-plane-group completion counters (layout in fz_swnmf_pipe.cu)
    unsigned long long* trace;   // experiment builds (FZ_TUNING): when CTA 0 saw each step complete
};

struct alignas(64) PhaseParams {
    CUtensorMap tm_x;     // X volume, box (8,8,8,8,1)
    CUtensorMap tm_g;     // dY volume (backward)
    const float* x;
    const float* gy;
    float* out;           // Y (forward) / dX (backward)
    const float* v0;
    float* saved;         // per window: [u_t (8T) | b_t (T) | pad | Gam (64) | r (8)], canonical window order
    float* oct;           // pass 1 -> pass 2 records
    float* fac;           // forward pass 2 -> pass 3
    float* mb;            // backward pass 2 -> pass 3
    float* b1;            // v_0 . v_0, written by forward pass 1 (three-launch scheme)
    int n0, n1, n2, G0, G1, G2, heads, B, C;
    int pow2, s2, s1, s0, sh;   // all of G2, G1, G0, heads are powers of two: their log2 (tile_coord without divisions)
    int tiles;            // B * heads * G0 * G1 * G2 = windows per set
    int t_begin, t_count; // the tiles (= windows of either set) this launch works on: whole (sample, head) sub-volumes
    int reverse;          // pass 3 walks its tiles backwards: the tail of pass 1 is what L2 still holds
    long long vox;
    int T, K, rec_floats, rec_head;
    float eps;
    PipeGeom pipe;
};

// tile index <-> coordinates.  tid = ((b * heads + h) * G0 + t0) * G1 * G2 + t1 * G2 + t2
struct TileCoord { int b, h, t0, t1, t2; };
__device__ __forceinline__ TileCoord tile_coord(const PhaseParams& P, int tid) {
    TileCoord c;
    if (P.pow2) {
        c.t2 = tid & (P.G2 - 1); tid >>= P.s2;
        c.t1 = tid & (P.G1 - 1); tid >>= P.s1;
        c.t0 = tid & (P.G0 - 1); tid >>= P.s0;
        c.h = tid & (P.heads - 1); c.b = tid >> P.sh;
        return c;
    }
    c.t2 = tid % P.G2; tid /= P.G2;
    c.t1 = tid % P.G1; tid /= P.G1;
    c.t0 = tid % P.G0; tid /= P.G0;
    c.h = tid % P.heads; c.b = tid / P.heads;
    return c;
}
__device__ __forceinline__ int tile_index(const PhaseParams& P, int b, int h, int t0, int t1, int t2) {
    return (((b * P.heads + h) * P.G0 + t0) * P.G1 + t1) * P.G2 + t2;
}
__device__ __forceinline__ int tile_index(const PhaseParams& P, const TileCoord& c) { return tile_index(P, c.b, c.h, c.t0, c.t1, c.t2); }
// Octant o = (o0,o1,o2) of tile t (voxels q_k in [4 o_k, 4 o_k + 4)) belongs to the shifted window
// (t + o) mod G: rolled coordinate (8 t_k + q_k + 4) mod n_k = 8 (t_k + o_k) + (q_k + 4 - 8 o_k).
__device__ __forceinline__ int shifted_window_of(const PhaseParams& P, const TileCoord& c, int o) {
    int w0 = c.t0 + (o >> 2); if (w0 >= P.G0) w0 -= P.G0;
    int w1 = c.t1 + ((o >> 1) & 1); if (w1 >= P.G1) w1 -= P.G1;
    int w2 = c.t2 + (o & 1); if (w2 >= P.G2) w2 -= P.G2;
    return tile_index(P, c.b, c.h, w0, w1, w2);
}
// ... and window w of the shifted set takes its octant o from tile (w - o) mod G.
__device__ __forceinline__ TileCoord source_coord_of(const PhaseParams& P, const TileCoord& c, int o) {
    TileCoord s = c;
    s.t0 = c.t0 - (o >> 2); if (s.t0 < 0) s.t0 += P.G0;
    s.t1 = c.t1 - ((o >> 1) & 1); if (s.t1 < 0) s.t1 += P.G1;
    s.t2 = c.t2 - (o & 1); if (s.t2 < 0) s.t2 += P.G2;
    return s;
}

// Where pass 1 leaves the records of tile c for pass 2, in units of tile records.  Three-launch scheme: the tile
// index.  Pipelined scheme: ring slot of the tile's plane-group (PipeGeom) times nA plus the tile's place in the group.
__device__ __forceinline__ long long rec_slot(const PhaseParams& P, const TileCoord& c) {
    if (!P.pipe.enabled) return tile_index(P, c);
    const int sv = c.b * P.heads + c.h;
    const int gang = sv >> P.pipe.gs_shift, svg = sv & (P.pipe.gs - 1);
    const int pos = c.t0 + 1 == P.G0 ? 0 : c.t0 + 1;
    const int slot = pos == 0 ? P.pipe.ring + (gang & 1) : ((gang * P.G0 + pos) & (P.pipe.ring - 1));
    return (long long)slot * P.pipe.nA + (svg * P.pipe.per_plane + c.t1 * P.G2 + c.t2);
}

// Lane layout inside a tile (one warp per tile): lane l works on octant o = l >> 2; with t = l & 3 its
// four chunks j = 0..3 are the 16-byte pieces (q0 = 4 o0 + j, q1 = 4 o1 + t, q2 = 4 o2 .. 4 o2 + 3),
// i.e. float4 index (within a channel row of 128 float4) 16 (4 o0 + j) + 2 (4 o1 + t) + o2.
__device__ __forceinline__ int chunk_f4(int lane, int j) {
    const int o0 = lane >> 4, o1 = (lane >> 3) & 1, o2 = (lane >> 2) & 1, t = lane & 3;
    return 16 * (4 * o0 + j) + 2 * (4 * o1 + t) + o2;
}
// the same chunk's float4 index in the column order of its SHIFTED window (q' = q + 4 - 8 o)
__device__ __forceinline__ int chunk_f4_shifted(int lane, int j) {
    const int o0 = lane >> 4, o1 = (lane >> 3) & 1, o2 = (lane >> 2) & 1, t = lane & 3;
    return 16 * (4 * (1 - o0) + j) + 2 * (4 * (1 - o1) + t) + (1 - o2);
}

// How a streaming warp sees one tile in shared memory.  fp32: an (8,8,8,8) box, rows of 32 bytes.  bf16 / fp16 activations:
// two tiles side by side along W travel as one (16,8,8,8) box -- again rows of 32 bytes, the row granularity TMA and the L2
// sectors like -- and a tile is one 16-byte column of that box.  ld(i, lane, j): the lane's chunk j of channel i as floats.
struct TileF32 {
    const float* p;
    __device__ __forceinline__ float4 ld(int i, int lane, int j) const {
        return reinterpret_cast<const float4*>(p)[i * 128 + chunk_f4(lane, j)];
    }
};
// four 16-bit values (two 32-bit words, the lower half first) as floats
__device__ __forceinline__ float4 widen4(uint2 r, const __nv_bfloat16*) {
    return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u),
                       __uint_as_float(r.y << 16), __uint_as_float(r.y & 0xffff0000u));
}
__device__ __forceinline__ float4 widen4(uint2 r, const __half*) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
template <typename E>             // E = __nv_bfloat16 or __half
struct Tile16 {
    const unsigned char* p;       // pair buffer + 16 * (which tile of the pair)
    __device__ __forceinline__ float4 ld(int i, int lane, int j) const {
        const int o0 = lane >> 4, o1 = (lane >> 3) & 1, o2 = (lane >> 2) & 1, t = lane & 3;
        const uint2 r = *reinterpret_cast<const uint2*>(p + (i * 64 + (4 * o0 + j) * 8 + 4 * o1 + t) * 32 + o2 * 8);
        return widen4(r, static_cast<const E*>(nullptr));
    }
};
// four neighbouring voxels of the output
__device__ __forceinline__ void store_out(float* p, float4 v, bool streaming) {
    if (streaming) __stcs(reinterpret_cast<float4*>(p), v);
    else *reinterpret_cast<float4*>(p) = v;
}
__device__ __forceinline__ void store_out(__nv_bfloat16* p, float4 v, bool streaming) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<const uint32_t*>(&a);
    r.y = *reinterpret_cast<const uint32_t*>(&b);
    if (streaming) __stcs(reinterpret_cast<uint2*>(p), r);
    else *reinterpret_cast<uint2*>(p) = r;
}
__device__ __forceinline__ void store_out(__half* p, float4 v, bool streaming) {
    const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<const uint32_t*>(&a);
    r.y = *reinterpret_cast<const uint32_t*>(&b);
    if (streaming) __stcs(reinterpret_cast<uint2*>(p), r);
    else *reinterpret_cast<uint2*>(p) = r;
}

template <int N, int CAP>
__device__ __forceinline__ void halve_vals(float (&v)[CAP], bool hi, int bit) {
    constexpr int m = (N + 1) / 2;
#pragma unroll
    for (int j = 0; j < N - m; ++j) {
        const float keep = hi ? v[j + m] : v[j], send = hi ? v[j] : v[j + m];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
    if (N & 1) v[m - 1] += __shfl_xor_sync(0xffffffffu, v[m - 1], bit);
}
template <int N, int CAP>
__device__ __forceinline__ void halve_idx(int (&id)[CAP], bool hi) {
    constexpr int m = (N + 1) / 2;
#pragma unroll
    for (int j = 0; j < N - m; ++j) id[j] = hi ? id[j + m] : id[j];
}
// where a lane's 15 reduced values of fwd_tile_gram go inside its tile's record
__device__ __forceinline__ void gram_destinations(int lane, int (&dst)[15]) {
    int id[kOctFloats];
#pragma unroll
    for (int s = 0; s < kOctFloats; ++s) id[s] = s;
    halve_idx<60, kOctFloats>(id, lane & 1);
    halve_idx<30, kOctFloats>(id, lane & 2);
#pragma unroll
    for (int s = 0; s < 15; ++s) dst[s] = (lane >> 2) * kOctFloats + id[s];
}

__device__ __forceinline__ float dot8(const float (&a)[8], const float (&b)[8]) {
    float s = a[0] * b[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) s = fmaf(a[j], b[j], s);
    return s;
}
__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
    const float4 a = __ldcg(reinterpret_cast<const float4*>(p)), b = __ldcg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ float pick8(const float (&a)[8], int row) {
    float v = a[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) v = (row == j) ? a[j] : v;
    return v;
}
__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// =====================================================================================================
// forward pass 1 of one tile: per-octant Gram partials (Gam, r, a_1 for both window sets) -> rec_out (480 floats)
// The tile buffer itself is the scratch area for the record once X sits in registers.
// =====================================================================================================
// scratch: where the record is assembled before it leaves, 16-byte pieces SPITCH float4 apart (1: a dense 1 920-byte area;
// 2: the 16-byte column of a bf16 pair buffer whose tile already sits in registers)
template <typename Tile, int SPITCH = 1>
__device__ __forceinline__ void fwd_tile_gram(const Tile tile, float* scratch, const float* v0s, const int (&dst)[15], int lane, float* rec_out) {
    f2 x[8][8];
    {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 a = tile.ld(i, lane, j);
                x[i][2 * j] = make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
                x[i][2 * j + 1] = make_float2(fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
            }
    }
    float pv[kOctFloats];
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
        f2 va[8], vb[8];     // v_0 at this lane's columns, in the unshifted / shifted window's column order
        {
            const float4* v4 = reinterpret_cast<const float4*>(v0s);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 a = v4[chunk_f4(lane, j)], b = v4[chunk_f4_shifted(lane, j)];
                va[2 * j] = make_float2(a.x, a.y); va[2 * j + 1] = make_float2(a.z, a.w);
                vb[2 * j] = make_float2(b.x, b.y); vb[2 * j + 1] = make_float2(b.z, b.w);
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            f2 sum = add2(x[i][0], x[i][1]);
            f2 a0 = mul2(x[i][0], va[0]), a1 = mul2(x[i][0], vb[0]);
#pragma unroll
            for (int kp = 1; kp < 8; ++kp) { a0 = fma2(x[i][kp], va[kp], a0); a1 = fma2(x[i][kp], vb[kp], a1); }
#pragma unroll
            for (int kp = 2; kp < 8; ++kp) sum = add2(sum, x[i][kp]);
            pv[36 + i] = sum.x + sum.y;
            pv[44 + i] = a0.x + a0.y;
            pv[52 + i] = a1.x + a1.y;
        }
    }
    // the four lanes of an octant add their partials: two halving levels, 15 values per lane remain
    halve_vals<60, kOctFloats>(pv, lane & 1, 1);
    halve_vals<30, kOctFloats>(pv, lane & 2, 2);
    __syncwarp();
#pragma unroll
    for (int s = 0; s < 15; ++s) scratch[(dst[s] >> 2) * (4 * SPITCH) + (dst[s] & 3)] = pv[s];
    __syncwarp();
    {
        const float4* s4 = reinterpret_cast<const float4*>(scratch);
        float4* o4 = reinterpret_cast<float4*>(rec_out);
        for (int q = lane; q < kTileRec / 4; q += 32) o4[q] = s4[q * SPITCH];
    }
    fence_proxy_async_smem();   // the buffer goes back to TMA
}
// fp32 tile: the tile buffer itself is the scratch area
__device__ __forceinline__ void fwd_tile_gram(float* tile, const float* v0s, const int (&dst)[15], int lane, float* rec_out) {
    fwd_tile_gram<TileF32, 1>(TileF32{tile}, tile, v0s, dst, lane, rec_out);
}

// =====================================================================================================
// forward pass 2 for one window (8 lanes, `gmask`): add its 8 octant records, run the T sweeps, write the saved
// record and the factors pass 3 needs.  sums: 64 floats of shared memory.
// =====================================================================================================
__device__ __forceinline__ int tri_index(int i, int j) {   // position of Gam(i,j), i <= j, in the packed upper triangle
    return i * 8 - (i * (i - 1)) / 2 + (j - i);
}

// All 32 lanes of the warp (four windows) run this together: the shuffles use the full mask and stay inside a window's 8
// lanes, so the four windows never diverge.  A window slot without work passes the index of any valid window and
// active = false (it computes along and stores nothing).
__device__ __forceinline__ void fwd_solve_window(const PhaseParams& P, float* sums, long long gwin, int set,
                                                 int lane, bool active, float b1) {
    constexpr unsigned gmask = 0xffffffffu;
    const int row = lane & 7;
    const float eps = P.eps;
    {
        // The 8 lanes of a window read its 8 octant records together (each record is 15 consecutive
        // float4, lane i takes float4 2i and 2i+1) and add them up on the fly: all 16 loads of a lane
        // are independent, and the sums (floats 8i .. 8i+7 in lane i) go to shared memory for the
        // row / full-vector views below.
        const int local = (int)(gwin - (long long)set * P.tiles);
        const TileCoord c = tile_coord(P, local);
        float4 va[8], vb[8];
#pragma unroll
        for (int o = 0; o < 8; ++o) {
            const long long src = rec_slot(P, set ? source_coord_of(P, c, o) : c);
            const float4* g4 = reinterpret_cast<const float4*>(P.oct + ((size_t)src * 8 + o) * kOctFloats);
            va[o] = __ldcg(g4 + 2 * row);
            vb[o] = row < 7 ? __ldcg(g4 + 2 * row + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float4 a0 = va[0], a1 = vb[0];
#pragma unroll
        for (int o = 1; o < 8; ++o) {
            a0.x += va[o].x; a0.y += va[o].y; a0.z += va[o].z; a0.w += va[o].w;
            a1.x += vb[o].x; a1.y += vb[o].y; a1.z += vb[o].z; a1.w += vb[o].w;
        }
        float4* d4 = reinterpret_cast<float4*>(sums);
        d4[2 * row] = a0; d4[2 * row + 1] = a1;
    }
    __syncwarp(gmask);

    float grow[8], r[8], a[8];
    {
        const float* sm = sums;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            grow[j] = sm[row <= j ? tri_index(row, j) : tri_index(j, row)];
            r[j] = sm[36 + j];
            a[j] = sm[44 + 8 * set + j];
        }
    }
    float* rec = (P.saved && active) ? P.saved + gwin * P.rec_floats : nullptr;
    if (rec) {
        float4* g4 = reinterpret_cast<float4*>(rec + P.rec_head);
        g4[2 * row] = make_float4(grow[0], grow[1], grow[2], grow[3]);
        g4[2 * row + 1] = make_float4(grow[4], grow[5], grow[6], grow[7]);
        if (row == 0) { g4[16] = make_float4(r[0], r[1], r[2], r[3]); g4[17] = make_float4(r[4], r[5], r[6], r[7]); }
    }
    float u[8], b = b1, rd = 0.f;
    for (int t = 0; t < P.T; ++t) {
        const float rb = rcp_nr(b + eps);
        const float erb = eps * rb;
#pragma unroll
        for (int j = 0; j < 8; ++j) u[j] = fmaxf(fmaf(a[j], rb, erb), 0.f);
        float d = u[0] * u[0];
#pragma unroll
        for (int j = 1; j < 8; ++j) d = fmaf(u[j], u[j], d);
        rd = rcp_nr(d + eps);
        if (rec && row == 0) {
            reinterpret_cast<float4*>(rec)[2 * t] = make_float4(u[0], u[1], u[2], u[3]);
            reinterpret_cast<float4*>(rec)[2 * t + 1] = make_float4(u[4], u[5], u[6], u[7]);
            rec[8 * P.T + t] = b;
        }
        if (t == P.T - 1) break;
        const float gi = dot8(grow, u);
        float gu[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) gu[j] = __shfl_sync(gmask, gi, (lane & 24) | j);
        const float sq = dot8(u, gu), q = dot8(u, r);
        b = (fmaf(2.f * eps, q, sq) + 512.f * eps * eps) * rd * rd;
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] = fmaf(eps, r[j], gu[j]) * rd;
    }
    if (row == 0 && active) {
        float4* f4 = reinterpret_cast<float4*>(P.fac + gwin * kFacF);
        f4[0] = make_float4(u[0], u[1], u[2], u[3]);
        f4[1] = make_float4(u[4], u[5], u[6], u[7]);
        f4[2] = make_float4(rd, 0.f, 0.f, 0.f);
    }
}

// =====================================================================================================
// forward pass 3 of one tile: y = 1/2 (u_0 v_0^T + u_1 v_1^T) voxel by voxel, v_s = relu(rd_s (X^T u_s + eps)),
// stored from registers
// =====================================================================================================
struct Fac { float u[8]; float rd; };
__device__ __forceinline__ Fac load_fac(const float* fac, long long wid) {
    Fac f;
    ld8(fac + wid * kFacF, f.u);
    f.rd = __ldcg(fac + wid * kFacF + 8);
    return f;
}

template <bool UNROLL, bool STREAM, typename Tile, typename OutT>
__device__ __forceinline__ void fwd_tile_apply_t(const PhaseParams& P, const Tile tile, const Fac& f0, const Fac& f1,
                                                 const TileCoord& c, int lane) {
    const float eps = P.eps;
    OutT* base = reinterpret_cast<OutT*>(P.out) + ((long long)c.b * P.C + c.h * 8) * P.vox;
    const f2 r0 = dup(f0.rd), e0 = dup(eps * f0.rd), r1 = dup(f1.rd), e1 = dup(eps * f1.rd);
#pragma unroll(UNROLL ? 4 : 1)
    for (int j = 0; j < 4; ++j) {
        f2 xa[8], xb[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 a = tile.ld(i, lane, j);
            xa[i] = make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
            xb[i] = make_float2(fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
        }
        f2 d0a = mul2(xa[0], dup(f0.u[0])), d0b = mul2(xb[0], dup(f0.u[0]));
        f2 d1a = mul2(xa[0], dup(f1.u[0])), d1b = mul2(xb[0], dup(f1.u[0]));
#pragma unroll
        for (int i = 1; i < 8; ++i) {
            d0a = fma2(xa[i], dup(f0.u[i]), d0a); d0b = fma2(xb[i], dup(f0.u[i]), d0b);
            d1a = fma2(xa[i], dup(f1.u[i]), d1a); d1b = fma2(xb[i], dup(f1.u[i]), d1b);
        }
        // v = relu(rd (c + eps)), already halved for the mean over the two window sets
        d0a = fma2(d0a, r0, e0); d0b = fma2(d0b, r0, e0); d1a = fma2(d1a, r1, e1); d1b = fma2(d1b, r1, e1);
        const f2 half = dup(0.5f);
        d0a = mul2(make_float2(fmaxf(d0a.x, 0.f), fmaxf(d0a.y, 0.f)), half);
        d0b = mul2(make_float2(fmaxf(d0b.x, 0.f), fmaxf(d0b.y, 0.f)), half);
        d1a = mul2(make_float2(fmaxf(d1a.x, 0.f), fmaxf(d1a.y, 0.f)), half);
        d1b = mul2(make_float2(fmaxf(d1b.x, 0.f), fmaxf(d1b.y, 0.f)), half);
        // voxel offset of the chunk: q0 = 4 o0 + j, q1 = 4 o1 + t, q2 = 4 o2
        const int q0 = 4 * (lane >> 4) + j, q1 = 4 * ((lane >> 3) & 1) + (lane & 3), q2 = 4 * ((lane >> 2) & 1);
        OutT* dstp = base + ((long long)(c.t0 * 8 + q0) * P.n1 + (c.t1 * 8 + q1)) * P.n2 + c.t2 * 8 + q2;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const f2 ya = fma2(dup(f1.u[i]), d1a, mul2(dup(f0.u[i]), d0a));
            const f2 yb = fma2(dup(f1.u[i]), d1b, mul2(dup(f0.u[i]), d0b));
            store_out(dstp + (long long)i * P.vox, make_float4(ya.x, ya.y, yb.x, yb.y), STREAM);
        }
    }
}

template <bool UNROLL, bool STREAM = false>
__device__ __forceinline__ void fwd_tile_apply(const PhaseParams& P, const float* tile, const Fac& f0, const Fac& f1,
                                               const TileCoord& c, int lane) {
    fwd_tile_apply_t<UNROLL, STREAM, TileF32, float>(P, TileF32{tile}, f0, f1, c, lane);
}

// =====================================================================================================
// backward pass 1 of one tile (X at `tile`, dY at `tile + 4096`): per octant and window set, lane-partials of
// w = G v_T / 2 + X cbar_T  and  e = qbar_T . v_T  -> rec_out (192 floats)
// =====================================================================================================
struct UT { float u[8]; float rd; };
__device__ __forceinline__ UT load_ut(const PhaseParams& P, long long wid) {
    UT f;
    ld8(P.saved + wid * P.rec_floats + 8 * (P.T - 1), f.u);
    float d = f.u[0] * f.u[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) d = fmaf(f.u[j], f.u[j], d);
    f.rd = rcp_nr(d + P.eps);
    return f;
}

template <typename Tile>
__device__ __forceinline__ void bwd_tile_reduce_t(const PhaseParams& P, const Tile xt, const Tile gt, const UT& f0, const UT& f1, int lane,
                                                  float* rec_out) {
    const float eps = P.eps;
    const int oct = lane >> 2;
    f2 w0[8], w1[8], e0 = make_float2(0.f, 0.f), e1 = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) { w0[i] = make_float2(0.f, 0.f); w1[i] = make_float2(0.f, 0.f); }
    const f2 half = dup(0.5f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        f2 xa[8], xb[8], ga[8], gb[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 a = xt.ld(i, lane, j), g = gt.ld(i, lane, j);
            xa[i] = make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
            xb[i] = make_float2(fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
            ga[i] = mul2(make_float2(g.x, g.y), half);       // G = dY / S
            gb[i] = mul2(make_float2(g.z, g.w), half);
        }
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const UT& f = s ? f1 : f0;
            f2 ca = mul2(xa[0], dup(f.u[0])), cb = mul2(xb[0], dup(f.u[0]));
            f2 ha = mul2(ga[0], dup(f.u[0])), hb = mul2(gb[0], dup(f.u[0]));
#pragma unroll
            for (int i = 1; i < 8; ++i) {
                ca = fma2(xa[i], dup(f.u[i]), ca); cb = fma2(xb[i], dup(f.u[i]), cb);
                ha = fma2(ga[i], dup(f.u[i]), ha); hb = fma2(gb[i], dup(f.u[i]), hb);
            }
            const f2 rd2 = dup(f.rd), er = dup(eps * f.rd);
            f2 va = fma2(ca, rd2, er), vb = fma2(cb, rd2, er);              // v_T
            va = make_float2(fmaxf(va.x, 0.f), fmaxf(va.y, 0.f));
            vb = make_float2(fmaxf(vb.x, 0.f), fmaxf(vb.y, 0.f));
            const f2 qa = mul2(ha, rd2), qb = mul2(hb, rd2);                // cbar_T = gv rd_T
            f2& e = s ? e1 : e0;
            e = fma2(ha, va, e); e = fma2(hb, vb, e);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                f2& w = s ? w1[i] : w0[i];
                w = fma2(ga[i], va, w); w = fma2(gb[i], vb, w);
                w = fma2(xa[i], qa, w); w = fma2(xb[i], qb, w);
            }
        }
    }
    // add over the 4 lanes of the octant; lane t = 0 writes both 12-float records
    float r0[9], r1[9];
#pragma unroll
    for (int i = 0; i < 8; ++i) { r0[i] = w0[i].x + w0[i].y; r1[i] = w1[i].x + w1[i].y; }
    r0[8] = e0.x + e0.y; r1[8] = e1.x + e1.y;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        r0[i] += __shfl_xor_sync(0xffffffffu, r0[i], 1); r0[i] += __shfl_xor_sync(0xffffffffu, r0[i], 2);
        r1[i] += __shfl_xor_sync(0xffffffffu, r1[i], 1); r1[i] += __shfl_xor_sync(0xffffffffu, r1[i], 2);
    }
    if ((lane & 3) == 0) {
        float4* o4 = reinterpret_cast<float4*>(rec_out + oct * 2 * kBwdOct);
        o4[0] = make_float4(r0[0], r0[1], r0[2], r0[3]); o4[1] = make_float4(r0[4], r0[5], r0[6], r0[7]);
        o4[2] = make_float4(r0[8], 0.f, 0.f, 0.f);
        o4[3] = make_float4(r1[0], r1[1], r1[2], r1[3]); o4[4] = make_float4(r1[4], r1[5], r1[6], r1[7]);
        o4[5] = make_float4(r1[8], 0.f, 0.f, 0.f);
    }
}

__device__ __forceinline__ void bwd_tile_reduce(const PhaseParams& P, const float* tile, const UT& f0, const UT& f1, int lane,
                                                float* rec_out) {
    bwd_tile_reduce_t(P, TileF32{tile}, TileF32{tile + 4096}, f0, f1, lane, rec_out);
}

// =====================================================================================================
// backward pass 2 for one window (8 lanes): the 8-vector recursion t = T .. 1 (fz_swnmf_gram.cuh header).
// stage: 8 x kBwdOct floats of shared memory.
// =====================================================================================================
__device__ __forceinline__ void bwd_solve_window(const PhaseParams& P, float (*stage)[kBwdOct], long long gwin, int set,
                                                 int lane, bool active) {
    constexpr unsigned gmask = 0xffffffffu;      // as fwd_solve_window: the four windows of a warp run together
    const int row = lane & 7;
    const float eps = P.eps;
    const int T = P.T;
    const float* rec = P.saved + gwin * P.rec_floats;
    float grow[8], r[8], u[8], unext[8], bcur, bnext = 0.f;
    {
        // lane i fetches octant i's (w, e) record; the saved record's pieces are fetched alongside
        const int local = (int)(gwin - (long long)set * P.tiles);
        const TileCoord c = tile_coord(P, local);
        const long long src = rec_slot(P, set ? source_coord_of(P, c, row) : c);
        const float4* g4 = reinterpret_cast<const float4*>(P.oct + (((size_t)src * 8 + row) * 2 + set) * kBwdOct);
        const float4 p0 = __ldcg(g4), p1 = __ldcg(g4 + 1), p2 = __ldcg(g4 + 2);
        ld8(rec + P.rec_head + 8 * row, grow);
        ld8(rec + P.rec_head + 64, r);
        ld8(rec + 8 * (T - 1), u);
        bcur = __ldcg(rec + 8 * T + (T - 1));
        if (T >= 2) { ld8(rec + 8 * (T - 2), unext); bnext = __ldcg(rec + 8 * T + (T - 2)); }
        float4* s4 = reinterpret_cast<float4*>(&stage[row][0]);
        s4[0] = p0; s4[1] = p1; s4[2] = p2;
    }
    __syncwarp(gmask);
    float w[8], e = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) w[j] = 0.f;
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        const float4* oc = reinterpret_cast<const float4*>(&stage[o][0]);
        const float4 a = oc[0], b = oc[1];
        w[0] += a.x; w[1] += a.y; w[2] += a.z; w[3] += a.w; w[4] += b.x; w[5] += b.y; w[6] += b.z; w[7] += b.w;
        e += stage[o][8];
    }
    const float rdT = rcp_nr(dot8(u, u) + eps);     // same instruction sequence as the forward's rd_T
    float mrow[8], mi = 0.f, ab[8], bbar;
#pragma unroll
    for (int j = 0; j < 8; ++j) mrow[j] = 0.f;
    {
        const float db = -e * rdT;
        const float rb = rcp_nr(bcur + eps);
        float bacc = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float ub = fmaf(2.f * db, u[j], w[j]);
            const float pb = (T == 1 && !(u[j] > 0.f)) ? 0.f : ub;
            ab[j] = pb * rb;
            bacc = fmaf(pb, u[j], bacc);
        }
        bbar = -bacc * rb;
    }
    float ruT[8], uT[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { uT[j] = u[j]; ruT[j] = u[j] * rdT; }
    for (int t = T - 2; t >= T - P.K; --t) {
#pragma unroll
        for (int j = 0; j < 8; ++j) u[j] = unext[j];
        bcur = bnext;
        if (t >= 1) { ld8(rec + 8 * (t - 1), unext); bnext = __ldcg(rec + 8 * T + (t - 1)); }   // one step ahead
        const float rd = rcp_nr(dot8(u, u) + eps);
        const float brd = 2.f * bbar * rd, kappa = brd * eps;
        float z[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) z[j] = fmaf(brd, u[j], ab[j]);
        {
            const float ur = pick8(u, row) * rd, ar = pick8(ab, row) * rd;
#pragma unroll
            for (int j = 0; j < 8; ++j) mrow[j] = fmaf(ur, z[j], fmaf(ar, u[j], mrow[j]));
            mi = fmaf(kappa, ur, fmaf(eps, ar, mi));
        }
        const float gzi = dot8(grow, z), gui = dot8(grow, u);
        float gz[8], gu[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            gz[j] = __shfl_sync(gmask, gzi, (lane & 24) | j);
            gu[j] = __shfl_sync(gmask, gui, (lane & 24) | j);
        }
        const float qv = rd * (dot8(z, gu) + eps * dot8(z, r) + kappa * dot8(u, r) + 512.f * kappa * eps);
        const float db = -qv * rd;
        const float rb = rcp_nr(bcur + eps);
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
        // truncated unroll: a_L = X v_{L-1} still reads X, v_{L-1} = rd (X^T u_{L-1} + eps 1) is a constant
        // u_{L-1} is the iterate prefetched by the last step of the sweep (or by the prologue when K == 1)
#pragma unroll
        for (int j = 0; j < 8; ++j) u[j] = unext[j];
        const float ar = pick8(ab, row) * rcp_nr(dot8(u, u) + eps);
#pragma unroll
        for (int j = 0; j < 8; ++j) mrow[j] = fmaf(ar, u[j], mrow[j]);
        mi = fmaf(eps, ar, mi);
    }
    if (!active) return;
    float* mb = P.mb + gwin * kMbF;
    float4* m4 = reinterpret_cast<float4*>(mb);
    m4[2 * row] = make_float4(mrow[0], mrow[1], mrow[2], mrow[3]);
    m4[2 * row + 1] = make_float4(mrow[4], mrow[5], mrow[6], mrow[7]);
    mb[64 + row] = mi;
    mb[72 + row] = (P.K >= T) ? pick8(ab, row) : 0.f;
    mb[80 + row] = pick8(ruT, row);
    mb[88 + row] = pick8(uT, row);
}

// The same recursion, ONE LANE PER WINDOW (three-launch scheme): all eight rows of M in registers, the Gram matrix packed,
// no shuffles; sums and products in the order of the 8-lane form (same bits).
__device__ __forceinline__ void bwd_solve_lane(const PhaseParams& P, long long gwin, int set, bool active) {
    const float eps = P.eps;
    const int T = P.T;
    const float* rec = P.saved + gwin * P.rec_floats;
    float G[36], r[8], u[8], unext[8], bcur, bnext = 0.f;
    {
        const float4* g4 = reinterpret_cast<const float4*>(rec + P.rec_head);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 a = __ldcg(g4 + 2 * i), b = __ldcg(g4 + 2 * i + 1);
            const float row[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int j = i; j < 8; ++j) G[tri_index(i, j)] = row[j];
        }
    }
    ld8(rec + P.rec_head + 64, r);
    ld8(rec + 8 * (T - 1), u);
    bcur = __ldcg(rec + 8 * T + (T - 1));
    if (T >= 2) { ld8(rec + 8 * (T - 2), unext); bnext = __ldcg(rec + 8 * T + (T - 2)); }
    float w[8], e = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) w[j] = 0.f;
    {
        const int local = (int)(gwin - (long long)set * P.tiles);
        const TileCoord c = tile_coord(P, local);
#pragma unroll
        for (int o = 0; o < 8; ++o) {
            const long long src = rec_slot(P, set ? source_coord_of(P, c, o) : c);
            const float4* g4 = reinterpret_cast<const float4*>(P.oct + (((size_t)src * 8 + o) * 2 + set) * kBwdOct);
            const float4 a = __ldcg(g4), b = __ldcg(g4 + 1), cc = __ldcg(g4 + 2);
            w[0] += a.x; w[1] += a.y; w[2] += a.z; w[3] += a.w; w[4] += b.x; w[5] += b.y; w[6] += b.z; w[7] += b.w;
            e += cc.x;
        }
    }
    const float rdT = rcp_nr(dot8(u, u) + eps);
    float M[8][8], mi[8], ab[8], bbar;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        mi[i] = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) M[i][j] = 0.f;
    }
    {
        const float db = -e * rdT;
        const float rb = rcp_nr(bcur + eps);
        float bacc = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float ub = fmaf(2.f * db, u[j], w[j]);
            const float pb = (T == 1 && !(u[j] > 0.f)) ? 0.f : ub;
            ab[j] = pb * rb;
            bacc = fmaf(pb, u[j], bacc);
        }
        bbar = -bacc * rb;
    }
    float ruT[8], uT[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { uT[j] = u[j]; ruT[j] = u[j] * rdT; }
    for (int t = T - 2; t >= T - P.K; --t) {
#pragma unroll
        for (int j = 0; j < 8; ++j) u[j] = unext[j];
        bcur = bnext;
        if (t >= 1) { ld8(rec + 8 * (t - 1), unext); bnext = __ldcg(rec + 8 * T + (t - 1)); }   // one step ahead
        const float rd = rcp_nr(dot8(u, u) + eps);
        const float brd = 2.f * bbar * rd, kappa = brd * eps;
        float z[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) z[j] = fmaf(brd, u[j], ab[j]);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float ur = u[i] * rd, ar = ab[i] * rd;
#pragma unroll
            for (int j = 0; j < 8; ++j) M[i][j] = fmaf(ur, z[j], fmaf(ar, u[j], M[i][j]));
            mi[i] = fmaf(kappa, ur, fmaf(eps, ar, mi[i]));
        }
        float gz[8], gu[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float sz = G[tri_index(0, i)] * z[0], su = G[tri_index(0, i)] * u[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) {
                const float gij = G[i <= j ? tri_index(i, j) : tri_index(j, i)];
                sz = fmaf(gij, z[j], sz);
                su = fmaf(gij, u[j], su);
            }
            gz[i] = sz; gu[i] = su;
        }
        const float qv = rd * (dot8(z, gu) + eps * dot8(z, r) + kappa * dot8(u, r) + 512.f * kappa * eps);
        const float db = -qv * rd;
        const float rb = rcp_nr(bcur + eps);
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
        // truncated unroll: a_L = X v_{L-1} still reads X, v_{L-1} = rd (X^T u_{L-1} + eps 1) is a constant
#pragma unroll
        for (int j = 0; j < 8; ++j) u[j] = unext[j];
        const float rdl = rcp_nr(dot8(u, u) + eps);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float ar = ab[i] * rdl;
#pragma unroll
            for (int j = 0; j < 8; ++j) M[i][j] = fmaf(ar, u[j], M[i][j]);
            mi[i] = fmaf(eps, ar, mi[i]);
        }
    }
    if (!active) return;
    float* mb = P.mb + gwin * kMbF;
    float4* m4 = reinterpret_cast<float4*>(mb);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        m4[2 * i] = make_float4(M[i][0], M[i][1], M[i][2], M[i][3]);
        m4[2 * i + 1] = make_float4(M[i][4], M[i][5], M[i][6], M[i][7]);
    }
    m4[16] = make_float4(mi[0], mi[1], mi[2], mi[3]); m4[17] = make_float4(mi[4], mi[5], mi[6], mi[7]);
    const bool full = P.K >= T;
    m4[18] = full ? make_float4(ab[0], ab[1], ab[2], ab[3]) : make_float4(0.f, 0.f, 0.f, 0.f);
    m4[19] = full ? make_float4(ab[4], ab[5], ab[6], ab[7]) : make_float4(0.f, 0.f, 0.f, 0.f);
    m4[20] = make_float4(ruT[0], ruT[1], ruT[2], ruT[3]); m4[21] = make_float4(ruT[4], ruT[5], ruT[6], ruT[7]);
    m4[22] = make_float4(uT[0], uT[1], uT[2], uT[3]); m4[23] = make_float4(uT[4], uT[5], uT[6], uT[7]);
}

// =====================================================================================================
// backward pass 3 of one tile (X at `tile`, dY at `tile + 4096`, its nine window records at `mbs`: 0 = unshifted,
// 1 + o = shifted window of octant o):
// dx = [x > 0] sum_s ( rd_s u_s (u_s . g)/2 + M_s x + m_s + abar1_s v0[col_s] ) voxel by voxel
// =====================================================================================================
// the nine window records of tile c, 9 x 25 float4 spread over the lanes, cp.async into `mbs`
__device__ __forceinline__ void bwd_fetch_records(const PhaseParams& P, float* mbs, int tid, const TileCoord& c, int lane) {
    for (int q = lane; q < 9 * (kMbF / 4); q += 32) {
        const int wdx = q / (kMbF / 4), part = q - wdx * (kMbF / 4);
        const long long wid = wdx == 0 ? (long long)tid : (long long)P.tiles + shifted_window_of(P, c, wdx - 1);
        cp_async16(mbs + wdx * kMbF + 4 * part, P.mb + wid * kMbF + 4 * part);
    }
}

template <bool STREAM, typename Tile, typename OutT>
__device__ __forceinline__ void bwd_tile_apply_t(const PhaseParams& P, const Tile xt, const Tile gt, const float* mbs, const float* v0s,
                                                 const TileCoord& c, int lane) {
    const int oct = lane >> 2;
    const float* mb0 = mbs;
    const float* mb1 = mb0 + (1 + oct) * kMbF;
    OutT* base = reinterpret_cast<OutT*>(P.out) + ((long long)c.b * P.C + c.h * 8) * P.vox;
    const f2 half = dup(0.5f);
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        f2 xa[8], xb[8];
        f2 h0a, h0b, h1a, h1b;      // gv = (u_s . g) / 2 for the two sets
        {
            float u0[8], u1[8];
            const float4* p0 = reinterpret_cast<const float4*>(mb0 + 88);
            const float4* p1 = reinterpret_cast<const float4*>(mb1 + 88);
            const float4 a0 = p0[0], b0 = p0[1], a1 = p1[0], b1 = p1[1];
            u0[0] = a0.x; u0[1] = a0.y; u0[2] = a0.z; u0[3] = a0.w; u0[4] = b0.x; u0[5] = b0.y; u0[6] = b0.z; u0[7] = b0.w;
            u1[0] = a1.x; u1[1] = a1.y; u1[2] = a1.z; u1[3] = a1.w; u1[4] = b1.x; u1[5] = b1.y; u1[6] = b1.z; u1[7] = b1.w;
            h0a = h0b = h1a = h1b = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 a = xt.ld(i, lane, j), g = gt.ld(i, lane, j);
                xa[i] = make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
                xb[i] = make_float2(fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
                const f2 ga = mul2(make_float2(g.x, g.y), half), gb = mul2(make_float2(g.z, g.w), half);
                h0a = fma2(ga, dup(u0[i]), h0a); h0b = fma2(gb, dup(u0[i]), h0b);
                h1a = fma2(ga, dup(u1[i]), h1a); h1b = fma2(gb, dup(u1[i]), h1b);
            }
        }
        // v_0 at the chunk's columns, in the column order of either window
        const float4 va4 = reinterpret_cast<const float4*>(v0s)[chunk_f4(lane, j)];
        const float4 vb4 = reinterpret_cast<const float4*>(v0s)[chunk_f4_shifted(lane, j)];
        const f2 v0a = make_float2(va4.x, va4.y), v0b = make_float2(va4.z, va4.w);
        const f2 v1a = make_float2(vb4.x, vb4.y), v1b = make_float2(vb4.z, vb4.w);
        const int q0 = 4 * (lane >> 4) + j, q1 = 4 * ((lane >> 3) & 1) + (lane & 3), q2 = 4 * ((lane >> 2) & 1);
        OutT* dstp = base + ((long long)(c.t0 * 8 + q0) * P.n1 + (c.t1 * 8 + q1)) * P.n2 + c.t2 * 8 + q2;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            // row i of both windows' M, and their m, abar_1, rd_T u_T entries
            const float4 ma0 = reinterpret_cast<const float4*>(mb0)[2 * i], mc0 = reinterpret_cast<const float4*>(mb0)[2 * i + 1];
            const float4 ma1 = reinterpret_cast<const float4*>(mb1)[2 * i], mc1 = reinterpret_cast<const float4*>(mb1)[2 * i + 1];
            const float m0 = mb0[64 + i] + mb1[64 + i];
            const float a10 = mb0[72 + i], a11 = mb1[72 + i], ru0 = mb0[80 + i], ru1 = mb1[80 + i];
            f2 ya = fma2(dup(a10), v0a, dup(m0)), yb = fma2(dup(a10), v0b, dup(m0));
            ya = fma2(dup(a11), v1a, ya); yb = fma2(dup(a11), v1b, yb);
            ya = fma2(dup(ru0), h0a, ya); yb = fma2(dup(ru0), h0b, yb);
            ya = fma2(dup(ru1), h1a, ya); yb = fma2(dup(ru1), h1b, yb);
            const float r0[8] = {ma0.x, ma0.y, ma0.z, ma0.w, mc0.x, mc0.y, mc0.z, mc0.w};
            const float r1[8] = {ma1.x, ma1.y, ma1.z, ma1.w, mc1.x, mc1.y, mc1.z, mc1.w};
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const f2 mm = dup(r0[q] + r1[q]);       // (M_0 + M_1) x
                ya = fma2(mm, xa[q], ya); yb = fma2(mm, xb[q], yb);
            }
            // ReLU adjoint (factorizer.py:44)
            ya.x = xa[i].x > 0.f ? ya.x : 0.f; ya.y = xa[i].y > 0.f ? ya.y : 0.f;
            yb.x = xb[i].x > 0.f ? yb.x : 0.f; yb.y = xb[i].y > 0.f ? yb.y : 0.f;
            store_out(dstp + (long long)i * P.vox, make_float4(ya.x, ya.y, yb.x, yb.y), STREAM);
        }
    }
}

template <bool STREAM = false>
__device__ __forceinline__ void bwd_tile_apply(const PhaseParams& P, const float* tile, const float* mbs, const float* v0s,
                                               const TileCoord& c, int lane) {
    bwd_tile_apply_t<STREAM, TileF32, float>(P, TileF32{tile}, TileF32{tile + 4096}, mbs, v0s, c, lane);
}

// ---- host helpers shared by both launch schemes ---------------------------------------------------------
// box (8,8,8,8,1) of fp32, or -- bf16 / fp16 activations -- (16,8,8,8,1) of 16-bit values: two tiles side by side along W
inline int make_tile_map(CUtensorMap* m, const void* ptr, const DevGeom& G) {
    if (reinterpret_cast<uintptr_t>(ptr) & 15) return fail(FZ_ERR_INVALID, "volume pointer %p is not 16-byte aligned", ptr);
    cuuint64_t dims[5] = {(cuuint64_t)G.n[2], (cuuint64_t)G.n[1], (cuuint64_t)G.n[0], (cuuint64_t)G.C, (cuuint64_t)G.B};
    const bool h16 = G.dtype != FZ_DTYPE_F32;
    const cuuint64_t e = h16 ? 2 : 4;
    cuuint64_t strides[4] = {(cuuint64_t)G.n[2] * e, (cuuint64_t)G.n[2] * G.n[1] * e, (cuuint64_t)G.vox * e,
                             (cuuint64_t)G.vox * G.C * e};
    cuuint32_t box[5] = {h16 ? 16u : 8u, 8, 8, 8, 1};
    const CUtensorMapDataType type = G.dtype == FZ_DTYPE_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                     : G.dtype == FZ_DTYPE_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    return encode_tiled_map(m, "volume tile", type, 5, ptr, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE);
}
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline int rec_head_for(int T) { return ((9 * T + 3) / 4) * 4; }

// everything of PhaseParams that depends only on the geometry and the solver (pointers are set by the caller)
inline void fill_common(PhaseParams& P, const DevGeom& G, const fz_solver& s, int K) {
    memset(&P, 0, sizeof(P));
    P.n0 = G.n[0]; P.n1 = G.n[1]; P.n2 = G.n[2];
    P.G0 = G.g[0]; P.G1 = G.g[1]; P.G2 = G.g[2];
    P.heads = G.heads; P.B = G.B; P.C = G.C; P.vox = G.vox;
    P.tiles = (int)G.mats_per_shift;
    {
        auto lg = [](int v) { int q = 0; while ((1 << q) < v) ++q; return (1 << q) == v ? q : -1; };
        P.s2 = lg(P.G2); P.s1 = lg(P.G1); P.s0 = lg(P.G0); P.sh = lg(P.heads);
        P.pow2 = P.s2 >= 0 && P.s1 >= 0 && P.s0 >= 0 && P.sh >= 0;
    }
    P.T = s.num_iters; P.K = K; P.rec_head = rec_head_for(s.num_iters); P.rec_floats = P.rec_head + 72;
    P.eps = s.eps;
}

}  // namespace oct
}  // namespace fz
